"""Per-env model (rg_mpc_env_model) without a GPU: the struct layout, the argument checks of the three entry points
(they return before any device call) and the host-side validation helper of BatchedMPCController.set_env_model."""
import ctypes
import math

import pytest
import torch

from robot_gym import cuda as rg
from robot_gym.controllers.mpc.batched_mpc_controller import validate_env_model


def test_env_model_symbols_and_layout(rg_lib):
    for name in ("rg_mpc_build_solve_model", "rg_control_step_model", "rg_control_step_graph_create_model"):
        assert name in rg.EXPORTED_SYMBOLS and hasattr(rg_lib, name)
    assert ctypes.sizeof(rg.MpcEnvModel) == 24
    assert rg.RG_STATUS_BAD_MODEL == 64


def test_env_model_entry_points_reject_bad_arguments_without_a_device(rg_lib):
    model = rg.MpcEnvModel()
    assert rg_lib.rg_mpc_build_solve_model(None, 4, None, None, None) == -1
    assert rg_lib.rg_mpc_build_solve_model(None, 0, None, ctypes.byref(model), None) == 0      # empty batch
    assert rg_lib.rg_control_step_model(None, None, 4, None, ctypes.byref(model), None) == -1
    handle = ctypes.c_void_p()
    assert rg_lib.rg_control_step_graph_create_model(None, None, 4, None, None, None, ctypes.byref(handle)) == -1
    # a misaligned model array is refused before the workspace is looked up
    io = rg.MpcIo(*([16] * 7), 16, None, None, None, None, 0, 0)
    model.mass = 8 * 1024 + 4
    assert rg_lib.rg_mpc_build_solve_model(ctypes.c_void_p(4096), 4, ctypes.byref(io), ctypes.byref(model), None) == -1
    assert b"8-byte aligned" in rg_lib.rg_last_error()
    # an aligned model on a workspace rg_mpc_setup never prepared: RG_ERR_WORKSPACE, no device access
    model.mass = 8 * 1024
    assert rg_lib.rg_mpc_build_solve_model(ctypes.c_void_p(4096), 4, ctypes.byref(io), ctypes.byref(model), None) == -4


def test_env_model_validation_matches_the_setup_checks():
    ok_i = torch.tensor([[0.07, 0, 0, 0, 0.25, 0, 0, 0, 0.25]] * 3, dtype=torch.float64)
    validate_env_model(mass=torch.tensor([1.0, 20.0, 40.0], dtype=torch.float64), inertia=ok_i,
                       friction_coeffs=torch.full((3, 4), 0.45, dtype=torch.float64))
    for bad in (0.0, -1.0, math.nan, math.inf):
        with pytest.raises(ValueError, match="mass"):
            validate_env_model(mass=torch.tensor([20.0, bad], dtype=torch.float64))
    nan_i = ok_i.clone(); nan_i[1, 4] = math.nan
    with pytest.raises(ValueError, match="finite"):
        validate_env_model(inertia=nan_i)
    sing = ok_i.clone(); sing[2] = torch.tensor([1.0, 2, 3, 2, 4, 6, 0, 0, 1], dtype=torch.float64)
    with pytest.raises(ValueError, match=r"invertible \(\|det\| >= 1e-300\).*row 2"):
        validate_env_model(inertia=sing)
    for bad in (0.0, -0.3, math.nan):
        mu = torch.full((2, 4), 0.5, dtype=torch.float64); mu[1, 3] = bad
        with pytest.raises(ValueError, match="friction"):
            validate_env_model(friction_coeffs=mu)
