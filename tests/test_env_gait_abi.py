"""Per-env gait (rg_gait_env_params) without a GPU: the struct layout, the exports, the argument checks of the two
entry points (they return before any device call), the validation helper of BatchedMPCController.set_env_gait and the
per-env rows of synthetic.desired_stance."""
import ctypes
import math

import numpy as np
import pytest
import torch

from robot_gym import cuda as rg
from robot_gym.controllers.mpc.batched_mpc_controller import validate_env_gait
from robot_gym.model.robots.descriptions import GAIT_SCHEDULES
from robot_gym.util import synthetic


def test_env_gait_symbols_and_layout(rg_lib):
    for name in ("rg_control_step_env", "rg_control_step_graph_create_env"):
        assert name in rg.EXPORTED_SYMBOLS and hasattr(rg_lib, name)
    assert ctypes.sizeof(rg.GaitEnvParams) == 32
    assert [f for f, _ in rg.GaitEnvParams._fields_] == ["stance_duration", "duty_factor", "initial_leg_phase",
                                                         "initial_leg_state"]


def _state():
    """A controller state whose pointers are all set and 16-byte aligned (never dereferenced: the calls below fail on
    their arguments before any device access)."""
    s = rg.ControllerState()
    for name, _ in rg.ControllerState._fields_:
        if name not in ("mpc_active_set", "solve_info", "motor_velocities", "motor_strength_ratios", "applied_motor_torques"):
            setattr(s, name, 16 * 1024)
    return s


def test_env_gait_entry_points_reject_bad_arguments_without_a_device(rg_lib):
    gait = rg.GaitEnvParams()
    s = _state()
    assert rg_lib.rg_control_step_env(None, None, 4, None, None, ctypes.byref(gait), None) == -1
    assert rg_lib.rg_control_step_env(None, None, 0, None, None, ctypes.byref(gait), None) == 0      # empty batch
    handle = ctypes.c_void_p()
    assert rg_lib.rg_control_step_graph_create_env(None, None, 4, None, None, ctypes.byref(gait), None,
                                                   ctypes.byref(handle)) == -1
    ws = ctypes.c_void_p(4096)
    for field, addr in (("stance_duration", 8 * 1024 + 4), ("duty_factor", 8 * 1024 + 2),
                        ("initial_leg_phase", 8 * 1024 + 1), ("initial_leg_state", 8 * 1024 + 2)):
        g = rg.GaitEnvParams()
        setattr(g, field, addr)
        assert rg_lib.rg_control_step_env(ws, ws, 4, ctypes.byref(s), None, ctypes.byref(g), None) == -1, field
        assert b"aligned" in rg_lib.rg_last_error(), field
        assert rg_lib.rg_control_step_graph_create_env(ws, ws, 4, ctypes.byref(s), None, ctypes.byref(g), None,
                                                       ctypes.byref(handle)) == -1, field
        assert handle.value is None
    # the model's checks still run first on the combined entry point
    model = rg.MpcEnvModel()
    model.mass = 8 * 1024 + 4
    assert rg_lib.rg_control_step_env(ws, ws, 4, ctypes.byref(s), ctypes.byref(model), ctypes.byref(gait), None) == -1
    assert b"8-byte aligned" in rg_lib.rg_last_error()


def _rows(n, **bad):
    good = dict(stance_duration=torch.full((n, 4), 0.3, dtype=torch.float64),
                duty_factor=torch.full((n, 4), 0.6, dtype=torch.float64),
                initial_leg_phase=torch.tensor([[0.9, 0.0, 0.0, 0.9]] * n, dtype=torch.float64),
                initial_leg_state=torch.tensor([[0, 1, 1, 0]] * n, dtype=torch.int32))
    good.update(bad)
    return good


def test_env_gait_validation_follows_the_row_rule():
    validate_env_gait(**_rows(3))
    validate_env_gait(duty_factor=torch.ones((2, 4), dtype=torch.float64))               # duty 1 (stand) is valid
    validate_env_gait(initial_leg_phase=torch.zeros((2, 4), dtype=torch.float64))
    cases = (("stance_duration", [0.0, -0.1, math.nan, math.inf], "stance_duration"),
             ("duty_factor", [0.0, -0.5, 1.5, 1.0 + 2 ** -52, math.nan], "duty_factor"),
             ("initial_leg_phase", [1.0, -1e-300, math.nan, math.inf], "initial_leg_phase"),
             ("initial_leg_state", [2, 3, -1], "initial_leg_state"))
    for field, values, match in cases:
        for v in values:
            rows = _rows(3)
            t = rows[field].clone()
            t[2, 1] = v
            with pytest.raises(ValueError, match=rf"{match}.*row 2"):
                validate_env_gait(**{field: t})


def test_desired_stance_takes_per_env_rows():
    rng = np.random.default_rng(3)
    n = 257
    stance = rng.uniform(0.1, 0.6, (n, 4))
    duty = rng.uniform(0.2, 1.0, (n, 4))
    duty[::7] = 1.0
    phase = rng.uniform(0.0, 1.0, (n, 4))
    state = rng.integers(0, 2, (n, 4)).astype(np.int32)
    t = np.concatenate([rng.integers(0, 2000, n - n // 2) * 0.001, rng.uniform(0.0, 3.0, n // 2)])
    got = synthetic.desired_stance(t, stance, duty, phase, state)
    for e in range(n):
        row = synthetic.desired_stance(t[e:e + 1], stance[e], duty[e], phase[e], [int(s) for s in state[e]])
        assert np.array_equal(got[e], row[0]), e
    # [4] rows keep their old meaning: the same row for every env
    sch = GAIT_SCHEDULES["bound"]
    one = synthetic.desired_stance(t, sch["STANCE_DURATION_SECONDS"], sch["DUTY_FACTOR"], sch["INIT_PHASE_FULL_CYCLE"],
                                   sch["INIT_LEG_STATE"])
    tiled = synthetic.desired_stance(t, *[np.tile(np.asarray([float(v) for v in sch[k]]), (n, 1)) for k in
                                          ("STANCE_DURATION_SECONDS", "DUTY_FACTOR", "INIT_PHASE_FULL_CYCLE")],
                                     np.tile(np.asarray([int(s) for s in sch["INIT_LEG_STATE"]]), (n, 1)))
    assert np.array_equal(one, tiled)


def test_state_sequence_with_env_gait_keeps_the_draws():
    from robot_gym.model.robots.descriptions import GHOST
    n = 64
    base = synthetic.make_state_sequence(n, 3, GHOST, seed=synthetic.SEED + 3)
    sch = GAIT_SCHEDULES["pace"]
    gait = dict(initial_leg_phase=np.tile(np.asarray(sch["INIT_PHASE_FULL_CYCLE"], dtype=np.float64), (n, 1)),
                initial_leg_state=np.tile(np.asarray([int(s) for s in sch["INIT_LEG_STATE"]]), (n, 1)))
    seq = synthetic.make_state_sequence(n, 3, GHOST, seed=synthetic.SEED + 3, env_gait=gait)
    for a, b in zip(base, seq):
        assert np.array_equal(a.com_velocity_body, b.com_velocity_body) and np.array_equal(a.time_since_reset, b.time_since_reset)
        flip_a = a.foot_contacts ^ a.planned_contacts
        flip_b = b.foot_contacts ^ b.planned_contacts
        assert np.array_equal(flip_a, flip_b)                        # the same contact noise on another schedule
    planned = synthetic.desired_stance(seq[1].time_since_reset - seq[0].time_since_reset, sch["STANCE_DURATION_SECONDS"],
                                       sch["DUTY_FACTOR"], sch["INIT_PHASE_FULL_CYCLE"], sch["INIT_LEG_STATE"])
    assert np.array_equal(seq[1].planned_contacts, planned)
