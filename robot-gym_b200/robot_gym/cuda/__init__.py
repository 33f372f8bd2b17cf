"""ctypes binding of ``librg_cuda.so`` (C ABI: include/rg_cuda.h) for PyTorch tensors.

PyTorch is plumbing here: it owns device memory and streams; every compute call goes through the
C ABI with raw device pointers.  There is NO CPU fallback: loading fails loudly when the library
is missing, and every wrapper refuses non-CUDA tensors.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_int, c_int32, c_size_t, c_uint64, c_void_p

from . import build as _build

RG_NUM_LEGS = 4
RG_NUM_MOTORS = 12
RG_ACTION_DIM = 60
RG_MAX_HORIZON = 20
RG_VEL_WINDOW_MAX = 64

RG_LEG_SWING, RG_LEG_STANCE, RG_LEG_EARLY_CONTACT, RG_LEG_LOSE_CONTACT = 0, 1, 2, 3
RG_INFO_IPM_ITERS, RG_INFO_POLISH_ROUNDS, RG_INFO_STATUS, RG_INFO_NUM_ACTIVE = 0, 1, 2, 3
RG_STATUS_POLISHED, RG_STATUS_IPM_CONVERGED, RG_STATUS_NO_STANCE, RG_STATUS_NUMERIC = 1, 2, 4, 8
RG_STATUS_ACTIVE_SET_ONLY = 16
RG_STATUS_BAD_WORKSPACE = 32
RG_STATUS_BAD_MODEL = 64

# every symbol include/rg_cuda.h declares (tests check the library exports all of them)
EXPORTED_SYMBOLS = (
    "rg_mpc_default_params", "rg_workspace_bytes", "rg_mpc_setup", "rg_mpc_release", "rg_mpc_build_solve",
    "rg_mpc_build_solve_warm", "rg_mpc_build_solve_io", "rg_mpc_build_solve_model",
    "rg_robot_calibrate_ik", "rg_robot_workspace_bytes", "rg_robot_setup",
    "rg_gait_step", "rg_com_velocity_update", "rg_swing_targets", "rg_leg_ik", "rg_leg_fk", "rg_state_from_sim",
    "rg_force_to_torque", "rg_pack_hybrid_action", "rg_control_step", "rg_control_step_graph_create", "rg_control_step_graph_launch", "rg_control_step_graph_destroy",
    "rg_control_step_model", "rg_control_step_graph_create_model", "rg_control_step_env", "rg_control_step_graph_create_env",
    "rg_mpc_build_solve_schedule", "rg_control_step_plan", "rg_control_step_graph_create_plan",
    "rg_mpc_build_solve_footholds", "rg_control_step_footholds", "rg_control_step_graph_create_footholds",
    "rg_hybrid_motor_torque", "rg_hybrid_motor_torque_ex",
    "rg_measure_fma_peak", "rg_launch_count", "rg_last_error", "rg_version",
)


class MpcParams(Structure):
    """``rg_mpc_params``."""
    _fields_ = [
        ("mass", c_double), ("inertia", c_double * 9), ("num_legs", c_int32), ("horizon", c_int32),
        ("dt", c_double), ("weights", c_double * 13), ("alpha", c_double),
        ("friction_coeffs", c_double * 4), ("gravity", c_double), ("fz_max", c_double),
        ("fz_min", c_double), ("desired_body_height", c_double), ("ipm_tol", c_double),
        ("max_ipm_iters", c_int32), ("max_polish_rounds", c_int32),
        ("cold_start_rounds", c_int32), ("cold_start_max_violations", c_int32),
        ("two_kernel_solve", c_int32), ("reserved_", c_int32),
    ]


class MpcIo(Structure):
    """``rg_mpc_io`` (device pointers + flags)."""
    _fields_ = [(name, c_void_p) for name in (
        "com_velocity_body", "base_rpy", "base_rpy_rate", "foot_contact_state", "foot_positions_base", "command",
        "com_height", "contact_forces", "horizon_forces", "solve_info", "active_set_io", "horizon_forces_f64")] + [
        ("zero_yaw", c_int32), ("reserved_", c_int32)]


class MpcEnvModel(Structure):
    """``rg_mpc_env_model``: per-env mass [N], inertia [N,9] and friction coefficients [N,4] (float64 device
    pointers, each may be NULL = the workspace's value)."""
    _fields_ = [("mass", c_void_p), ("inertia", c_void_p), ("friction_coeffs", c_void_p)]


class GaitEnvParams(Structure):
    """``rg_gait_env_params``: per-env stance_duration, duty_factor, initial_leg_phase (float64 [N,4]) and
    initial_leg_state (int32 [N,4]) device pointers, each may be NULL = the robot workspace's value."""
    _fields_ = [("stance_duration", c_void_p), ("duty_factor", c_void_p), ("initial_leg_phase", c_void_p),
                ("initial_leg_state", c_void_p)]


class LegChain(Structure):
    """``rg_leg_chain``."""
    _fields_ = [
        ("p", (c_double * 3) * 3), ("r", (c_double * 9) * 3), ("axis", (c_double * 3) * 3),
        ("toe", c_double * 3), ("ik_sign_hip", c_double), ("ik_sign_knee", c_double),
    ]


class RobotParams(Structure):
    """``rg_robot_params``."""
    _fields_ = [
        ("legs", LegChain * 4), ("hip_positions", (c_double * 3) * 4),
        ("motor_offset", c_double * 12), ("motor_direction", c_double * 12),
        ("motor_kp", c_double * 12), ("motor_kd", c_double * 12),
        ("stance_duration", c_double * 4), ("duty_factor", c_double * 4),
        ("initial_leg_phase", c_double * 4), ("initial_leg_state", c_int32 * 4),
        ("contact_detection_phase_threshold", c_double),
        ("desired_height", c_double), ("foot_clearance", c_double), ("swing_kp", c_double * 3),
        ("swing_max_clearance", c_double), ("velocity_window", c_int32),
    ]


class ControllerState(Structure):
    """``rg_controller_state`` (all device pointers)."""
    _fields_ = [(name, c_void_p) for name in (
        "time_since_reset", "foot_contacts", "base_velocity_world", "base_orientation_xyzw", "base_rpy",
        "base_rpy_rate", "foot_positions_base", "motor_angles", "command",
        "vel_window", "vel_window_sum", "vel_window_corr", "vel_window_count", "vel_window_head",
        "last_leg_state", "phase_switch_foot_local_position", "swing_joint_angles", "swing_joint_valid",
        "mpc_active_set",
        "desired_leg_state", "leg_state", "normalized_phase", "mpc_contact_state", "swing_foot_target",
        "com_velocity_body", "contact_forces", "motor_torques", "solve_info", "action",
        "motor_velocities", "motor_strength_ratios", "applied_motor_torques")]


class RgCudaError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"rg_cuda error {code}: {message}")
        self.code = code


_lib = None


def library_path() -> str:
    return _build.LIB_PATH


def load(build_if_missing: bool = False):
    """Load librg_cuda.so.  Raises (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if not os.path.exists(path):
        if build_if_missing:
            _build.build()
        else:
            raise RuntimeError(
                f"{path} is missing: build it with `python -m robot_gym.cuda.build` "
                "(or __graft_entry__.build()). There is no CPU fallback for the controller kernels.")
    lib = ctypes.CDLL(path)
    lib.rg_last_error.restype = c_char_p
    lib.rg_version.restype = c_char_p
    lib.rg_launch_count.restype = c_uint64
    lib.rg_mpc_default_params.argtypes = [POINTER(MpcParams), c_double, POINTER(c_double), c_double, c_int]
    lib.rg_workspace_bytes.argtypes = [c_int, c_int, c_int, POINTER(c_size_t)]
    lib.rg_mpc_setup.argtypes = [POINTER(MpcParams), c_void_p, c_size_t, c_void_p]
    lib.rg_mpc_release.argtypes = [c_void_p]
    lib.rg_mpc_build_solve.argtypes = [c_void_p, c_int] + [c_void_p] * 10 + [c_void_p]
    lib.rg_mpc_build_solve_warm.argtypes = [c_void_p, c_int] + [c_void_p] * 11 + [c_void_p]
    lib.rg_mpc_build_solve_io.argtypes = [c_void_p, c_int, POINTER(MpcIo), c_void_p]
    lib.rg_mpc_build_solve_model.argtypes = [c_void_p, c_int, POINTER(MpcIo), POINTER(MpcEnvModel), c_void_p]
    lib.rg_robot_calibrate_ik.argtypes = [POINTER(RobotParams), POINTER(c_double)]
    lib.rg_robot_workspace_bytes.argtypes = [POINTER(c_size_t)]
    lib.rg_robot_setup.argtypes = [POINTER(RobotParams), c_void_p, c_size_t, c_void_p]
    lib.rg_gait_step.argtypes = [c_void_p, c_int] + [c_void_p] * 5 + [c_void_p]
    lib.rg_com_velocity_update.argtypes = [c_void_p, c_int] + [c_void_p] * 9 + [c_void_p]
    lib.rg_swing_targets.argtypes = [c_void_p, c_int] + [c_void_p] * 10 + [c_void_p]
    lib.rg_leg_ik.argtypes = [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.rg_leg_fk.argtypes = [c_void_p, c_int, c_void_p, c_void_p, c_void_p]
    lib.rg_state_from_sim.argtypes = [c_void_p, c_int] + [c_void_p] * 7 + [c_void_p]
    lib.rg_force_to_torque.argtypes = [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.rg_pack_hybrid_action.argtypes = [c_void_p, c_int] + [c_void_p] * 5 + [c_void_p]
    lib.rg_control_step.argtypes = [c_void_p, c_void_p, c_int, POINTER(ControllerState), c_void_p]
    lib.rg_control_step_graph_create.argtypes = [c_void_p, c_void_p, c_int, POINTER(ControllerState), c_void_p, POINTER(c_void_p)]
    lib.rg_control_step_graph_launch.argtypes = [c_void_p, c_void_p]
    lib.rg_control_step_graph_destroy.argtypes = [c_void_p]
    lib.rg_control_step_model.argtypes = [c_void_p, c_void_p, c_int, POINTER(ControllerState), POINTER(MpcEnvModel), c_void_p]
    lib.rg_control_step_graph_create_model.argtypes = [c_void_p, c_void_p, c_int, POINTER(ControllerState), POINTER(MpcEnvModel),
                                                       c_void_p, POINTER(c_void_p)]
    lib.rg_control_step_env.argtypes = [c_void_p, c_void_p, c_int, POINTER(ControllerState), POINTER(MpcEnvModel),
                                        POINTER(GaitEnvParams), c_void_p]
    lib.rg_control_step_graph_create_env.argtypes = [c_void_p, c_void_p, c_int, POINTER(ControllerState), POINTER(MpcEnvModel),
                                                     POINTER(GaitEnvParams), c_void_p, POINTER(c_void_p)]
    lib.rg_mpc_build_solve_schedule.argtypes = [c_void_p, c_int, POINTER(MpcIo), POINTER(MpcEnvModel), c_void_p, c_void_p]
    lib.rg_control_step_plan.argtypes = [c_void_p, c_void_p, c_int, POINTER(ControllerState), POINTER(MpcEnvModel),
                                         POINTER(GaitEnvParams), c_void_p, c_void_p]
    lib.rg_control_step_graph_create_plan.argtypes = [c_void_p, c_void_p, c_int, POINTER(ControllerState), POINTER(MpcEnvModel),
                                                      POINTER(GaitEnvParams), c_void_p, c_void_p, POINTER(c_void_p)]
    lib.rg_mpc_build_solve_footholds.argtypes = [c_void_p, c_int, POINTER(MpcIo), POINTER(MpcEnvModel), c_void_p, c_void_p,
                                                 c_void_p]
    lib.rg_control_step_footholds.argtypes = [c_void_p, c_void_p, c_int, POINTER(ControllerState), POINTER(MpcEnvModel),
                                              POINTER(GaitEnvParams), c_void_p, c_void_p, c_void_p]
    lib.rg_control_step_graph_create_footholds.argtypes = [c_void_p, c_void_p, c_int, POINTER(ControllerState),
                                                           POINTER(MpcEnvModel), POINTER(GaitEnvParams), c_void_p, c_void_p,
                                                           c_void_p, POINTER(c_void_p)]
    lib.rg_hybrid_motor_torque.argtypes = [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.rg_hybrid_motor_torque_ex.argtypes = [c_void_p, c_int] + [c_void_p] * 6 + [c_void_p]
    lib.rg_measure_fma_peak.argtypes = [c_int, c_int, POINTER(c_double)]
    for name in EXPORTED_SYMBOLS:
        fn = getattr(lib, name)
        if name not in ("rg_last_error", "rg_version", "rg_launch_count"):
            fn.restype = c_int
    _lib = lib
    return lib


def check(code: int):
    if code != 0:
        raise RgCudaError(code, load().rg_last_error().decode())


def measure_fma_peak(fp64: bool, iters: int = 1 << 15) -> float:
    """Measured CUDA-core FMA peak in TFLOP/s (diagnostic; synchronises the device)."""
    out = c_double()
    check(load().rg_measure_fma_peak(1 if fp64 else 0, int(iters), ctypes.byref(out)))
    return float(out.value)


def launch_count() -> int:
    return int(load().rg_launch_count())


# ------------------------------------------------------------------------------------------ tensors
def _ptr(t, dtype, shape_tail=None, allow_none=False, n=None, device=None, align=1):
    """Device pointer of a contiguous CUDA tensor after dtype / shape / device / alignment checks.
    ``n``: required leading dimension (the kernels index n_env rows: a shorter tensor would be read out of
    bounds); ``device``: the device the call runs on; ``align``: required pointer alignment in bytes."""
    import torch
    if t is None:
        if allow_none:
            return None
        raise ValueError("tensor argument is None")
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError("rg_cuda wrappers take CUDA tensors only (no CPU fallback)")
    if t.dtype != dtype:
        raise TypeError(f"expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError("tensor must be contiguous")
    if shape_tail is not None and tuple(t.shape[1:]) != tuple(shape_tail):
        raise ValueError(f"expected shape [N,{','.join(map(str, shape_tail))}], got {tuple(t.shape)}")
    if n is not None and (t.dim() == 0 or t.shape[0] != n):
        raise ValueError(f"expected {n} rows (one per env), got shape {tuple(t.shape)}")
    if device is not None:
        want = torch.device(device)
        want_index = torch.cuda.current_device() if want.index is None else want.index
        if t.device.type != want.type or t.device.index != want_index:
            raise ValueError(f"tensor lives on {t.device}, the call runs on {want.type}:{want_index}")
    if align > 1 and t.data_ptr() % align:
        raise ValueError(f"tensor storage must be {align}-byte aligned")
    return c_void_p(t.data_ptr())


def current_stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def default_mpc_params(mass, inertia9, desired_body_height, horizon=10) -> MpcParams:
    p = MpcParams()
    arr = (c_double * 9)(*[float(v) for v in inertia9])
    check(load().rg_mpc_default_params(ctypes.byref(p), float(mass), arr, float(desired_body_height), int(horizon)))
    return p


class MpcWorkspace:
    """Device-resident parameter block + horizon tables prepared by ``rg_mpc_setup``, followed by the fallback
    queue of the two-kernel solve for batches of up to ``max_envs`` envs (4 bytes each).  Larger batches are
    still solved, by the single complete kernel.  One solve at a time per workspace: concurrent solves on
    different streams need a workspace each."""

    def __init__(self, params: MpcParams, device="cuda", max_envs=65536):
        import torch
        lib = load()
        nbytes = c_size_t()
        check(lib.rg_workspace_bytes(int(max_envs), params.horizon, params.num_legs, ctypes.byref(nbytes)))
        self.params = params
        self.horizon = int(params.horizon)
        self.max_envs = int(max_envs)
        self.buffer = torch.zeros(nbytes.value, dtype=torch.uint8, device=device)
        with torch.cuda.device(self.buffer.device):
            check(lib.rg_mpc_setup(ctypes.byref(params), c_void_p(self.buffer.data_ptr()), nbytes.value,
                                   current_stream_ptr()))

    @property
    def ptr(self):
        return c_void_p(self.buffer.data_ptr())

    def __del__(self):
        try:                       # the buffer's memory is about to return to the allocator
            load().rg_mpc_release(c_void_p(self.buffer.data_ptr()))
        except Exception:
            pass


class RobotWorkspace:
    """Device image of the robot model (leg chains, gait, gains) prepared by ``rg_robot_setup``."""

    def __init__(self, params: RobotParams, device="cuda"):
        import torch
        lib = load()
        nbytes = c_size_t()
        check(lib.rg_robot_workspace_bytes(ctypes.byref(nbytes)))
        self.params = params
        self.buffer = torch.zeros(nbytes.value, dtype=torch.uint8, device=device)
        with torch.cuda.device(self.buffer.device):
            check(lib.rg_robot_setup(ctypes.byref(params), c_void_p(self.buffer.data_ptr()), nbytes.value,
                                     current_stream_ptr()))

    @property
    def ptr(self):
        return c_void_p(self.buffer.data_ptr())


def calibrate_ik(params: RobotParams, reference_motor_angles) -> None:
    arr = (c_double * 12)(*[float(v) for v in reference_motor_angles])
    check(load().rg_robot_calibrate_ik(ctypes.byref(params), arr))


def mpc_build_solve(ws: MpcWorkspace, com_velocity_body, base_rpy, base_rpy_rate, foot_contact_state,
                    foot_positions_base, command, com_height=None, contact_forces=None,
                    horizon_forces=None, solve_info=None, want_horizon=False, want_info=True, active_set=None,
                    zero_yaw=False, horizon_forces_f64=None, env_model=None, contact_schedule=None,
                    foothold_plan=None):
    """``rg_mpc_build_solve`` (``rg_mpc_build_solve_warm`` when ``active_set`` -- an ``[N, 4*horizon]`` int16 tensor
    initialised to -1, see ``new_active_set`` -- is given) on the current stream.  ``base_rpy`` is used as given:
    pass a yaw-aligned attitude (yaw = 0) to reproduce TorqueStanceLegController (the controller's fused step
    zeroes it itself) or set ``zero_yaw``.  ``horizon_forces_f64``: optional ``[N,h,12]`` float64 output (the
    unrounded solution; goes through ``rg_mpc_build_solve_io``).  ``env_model``: per-env body and ground for this
    solve (``rg_mpc_build_solve_model``), a dict or an object with ``mass`` [N], ``inertia`` [N,9] or [N,3,3] and
    ``friction_coeffs`` [N,4] float64 CUDA tensors, any of them None (= the workspace's value); an env whose row fails
    the workspace checks gets zero forces and RG_STATUS_BAD_MODEL.  ``contact_schedule``: the planned stance of every
    leg at every horizon step, an ``[N,h,4]`` uint8 or bool CUDA tensor (nonzero = stance; ``rg_mpc_build_solve_schedule``);
    ``foot_contact_state`` is then not read and may be None.  ``foothold_plan``: the position of every foot at every
    horizon step, an ``[N,h,12]`` or ``[N,h,4,3]`` float32 CUDA tensor in the frame of ``foot_positions_base``, used as
    the QP's per-step lever arms (``rg_mpc_build_solve_footholds``); it needs ``contact_schedule``, and
    ``foot_positions_base`` is then not read and may be None.  Returns (contact_forces, horizon_forces, solve_info)."""
    import torch
    if foothold_plan is not None and contact_schedule is None:
        raise ValueError("mpc_build_solve: foothold_plan needs contact_schedule")
    n = base_rpy.shape[0]
    dev = base_rpy.device
    if ws.buffer.device != dev:
        raise ValueError(f"workspace lives on {ws.buffer.device}, inputs on {dev}")
    if contact_forces is None:
        contact_forces = torch.empty((n, 12), dtype=torch.float32, device=dev)
    if horizon_forces is None and want_horizon:
        horizon_forces = torch.empty((n, ws.horizon, 12), dtype=torch.float32, device=dev)
    if solve_info is None and want_info:
        solve_info = torch.empty((n, 4), dtype=torch.int32, device=dev)
    P = lambda t, dtype, tail, **kw: _ptr(t, dtype, tail, n=n, device=dev, **kw)
    hf = None if horizon_forces is None else P(horizon_forces.view(n, ws.horizon * 12), torch.float32, (ws.horizon * 12,))
    args = (ws.ptr, n,
            P(com_velocity_body, torch.float32, (3,)), P(base_rpy, torch.float32, (3,)),
            P(base_rpy_rate, torch.float32, (3,)),
            P(foot_contact_state, torch.uint8, (4,), align=4, allow_none=contact_schedule is not None),
            P(None if foot_positions_base is None else foot_positions_base.view(n, 12), torch.float32, (12,), align=16,
              allow_none=foothold_plan is not None), P(command, torch.float32, (3,)),
            P(com_height, torch.float32, (), allow_none=True),
            P(contact_forces, torch.float32, (12,)), hf,
            P(solve_info, torch.int32, (4,), allow_none=True))
    model = None if env_model is None else env_model_struct(env_model, n, dev)
    schedule = None
    if contact_schedule is not None:
        if isinstance(contact_schedule, torch.Tensor) and contact_schedule.dtype == torch.bool:
            contact_schedule = contact_schedule.view(torch.uint8)
        schedule = P(contact_schedule, torch.uint8, (ws.horizon, 4), align=4)
    feet = None
    if foothold_plan is not None:
        if isinstance(foothold_plan, torch.Tensor) and tuple(foothold_plan.shape[1:]) == (ws.horizon, 4, 3):
            foothold_plan = foothold_plan.view(foothold_plan.shape[0], ws.horizon, 12)
        feet = P(foothold_plan, torch.float32, (ws.horizon, 12), align=16)
    with torch.cuda.device(dev):
        if zero_yaw or horizon_forces_f64 is not None or model is not None or schedule is not None:
            io = MpcIo(*[a if a is None or isinstance(a, int) else a.value for a in args[2:]],
                       None if active_set is None else P(active_set, torch.int16, (4 * ws.horizon,)).value,
                       None if horizon_forces_f64 is None else P(horizon_forces_f64.view(n, ws.horizon * 12), torch.float64, (ws.horizon * 12,)).value,
                       1 if zero_yaw else 0, 0)
            if feet is not None:
                check(load().rg_mpc_build_solve_footholds(ws.ptr, n, ctypes.byref(io),
                                                          None if model is None else ctypes.byref(model), schedule, feet,
                                                          current_stream_ptr()))
            elif schedule is not None:
                check(load().rg_mpc_build_solve_schedule(ws.ptr, n, ctypes.byref(io),
                                                         None if model is None else ctypes.byref(model), schedule,
                                                         current_stream_ptr()))
            elif model is None:
                check(load().rg_mpc_build_solve_io(ws.ptr, n, ctypes.byref(io), current_stream_ptr()))
            else:
                check(load().rg_mpc_build_solve_model(ws.ptr, n, ctypes.byref(io), ctypes.byref(model), current_stream_ptr()))
        elif active_set is None:
            check(load().rg_mpc_build_solve(*args, current_stream_ptr()))
        else:
            check(load().rg_mpc_build_solve_warm(*args, P(active_set, torch.int16, (4 * ws.horizon,)), current_stream_ptr()))
    return contact_forces, horizon_forces, solve_info


def env_model_struct(env_model, n, device) -> MpcEnvModel:
    """``MpcEnvModel`` of a dict / object with ``mass`` [N], ``inertia`` [N,9] or [N,3,3], ``friction_coeffs`` [N,4]
    float64 CUDA tensors (any may be None or absent), after the ``_ptr`` checks.  The tensors must outlive the solve."""
    import torch
    get = env_model.get if isinstance(env_model, dict) else lambda k: getattr(env_model, k, None)
    mass, inertia, mu = get("mass"), get("inertia"), get("friction_coeffs")
    if inertia is not None and isinstance(inertia, torch.Tensor) and inertia.dim() == 3:
        if tuple(inertia.shape[1:]) != (3, 3):
            raise ValueError(f"expected inertia [N,9] or [N,3,3], got {tuple(inertia.shape)}")
        inertia = inertia.view(inertia.shape[0], 9) if inertia.is_contiguous() else inertia
    P = lambda t, tail: _ptr(t, torch.float64, tail, allow_none=True, n=n, device=device, align=8)
    m = MpcEnvModel()
    m.mass, m.inertia, m.friction_coeffs = P(mass, ()), P(inertia, (9,)), P(mu, (4,))
    return m


def new_active_set(n_env, horizon, device="cuda"):
    """Warm-start buffer of ``rg_mpc_build_solve_warm``: ``[N, 4*horizon]`` 16-bit words, all RG_ACTIVE_SET_UNKNOWN
    (torch has no uint16 arithmetic: int16 -1 is the same bit pattern 0xFFFF)."""
    import torch
    return torch.full((n_env, 4 * horizon), -1, dtype=torch.int16, device=device)
