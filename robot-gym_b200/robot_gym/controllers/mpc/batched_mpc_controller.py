"""Batched drop-in for ``MPCController`` (robot_gym/controllers/mpc/mpc_controller.py:14-113).

Same interface -- ``update_controller_params`` / ``get_action`` / ``reset`` / ``kinematics_model`` /
``get_standing_action`` / ``MOTOR_CONTROL_MODE`` -- but one instance drives N independent envs whose
state lives in CUDA tensors, and every numerical step (gait generator, COM velocity estimator,
Raibert swing controller, leg IK, convex-MPC stance QP, force -> torque, hybrid action packing)
runs in the sm_100a kernels behind ``robot_gym.cuda`` (C ABI: include/rg_cuda.h).  The third-party
``mpc_controller`` / ``mpc_osqp`` / PyBullet calls of the reference are not used.

There is no CPU path: constructing the controller without the CUDA library or a CUDA device raises.
"""
from __future__ import annotations

import ctypes
from ctypes import c_void_p

import numpy as np
import torch

from robot_gym import cuda as rg
from robot_gym.controllers.controller import Controller
from robot_gym.controllers.mpc.batched_kinematics import BatchedKinematics, robot_params_from_description
from robot_gym.controllers.mpc.leg_state import LegState
from robot_gym.model.robots.descriptions import MOTOR_CONTROL_HYBRID


class _LegControllerHandle:
    """Stands in for ``_mpc_controller.swing_leg_controller`` / ``.stance_leg_controller``: the
    reference adapter writes ``desired_speed`` / ``desired_twisting_speed`` onto both
    (mpc_controller.py:97-100).  Here both handles alias the controller's [N,3] command tensor."""

    def __init__(self, owner):
        self._owner = owner

    @property
    def desired_speed(self):
        cmd = self._owner.command
        return torch.stack([cmd[:, 0], cmd[:, 1], torch.zeros_like(cmd[:, 0])], dim=1)

    @desired_speed.setter
    def desired_speed(self, value):
        v = torch.as_tensor(value, dtype=torch.float32, device=self._owner.device)
        self._owner.command[:, 0] = v[..., 0]
        self._owner.command[:, 1] = v[..., 1]

    @property
    def desired_twisting_speed(self):
        return self._owner.command[:, 2]

    @desired_twisting_speed.setter
    def desired_twisting_speed(self, value):
        self._owner.command[:, 2] = torch.as_tensor(value, dtype=torch.float32, device=self._owner.device)


class _LocomotionHandle:
    def __init__(self, owner):
        self.swing_leg_controller = _LegControllerHandle(owner)
        self.stance_leg_controller = _LegControllerHandle(owner)


class BatchedMPCController(Controller):

    MOTOR_CONTROL_MODE = MOTOR_CONTROL_HYBRID      # mpc_controller.py:16

    GRAPH_MAX_ENVS = 2048          # below this a control step is launch-bound: replay it as one CUDA graph

    def __init__(self, robot, get_time_since_reset, horizon=10, mpc_overrides=None, squeeze_single=True,
                 warm_start=True, use_graph=None, contact_plan=False, foothold_plan=False):
        """``robot``: batched state provider with the getter names of robot.py (see
        ``SyntheticRobotBatch``); ``get_time_since_reset``: callable returning a float or an
        ``[N]`` float64 tensor (Simulation.GetTimeSinceReset, core/simulation.py:141-142).
        ``warm_start``: seed each stance QP with the active set the same env verified one control step
        earlier (``rg_mpc_build_solve_warm``); the optimum is unique, so the forces do not depend on it.
        ``contact_plan``: plan the stance QP over each env's gait schedule -- the desired stance of every leg at every
        horizon step (``rg_control_step_plan``) -- instead of holding the current contact row over the horizon.  The
        schedule the step solved against is ``mpc_contact_schedule`` ([N, horizon, 4] uint8, row 0 = ``mpc_contact_state``).
        ``foothold_plan`` (needs ``contact_plan``): take the QP's lever arms at every horizon step from the predicted
        footholds (``rg_control_step_footholds``): a planted foot moves back at the commanded velocity, and a leg that
        touches down inside the horizon lands at its Raibert foothold.  The footholds the step solved against are
        ``mpc_foothold_plan`` ([N, horizon, 4, 3] float32, in the frame of the feet's base positions)."""
        if foothold_plan and not contact_plan:
            raise ValueError("foothold_plan=True needs contact_plan=True (the footholds follow the contact schedule)")
        if not torch.cuda.is_available():
            raise RuntimeError("BatchedMPCController needs a CUDA device (no CPU fallback)")
        rg.load()
        self._adapter = None
        if not hasattr(robot, "num_envs"):
            # a stock (PyBullet-backed) Robot, as Simulation.build_world passes it (core/simulation.py:117):
            # N = 1 behind the batched getter surface
            from robot_gym.model.robots.pybullet_adapter import PyBulletRobotAdapter
            robot = self._adapter = PyBulletRobotAdapter(robot)
        super().__init__(robot, get_time_since_reset)
        self._constants = robot.GetCtrlConstants()
        self.device = torch.device(getattr(robot, "device", "cuda"))
        self.num_envs = int(getattr(robot, "num_envs", 1))
        self.horizon = int(horizon)
        self._squeeze_single = bool(squeeze_single)
        n, dev = self.num_envs, self.device
        # one graph launch per step instead of three kernel launches (rg_control_step_graph_*): default for small batches
        self._use_graph = (n <= self.GRAPH_MAX_ENVS) if use_graph is None else bool(use_graph)
        self._graph = None
        self._graph_invalidations = 0
        self.env_mass = self.env_inertia = self.env_friction_coeffs = None   # per-env model (set_env_model)
        self._env_model = None
        # per-env gait (set_env_gait)
        self.env_stance_duration = self.env_duty_factor = self.env_initial_leg_phase = self.env_initial_leg_state = None
        self._env_gait = None

        # --- C-ABI workspaces (the analogue of _setup_controller, mpc_controller.py:28-66)
        c = self._constants
        self.mpc_params = rg.default_mpc_params(c.MPC_BODY_MASS, c.MPC_BODY_INERTIA, c.MPC_BODY_HEIGHT, self.horizon)
        for key, value in (mpc_overrides or {}).items():
            field = getattr(self.mpc_params, key)
            if hasattr(field, "__len__"):
                for i, v in enumerate(value):
                    field[i] = v
            else:
                setattr(self.mpc_params, key, value)
        self.robot_params = robot_params_from_description(robot, c)
        with torch.cuda.device(dev):
            self._mpc_ws = rg.MpcWorkspace(self.mpc_params, device=dev, max_envs=n)
            self._robot_ws = rg.RobotWorkspace(self.robot_params, device=dev)
        self._kinematics = BatchedKinematics(self._robot_ws, dev)
        self._window = int(self.robot_params.velocity_window)

        # --- persistent controller state + outputs
        f32, f64, i32, u8 = torch.float32, torch.float64, torch.int32, torch.uint8
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)
        self.command = z((n, 3), f32)
        self.vel_window = z((n, 3, self._window), f64)
        self.vel_window_sum = z((n, 3), f64)
        self.vel_window_corr = z((n, 3), f64)
        self.vel_window_count = z((n,), i32)
        self.vel_window_head = z((n,), i32)
        self.last_leg_state = z((n, 4), i32)
        self.phase_switch_foot_local_position = z((n, 12), f32)
        self.swing_joint_angles = z((n, 12), f32)
        self.swing_joint_valid = z((n, 4), u8)
        self.desired_leg_state = z((n, 4), i32)
        self.leg_state = z((n, 4), i32)
        self.normalized_phase = z((n, 4), f64)
        self.mpc_contact_state = z((n, 4), u8)
        self.swing_foot_target = z((n, 12), f32)
        self.com_velocity_body = z((n, 3), f32)
        self.contact_forces = z((n, 12), f32)
        self.motor_torques = z((n, 12), f32)
        self.solve_info = z((n, 4), i32)
        self.mpc_active_set = rg.new_active_set(n, self.horizon, dev) if warm_start else None
        self.mpc_contact_schedule = z((n, self.horizon, 4), u8) if contact_plan else None
        self.mpc_foothold_plan = z((n, self.horizon, 4, 3), f32) if foothold_plan else None
        self.action = z((n, 60), f32)
        self.reset_time = z((n,), f64)
        self.time_since_reset = z((n,), f64)
        self._mpc_controller = _LocomotionHandle(self)
        self._state = self._build_state()
        self._input_cache = {}
        self.update_controller_params(self.get_standing_action())
        self.reset()

    # ------------------------------------------------------------------ reference interface
    @property
    def kinematics_model(self):                    # mpc_controller.py:24-26 (used by robot.py:94-102)
        return self._kinematics

    @staticmethod
    def setup_ui_params(pybullet_client):          # mpc_controller.py:68-73
        return tuple(pybullet_client.addUserDebugParameter(name, -2., 2., 0.) for name in ("Vx", "Vy", "Wz"))

    @staticmethod
    def read_ui_params(pybullet_client, ui):       # mpc_controller.py:75-81
        return tuple(pybullet_client.readUserDebugParameter(handle) for handle in ui)

    @staticmethod
    def get_standing_action():                     # mpc_controller.py:111-113
        return 0., 0.

    def update_controller_params(self, params):
        """(vx, wz) / (vx, vy, wz) as scalars (broadcast to every env) or an [N,2] / [N,3] tensor;
        the per-robot command offsets are added exactly as mpc_controller.py:83-100 does."""
        c = self._constants
        if isinstance(params, torch.Tensor) and params.dim() == 2:
            p = params.to(device=self.device, dtype=torch.float32)
            if p.shape[0] != self.num_envs or p.shape[1] not in (2, 3):
                raise ValueError(f"expected [{self.num_envs},2] or [{self.num_envs},3], got {tuple(p.shape)}")
            vx, wz = p[:, 0], p[:, -1]
            vy = p[:, 1] if p.shape[1] == 3 else torch.zeros_like(vx)
        else:
            if len(params) == 2:
                vx, wz = params
                vy = 0.
            elif len(params) == 3:
                vx, vy, wz = params
            else:
                raise ValueError("params must have 2 or 3 entries")
        self.command[:, 0] = torch.as_tensor(vx, dtype=torch.float32, device=self.device) + float(c.VX_OFFSET)
        self.command[:, 1] = torch.as_tensor(vy, dtype=torch.float32, device=self.device) + float(c.VY_OFFSET)
        self.command[:, 2] = torch.as_tensor(wz, dtype=torch.float32, device=self.device) + float(c.WZ_OFFSET)

    def _clock(self):
        t = self.get_time_since_reset()
        if isinstance(t, torch.Tensor):
            return t.to(device=self.device, dtype=torch.float64).expand(self.num_envs)
        return torch.full((self.num_envs,), float(t), dtype=torch.float64, device=self.device)

    def reset(self, env_ids=None):
        """LocomotionController.reset (mpc_controller.py:108-109): reset_time = clock(); gait, estimator,
        swing (latch = current feet, joint-angle store cleared) and stance state are re-armed.  The leg states
        start from INIT_LEG_STATE, or with a per-env gait (``set_env_gait``) from each env's own
        ``env_initial_leg_state`` row.  ``env_ids`` (LongTensor) restricts the reset to a subset of envs."""
        sel = slice(None) if env_ids is None else env_ids
        if self._adapter is not None:
            self._adapter.refresh()
        self.reset_time[sel] = self._clock()[sel]
        self.vel_window[sel] = 0
        self.vel_window_sum[sel] = 0
        self.vel_window_corr[sel] = 0
        self.vel_window_count[sel] = 0
        self.vel_window_head[sel] = 0
        self.last_leg_state[sel] = -1       # "aliased" marker: the first update never latches
        feet = self._robot.GetFootPositionsInBaseFrame().reshape(self.num_envs, 12)
        self.phase_switch_foot_local_position[sel] = feet[sel].to(torch.float32)
        self.swing_joint_valid[sel] = 0
        if self.mpc_active_set is not None:
            self.mpc_active_set[sel] = -1   # RG_ACTIVE_SET_UNKNOWN
        if self._env_gait is None:
            init_state = torch.tensor([int(s) for s in self._constants.INIT_LEG_STATE], dtype=torch.int32, device=self.device)
        else:                               # OpenloopGaitGenerator.reset with each env's own initial_leg_state
            init_state = self.env_initial_leg_state[sel]
        self.desired_leg_state[sel] = init_state
        self.leg_state[sel] = init_state
        self.normalized_phase[sel] = 0

    def get_action(self):
        """``update()`` + ``get_action()`` of the third-party glue in one fused C-ABI call
        (mpc_controller.py:102-106).  Returns the [N,60] hybrid command tensor (N == 1: a [60]
        float32 numpy array, what Simulation.ApplyStepAction consumes)."""
        self.step()
        if self.num_envs == 1 and self._squeeze_single:
            return self.action[0].cpu().numpy()
        return self.action

    # ------------------------------------------------------------------ batched step
    # (field of rg_controller_state, robot getter, dtype, trailing shape, pointer alignment)
    _ROBOT_INPUTS = (
        ("foot_contacts", "GetFootContacts", torch.uint8, (4,), 4),
        ("base_velocity_world", "GetBaseVelocity", torch.float32, (3,), 4),
        ("base_orientation_xyzw", "GetTrueBaseOrientation", torch.float32, (4,), 4),
        ("base_rpy", "GetBaseRollPitchYaw", torch.float32, (3,), 4),
        ("base_rpy_rate", "GetBaseRollPitchYawRate", torch.float32, (3,), 4),
        ("foot_positions_base", "GetFootPositionsInBaseFrame", torch.float32, (12,), 16),
        ("motor_angles", "GetMotorAngles", torch.float32, (12,), 4),
    )

    def _build_state(self):
        """The ``rg_controller_state`` of this controller, built ONCE: every pointer to a controller-owned
        tensor is fixed for the controller's lifetime; ``step`` only refreshes the robot-provided inputs whose
        storage changed since the previous step."""
        n, dev = self.num_envs, self.device
        f32, f64, i32, u8 = torch.float32, torch.float64, torch.int32, torch.uint8
        P = lambda t, dtype, tail=None, **kw: rg._ptr(t, dtype, tail, n=n, device=dev, **kw)
        st = rg.ControllerState()
        st.time_since_reset = P(self.time_since_reset, f64)
        st.command = P(self.command, f32, (3,))
        st.vel_window = P(self.vel_window, f64)
        st.vel_window_sum = P(self.vel_window_sum, f64)
        st.vel_window_corr = P(self.vel_window_corr, f64)
        st.vel_window_count = P(self.vel_window_count, i32)
        st.vel_window_head = P(self.vel_window_head, i32)
        st.last_leg_state = P(self.last_leg_state, i32)
        st.phase_switch_foot_local_position = P(self.phase_switch_foot_local_position, f32)
        st.swing_joint_angles = P(self.swing_joint_angles, f32)
        st.swing_joint_valid = P(self.swing_joint_valid, u8)
        st.mpc_active_set = P(self.mpc_active_set, torch.int16, allow_none=True)
        st.desired_leg_state = P(self.desired_leg_state, i32)
        st.leg_state = P(self.leg_state, i32)
        st.normalized_phase = P(self.normalized_phase, f64)
        st.mpc_contact_state = P(self.mpc_contact_state, u8, align=4)
        st.swing_foot_target = P(self.swing_foot_target, f32)
        st.com_velocity_body = P(self.com_velocity_body, f32)
        st.contact_forces = P(self.contact_forces, f32)
        st.motor_torques = P(self.motor_torques, f32)
        st.solve_info = P(self.solve_info, i32)
        st.action = P(self.action, f32)
        return st

    def _refresh_inputs(self):
        """Pull the robot getters (robot.py:79-236,389-397).  A tensor whose storage, shape and dtype are the ones
        validated last step is not validated again; anything new is checked for dtype, contiguity, [N, ...]
        shape, device and alignment before its pointer reaches a kernel.  Returns True if any pointer changed."""
        n, cache, st = self.num_envs, self._input_cache, self._state
        changed = False
        for field, getter, dtype, tail, align in self._ROBOT_INPUTS:
            t = getattr(self._robot, getter)()
            if field == "foot_positions_base" and isinstance(t, torch.Tensor) and t.dim() == 3:
                t = t.view(n, 12) if t.is_contiguous() else t.reshape(n, 12)
            key = (t.data_ptr(), t.shape, t.dtype) if isinstance(t, torch.Tensor) else None
            if key is None or cache.get(field) != key:
                setattr(st, field, rg._ptr(t, dtype, tail, n=n, device=self.device, align=align))
                cache[field] = (t.data_ptr(), t.shape, t.dtype)
                changed = True
            cache[field + "_ref"] = t          # keep the storage alive until the kernels have consumed it
        return changed

    def attach_torque_consumer(self, motor_velocities_getter, strength_ratios=None, applied_motor_torques=None):
        """Fuse the HYBRID motor model of the first physics tick into the step's epilogue (SURVEY.md 8f row 1):
        ``applied_motor_torques`` [N,12] = strength_ratios * (-kp (q - q_des) - kd (qd - qd_des) + tau) *
        MOTOR_DIRECTION (simple_motor.py:128-140, robot.py:291-292) is written by the same launch that packs the
        command, so a GPU physics step never reads the [N,60] command back.  Returns the output tensor."""
        n, dev, f32 = self.num_envs, self.device, torch.float32
        if applied_motor_torques is None:
            applied_motor_torques = torch.zeros((n, 12), dtype=f32, device=dev)
        self.applied_motor_torques = applied_motor_torques
        self._motor_velocities_getter = motor_velocities_getter
        self._strength_ratios = strength_ratios
        self._destroy_graph()                                  # the captured step does not write the torques yet
        self._state.applied_motor_torques = rg._ptr(applied_motor_torques, f32, (12,), n=n, device=dev)
        self._state.motor_strength_ratios = rg._ptr(strength_ratios, f32, (12,), allow_none=True, n=n, device=dev)
        return applied_motor_torques

    def step(self):
        if self._adapter is not None:
            self._adapter.refresh()
        torch.sub(self._clock(), self.reset_time, out=self.time_since_reset)
        changed = self._refresh_inputs()
        if getattr(self, "_motor_velocities_getter", None) is not None:
            qd = self._motor_velocities_getter()
            key = (qd.data_ptr(), qd.shape, qd.dtype)
            if self._input_cache.get("motor_velocities") != key:
                self._state.motor_velocities = rg._ptr(qd, torch.float32, (12,), n=self.num_envs, device=self.device)
                self._input_cache["motor_velocities"] = key
                changed = True
            self._input_cache["motor_velocities_ref"] = qd
        lib = rg.load()
        with torch.cuda.device(self.device):
            if not self._use_graph:
                self._eager_step(lib)
            else:
                if changed and self._graph is not None:          # a buffer moved: the captured pointers are stale
                    self._destroy_graph()
                    self._graph_invalidations += 1
                    if self._graph_invalidations >= 3:            # a provider that hands out fresh tensors every step
                        self._use_graph = False
                        self._eager_step(lib)
                        return self.action
                if self._graph is None:
                    # creating the graph executes this step eagerly (and synchronises once)
                    handle = ctypes.c_void_p()
                    if self.mpc_foothold_plan is not None:
                        rg.check(lib.rg_control_step_graph_create_footholds(
                            self._mpc_ws.ptr, self._robot_ws.ptr, self.num_envs, ctypes.byref(self._state),
                            self._env_model_ref(), self._env_gait_ref(), self._schedule_ptr(), self._footholds_ptr(),
                            rg.current_stream_ptr(), ctypes.byref(handle)))
                    elif self.mpc_contact_schedule is not None:
                        rg.check(lib.rg_control_step_graph_create_plan(self._mpc_ws.ptr, self._robot_ws.ptr, self.num_envs,
                                                                       ctypes.byref(self._state), self._env_model_ref(),
                                                                       self._env_gait_ref(), self._schedule_ptr(),
                                                                       rg.current_stream_ptr(), ctypes.byref(handle)))
                    elif self._env_model is None and self._env_gait is None:
                        rg.check(lib.rg_control_step_graph_create(self._mpc_ws.ptr, self._robot_ws.ptr, self.num_envs,
                                                                  ctypes.byref(self._state), rg.current_stream_ptr(),
                                                                  ctypes.byref(handle)))
                    else:
                        rg.check(lib.rg_control_step_graph_create_env(self._mpc_ws.ptr, self._robot_ws.ptr, self.num_envs,
                                                                      ctypes.byref(self._state), self._env_model_ref(),
                                                                      self._env_gait_ref(), rg.current_stream_ptr(),
                                                                      ctypes.byref(handle)))
                    self._graph = handle
                else:
                    rg.check(lib.rg_control_step_graph_launch(self._graph, rg.current_stream_ptr()))
        return self.action

    def _eager_step(self, lib):
        if self.mpc_foothold_plan is not None:
            rg.check(lib.rg_control_step_footholds(self._mpc_ws.ptr, self._robot_ws.ptr, self.num_envs,
                                                   ctypes.byref(self._state), self._env_model_ref(), self._env_gait_ref(),
                                                   self._schedule_ptr(), self._footholds_ptr(), rg.current_stream_ptr()))
        elif self.mpc_contact_schedule is not None:
            rg.check(lib.rg_control_step_plan(self._mpc_ws.ptr, self._robot_ws.ptr, self.num_envs, ctypes.byref(self._state),
                                              self._env_model_ref(), self._env_gait_ref(), self._schedule_ptr(),
                                              rg.current_stream_ptr()))
        elif self._env_model is None and self._env_gait is None:
            rg.check(lib.rg_control_step(self._mpc_ws.ptr, self._robot_ws.ptr, self.num_envs,
                                         ctypes.byref(self._state), rg.current_stream_ptr()))
        else:
            rg.check(lib.rg_control_step_env(self._mpc_ws.ptr, self._robot_ws.ptr, self.num_envs, ctypes.byref(self._state),
                                             self._env_model_ref(), self._env_gait_ref(), rg.current_stream_ptr()))

    def _schedule_ptr(self):
        return rg._ptr(self.mpc_contact_schedule, torch.uint8, (self.horizon, 4), n=self.num_envs, device=self.device, align=4)

    def _footholds_ptr(self):
        return rg._ptr(self.mpc_foothold_plan, torch.float32, (self.horizon, 4, 3), n=self.num_envs, device=self.device,
                       align=16)

    def _env_model_ref(self):
        return None if self._env_model is None else ctypes.byref(self._env_model)

    def _env_gait_ref(self):
        return None if self._env_gait is None else ctypes.byref(self._env_gait)

    # ------------------------------------------------------------------ per-env body and ground
    def set_env_model(self, mass=None, inertia=None, friction_coeffs=None, env_ids=None):
        """Per-env mass [N] (kg), body-frame inertia [N,9] / [N,3,3] and friction coefficients [N,4] (one per
        pyramid row) for the stance solve -- what each reference process passes to its own ``ConvexMpc(mass,
        inertia, ...)`` and to ``compute_contact_forces(..., friction, ...)``.  The force bounds follow the mass with
        the workspace's ratios (fz_max / mass, fz_min / mass).  Scalars and shorter leading shapes broadcast; with
        ``env_ids`` only those rows are written.  The first call allocates controller-owned float64 tensors
        (``env_mass``, ``env_inertia``, ``env_friction_coeffs``) filled with the robot's constants and drops the
        captured step graph once; later calls write into them in place, so a captured graph stays valid.
        Raises ``ValueError`` (before anything is written) for a mass that is not > 0 and finite, an inertia that is
        not finite or not invertible, or a friction coefficient that is not > 0.  Synchronises once."""
        n, dev, f64 = self.num_envs, self.device, torch.float64
        if self._env_model is None:
            p = self.mpc_params                       # the workspace's own values: robot constants + mpc_overrides
            self.env_mass = torch.full((n,), float(p.mass), dtype=f64, device=dev)
            self.env_inertia = torch.tensor([float(v) for v in p.inertia], dtype=f64, device=dev).repeat(n, 1)
            self.env_friction_coeffs = torch.tensor([float(v) for v in p.friction_coeffs], dtype=f64, device=dev).repeat(n, 1)
            model = rg.MpcEnvModel()
            model.mass = rg._ptr(self.env_mass, f64, (), n=n, device=dev, align=8)
            model.inertia = rg._ptr(self.env_inertia, f64, (9,), n=n, device=dev, align=8)
            model.friction_coeffs = rg._ptr(self.env_friction_coeffs, f64, (4,), n=n, device=dev, align=8)
            self._env_model = model
            self._destroy_graph()                     # the captured step was the model-free one
        sel = slice(None) if env_ids is None else torch.as_tensor(env_ids, device=dev, dtype=torch.long)
        rows = n if env_ids is None else int(sel.numel())
        new = {}
        if mass is not None:
            new["mass"] = torch.as_tensor(mass, dtype=f64, device=dev).expand(rows)
        if inertia is not None:
            i = torch.as_tensor(inertia, dtype=f64, device=dev)
            new["inertia"] = (i.reshape(*i.shape[:-2], 9) if i.dim() >= 2 and tuple(i.shape[-2:]) == (3, 3) else i).expand(rows, 9)
        if friction_coeffs is not None:
            new["friction_coeffs"] = torch.as_tensor(friction_coeffs, dtype=f64, device=dev).expand(rows, 4)
        validate_env_model(**new)
        if "mass" in new:
            self.env_mass[sel] = new["mass"]
        if "inertia" in new:
            self.env_inertia[sel] = new["inertia"]
        if "friction_coeffs" in new:
            self.env_friction_coeffs[sel] = new["friction_coeffs"]

    # ------------------------------------------------------------------ per-env gait
    def set_env_gait(self, stance_duration=None, duty_factor=None, initial_leg_phase=None, initial_leg_state=None,
                     schedule=None, env_ids=None):
        """Per-env ``OpenloopGaitGenerator(stance_duration, duty_factor, initial_leg_phase, initial_leg_state)``
        arguments, each [N,4] (leg order FR, FL, RR, RL) -- what each reference process passes to its own gait
        generator (mpc_controller.py:30-35).  ``schedule`` (a name of ``descriptions.GAIT_SCHEDULES``: trot, pace,
        bound, walk, stand) supplies all four instead.  Scalars and [4] rows broadcast; with ``env_ids`` only those rows
        are written.  The stance duration also sets the Raibert foothold of the swing legs.

        The first call allocates controller-owned tensors (``env_stance_duration``, ``env_duty_factor``,
        ``env_initial_leg_phase`` float64 and ``env_initial_leg_state`` int32, [N,4]) filled with the robot's gait
        constants and drops the captured step graph once; later calls write into them in place, so a captured graph
        stays valid.  Raises ``ValueError`` before anything is written for a stance duration that is not > 0 and
        finite, a duty factor outside (0, 1], a phase outside [0, 1) or a state other than SWING / STANCE.

        The new timing applies from the next step, at each env's current clock (``time_since_reset``): this call
        does not reset.  A task that wants the envs to start a fresh cycle calls ``reset(env_ids)`` after it, which
        re-arms their leg states from the new ``initial_leg_state`` rows.  Synchronises once."""
        from robot_gym.model.robots.descriptions import GAIT_SCHEDULES
        n, dev, f64, i32 = self.num_envs, self.device, torch.float64, torch.int32
        given = dict(stance_duration=stance_duration, duty_factor=duty_factor, initial_leg_phase=initial_leg_phase,
                     initial_leg_state=initial_leg_state)
        if schedule is not None:
            if any(v is not None for v in given.values()):
                raise ValueError("set_env_gait: pass either schedule= or the gait arrays, not both")
            if schedule not in GAIT_SCHEDULES:
                raise ValueError(f"unknown gait schedule {schedule!r}; expected one of {tuple(GAIT_SCHEDULES)}")
            given = _gait_rows(GAIT_SCHEDULES[schedule])
        sel = slice(None) if env_ids is None else torch.as_tensor(env_ids, device=dev, dtype=torch.long)
        rows = n if env_ids is None else int(sel.numel())
        new = {}
        for key, value in given.items():
            if value is None:
                continue
            if key == "initial_leg_state":
                t = torch.as_tensor(value if isinstance(value, torch.Tensor) else np.asarray(value), device=dev)
                if t.is_floating_point() and not torch.equal(t, t.round()):
                    raise ValueError("env gait: initial_leg_state must hold integer leg states")
                new[key] = t.to(i32).expand(rows, 4)
            else:
                new[key] = torch.as_tensor(value, dtype=f64, device=dev).expand(rows, 4)
        validate_env_gait(**new)
        if self._env_gait is None:
            c = _gait_rows(self._constants)            # the robot workspace's own gait (robot_params_from_description)
            self.env_stance_duration = torch.tensor(c["stance_duration"], dtype=f64, device=dev).repeat(n, 1)
            self.env_duty_factor = torch.tensor(c["duty_factor"], dtype=f64, device=dev).repeat(n, 1)
            self.env_initial_leg_phase = torch.tensor(c["initial_leg_phase"], dtype=f64, device=dev).repeat(n, 1)
            self.env_initial_leg_state = torch.tensor(c["initial_leg_state"], dtype=i32, device=dev).repeat(n, 1)
            gait = rg.GaitEnvParams()
            gait.stance_duration = rg._ptr(self.env_stance_duration, f64, (4,), n=n, device=dev, align=8)
            gait.duty_factor = rg._ptr(self.env_duty_factor, f64, (4,), n=n, device=dev, align=8)
            gait.initial_leg_phase = rg._ptr(self.env_initial_leg_phase, f64, (4,), n=n, device=dev, align=8)
            gait.initial_leg_state = rg._ptr(self.env_initial_leg_state, i32, (4,), n=n, device=dev, align=4)
            self._env_gait = gait
            self._destroy_graph()                     # the captured step was the gait-free one
        for key, value in new.items():
            getattr(self, "env_" + key)[sel] = value

    def _destroy_graph(self):
        if self._graph is not None:
            try:
                rg.load().rg_control_step_graph_destroy(self._graph)
            finally:
                self._graph = None

    def __del__(self):
        try:
            self._destroy_graph()
        except Exception:
            pass

    def unverified_count(self):
        """Number of envs (device scalar, no synchronisation) whose last stance QP did NOT end in a verified KKT
        point (neither RG_STATUS_POLISHED nor RG_STATUS_NO_STANCE; an env with RG_STATUS_BAD_MODEL counts).  The reference's OSQP path returns forces only
        on OSQP_SOLVED; here such an env still gets forces -- the best interior-point iterate, feasible by
        construction -- and this counter is the signal: 0 in every batch measured so far."""
        status = self.solve_info[:, rg.RG_INFO_STATUS]
        return ((status & (rg.RG_STATUS_POLISHED | rg.RG_STATUS_NO_STANCE)) == 0).sum()

    # ------------------------------------------------------------------ rollout statistics
    def rollout_stats(self):
        """Per-rank statistics vector for the multi-GPU all-gather (SURVEY.md 8e):
        [solves, sum ipm iters, max ipm iters, sum polish rounds, polished count, no-stance count,
         numeric-flag count, sum |f|_1]  (float64, on device)."""
        info = self.solve_info
        status = info[:, rg.RG_INFO_STATUS]
        iters = info[:, rg.RG_INFO_IPM_ITERS].to(torch.float64)
        return torch.stack([
            torch.tensor(float(self.num_envs), dtype=torch.float64, device=self.device),
            iters.sum(), iters.max(),
            info[:, rg.RG_INFO_POLISH_ROUNDS].to(torch.float64).sum(),
            ((status & rg.RG_STATUS_POLISHED) != 0).to(torch.float64).sum(),
            ((status & rg.RG_STATUS_NO_STANCE) != 0).to(torch.float64).sum(),
            ((status & rg.RG_STATUS_NUMERIC) != 0).to(torch.float64).sum(),
            self.contact_forces.abs().to(torch.float64).sum(),
        ])


def validate_env_model(mass=None, inertia=None, friction_coeffs=None):
    """The checks rg_mpc_setup makes on one parameter set, applied to every row of a per-env model (float64 tensors
    on any device: mass [..], inertia [.., 9], friction_coeffs [.., 4]).  Raises ValueError naming the first failing
    row; the kernels flag such a row with RG_STATUS_BAD_MODEL instead."""
    def fail(what, bad):
        idx = torch.nonzero(bad.reshape(bad.shape[0], -1).any(dim=1) if bad.dim() else bad.reshape(1)).flatten()
        if idx.numel():
            raise ValueError(f"env model: {what} (first bad row {int(idx[0])})")
    if mass is not None:
        m = mass.to(torch.float64).reshape(-1)
        fail("mass must be > 0 and finite", ~((m > 0) & torch.isfinite(m)))
    if inertia is not None:
        i = inertia.to(torch.float64).reshape(-1, 9)
        fail("inertia must be finite", ~torch.isfinite(i))
        det = (i[:, 0] * (i[:, 4] * i[:, 8] - i[:, 5] * i[:, 7]) + i[:, 1] * (i[:, 5] * i[:, 6] - i[:, 3] * i[:, 8]) +
               i[:, 2] * (i[:, 3] * i[:, 7] - i[:, 4] * i[:, 6]))
        fail("inertia must be invertible (|det| >= 1e-300)", ~(det.abs() >= 1e-300))
    if friction_coeffs is not None:
        f = friction_coeffs.to(torch.float64).reshape(-1, 4)
        fail("friction coefficients must be > 0", ~(f > 0))


def _gait_rows(ctrl):
    """The four OpenloopGaitGenerator arguments of a ctrl-constants module or a GAIT_SCHEDULES entry, as [4] lists."""
    get = ctrl.get if isinstance(ctrl, dict) else lambda k: getattr(ctrl, k)
    return dict(stance_duration=[float(v) for v in get("STANCE_DURATION_SECONDS")],
                duty_factor=[float(v) for v in get("DUTY_FACTOR")],
                initial_leg_phase=[float(v) for v in get("INIT_PHASE_FULL_CYCLE")],
                initial_leg_state=[int(v) for v in get("INIT_LEG_STATE")])


def validate_env_gait(stance_duration=None, duty_factor=None, initial_leg_phase=None, initial_leg_state=None):
    """The row rule of rg_gait_env_params (include/rg_cuda.h) on [.., 4] tensors on any device: stance_duration > 0
    and finite, 0 < duty_factor <= 1, 0 <= initial_leg_phase < 1, initial_leg_state SWING (0) or STANCE (1).
    Raises ValueError naming the first failing row; the control step holds such an env in stance instead."""
    def fail(what, bad):
        idx = torch.nonzero(bad.reshape(-1, 4).any(dim=1)).flatten()
        if idx.numel():
            raise ValueError(f"env gait: {what} (first bad row {int(idx[0])})")
    if stance_duration is not None:
        s = stance_duration.to(torch.float64)
        fail("stance_duration must be > 0 and finite", ~((s > 0) & torch.isfinite(s)))
    if duty_factor is not None:
        d = duty_factor.to(torch.float64)
        fail("duty_factor must lie in (0, 1]", ~((d > 0) & (d <= 1)))
    if initial_leg_phase is not None:
        p = initial_leg_phase.to(torch.float64)
        fail("initial_leg_phase must lie in [0, 1)", ~((p >= 0) & (p < 1)))
    if initial_leg_state is not None:
        st = initial_leg_state
        fail("initial_leg_state must be SWING (0) or STANCE (1)", ~((st == int(LegState.SWING)) | (st == int(LegState.STANCE))))


def shard_bounds(n_total, rank, world_size):
    """Contiguous env range [lo, hi) of ``rank`` (SURVEY.md 8e): sizes differ by at most one."""
    base, rem = divmod(int(n_total), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def gather_rollout_stats(local_stats, group=None):
    """all_gather of the small per-rank stats vector -- the ONLY collective on this path (NCCL on
    GPUs, gloo in the CPU tests).  Returns a [world_size, len(stats)] tensor on every rank."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return local_stats.unsqueeze(0)
    out = [torch.empty_like(local_stats) for _ in range(dist.get_world_size(group))]
    dist.all_gather(out, local_stats, group=group)
    return torch.stack(out)


def reduce_rollout_stats(gathered):
    """Whole-job summary of gathered [R,8] stats: sums except column 2 (max)."""
    total = gathered.sum(dim=0)
    total[2] = gathered[:, 2].max()
    return total
