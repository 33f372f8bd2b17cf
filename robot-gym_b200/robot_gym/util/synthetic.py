"""Seeded synthetic robot states of the shape BASELINE.json names (SURVEY.md section 8d).

Generated once on the CPU at full size with ``numpy.random.default_rng(20261017)`` and sliced per
rank, so results are invariant to the GPU count.  No physics: this plays the role the reference's
unused ``MockEnvironment`` (agents/ppo/tools/mock_environment.py:20-80) hints at -- a seeded state
source behind the robot getter names of robot.py:71-264,367-397.
"""
from __future__ import annotations

import dataclasses

import numpy as np

SEED = 20261017

# Nominal ghost foot positions in the base frame at INIT_MOTOR_ANGLES (URDF forward kinematics,
# SURVEY.md App. B.1; reproduced by tests/test_kinematics.py from the leg chains).
GHOST_NOMINAL_FEET = np.array([[0.2153, -0.1600, -0.3904], [0.2161, 0.1550, -0.3910],
                               [-0.2247, -0.1600, -0.3904], [-0.2239, 0.1550, -0.3910]])


@dataclasses.dataclass
class SyntheticStates:
    """Host (numpy) arrays, env-major; dtypes are the ones the C ABI takes."""
    time_since_reset: np.ndarray        # [N]    f64
    foot_contacts: np.ndarray           # [N,4]  u8   measured contacts
    planned_contacts: np.ndarray        # [N,4]  u8   desired stance from the gait at t0
    base_velocity_world: np.ndarray     # [N,3]  f32
    base_orientation_xyzw: np.ndarray   # [N,4]  f32
    base_rpy: np.ndarray                # [N,3]  f32  (yaw = 0)
    base_rpy_rate: np.ndarray           # [N,3]  f32
    com_velocity_body: np.ndarray       # [N,3]  f32
    foot_positions_base: np.ndarray     # [N,12] f32
    motor_angles: np.ndarray            # [N,12] f32
    command: np.ndarray                 # [N,3]  f32  (vx, vy, wz) incl. robot offsets
    com_height: np.ndarray              # [N]    f32

    def slice(self, start, stop):
        return SyntheticStates(**{f.name: getattr(self, f.name)[start:stop] for f in dataclasses.fields(self)})

    def __len__(self):
        return len(self.time_since_reset)


def desired_stance(time_s, stance_duration, duty_factor, init_phase, init_state):
    """Vectorised planned-stance flags of the open-loop gait at time ``time_s`` [N] -> [N,4] bool.  Each gait
    argument is one [4] row for every env or [N,4] rows, one per env."""
    rows = lambda a: a if a.ndim == 2 else a[None, :]
    t = np.asarray(time_s, dtype=np.float64)[:, None]
    stance = rows(np.asarray(stance_duration, dtype=np.float64))
    duty = rows(np.asarray(duty_factor, dtype=np.float64))
    phase0 = rows(np.asarray(init_phase, dtype=np.float64))
    init = np.asarray(init_state).astype(np.int64) if np.ndim(init_state) == 2 else np.asarray([int(s) for s in init_state])[None, :]
    period = stance / duty
    ph = np.fmod(t + phase0 * period, period) / period
    ratio = np.where(init == 0, 1.0 - duty, duty)
    in_init = ph < ratio
    return np.where(in_init, init == 1, init != 1)


def planned_contact_schedule(time_s, dt, horizon, stance_duration, duty_factor, init_phase, init_state):
    """Contact schedule of the open-loop gait over an MPC horizon: ``[N, horizon, 4]`` uint8, row k the planned stance
    at ``t + k * dt`` (each product and sum rounded separately, as the control step's prologue evaluates it).  The
    gait arguments are as for ``desired_stance``."""
    t = np.asarray(time_s, dtype=np.float64)
    rows = [desired_stance(t + float(k) * float(dt), stance_duration, duty_factor, init_phase, init_state)
            for k in range(int(horizon))]
    return np.stack(rows, axis=1).astype(np.uint8)


def euler_to_quat_xyzw(rpy):
    r, p, y = rpy[:, 0] * 0.5, rpy[:, 1] * 0.5, rpy[:, 2] * 0.5
    cr, sr, cp, sp, cy, sy = np.cos(r), np.sin(r), np.cos(p), np.sin(p), np.cos(y), np.sin(y)
    return np.stack([sr * cp * cy - cr * sp * sy, cr * sp * cy + sr * cp * sy,
                     cr * cp * sy - sr * sp * cy, cr * cp * cy + sr * sp * sy], axis=1)


def make_states(n_env, description, schedule_ctrl=None, all_stance=False, nominal_feet=None,
                nominal_motor_angles=None, seed=SEED, flip_contact_fraction=0.05):
    """BASELINE config 2/3 inputs for ``n_env`` envs (ghost parameters by default).

    roll, pitch ~U(-0.2,0.2), yaw = 0; com_z ~U(0.37,0.47); v_body, w_body ~U(-0.5,0.5)^3;
    feet = nominal + U(-0.05,0.05)^3; vx ~U(0,0.35), wz ~U(-0.4,0.4) (go_env.py:102-103), vy = 0,
    plus the robot's command offsets (ghost/ctrl_constants.py:39-41); planned contacts from the
    gait at t0 ~U(0,0.5 s) on the 1 ms grid; measured contacts = planned with 5 % flipped;
    motor angles = nominal + U(-0.1,0.1).
    """
    ctrl = schedule_ctrl or description.GetCtrlConstants()
    const = description.GetConstants()
    rng = np.random.default_rng(seed)
    n = int(n_env)
    rpy = np.zeros((n, 3))
    rpy[:, :2] = rng.uniform(-0.2, 0.2, (n, 2))
    com_z = rng.uniform(0.37, 0.47, n) - 0.42 + float(ctrl.MPC_BODY_HEIGHT)
    v_body = rng.uniform(-0.5, 0.5, (n, 3))
    w_body = rng.uniform(-0.5, 0.5, (n, 3))
    feet0 = GHOST_NOMINAL_FEET if nominal_feet is None else np.asarray(nominal_feet)
    feet = feet0[None] + rng.uniform(-0.05, 0.05, (n, 4, 3))
    vx = rng.uniform(0.0, 0.35, n)
    wz = rng.uniform(-0.4, 0.4, n)
    cmd = np.stack([vx + ctrl.VX_OFFSET, np.zeros(n) + ctrl.VY_OFFSET, wz + ctrl.WZ_OFFSET], axis=1)
    step = rng.integers(0, 500, n)
    t0 = step * 0.001                                   # Simulation.GetTimeSinceReset: step_counter * 0.001
    if all_stance:
        planned = np.ones((n, 4), dtype=bool)
    else:
        planned = desired_stance(t0, ctrl.STANCE_DURATION_SECONDS, ctrl.DUTY_FACTOR,
                                 ctrl.INIT_PHASE_FULL_CYCLE, ctrl.INIT_LEG_STATE)
    flip = rng.uniform(0, 1, (n, 4)) < flip_contact_fraction
    measured = np.logical_xor(planned, flip)
    q0 = const.INIT_MOTOR_ANGLES if nominal_motor_angles is None else nominal_motor_angles
    motor = np.asarray(q0, dtype=np.float64)[None] + rng.uniform(-0.1, 0.1, (n, 12))
    quat = euler_to_quat_xyzw(rpy)
    # world-frame velocity consistent with the body-frame sample: v_world = R(q) v_body
    x, y, z, w = quat.T
    rot = np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                    2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                    2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], axis=1).reshape(n, 3, 3)
    v_world = np.einsum("nij,nj->ni", rot, v_body)
    f32 = np.float32
    return SyntheticStates(
        time_since_reset=t0.astype(np.float64),
        foot_contacts=measured.astype(np.uint8),
        planned_contacts=planned.astype(np.uint8),
        base_velocity_world=v_world.astype(f32),
        base_orientation_xyzw=quat.astype(f32),
        base_rpy=rpy.astype(f32),
        base_rpy_rate=w_body.astype(f32),
        com_velocity_body=v_body.astype(f32),
        foot_positions_base=feet.reshape(n, 12).astype(f32),
        motor_angles=motor.astype(f32),
        command=cmd.astype(f32),
        com_height=com_z.astype(f32),
    )


OFF_NOMINAL_FAMILIES = ("tilted", "steep_pitch", "fast", "landing", "liftoff", "feet_far", "feet_coincident",
                        "feet_colinear", "feet_high", "patterns")


def make_off_nominal_states(n_env, family, description=None, seed=SEED):
    """States an RL batch reaches and ``make_states`` does not: ``make_states(n_env, description, seed=seed)`` with
    the fields of one family overridden by float32 draws from a generator seeded with (seed, family index).

    tilted: roll, pitch ~U(-1,1), yaw ~U(-3,3).  steep_pitch: roll ~U(-0.3,0.3), |pitch| ~U(1.3,1.5) with a random
    sign (cos(pitch) >= 0.07: the entries of T(rpy) reach ~14).  fast: v_body ~U(-3,3)^3, rates ~U(-6,6)^3, command
    (vx, vy, wz) ~U(+-2, +-1, +-3) plus the robot's offsets.  landing: v_z ~U(-3,-1.5), four feet in stance.
    liftoff: v_z ~U(1,3).  feet_far: feet + U(-0.2,0.2) per coordinate.  feet_coincident: foot 3 := foot 0,
    foot 1 := foot 2, four feet in stance.  feet_colinear: every foot y := 0, four feet in stance (no roll
    authority).  feet_high: every foot z ~U(-0.02,0.02) (estimated CoM height near 0).  patterns: contact pattern =
    env index mod 16 (bit l = leg l), v_body ~U(-2,2)^3.  v_z is the body-frame z velocity; the world-frame
    velocity and the quaternion are recomputed from the overridden body velocity and attitude.  Measured contacts
    equal the planned ones wherever a family sets the contact pattern."""
    if family not in OFF_NOMINAL_FAMILIES:
        raise ValueError(f"unknown family {family!r}; expected one of {OFF_NOMINAL_FAMILIES}")
    if description is None:
        from robot_gym.model.robots.descriptions import GHOST
        description = GHOST
    ctrl = description.GetCtrlConstants()
    st = make_states(n_env, description, seed=seed)
    n = len(st)
    rng = np.random.default_rng((int(seed), OFF_NOMINAL_FAMILIES.index(family)))
    rpy = st.base_rpy.astype(np.float64)
    v_body = st.com_velocity_body.astype(np.float64)
    feet = st.foot_positions_base.astype(np.float64).reshape(n, 4, 3)
    contacts = None
    if family == "tilted":
        rpy[:, :2] = rng.uniform(-1.0, 1.0, (n, 2))
        rpy[:, 2] = rng.uniform(-3.0, 3.0, n)
    elif family == "steep_pitch":
        rpy[:, 0] = rng.uniform(-0.3, 0.3, n)
        rpy[:, 1] = rng.uniform(1.3, 1.5, n) * rng.choice([-1.0, 1.0], n)
    elif family == "fast":
        v_body = rng.uniform(-3.0, 3.0, (n, 3))
        st.base_rpy_rate = rng.uniform(-6.0, 6.0, (n, 3)).astype(np.float32)
        cmd = rng.uniform(-1.0, 1.0, (n, 3)) * np.array([2.0, 1.0, 3.0])
        st.command = (cmd + np.array([ctrl.VX_OFFSET, ctrl.VY_OFFSET, ctrl.WZ_OFFSET])).astype(np.float32)
    elif family == "landing":
        v_body[:, 2] = rng.uniform(-3.0, -1.5, n)
        contacts = np.ones((n, 4), dtype=bool)
    elif family == "liftoff":
        v_body[:, 2] = rng.uniform(1.0, 3.0, n)
    elif family == "feet_far":
        feet = feet + rng.uniform(-0.2, 0.2, (n, 4, 3))
    elif family == "feet_coincident":
        feet[:, 3] = feet[:, 0]
        feet[:, 1] = feet[:, 2]
        contacts = np.ones((n, 4), dtype=bool)
    elif family == "feet_colinear":
        feet[:, :, 1] = 0.0
        contacts = np.ones((n, 4), dtype=bool)
    elif family == "feet_high":
        feet[:, :, 2] = rng.uniform(-0.02, 0.02, (n, 4))
    elif family == "patterns":
        contacts = ((np.arange(n)[:, None] % 16) >> np.arange(4)[None, :]) & 1 != 0
        v_body = rng.uniform(-2.0, 2.0, (n, 3))
    if contacts is not None:
        st.planned_contacts = contacts.astype(np.uint8)
        st.foot_contacts = contacts.astype(np.uint8)
    rpy32 = rpy.astype(np.float32)
    quat = euler_to_quat_xyzw(rpy32.astype(np.float64))
    x, y, z, w = quat.T
    rot = np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                    2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                    2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], axis=1).reshape(n, 3, 3)
    st.base_rpy = rpy32
    st.base_orientation_xyzw = quat.astype(np.float32)
    st.com_velocity_body = v_body.astype(np.float32)
    st.base_velocity_world = np.einsum("nij,nj->ni", rot, v_body).astype(np.float32)
    st.foot_positions_base = np.ascontiguousarray(feet.reshape(n, 12).astype(np.float32))
    return st


def make_state_sequence(n_env, n_steps, description, schedule_ctrl=None, seed=SEED, control_dt_ticks=10, env_gait=None):
    """``n_steps`` consecutive control steps for ``n_env`` envs: every step draws a fresh random
    state (no physics), while the clock advances like Simulation's: t = step_counter * 0.001 with
    ACTION_REPEAT = 10 ticks per control step (core/sim_constants.py:7,11) from a per-env start.
    ``env_gait``: per-env gait rows for the planned (and so the measured) contacts, a dict with any of
    ``stance_duration``, ``duty_factor``, ``initial_leg_phase``, ``initial_leg_state`` as [N,4] arrays (a missing
    key takes the schedule's row); the random draws do not depend on it."""
    ctrl = schedule_ctrl or description.GetCtrlConstants()
    g = env_gait or {}
    gait = (g.get("stance_duration", ctrl.STANCE_DURATION_SECONDS), g.get("duty_factor", ctrl.DUTY_FACTOR),
            g.get("initial_leg_phase", ctrl.INIT_PHASE_FULL_CYCLE), g.get("initial_leg_state", ctrl.INIT_LEG_STATE))
    rng = np.random.default_rng(seed + 1)
    start = rng.integers(0, 500, int(n_env))
    seq = []
    for k in range(int(n_steps)):
        st = make_states(n_env, description, schedule_ctrl=ctrl, seed=seed + 17 * (k + 1))
        tick = start + control_dt_ticks * k
        st.time_since_reset = (tick * 0.001).astype(np.float64)
        planned = desired_stance(st.time_since_reset - start * 0.001, *gait)
        flip = np.random.default_rng(seed + 31 * (k + 1)).uniform(0, 1, planned.shape) < 0.08
        st.planned_contacts = planned.astype(np.uint8)
        st.foot_contacts = np.logical_xor(planned, flip).astype(np.uint8)
        seq.append(st)
    return seq


CHUNK = 4096


def make_states_sharded(lo, hi, description, schedule_ctrl=None, seed=SEED, **kwargs):
    """Envs [lo, hi) of an unbounded, PREFIX-STABLE global batch: the batch is the concatenation of 4096-env chunks,
    chunk c drawn by ``make_states(4096, ..., seed=seed + c)``.  A rank's shard therefore does not depend on how
    many ranks (or envs) the job has -- rank 0 of a 1-, 2-, 4- or 8-GPU run solves exactly the same first chunk,
    which is ``make_states(4096, description)`` itself, the single-GPU benchmark batch."""
    lo, hi = int(lo), int(hi)
    parts = []
    for c in range(lo // CHUNK, (max(hi, lo + 1) - 1) // CHUNK + 1):
        st = make_states(CHUNK, description, schedule_ctrl=schedule_ctrl, seed=seed + c, **kwargs)
        a, b = max(lo, c * CHUNK) - c * CHUNK, min(hi, (c + 1) * CHUNK) - c * CHUNK
        parts.append(st.slice(a, b))
    return SyntheticStates(**{f.name: np.concatenate([getattr(p, f.name) for p in parts]) for f in dataclasses.fields(SyntheticStates)})
