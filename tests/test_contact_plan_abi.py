"""Contact schedules (rg_mpc_build_solve_schedule, rg_control_step_plan) without a GPU: the exports and argument types,
the alignment checks of the three entry points (they return before any device call), the schedule-form reference QP
(a tiled schedule is the oracle's own QP; random schedules solve and pass the KKT certificate) and the gait's planned
stance over the horizon (the restated generator against synthetic.desired_stance / planned_contact_schedule)."""
import ctypes

import numpy as np
import pytest

from contact_plan_reference import (build_qp_schedule, c_compute_contact_forces_schedule, com_height_row,
                                    compute_contact_forces_schedule, desired_leg_state_at, random_schedules, schedule_of)
from oracle import c_oracle
from oracle import convex_mpc, locomotion
from robot_gym import cuda as rg
from robot_gym.model.robots.descriptions import GAIT_SCHEDULES, GHOST
from robot_gym.util import synthetic

HEIGHT = GHOST.GetCtrlConstants().MPC_BODY_HEIGHT
NAMES = ("rg_mpc_build_solve_schedule", "rg_control_step_plan", "rg_control_step_graph_create_plan")


def test_contact_plan_symbols_and_argtypes(rg_lib):
    for name in NAMES:
        assert name in rg.EXPORTED_SYMBOLS and hasattr(rg_lib, name)
    assert len(rg_lib.rg_mpc_build_solve_schedule.argtypes) == 6
    assert len(rg_lib.rg_control_step_plan.argtypes) == 8
    assert len(rg_lib.rg_control_step_graph_create_plan.argtypes) == 9


def _state():
    s = rg.ControllerState()
    for name, _ in rg.ControllerState._fields_:
        if name not in ("mpc_active_set", "solve_info", "motor_velocities", "motor_strength_ratios", "applied_motor_torques"):
            setattr(s, name, 16 * 1024)
    return s


def test_misaligned_schedule_is_rejected_before_any_launch(rg_lib):
    io = rg.MpcIo()
    for name, _ in rg.MpcIo._fields_[:12]:
        setattr(io, name, 16 * 1024)
    io.foot_contact_state = None                      # not read with a schedule
    ws = ctypes.c_void_p(4096)
    for addr in (8 * 1024 + 1, 8 * 1024 + 2, 8 * 1024 + 3):
        assert rg_lib.rg_mpc_build_solve_schedule(ws, 4, ctypes.byref(io), None, ctypes.c_void_p(addr), None) == -1
        assert b"contact_schedule must be 4-byte aligned" in rg_lib.rg_last_error()
    # without a schedule the contact row is required, as for rg_mpc_build_solve_model
    assert rg_lib.rg_mpc_build_solve_schedule(ws, 4, ctypes.byref(io), None, None, None) == -1
    assert b"NULL argument" in rg_lib.rg_last_error()
    assert rg_lib.rg_mpc_build_solve_schedule(ws, 0, ctypes.byref(io), None, ctypes.c_void_p(8 * 1024 + 1), None) == 0
    s = _state()
    handle = ctypes.c_void_p()
    for addr in (8 * 1024 + 1, 8 * 1024 + 2):
        assert rg_lib.rg_control_step_plan(ws, ws, 4, ctypes.byref(s), None, None, ctypes.c_void_p(addr), None) == -1
        assert b"contact_schedule_out must be 4-byte aligned" in rg_lib.rg_last_error()
        assert rg_lib.rg_control_step_graph_create_plan(ws, ws, 4, ctypes.byref(s), None, None, ctypes.c_void_p(addr),
                                                        None, ctypes.byref(handle)) == -1
        assert handle.value is None
    # the model and gait checks still run on the plan entry point
    g = rg.GaitEnvParams()
    g.duty_factor = 8 * 1024 + 4
    assert rg_lib.rg_control_step_plan(ws, ws, 4, ctypes.byref(s), None, ctypes.byref(g), ctypes.c_void_p(8 * 1024), None) == -1
    assert b"8-byte aligned" in rg_lib.rg_last_error()


def _args(st, i):
    return (st.com_velocity_body[i].astype(np.float64), st.base_rpy[i].astype(np.float64),
            st.base_rpy_rate[i].astype(np.float64))


def _rest(st, i):
    return (st.foot_positions_base[i].astype(np.float64), [0, 0, HEIGHT], [float(st.command[i, 0]), float(st.command[i, 1]), 0.0],
            [0, 0, 0], [0, 0, float(st.command[i, 2])])


@pytest.mark.parametrize("horizon", [5, 10, 20])
def test_tiled_schedule_is_the_oracle_qp(horizon):
    st = synthetic.make_states(6, GHOST, seed=900 + horizon)
    mp = convex_mpc.MpcParams(horizon=horizon)
    for i in range(len(st)):
        tiled = np.tile(st.planned_contacts[i][None, :], (horizon, 1))
        a = convex_mpc.build_qp(mp, *_args(st, i), st.planned_contacts[i], *_rest(st, i))
        b = build_qp_schedule(mp, *_args(st, i), tiled, *_rest(st, i))
        for f in ("p_mat", "q_vec", "c_mat", "lb", "ub", "x0"):
            np.testing.assert_array_equal(getattr(a, f), getattr(b, f))
        assert a.com_z == b.com_z
        if i < 2:
            np.testing.assert_array_equal(convex_mpc.compute_contact_forces(mp, *_args(st, i), st.planned_contacts[i], *_rest(st, i)),
                                          compute_contact_forces_schedule(mp, *_args(st, i), tiled, *_rest(st, i)))


@pytest.mark.parametrize("horizon,n", [(5, 12), (10, 8), (20, 4)])
def test_random_schedules_solve_and_certify(horizon, n):
    rng = np.random.default_rng(77 + horizon)
    st = synthetic.make_states(n, GHOST, seed=800 + horizon)
    sched = random_schedules(n, horizon, rng)
    sched[1] = 0                                                 # one all-zero schedule
    mp = convex_mpc.MpcParams(horizon=horizon)
    for i in range(n):
        f, info = compute_contact_forces_schedule(mp, *_args(st, i), sched[i], *_rest(st, i), return_info=True)
        qp = info["qp"]
        swing = np.repeat(sched[i] == 0, 3, axis=1).reshape(-1)
        assert np.all(f[swing] == 0.0)
        row = com_height_row(sched[i])
        if row.any():
            assert info["polished"], i
            cert = convex_mpc.kkt_certificate(qp.p_mat, qp.q_vec, qp.c_mat, qp.lb, qp.ub, info["x"], act_tol=1e-8)
            qs = max(1.0, float(np.abs(qp.q_vec).max()))
            assert cert["primal"] <= 1e-8 * mp.fz_max and cert["stationarity"] <= 1e-6 * qs, (i, cert)
            # com height over the first non-empty row
            feet_w = (convex_mpc.foot_rotation_xyz(_args(st, i)[1]) @ st.foot_positions_base[i].astype(np.float64).reshape(4, 3).T).T
            assert qp.com_z == abs(float(np.sum(feet_w[row != 0, 2])) / int((row != 0).sum()))
        else:
            assert not f.any()


@pytest.mark.parametrize("horizon,n", [(5, 40), (10, 24), (20, 8)])
def test_c_oracle_matches_the_numpy_oracle_on_schedules(horizon, n):
    """The C schedule oracle against the numpy one: random rows (all 16 patterns), flight rows, an empty row 0 every
    7th env, one all-zero schedule; and a tiled schedule is the C oracle's own result for the contact row."""
    rng = np.random.default_rng(300 + horizon)
    st = synthetic.make_states(n, GHOST, seed=310 + horizon)
    sched = random_schedules(n, horizon, rng)
    sched[2] = 0
    sched[3] = ((np.arange(horizon)[:, None] % 16) >> np.arange(4)) & 1     # row k: pattern k mod 16
    mp = convex_mpc.MpcParams(horizon=horizon)
    for i in range(n):
        ref = compute_contact_forces_schedule(mp, *_args(st, i), sched[i], *_rest(st, i))
        got = c_compute_contact_forces_schedule(mp, *_args(st, i), sched[i], *_rest(st, i))
        assert np.abs(got - ref).max() <= 1e-6 * max(1.0, np.abs(ref).max()), i
        tiled = np.tile(st.planned_contacts[i][None, :], (horizon, 1))
        np.testing.assert_array_equal(c_compute_contact_forces_schedule(mp, *_args(st, i), tiled, *_rest(st, i)),
                                      c_oracle.compute_contact_forces(mp, *_args(st, i), st.planned_contacts[i], *_rest(st, i)))


def _gait_rows(name):
    s = GAIT_SCHEDULES[name]
    return (np.asarray(s["STANCE_DURATION_SECONDS"], dtype=np.float64), np.asarray(s["DUTY_FACTOR"], dtype=np.float64),
            np.asarray(s["INIT_PHASE_FULL_CYCLE"], dtype=np.float64), np.asarray([int(v) for v in s["INIT_LEG_STATE"]]))


class _NoContacts:
    num_legs = 4

    def GetFootContacts(self):
        return np.zeros(4, dtype=np.uint8)


@pytest.mark.parametrize("horizon", [5, 10, 20])
def test_desired_leg_state_at_matches_desired_stance(horizon):
    rng = np.random.default_rng(horizon)
    dt = 0.025
    n = 200
    t = rng.integers(0, 5000, n) * 0.001
    t[n // 2:] = rng.uniform(0.0, 7.0, n - n // 2)              # non-grid times
    gaits = [_gait_rows(name) for name in GAIT_SCHEDULES]
    stance = rng.uniform(0.1, 0.6, (n, 4)); duty = 1.0 - rng.uniform(0.0, 0.8, (n, 4)); duty[:, 0][::5] = 1.0
    phase = rng.uniform(0.0, 1.0, (n, 4)); state = rng.integers(0, 2, (n, 4))
    for e, g in enumerate(gaits):
        stance[e], duty[e], phase[e], state[e] = g
    for name, g in zip(GAIT_SCHEDULES, gaits):                   # one row for every env
        plan = synthetic.planned_contact_schedule(t, dt, horizon, *g)
        gen = locomotion.OpenloopGaitGenerator(_NoContacts(), *g)
        for e in range(0, n, 7):
            np.testing.assert_array_equal(plan[e], schedule_of(gen, float(t[e]), dt, horizon), err_msg=name)
    plan = synthetic.planned_contact_schedule(t, dt, horizon, stance, duty, phase, state)   # [N,4] rows
    for e in range(n):
        gen = locomotion.OpenloopGaitGenerator(_NoContacts(), stance[e], duty[e], phase[e], state[e])
        for k in range(horizon):
            want = synthetic.desired_stance(np.array([t[e] + float(k) * dt]), stance[e], duty[e], phase[e], state[e])[0]
            got = [s == locomotion.STANCE for s in desired_leg_state_at(gen, float(t[e]) + float(k) * dt)]
            assert list(want) == got and list(plan[e, k].astype(bool)) == got, (e, k)
        gen.update(float(t[e]))                                  # row 0 is the generator's own desired state
        assert [s == locomotion.STANCE for s in gen.desired_leg_state] == list(plan[e, 0].astype(bool))
