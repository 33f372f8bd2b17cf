"""Foothold plans (rg_mpc_build_solve_footholds, rg_control_step_footholds) without a GPU: the exports and argument
types, the argument checks of the three entry points (they return before any device call), the per-step-B reference QP
(held rows are the schedule's QP; the condensed form 2 alpha I + W^T K W with W = blkdiag_t(B_nu,t) is the dense QP for
any footholds; random plans solve and pass the KKT certificate) and the foothold rule of the control step."""
import ctypes

import numpy as np
import pytest

from contact_plan_reference import build_qp_schedule, compute_contact_forces_schedule, random_schedules
from foothold_plan_reference import (build_qp_footholds, compute_contact_forces_footholds, predict_footholds,
                                     raibert_end, random_footholds, structured_qp)
from oracle import convex_mpc, locomotion
from robot_gym import cuda as rg
from robot_gym.model.robots.descriptions import GHOST
from robot_gym.util import synthetic

HEIGHT = GHOST.GetCtrlConstants().MPC_BODY_HEIGHT
NAMES = ("rg_mpc_build_solve_footholds", "rg_control_step_footholds", "rg_control_step_graph_create_footholds")


def test_foothold_plan_symbols_and_argtypes(rg_lib):
    for name in NAMES:
        assert name in rg.EXPORTED_SYMBOLS and hasattr(rg_lib, name)
    assert len(rg_lib.rg_mpc_build_solve_footholds.argtypes) == 7
    assert len(rg_lib.rg_control_step_footholds.argtypes) == 9
    assert len(rg_lib.rg_control_step_graph_create_footholds.argtypes) == 10


def _state():
    s = rg.ControllerState()
    for name, _ in rg.ControllerState._fields_:
        if name not in ("mpc_active_set", "solve_info", "motor_velocities", "motor_strength_ratios", "applied_motor_torques"):
            setattr(s, name, 16 * 1024)
    return s


def test_bad_foothold_arguments_are_rejected_before_any_launch(rg_lib):
    io = rg.MpcIo()
    for name, _ in rg.MpcIo._fields_[:12]:
        setattr(io, name, 16 * 1024)
    io.foot_contact_state = None                      # not read with a schedule
    io.foot_positions_base = None                     # not read with a foothold plan
    ws = ctypes.c_void_p(4096)
    sched = ctypes.c_void_p(8 * 1024)
    for addr in (8 * 1024 + 4, 8 * 1024 + 8, 8 * 1024 + 12, 8 * 1024 + 1):
        assert rg_lib.rg_mpc_build_solve_footholds(ws, 4, ctypes.byref(io), None, sched, ctypes.c_void_p(addr), None) == -1
        assert b"foothold_plan must be 16-byte aligned" in rg_lib.rg_last_error()
    # a plan needs a schedule
    assert rg_lib.rg_mpc_build_solve_footholds(ws, 4, ctypes.byref(io), None, None, ctypes.c_void_p(8 * 1024), None) == -1
    assert b"needs a contact schedule" in rg_lib.rg_last_error()
    # without a plan the current feet are required, as for rg_mpc_build_solve_schedule
    assert rg_lib.rg_mpc_build_solve_footholds(ws, 4, ctypes.byref(io), None, sched, None, None) == -1
    assert b"NULL argument" in rg_lib.rg_last_error()
    # the schedule checks still run
    assert rg_lib.rg_mpc_build_solve_footholds(ws, 4, ctypes.byref(io), None, ctypes.c_void_p(8 * 1024 + 2),
                                               ctypes.c_void_p(8 * 1024), None) == -1
    assert b"contact_schedule must be 4-byte aligned" in rg_lib.rg_last_error()
    # an empty batch: nothing to validate, nothing to launch
    assert rg_lib.rg_mpc_build_solve_footholds(ws, 0, ctypes.byref(io), None, None, ctypes.c_void_p(8 * 1024 + 1), None) == 0
    assert rg_lib.rg_control_step_footholds(ws, ws, 0, None, None, None, None, ctypes.c_void_p(8 * 1024 + 1), None) == 0
    s = _state()
    handle = ctypes.c_void_p()
    for addr in (8 * 1024 + 4, 8 * 1024 + 8):
        assert rg_lib.rg_control_step_footholds(ws, ws, 4, ctypes.byref(s), None, None, sched, ctypes.c_void_p(addr),
                                                None) == -1
        assert b"foothold_plan_out must be 16-byte aligned" in rg_lib.rg_last_error()
        assert rg_lib.rg_control_step_graph_create_footholds(ws, ws, 4, ctypes.byref(s), None, None, sched,
                                                             ctypes.c_void_p(addr), None, ctypes.byref(handle)) == -1
        assert handle.value is None
    assert rg_lib.rg_control_step_footholds(ws, ws, 4, ctypes.byref(s), None, None, None, ctypes.c_void_p(8 * 1024),
                                            None) == -1
    assert b"needs contact_schedule_out" in rg_lib.rg_last_error()
    assert rg_lib.rg_control_step_graph_create_footholds(ws, ws, 4, ctypes.byref(s), None, None, None,
                                                         ctypes.c_void_p(8 * 1024), None, ctypes.byref(handle)) == -1
    assert handle.value is None


def _args(st, i):
    return (st.com_velocity_body[i].astype(np.float64), st.base_rpy[i].astype(np.float64),
            st.base_rpy_rate[i].astype(np.float64))


def _desired(st, i):
    return ([0, 0, HEIGHT], [float(st.command[i, 0]), float(st.command[i, 1]), 0.0], [0, 0, 0], [0, 0, float(st.command[i, 2])])


def _rel(a, b):
    return float(np.abs(a - b).max() / max(1.0, np.abs(b).max()))


@pytest.mark.parametrize("horizon", [5, 10, 20])
def test_held_rows_are_the_schedule_qp(horizon):
    st = synthetic.make_states(6, GHOST, seed=40 + horizon)
    sched = random_schedules(6, horizon, np.random.default_rng(horizon))
    mp = convex_mpc.MpcParams(horizon=horizon)
    for i in range(len(st)):
        feet = st.foot_positions_base[i].astype(np.float64)
        held = np.tile(feet.reshape(1, 12), (horizon, 1))
        a = build_qp_schedule(mp, *_args(st, i), sched[i], feet, *_desired(st, i))
        b = build_qp_footholds(mp, *_args(st, i), sched[i], held, *_desired(st, i))
        assert _rel(b.p_mat, a.p_mat) <= 1e-12 and _rel(b.q_vec, a.q_vec) <= 1e-12
        for f in ("c_mat", "lb", "ub", "x0"):
            np.testing.assert_array_equal(getattr(a, f), getattr(b, f))


@pytest.mark.parametrize("horizon", [5, 10, 20])
def test_per_step_lever_arms_keep_the_closed_form_condensing(horizon):
    """The condensed QP of the kernel -- P = 2 alpha I + W^T K W, q = W^T g~ with K and g~ independent of B -- holds
    with W = blkdiag_t(B_nu,t) for any footholds: against the dense QP built from per-step exponentials."""
    n = 4
    rng = np.random.default_rng(10 + horizon)
    st = synthetic.make_states(n, GHOST, seed=20 + horizon)
    sched = random_schedules(n, horizon, rng)
    sched[:, 0] = 1
    feet = random_footholds(st.foot_positions_base, horizon, rng)
    mp = convex_mpc.MpcParams(horizon=horizon)
    for i in range(n):
        qp = build_qp_footholds(mp, *_args(st, i), sched[i], feet[i], *_desired(st, i))
        p_s, q_s = structured_qp(mp, qp, _args(st, i)[1], feet[i])
        assert _rel(p_s, qp.p_mat) <= 1e-10 and _rel(q_s, qp.q_vec) <= 1e-10, (i, _rel(p_s, qp.p_mat), _rel(q_s, qp.q_vec))
        # and the per-step lever arms matter: the single-B QP of the current feet is a different problem
        held = build_qp_schedule(mp, *_args(st, i), sched[i], st.foot_positions_base[i].astype(np.float64), *_desired(st, i))
        assert _rel(held.p_mat, qp.p_mat) > 1e-4


@pytest.mark.parametrize("horizon,n", [(5, 10), (10, 6), (20, 3)])
def test_random_footholds_solve_and_certify(horizon, n):
    rng = np.random.default_rng(70 + horizon)
    st = synthetic.make_states(n, GHOST, seed=71 + horizon)
    sched = random_schedules(n, horizon, rng)
    sched[1] = 0                                                 # one all-zero schedule
    feet = random_footholds(st.foot_positions_base, horizon, rng)
    mp = convex_mpc.MpcParams(horizon=horizon)
    for i in range(n):
        f, info = compute_contact_forces_footholds(mp, *_args(st, i), sched[i], feet[i], *_desired(st, i), return_info=True)
        swing = np.repeat(sched[i] == 0, 3, axis=1).reshape(-1)
        assert np.all(f[swing] == 0.0)
        if not sched[i].any():
            assert not f.any()
            continue
        qp = info["qp"]
        assert info["polished"], i
        cert = convex_mpc.kkt_certificate(qp.p_mat, qp.q_vec, qp.c_mat, qp.lb, qp.ub, info["x"], act_tol=1e-8)
        qs = max(1.0, float(np.abs(qp.q_vec).max()))
        assert cert["primal"] <= 1e-8 * mp.fz_max and cert["stationarity"] <= 1e-6 * qs, (i, cert)
        # swing entries of the plan do not matter
        moved = feet[i].copy()
        moved[sched[i] == 0] += 0.3
        g = compute_contact_forces_footholds(mp, *_args(st, i), sched[i], moved, *_desired(st, i))
        assert _rel(g, f) <= 1e-9
        # the com height is the one of the first stance row's feet
        r = int(np.flatnonzero(sched[i].any(axis=1))[0])
        feet_w = (convex_mpc.foot_rotation_xyz(_args(st, i)[1]) @ feet[i, r].astype(np.float64).T).T
        assert qp.com_z == abs(float(np.sum(feet_w[sched[i, r] != 0, 2])) / int((sched[i, r] != 0).sum()))


def test_held_rows_solve_the_schedule_qp():
    horizon = 10
    st = synthetic.make_states(3, GHOST, seed=5)
    sched = random_schedules(3, horizon, np.random.default_rng(5))
    sched[:, 0] = 1
    mp = convex_mpc.MpcParams(horizon=horizon)
    for i in range(3):
        feet = st.foot_positions_base[i].astype(np.float64)
        a = compute_contact_forces_schedule(mp, *_args(st, i), sched[i], feet, *_desired(st, i))
        b = compute_contact_forces_footholds(mp, *_args(st, i), sched[i], np.tile(feet, (horizon, 1)), *_desired(st, i))
        assert _rel(b, a) <= 1e-9


def test_foothold_rule():
    h, dt = 10, 0.025
    rng = np.random.default_rng(3)
    feet = rng.uniform(-0.3, 0.3, (4, 3)).astype(np.float32)
    cmd = np.array([0.35, -0.1, 0.2], dtype=np.float32)
    ends = rng.uniform(-0.3, 0.3, (4, 3))
    sched = np.ones((h, 4), dtype=np.uint8)
    sched[0:4, 1] = 0                                          # leg 1 touches down at row 4
    sched[3:, 2] = 0                                           # leg 2 lifts off at row 3 and stays up
    sched[2:5, 3] = 0                                          # leg 3: stance, swing, touchdown at row 5
    out = predict_footholds(sched, feet, cmd, ends, dt)
    v = np.array([float(cmd[0]), float(cmd[1]), 0.0])
    for k in range(h):
        # a held stance leg moves back by k dt v
        np.testing.assert_array_equal(out[k, 0], (feet[0].astype(np.float64) - float(k) * dt * v).astype(np.float32))
        np.testing.assert_array_equal(out[k, 2], (feet[2].astype(np.float64) - float(k) * dt * v).astype(np.float32))
    for k in range(4, h):                                      # the touchdown row takes the Raibert point
        np.testing.assert_array_equal(out[k, 1], (ends[1] - float(k - 4) * dt * v).astype(np.float32))
    for k in range(5, h):
        np.testing.assert_array_equal(out[k, 3], (ends[3] - float(k - 5) * dt * v).astype(np.float32))
    assert out[4, 1, 2] == np.float32(ends[1][2])              # flat ground: z of the Raibert point
    # an invalid gait row holds the current feet
    held = predict_footholds(sched, feet, cmd, ends, dt, valid=False)
    assert np.array_equal(held, np.broadcast_to(feet, (h, 4, 3)))
    # a stand with zero command holds the feet bitwise
    stand = predict_footholds(np.ones((h, 4)), feet, np.zeros(3, np.float32), ends, dt)
    assert stand.tobytes() == np.broadcast_to(feet, (h, 4, 3)).astype(np.float32).tobytes()


def test_raibert_end_is_the_swing_controllers_target():
    """raibert_end against the oracle swing controller's foot target at the end of its swing (phase 1)."""
    from oracle import kinematics

    robot = kinematics.OracleRobot(GHOST)
    c = GHOST.GetCtrlConstants()
    rng = np.random.default_rng(9)
    for _ in range(4):
        rpy_rate = rng.uniform(-0.5, 0.5, 3)
        robot.set_state(base_velocity=np.zeros(3), base_orientation=np.array([0.0, 0.0, 0.0, 1.0]),
                        base_rpy=np.zeros(3), base_rpy_rate=rpy_rate, foot_positions=np.tile([0.0, 0.0, -HEIGHT], 4),
                        foot_contacts=np.zeros(4, np.uint8), motor_angles=np.zeros(12))

        class Est:
            com_velocity_body_frame = rng.uniform(-0.5, 0.5, 3)

        class Gait:
            stance_duration = list(rng.uniform(0.1, 0.4, 4))
            leg_state = [locomotion.SWING] * 4
            desired_leg_state = [locomotion.SWING] * 4
            normalized_phase = [1.0] * 4

        speed, twist = rng.uniform(-0.5, 0.5, 2), float(rng.uniform(-0.5, 0.5))
        swing = locomotion.RaibertSwingLegController(robot, Gait, Est, (speed[0], speed[1]), twist, c.MPC_BODY_HEIGHT,
                                                     0.01)
        swing.get_action()
        hips = robot.GetHipPositionsInBaseFrame()
        for leg in range(4):
            end = raibert_end(Est.com_velocity_body_frame, rpy_rate[2], speed, twist, hips[leg], Gait.stance_duration[leg],
                              c.MPC_BODY_HEIGHT - 0.01)
            np.testing.assert_allclose(swing.foot_targets[leg], end, rtol=0, atol=1e-12)


def test_controller_foothold_plan_needs_the_contact_plan():
    from robot_gym.controllers.mpc.batched_mpc_controller import BatchedMPCController

    with pytest.raises(ValueError, match="contact_plan"):
        BatchedMPCController(None, None, foothold_plan=True)


def test_mpc_build_solve_foothold_plan_needs_a_schedule():
    with pytest.raises(ValueError, match="contact_schedule"):
        rg.mpc_build_solve(None, None, None, None, None, None, None, foothold_plan=object())
