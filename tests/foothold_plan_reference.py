"""Reference of the stance QP planned over predicted footholds, restated on the oracle's own routines.

``oracle.convex_mpc.build_qp`` builds one continuous-time B from the current feet and one exponential ``(A_exp,
B_exp)`` for the whole horizon.  The foothold form builds them per step, as convex MPC does with predicted footholds
(Di Carlo et al. 2018): ``calculate_b_mat`` from row k's feet and ``calculate_exponentials`` for every step k, and the
stacked ``B_qp[i, j] = A_exp^(i-j) B_exp,j``.  The com height is taken over the stance feet of row r* of the plan, the
row the schedule form takes it from (include/rg_cuda.h, rg_mpc_build_solve_footholds).  The bounds are the schedule's
(``contact_plan_reference.build_qp_schedule``), and the solve and the certificate are the oracle's.  This shares no
shortcut with the kernel's condensing.  Also here: the foothold rule of the control step's prologue
(rg_control_step_footholds), with the Raibert point in the arithmetic of ``oracle.locomotion.RaibertSwingLegController``.
Test infrastructure only.
"""
from __future__ import annotations

import multiprocessing
import os

import numpy as np

from contact_plan_reference import build_qp_schedule, schedule_of
from oracle import convex_mpc, locomotion

K = convex_mpc.K_STATE_DIM


def first_stance_row(schedule):
    """r*: row 0, or the first row with a stance foot (row 0 if none)."""
    nonempty = np.flatnonzero((np.asarray(schedule) != 0).any(axis=1))
    return int(nonempty[0]) if len(nonempty) else 0


def build_qp_footholds(params, com_velocity, rpy, angular_velocity, schedule, footholds, desired_com_position,
                       desired_com_velocity, desired_rpy, desired_angular_velocity, com_position=None):
    """The dense QP over a ``[h, 4]`` schedule with one B per step from ``footholds`` ([h, 12] or [h, 4, 3], base frame
    of the current step).  As the oracle's B, every column is built from the given feet, swing blocks' included: their
    forces are pinned to zero by the bounds, so the solution does not depend on them."""
    h, k, dt = params.horizon, params.num_legs, params.dt
    schedule = np.asarray(schedule)
    feet = np.asarray(footholds, dtype=np.float64).reshape(h, k, 3)
    rpy = np.asarray(rpy, dtype=np.float64)
    rf = convex_mpc.foot_rotation_xyz(rpy)
    r_star = first_stance_row(schedule)
    # the schedule form supplies x_ref, the bounds, C and (through its own feet argument) the com height of row r*
    qp = build_qp_schedule(params, com_velocity, rpy, angular_velocity, schedule, feet[r_star].reshape(-1),
                           desired_com_position, desired_com_velocity, desired_rpy, desired_angular_velocity,
                           com_position)
    x_ref = np.zeros(K * h)
    for i in range(h):
        o = i * K
        x_ref[o:o + K] = [desired_rpy[0], desired_rpy[1], rpy[2] + dt * (i + 1) * desired_angular_velocity[2],
                          dt * (i + 1) * desired_com_velocity[0], dt * (i + 1) * desired_com_velocity[1],
                          desired_com_position[2], 0.0, 0.0, desired_angular_velocity[2], desired_com_velocity[0],
                          desired_com_velocity[1], 0.0, -params.gravity]
    a_mat = convex_mpc.calculate_a_mat(rpy)
    rot = convex_mpc.rpy_to_rot_zyx(rpy)
    inv_inertia = np.linalg.inv(np.asarray(params.inertia, dtype=np.float64).reshape(3, 3))
    inv_inertia_world = rot @ inv_inertia @ rot.T
    m = 3 * k
    b_exps = []
    a_exp = None
    for step in range(h):
        feet_world = (rf @ feet[step].T).T
        b_mat = convex_mpc.calculate_b_mat(1.0 / params.mass, inv_inertia_world, feet_world)
        a_exp, b_exp = convex_mpc.calculate_exponentials(a_mat, b_mat, dt)
        b_exps.append(b_exp)
    a_pows = [np.eye(K)]
    for _ in range(h):
        a_pows.append(a_exp @ a_pows[-1])
    a_qp = np.vstack(a_pows[1:])
    b_qp = np.zeros((K * h, m * h))
    for i in range(h):
        for j in range(i + 1):
            b_qp[i * K:(i + 1) * K, j * m:(j + 1) * m] = a_pows[i - j] @ b_exps[j]
    big_l = np.tile(np.asarray(params.weights, dtype=np.float64), h)
    qp.p_mat = 2.0 * (b_qp.T @ (big_l[:, None] * b_qp) + params.alpha * np.eye(m * h))
    qp.q_vec = 2.0 * b_qp.T @ (big_l * (a_qp @ qp.x0 - x_ref))
    qp.b_qp = b_qp
    qp.state_error = a_qp @ qp.x0 - x_ref
    return qp


def compute_contact_forces_footholds(params, com_velocity, rpy, angular_velocity, schedule, footholds,
                                     desired_com_position, desired_com_velocity, desired_rpy, desired_angular_velocity,
                                     com_position=None, return_info=False):
    """The negated solution (3 k h values) of the foothold-plan QP."""
    qp = build_qp_footholds(params, com_velocity, rpy, angular_velocity, schedule, footholds, desired_com_position,
                            desired_com_velocity, desired_rpy, desired_angular_velocity, com_position)
    if not (np.asarray(schedule) != 0).any():
        x, info = np.zeros(len(qp.q_vec)), {"polished": True}
    else:
        x, info = convex_mpc.solve_qp(qp.p_mat, qp.q_vec, qp.c_mat, qp.lb, qp.ub)
    if return_info:
        info["qp"] = qp
        info["x"] = x
        return -x, info
    return -x


def structured_qp(params, qp, rpy, footholds):
    """P = 2 alpha I + W^T K W and q = W^T g~ with W = blkdiag_t(B_nu,t): K and g~ from their closed forms over the
    horizon (they do not depend on B), B_nu,t = [I_w^-1 [r_t]x ; I / m] from row t's feet.  ``qp``: a dense QP of
    ``build_qp_footholds`` (its free-response error A_qp x0 - x_ref is the only thing taken from it)."""
    h, k, dt = params.horizon, params.num_legs, params.dt
    w = np.asarray(params.weights, dtype=np.float64)
    l_rho, l_nu = np.diag(w[0:6]), np.diag(w[6:12])
    a_mat = convex_mpc.calculate_a_mat(np.asarray(rpy, dtype=np.float64))
    g6 = np.zeros((6, 6))
    g6[0:3, 0:3] = a_mat[0:3, 6:9]                           # T(rpy): angular velocity -> rpy rate
    g6[3:6, 3:6] = np.eye(3)
    kmat = np.zeros((6 * h, 6 * h))
    for j in range(h):
        for c in range(h):
            blk = np.zeros((6, 6))
            for i in range(max(j, c), h):
                blk += 2.0 * (dt * dt * l_nu + dt ** 4 * (i - j + 0.5) * (i - c + 0.5) * g6.T @ l_rho @ g6)
            kmat[6 * j:6 * j + 6, 6 * c:6 * c + 6] = blk
    e = qp.state_error.reshape(h, K)
    g_t = np.zeros(6 * h)
    for j in range(h):
        for i in range(j, h):
            g_t[6 * j:6 * j + 6] += 2.0 * (dt * l_nu @ e[i, 6:12] + dt * dt * (i - j + 0.5) * g6.T @ l_rho @ e[i, 0:6])
    rpy = np.asarray(rpy, dtype=np.float64)
    rot = convex_mpc.rpy_to_rot_zyx(rpy)
    iw = rot @ np.linalg.inv(np.asarray(params.inertia, dtype=np.float64).reshape(3, 3)) @ rot.T
    rf = convex_mpc.foot_rotation_xyz(rpy)
    feet = np.asarray(footholds, dtype=np.float64).reshape(h, k, 3)
    wmat = np.zeros((6 * h, 3 * k * h))
    for t in range(h):
        for leg in range(k):
            r = rf @ feet[t, leg]
            col = 3 * (k * t + leg)
            wmat[6 * t:6 * t + 3, col:col + 3] = iw @ convex_mpc.skew(r)
            wmat[6 * t + 3:6 * t + 6, col:col + 3] = np.eye(3) / params.mass
    p_mat = 2.0 * params.alpha * np.eye(3 * k * h) + wmat.T @ kmat @ wmat
    return p_mat, wmat.T @ g_t


# ------------------------------------------------------------------------------------------ the foothold rule
def raibert_end(com_velocity, yaw_dot, desired_speed, desired_twisting_speed, hip_offset, stance_duration,
                desired_height_minus_clearance):
    """The end point of ``RaibertSwingLegController.get_action``'s swing trajectory for one leg, in its arithmetic."""
    com_velocity = np.array((com_velocity[0], com_velocity[1], 0))
    twisting_vector = np.array((-hip_offset[1], hip_offset[0], 0))
    hip_horizontal_velocity = com_velocity + yaw_dot * twisting_vector
    target_hip_horizontal_velocity = (np.array((desired_speed[0], desired_speed[1], 0)) +
                                      desired_twisting_speed * twisting_vector)
    return (hip_horizontal_velocity * stance_duration / 2 -
            locomotion._KP * (target_hip_horizontal_velocity - hip_horizontal_velocity)
            ) - np.array((0, 0, desired_height_minus_clearance)) + np.array((hip_offset[0], hip_offset[1], 0))


def predict_footholds(schedule, feet, command, ends, dt, valid=True):
    """[h, 4, 3] float32 footholds of one env (rg_control_step_footholds): a planted foot moves back by (k - k_a) dt v,
    v = (command[0], command[1], 0); a touchdown at k (swing at k - 1, stance at k) re-anchors the foot at its Raibert
    point ``ends[leg]``.  Each product and difference is rounded separately in double.  ``valid`` False: held rows."""
    schedule = np.asarray(schedule) != 0
    h = schedule.shape[0]
    feet = np.asarray(feet, dtype=np.float64).reshape(4, 3)
    out = np.zeros((h, 4, 3), dtype=np.float32)
    v = (float(command[0]), float(command[1]))
    for leg in range(4):
        anchor, k_a = [float(x) for x in feet[leg]], 0
        for k in range(h):
            if not valid:
                out[k, leg] = feet[leg]
                continue
            if k >= 1 and schedule[k, leg] and not schedule[k - 1, leg]:
                anchor, k_a = [float(x) for x in ends[leg]], k
            back = float(k - k_a) * dt
            out[k, leg] = (anchor[0] - back * v[0], anchor[1] - back * v[1], anchor[2])
    return out


def foothold_planning_solver(clock, dt, h, solver=None):
    """An ``mpc_solver`` for ``locomotion.TorqueStanceLegController`` that plans over the schedule of ``solve.gen`` and
    over the footholds predicted from it (``predict_footholds``), at the controller's clock.  Set ``solve.gen`` (the
    gait generator), ``solve.robot`` (hip offsets) and ``solve.swing_height`` (desired height - foot clearance) once
    the controller is built.  The velocity estimate enters the Raibert point rounded to float32, as the control step
    stores it."""
    def solve(params, com_velocity, rpy, angular_velocity, contacts, feet, desired_com_position, desired_com_velocity,
              desired_rpy, desired_angular_velocity, **kw):
        sched = schedule_of(solve.gen, clock(), dt, h)
        assert np.array_equal(sched[0], (np.asarray(contacts) != 0).astype(np.uint8))
        vel = np.asarray(com_velocity, dtype=np.float32).astype(np.float64)
        hips = solve.robot.GetHipPositionsInBaseFrame()
        ends = [raibert_end(vel, float(angular_velocity[2]), desired_com_velocity, float(desired_angular_velocity[2]),
                            hips[leg], solve.gen.stance_duration[leg], solve.swing_height) for leg in range(4)]
        plan = predict_footholds(sched, feet, desired_com_velocity, ends, dt)
        solve.last_schedule, solve.last_footholds = sched, plan
        return (solver or compute_contact_forces_footholds)(params, com_velocity, rpy, angular_velocity, sched,
                                                            plan.astype(np.float64), desired_com_position,
                                                            desired_com_velocity, desired_rpy, desired_angular_velocity,
                                                            **kw)
    solve.last_schedule = solve.last_footholds = None
    solve.gen = solve.robot = solve.swing_height = None
    return solve


def random_footholds(feet, h, rng, spread=0.08):
    """[n, h, 4, 3] float32 footholds: the current feet moved by up to ``spread`` m per axis, a different offset per row."""
    feet = np.asarray(feet, dtype=np.float32).reshape(-1, 1, 4, 3)
    return (feet + rng.uniform(-spread, spread, (feet.shape[0], h, 4, 3))).astype(np.float32)


# ------------------------------------------------------------------------------------------ batches
def oracle_args(states, i, schedule, footholds, desired_height):
    cmd = states.command[i].astype(np.float64)
    return (states.com_velocity_body[i].astype(np.float64), states.base_rpy[i].astype(np.float64),
            states.base_rpy_rate[i].astype(np.float64), schedule, np.asarray(footholds, dtype=np.float64),
            [0.0, 0.0, desired_height], [cmd[0], cmd[1], 0.0], [0.0, 0.0, 0.0], [0.0, 0.0, cmd[2]])


def _solve_one(job):
    params, args = job
    f, info = compute_contact_forces_footholds(params, *args, return_info=True)
    return f, bool(info.get("polished", False))


def _kkt_one(job):
    params, args, x = job
    qp = build_qp_footholds(params, *args)
    cert = convex_mpc.kkt_certificate(qp.p_mat, qp.q_vec, qp.c_mat, qp.lb, qp.ub, x, act_tol=1e-8)
    return cert["primal"], cert["stationarity"], cert["dual_sign"], max(1.0, float(np.abs(qp.q_vec).max()))


def _pool_map(fn, jobs, processes):
    n_proc = processes or min(len(jobs), os.cpu_count() or 1, 32)
    if n_proc <= 1:
        return [fn(j) for j in jobs]
    with multiprocessing.get_context("fork").Pool(n_proc) as pool:
        return pool.map(fn, jobs, chunksize=max(1, len(jobs) // (4 * n_proc)))


def solve_batch_footholds(params, states, schedules, footholds, desired_height, processes=None):
    """The dense reference for a batch: (horizon forces [N, 12 h], verified [N])."""
    jobs = [(params, oracle_args(states, i, schedules[i], footholds[i], desired_height)) for i in range(len(schedules))]
    out = _pool_map(_solve_one, jobs, processes)
    return np.stack([o[0] for o in out]), np.array([o[1] for o in out])


def kkt_batch_footholds(params, states, schedules, footholds, solutions, desired_height, processes=None):
    """KKT certificates on the per-step-B QP of the float64 solutions [N, 3 k h] (the QP variables, i.e. the negated
    forces).  Returns [N, 4]: primal residual, stationarity, multiplier-sign violation and max(1, |q|_inf)."""
    jobs = [(params, oracle_args(states, i, schedules[i], footholds[i], desired_height), solutions[i])
            for i in range(len(schedules))]
    return np.array(_pool_map(_kkt_one, jobs, processes))
