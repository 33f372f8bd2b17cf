"""Reference of the stance QP planned over a contact schedule, restated on the oracle's own routines.

``oracle.convex_mpc.build_qp`` holds one contact row over the horizon: it tiles the row into the (horizon x legs)
matrix that ``calculate_constraint_bounds`` (``CalculateConstraintBounds``) takes.  The schedule form hands that
routine the schedule itself, and takes the com height over the stance feet of row 0, or of the first row with a
stance foot when row 0 has none (include/rg_cuda.h, rg_mpc_build_solve_schedule).  Everything else -- dynamics,
weights, condensing, the polished solve -- is the oracle's.  Test infrastructure only.
"""
from __future__ import annotations

import ctypes
import hashlib
import math
import multiprocessing
import os
import subprocess
import tempfile

import numpy as np

from oracle import c_oracle, convex_mpc, locomotion

_C_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "c", "mpc_plan_oracle.c")
_C_ORACLE_SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "c", "mpc_oracle.c")
_c_lib = None


def c_load():
    """The C schedule oracle (tests/c/mpc_plan_oracle.c), compiled once into the temporary directory: the source tree
    may be read-only."""
    global _c_lib
    if _c_lib is None:
        h = hashlib.sha256()
        for path in (_C_SRC, _C_ORACLE_SRC):
            with open(path, "rb") as fh:
                h.update(fh.read())
        lib_path = os.path.join(tempfile.gettempdir(), f"rg_mpc_plan_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(lib_path):
            tmp = f"{lib_path}.{os.getpid()}"
            subprocess.run(["gcc", "-O3", "-pthread", "-fPIC", "-Wall", "-Wno-unused-variable", "-shared", "-o", tmp, _C_SRC,
                            "-lm"], check=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
            os.replace(tmp, lib_path)
        lib = ctypes.CDLL(lib_path)
        lib.rgo_compute_contact_forces_schedule.restype = ctypes.c_int
        lib.rgo_compute_contact_forces_schedule.argtypes = [ctypes.POINTER(c_oracle.RgoParams)] + [ctypes.c_void_p] * 12
        lib.rgo_scratch_doubles.restype = ctypes.c_size_t
        lib.rgo_scratch_doubles.argtypes = [ctypes.c_int, ctypes.c_int]
        _c_lib = lib
    return _c_lib


def c_compute_contact_forces_schedule(params, com_velocity, rpy, angular_velocity, schedule, foot_positions_base,
                                      desired_com_position, desired_com_velocity, desired_rpy, desired_angular_velocity,
                                      com_position=None):
    """``compute_contact_forces_schedule`` through the C oracle: same arguments, the negated solution (3 k h doubles)."""
    lib = c_load()
    p = c_oracle.params_from(params)
    d = lambda a: np.ascontiguousarray(np.asarray(a, dtype=np.float64))
    ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    cv, r3, w3, ft = d(com_velocity), d(rpy), d(angular_velocity), d(foot_positions_base).reshape(-1)
    sc = np.ascontiguousarray(np.asarray(schedule).astype(np.int32).reshape(params.horizon, params.num_legs))
    dp, dv, dr, dw = d(desired_com_position), d(desired_com_velocity), d(desired_rpy), d(desired_angular_velocity)
    cp = d(com_position) if com_position is not None and len(com_position) == 3 else None
    out = np.zeros(3 * params.num_legs * params.horizon, dtype=np.float64)
    scratch = np.zeros(int(lib.rgo_scratch_doubles(params.horizon, params.num_legs)), dtype=np.float64)
    lib.rgo_compute_contact_forces_schedule(ctypes.byref(p), ptr(cv), ptr(r3), ptr(w3), ptr(sc), ptr(ft), ptr(dp), ptr(dv),
                                            ptr(dr), ptr(dw), ptr(cp) if cp is not None else None, ptr(out), ptr(scratch))
    return out


def com_height_row(schedule):
    """The row whose stance feet give the com height: row 0, or the first row with a stance foot (row 0 if none)."""
    schedule = np.asarray(schedule)
    nonempty = np.flatnonzero((schedule != 0).any(axis=1))
    return schedule[nonempty[0] if len(nonempty) else 0]


def build_qp_schedule(params, com_velocity, rpy, angular_velocity, schedule, foot_positions_base, desired_com_position,
                      desired_com_velocity, desired_rpy, desired_angular_velocity, com_position=None):
    """``convex_mpc.build_qp`` with a ``[h, 4]`` contact schedule in place of the tiled contact row."""
    schedule = np.asarray(schedule)
    assert schedule.shape == (params.horizon, params.num_legs), schedule.shape
    qp = convex_mpc.build_qp(params, com_velocity, rpy, angular_velocity, com_height_row(schedule), foot_positions_base,
                             desired_com_position, desired_com_velocity, desired_rpy, desired_angular_velocity,
                             com_position)
    qp.lb, qp.ub = convex_mpc.calculate_constraint_bounds((schedule != 0).astype(np.float64), params.fz_max,
                                                          params.fz_min, params.friction_coeffs[0], params.horizon)
    return qp


def compute_contact_forces_schedule(params, com_velocity, rpy, angular_velocity, schedule, foot_positions_base,
                                    desired_com_position, desired_com_velocity, desired_rpy, desired_angular_velocity,
                                    com_position=None, return_info=False):
    """``convex_mpc.compute_contact_forces`` over a contact schedule: the negated QP solution (3 k h values)."""
    qp = build_qp_schedule(params, com_velocity, rpy, angular_velocity, schedule, foot_positions_base,
                           desired_com_position, desired_com_velocity, desired_rpy, desired_angular_velocity,
                           com_position)
    if not (np.asarray(schedule) != 0).any():     # every force pinned to zero (the solve's NO_STANCE)
        x, info = np.zeros(len(qp.q_vec)), {"polished": True}
    else:
        x, info = convex_mpc.solve_qp(qp.p_mat, qp.q_vec, qp.c_mat, qp.lb, qp.ub)
    if return_info:
        info["qp"] = qp
        info["x"] = x
        return -x, info
    return -x


def desired_leg_state_at(gen, t):
    """The desired leg states of an ``oracle.locomotion.OpenloopGaitGenerator`` at time ``t``: ``update(t)`` in
    CPython float order, without contact detection and without touching the generator's state."""
    out = []
    for leg in range(len(gen._stance_duration)):
        period = gen._stance_duration[leg] / gen._duty_factor[leg]
        aug = t + gen._initial_leg_phase[leg] * period
        ph = math.fmod(aug, period) / period
        ratio = gen._initial_state_ratio_in_cycle[leg]
        out.append(gen._initial_leg_state[leg] if ph < ratio else gen._next_leg_state[leg])
    return out


def schedule_of(gen, t, dt, h):
    """``[h, 4]`` uint8 planned-stance rows of a generator at t + k dt (each product and sum separately rounded)."""
    return np.array([[s == locomotion.STANCE for s in desired_leg_state_at(gen, t + float(k) * dt)] for k in range(h)],
                    dtype=np.uint8)


def planning_solver(clock, dt, h, solver=None):
    """An ``mpc_solver`` for ``locomotion.TorqueStanceLegController`` that plans over the schedule of the generator
    ``solve.gen`` (set it once the controller is built) at the controller's clock: the contact row it is handed is
    replaced by the schedule, whose row 0 equals it."""
    def solve(params, com_velocity, rpy, angular_velocity, contacts, feet, *args, **kw):
        sched = schedule_of(solve.gen, clock(), dt, h)
        assert np.array_equal(sched[0], (np.asarray(contacts) != 0).astype(np.uint8))
        solve.last_schedule = sched
        return (solver or compute_contact_forces_schedule)(params, com_velocity, rpy, angular_velocity, sched, feet,
                                                           *args, **kw)
    solve.last_schedule = None
    solve.gen = None
    return solve


def random_schedules(n, h, rng):
    """Random [n, h, 4] schedules: any of the 16 patterns per row, flight rows, and an empty row 0 every 7th env."""
    sched = rng.integers(0, 16, (n, h))
    sched[rng.uniform(size=(n, h)) < 0.1] = 0
    sched[::7, 0] = 0
    return ((sched[..., None] >> np.arange(4)) & 1).astype(np.uint8)


def _solve_one(job):
    params, args, com_position = job
    f, info = compute_contact_forces_schedule(params, *args, com_position=com_position, return_info=True)
    return f, bool(info.get("polished", False))


def _solve_one_c(job):
    params, args, com_position = job
    return c_compute_contact_forces_schedule(params, *args, com_position=com_position), True


def oracle_args(states, i, schedule, desired_height):
    """The arguments of the schedule solvers for env i of ``synthetic`` states."""
    cmd = states.command[i].astype(np.float64)
    return (states.com_velocity_body[i].astype(np.float64), states.base_rpy[i].astype(np.float64),
            states.base_rpy_rate[i].astype(np.float64), schedule, states.foot_positions_base[i].astype(np.float64).reshape(12),
            [0.0, 0.0, desired_height], [cmd[0], cmd[1], 0.0], [0.0, 0.0, 0.0], [0.0, 0.0, cmd[2]])


def solve_batch_schedule(params, states, schedules, desired_height, processes=None, use_c=False):
    """The numpy reference (or, with ``use_c``, the C oracle) for a batch of ``synthetic`` states over ``[N, h, 4]``
    schedules, in parallel processes.  Returns (horizon forces [N, 12 h], verified [N]; the C oracle has no verdict:
    True)."""
    jobs = [(params, oracle_args(states, i, schedules[i], desired_height), None) for i in range(len(schedules))]
    fn = _solve_one_c if use_c else _solve_one
    if use_c:
        c_load()                                   # compiled once, before the workers fork
    n_proc = processes or min(len(jobs), os.cpu_count() or 1, 32)
    if n_proc <= 1:
        out = [fn(j) for j in jobs]
    else:
        with multiprocessing.get_context("fork").Pool(n_proc) as pool:
            out = pool.map(fn, jobs, chunksize=max(1, len(jobs) // (4 * n_proc)))
    return np.stack([o[0] for o in out]), np.array([o[1] for o in out])


def _kkt_one(job):
    params, args, x = job
    qp = build_qp_schedule(params, *args)
    cert = convex_mpc.kkt_certificate(qp.p_mat, qp.q_vec, qp.c_mat, qp.lb, qp.ub, x, act_tol=1e-8)
    return cert["primal"], cert["stationarity"], cert["dual_sign"], max(1.0, float(np.abs(qp.q_vec).max()))


def kkt_batch(params, states, schedules, solutions, desired_height, processes=None):
    """KKT certificates (``convex_mpc.kkt_certificate`` on the schedule's QP) of the float64 solutions [N, 3 k h] (the
    QP variables, i.e. the negated forces), in parallel processes.  Returns [N, 4]: primal residual, stationarity,
    multiplier-sign violation and max(1, |q|_inf)."""
    jobs = [(params, oracle_args(states, i, schedules[i], desired_height), solutions[i]) for i in range(len(schedules))]
    n_proc = processes or min(len(jobs), os.cpu_count() or 1, 32)
    if n_proc <= 1:
        return np.array([_kkt_one(j) for j in jobs])
    with multiprocessing.get_context("fork").Pool(n_proc) as pool:
        return np.array(pool.map(_kkt_one, jobs, chunksize=max(1, len(jobs) // (4 * n_proc))))
