"""Stance QP planned over a contact schedule (rg_mpc_build_solve_schedule) and the control step that plans over each
env's gait (rg_control_step_plan, BatchedMPCController(contact_plan=True)).

  * random schedules (every pattern per row, flight rows, empty row 0) x h = 5 / 10 / 20 on trot / pace / bound states,
    4096 envs, against the C schedule oracle (the numpy one re-checks suspects), with a KKT certificate for every env
    with a stance block;
  * a schedule that tiles the contact row is bitwise the solve without one: both kernel paths, with and without a
    per-env model, warm and cold;
  * the two-kernel and the one-kernel schedule solves on a 4096-env batch at every horizon: bitwise for every env,
    queued ones included, and repeatable; warm equals cold to 1e-9;
  * all-zero schedules, and an empty row 0 with stance later;
  * the schedule the prologue writes, byte for byte, on both prologue mappings, for the workspace gait and random
    per-env gaits; row 0 is mpc_contact_state; invalid gait rows plan all-stance without touching their neighbours;
  * the planning control step against a restated oracle controller on a five-schedule batch, eager and graph, warm
    and cold; graph replay equals eager bitwise; contact_plan=False is the controller without the argument."""
import dataclasses
import multiprocessing
import os

import numpy as np
import pytest
import torch

from contact_plan_reference import (build_qp_schedule, c_compute_contact_forces_schedule, compute_contact_forces_schedule,
                                    kkt_batch, oracle_args, planning_solver, random_schedules, schedule_of,
                                    solve_batch_schedule)
from oracle import convex_mpc as cm
from oracle import kinematics, locomotion
from robot_gym import cuda as rg
from robot_gym.controllers.mpc.batched_mpc_controller import BatchedMPCController
from robot_gym.model.robots.descriptions import GAIT_SCHEDULES, GHOST, with_gait
from robot_gym.model.robots.synthetic_robot import SyntheticRobotBatch
from robot_gym.util import synthetic

pytestmark = pytest.mark.gpu
REL_TOL = 1e-4
RECHECK = 1e-5            # C oracle vs kernel beyond this: the numpy oracle arbitrates (as tests/test_gpu_off_nominal.py)
HEIGHT = GHOST.GetCtrlConstants().MPC_BODY_HEIGHT
INPUTS = ("com_velocity_body", "base_rpy", "base_rpy_rate", "planned_contacts", "foot_positions_base", "command")
SCHEDULES = tuple(GAIT_SCHEDULES)
KEYS = ("stance_duration", "duty_factor", "initial_leg_phase", "initial_leg_state")
DT = 0.025


def _dev(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _params(horizon, **overrides):
    ctrl = GHOST.GetCtrlConstants()
    p = rg.default_mpc_params(ctrl.MPC_BODY_MASS, ctrl.MPC_BODY_INERTIA, ctrl.MPC_BODY_HEIGHT, horizon)
    for k, v in overrides.items():
        setattr(p, k, v)
    return p


def _solve(dev, st, horizon, schedule=None, ws=None, active_set=None, model=None, **overrides):
    """(float32 forces [N,h,12], float64 forces [N,h,12], solve_info [N,4]) of one solve."""
    n = len(st)
    ws = ws or rg.MpcWorkspace(_params(horizon, **overrides), device=dev, max_envs=max(1, n))
    h64 = torch.empty((n, horizon, 12), dtype=torch.float64, device=dev)
    inputs = [_dev(getattr(st, k), dev) for k in INPUTS]
    if schedule is not None:
        inputs[3] = None                                     # the contact row is not read with a schedule
    f, hf, info = rg.mpc_build_solve(ws, *inputs, want_horizon=True, horizon_forces_f64=h64, active_set=active_set,
                                     env_model=model, zero_yaw=False,
                                     contact_schedule=None if schedule is None else _dev(schedule, dev))
    torch.cuda.synchronize()
    hf = hf.cpu().numpy()
    np.testing.assert_array_equal(f.cpu().numpy(), hf[:, 0, :])
    return hf, h64.cpu().numpy(), info.cpu().numpy()


def _concat(states):
    return synthetic.SyntheticStates(**{f.name: np.concatenate([getattr(s, f.name) for s in states])
                                        for f in dataclasses.fields(synthetic.SyntheticStates)})


def _gait_states(n, seed, names=("trot", "pace", "bound")):
    per = -(-n // len(names))
    return _concat([synthetic.make_states(per, with_gait(GHOST, g), seed=seed + k) for k, g in enumerate(names)]).slice(0, n)


def _oracle_args(st, i, sched):
    return (st.com_velocity_body[i].astype(np.float64), st.base_rpy[i].astype(np.float64),
            st.base_rpy_rate[i].astype(np.float64), sched, st.foot_positions_base[i].astype(np.float64),
            [0, 0, HEIGHT], [float(st.command[i, 0]), float(st.command[i, 1]), 0.0], [0, 0, 0], [0, 0, float(st.command[i, 2])])


# ------------------------------------------------------------------------------------- 1. against the reference
@pytest.mark.parametrize("horizon", [5, 10, 20])
def test_random_schedules_against_the_reference(rg_lib, cuda_device, horizon):
    """4096 envs (above one wave: the lean kernel and the fallback queue run) against the C oracle; envs where the
    two differ beyond RECHECK are re-solved by the numpy oracle.  KKT certificate for every env with a stance block."""
    n = 4096
    rng = np.random.default_rng(500 + horizon)
    st = _gait_states(n, seed=600 + horizon)
    sched = random_schedules(n, horizon, rng)
    sched[3] = 0                                                  # one all-zero schedule
    mp = cm.MpcParams(horizon=horizon)
    ref, _ = solve_batch_schedule(mp, st, sched, HEIGHT, use_c=True)
    hf, h64, info = _solve(cuda_device, st, horizon, schedule=sched)
    status = info[:, rg.RG_INFO_STATUS]
    assert np.all(status & rg.RG_STATUS_POLISHED), np.flatnonzero((status & rg.RG_STATUS_POLISHED) == 0)
    assert status[3] == rg.RG_STATUS_NO_STANCE | rg.RG_STATUS_POLISHED and not h64[3].any()
    assert (info[:, rg.RG_INFO_IPM_ITERS] > 0).any()              # the fallback queue was not empty
    swing = np.repeat(sched == 0, 3, axis=2).reshape(n, horizon, 12)
    assert np.all(hf[swing] == 0.0) and np.all(h64[swing] == 0.0)
    gpu = h64.reshape(n, -1)
    rel = np.abs(gpu - ref).max(axis=1) / np.maximum(1.0, np.abs(ref).max(axis=1))
    suspects = np.flatnonzero(rel > RECHECK)
    assert len(suspects) <= max(8, n // 200), (len(suspects), float(rel.max()))
    for i in suspects:
        exact = compute_contact_forces_schedule(mp, *oracle_args(st, int(i), sched[i], HEIGHT))
        rel[i] = np.abs(gpu[i] - exact).max() / max(1.0, np.abs(exact).max())
    assert rel.max() < REL_TOL, (int(rel.argmax()), float(rel.max()))
    stance = sched.any(axis=(1, 2))
    idx = np.flatnonzero(stance)
    cert = kkt_batch(mp, _take(st, idx), sched[idx], -gpu[idx], HEIGHT)
    assert np.all(cert[:, 0] <= 1e-8 * mp.fz_max), float(cert[:, 0].max())
    assert np.all(cert[:, 1] <= 1e-6 * cert[:, 3]) and np.all(cert[:, 2] <= 1e-6 * cert[:, 3])
    print(f"[schedule h={horizon}] worst force {rel.max():.1e} rel ({len(suspects)} re-checked), worst stationarity "
          f"{(cert[:, 1] / cert[:, 3]).max():.1e}, rounds {info[:, rg.RG_INFO_POLISH_ROUNDS].mean():.2f}, "
          f"queued {int((info[:, rg.RG_INFO_IPM_ITERS] > 0).sum())}")


def _take(st, idx):
    return synthetic.SyntheticStates(**{f.name: getattr(st, f.name)[idx] for f in dataclasses.fields(synthetic.SyntheticStates)})


def test_empty_first_row_takes_the_com_height_of_the_first_stance_row(rg_lib, cuda_device):
    n, horizon = 64, 10
    st = _gait_states(n, seed=31)
    rng = np.random.default_rng(5)
    sched = random_schedules(n, horizon, rng)
    sched[:, 0] = 0
    sched[:, 1] = 0
    sched[:, 3] |= 1                                              # stance from row 3 on, at least
    ref, _ = solve_batch_schedule(cm.MpcParams(horizon=horizon), st, sched, HEIGHT)
    hf, h64, info = _solve(cuda_device, st, horizon, schedule=sched)
    assert not hf[:, :2].any() and np.all(info[:, rg.RG_INFO_STATUS] & rg.RG_STATUS_POLISHED)
    rel = np.abs(h64.reshape(n, -1) - ref).max(axis=1) / np.maximum(1.0, np.abs(ref).max(axis=1))
    assert rel.max() < REL_TOL
    # the height matters: taking it from the (empty) first row would be a different QP
    qp = build_qp_schedule(cm.MpcParams(horizon=horizon), *_oracle_args(st, 0, sched[0]))
    assert qp.com_z > 0.2


# ------------------------------------------------------------------------------------- 2. tiled = no schedule
@pytest.mark.parametrize("horizon", [5, 10, 20])
@pytest.mark.parametrize("two_kernel", [0, 1])
@pytest.mark.parametrize("with_model", [False, True])
def test_tiled_schedule_is_bitwise_the_solve_without_one(rg_lib, cuda_device, horizon, two_kernel, with_model):
    n = 4096                                                      # above one wave at every horizon: lean + fallback
    st = _gait_states(n, seed=70 + horizon, names=SCHEDULES)
    tiled = np.repeat(st.planned_contacts[:, None, :], horizon, axis=1)
    model = None
    if with_model:
        rng = np.random.default_rng(3)
        ctrl = GHOST.GetCtrlConstants()
        model = dict(mass=_dev(ctrl.MPC_BODY_MASS * rng.uniform(0.8, 1.3, n), cuda_device),
                     friction_coeffs=_dev(rng.uniform(0.3, 0.9, (n, 4)), cuda_device))
    outs = []
    for sched in (None, tiled):
        ws = rg.MpcWorkspace(_params(horizon, two_kernel_solve=two_kernel), device=cuda_device, max_envs=n)
        act = rg.new_active_set(n, horizon, cuda_device)
        cold = _solve(cuda_device, st, horizon, schedule=sched, ws=ws, active_set=act, model=model)
        a1 = act.cpu().numpy().copy()
        warm = _solve(cuda_device, st, horizon, schedule=sched, ws=ws, active_set=act, model=model)
        outs.append((cold, a1, warm, act.cpu().numpy()))
    (c0, a0, w0, b0), (c1, a1, w1, b1) = outs
    for x, y in zip(c0 + w0, c1 + w1):
        assert x.tobytes() == y.tobytes()
    assert np.array_equal(a0, a1) and np.array_equal(b0, b1)


# ------------------------------------------------------------------------------------- 3. kernel paths, warm vs cold
@pytest.mark.parametrize("horizon", [5, 10, 20])
def test_two_kernel_and_one_kernel_plan_solves_agree(rg_lib, cuda_device, horizon):
    """Bitwise equal for every env, the ones the lean kernel queues included, and repeatable: a second two-kernel
    solve on a fresh workspace (another queue order) gives the same bits."""
    n = 4096
    st = _gait_states(n, seed=41, names=SCHEDULES)
    sched = random_schedules(n, horizon, np.random.default_rng(41 + horizon))
    res = []
    for tk in (0, 1, 1):
        ws = rg.MpcWorkspace(_params(horizon, two_kernel_solve=tk), device=cuda_device, max_envs=n)
        res.append(_solve(cuda_device, st, horizon, schedule=sched, ws=ws))
    assert np.all(res[0][2][:, rg.RG_INFO_STATUS] & rg.RG_STATUS_POLISHED)
    queued = res[1][2][:, rg.RG_INFO_IPM_ITERS] > 0
    assert queued.any()
    for other in res[1:]:
        for x, y in zip(res[0][:2], other[:2]):
            assert x.tobytes() == y.tobytes(), np.flatnonzero((x != y).reshape(n, -1).any(axis=1))[:8]
        assert np.array_equal(res[0][2][:, rg.RG_INFO_STATUS], other[2][:, rg.RG_INFO_STATUS])
    assert res[1][2].tobytes() == res[2][2].tobytes()
    print(f"[two vs one kernel h={horizon}] {int(queued.sum())} queued envs, all bitwise")
    ws = rg.MpcWorkspace(_params(horizon), device=cuda_device, max_envs=n)
    act = rg.new_active_set(n, horizon, cuda_device)
    cold = _solve(cuda_device, st, horizon, schedule=sched, ws=ws, active_set=act)
    warm = _solve(cuda_device, st, horizon, schedule=sched, ws=ws, active_set=act)
    assert np.all(warm[2][:, rg.RG_INFO_STATUS] & rg.RG_STATUS_POLISHED)
    stance = sched.any(axis=(1, 2))
    assert np.all(warm[2][stance, rg.RG_INFO_POLISH_ROUNDS] <= cold[2][stance, rg.RG_INFO_POLISH_ROUNDS])
    scale = np.maximum(1.0, np.abs(cold[1]).reshape(n, -1).max(axis=1))
    assert (np.abs(warm[1] - cold[1]).reshape(n, -1).max(axis=1) / scale).max() < 1e-9


# ------------------------------------------------------------------------------------- 5. the prologue's schedule
def _random_gait(n, rng):
    stance = rng.uniform(0.1, 0.6, (n, 4))
    duty = 1.0 - rng.uniform(0.0, 0.8, (n, 4))
    duty[rng.uniform(size=(n, 4)) < 0.1] = 1.0
    phase = rng.uniform(0.0, 1.0, (n, 4))
    state = rng.integers(0, 2, (n, 4)).astype(np.int32)
    return dict(stance_duration=stance, duty_factor=duty, initial_leg_phase=phase, initial_leg_state=state)


def _ws_gait():
    c = GHOST.GetCtrlConstants()
    return dict(stance_duration=np.tile(np.asarray(c.STANCE_DURATION_SECONDS, dtype=np.float64), (1, 1)),
                duty_factor=np.tile(np.asarray(c.DUTY_FACTOR, dtype=np.float64), (1, 1)),
                initial_leg_phase=np.tile(np.asarray(c.INIT_PHASE_FULL_CYCLE, dtype=np.float64), (1, 1)),
                initial_leg_state=np.asarray([[int(v) for v in c.INIT_LEG_STATE]]))


class _NoContacts:
    num_legs = 4

    def GetFootContacts(self):
        return np.zeros(4, dtype=np.uint8)


@pytest.mark.parametrize("per_env", [False, True])
@pytest.mark.parametrize("n", [6000, 40000])                     # per-(env, leg) prologue / per-env prologue
def test_prologue_schedule_bytes(rg_lib, cuda_device, n, per_env):
    horizon = 20 if per_env else 10
    rng = np.random.default_rng(n + per_env)
    st = synthetic.make_states(n, GHOST, seed=72)
    robot = SyntheticRobotBatch(GHOST, st, device=cuda_device)
    clock = {"t": torch.zeros(n, dtype=torch.float64, device=cuda_device)}
    ctl = BatchedMPCController(robot, lambda: clock["t"], horizon=horizon, contact_plan=True, use_graph=False)
    gait = _random_gait(n, rng) if per_env else _ws_gait()
    if per_env:
        ctl.set_env_gait(**gait)
    for k in range(2):
        t = rng.integers(0, 5000, n) * 0.001
        odd = rng.uniform(size=n) < 0.5
        t[odd] = rng.uniform(0.0, 7.0, int(odd.sum()))
        clock["t"] = torch.from_numpy(t).to(cuda_device)
        ctl.get_action()
        torch.cuda.synchronize()
        got = ctl.mpc_contact_schedule.cpu().numpy()
        want = synthetic.planned_contact_schedule(t, DT, horizon, *[gait[key] for key in KEYS])
        assert np.array_equal(got, want)
        assert np.array_equal(got[:, 0], ctl.mpc_contact_state.cpu().numpy())
        for e in range(0, n, max(1, n // 64)):                    # the restated generator on a sample
            g = locomotion.OpenloopGaitGenerator(_NoContacts(), *[gait[key][e if per_env else 0] for key in KEYS])
            assert np.array_equal(got[e], schedule_of(g, float(t[e]), DT, horizon)), e
        assert int(ctl.unverified_count()) == 0
    if per_env:                                                   # invalid rows: all-stance, neighbours untouched
        bad = np.arange(5, n, 997)
        ctl.env_duty_factor[torch.from_numpy(bad).to(cuda_device), 1] = 1.5
        ctl.get_action()
        torch.cuda.synchronize()
        got2 = ctl.mpc_contact_schedule.cpu().numpy()
        assert np.all(got2[bad] == 1)
        ok = np.setdiff1d(np.arange(n), bad)
        assert np.array_equal(got2[ok], want[ok])


# ------------------------------------------------------------------------------------- 6. the whole control step
N_STEP_ENVS, N_STEPS = 260, 10


def _mixed_gait(n):
    group = np.arange(n) % len(SCHEDULES)
    rows = [GAIT_SCHEDULES[SCHEDULES[g]] for g in group]
    return dict(stance_duration=np.array([r["STANCE_DURATION_SECONDS"] for r in rows], dtype=np.float64),
                duty_factor=np.array([r["DUTY_FACTOR"] for r in rows], dtype=np.float64),
                initial_leg_phase=np.array([r["INIT_PHASE_FULL_CYCLE"] for r in rows], dtype=np.float64),
                initial_leg_state=np.array([[int(v) for v in r["INIT_LEG_STATE"]] for r in rows], dtype=np.int32)), group


def _reference_env(args):
    """One restated LocomotionController with the planning solver, for env e over the whole sequence."""
    seq, e, name = args
    orobot = kinematics.OracleRobot(GHOST)
    clock = {"t": 0.0}

    def load(k):
        s = seq[k]
        orobot.set_state(base_velocity=s.base_velocity_world[e].astype(np.float64),
                         base_orientation=s.base_orientation_xyzw[e].astype(np.float64),
                         base_rpy=s.base_rpy[e].astype(np.float64), base_rpy_rate=s.base_rpy_rate[e].astype(np.float64),
                         foot_positions=s.foot_positions_base[e].astype(np.float64), foot_contacts=s.foot_contacts[e],
                         motor_angles=s.motor_angles[e].astype(np.float64))
        clock["t"] = float(s.time_since_reset[e])
    load(0)
    solver = planning_solver(lambda: octl._time_since_reset, DT, 10, solver=c_compute_contact_forces_schedule)   # the time the generator was updated with
    octl = locomotion.build_mpc_controller(orobot, lambda: clock["t"], with_gait(GHOST, name).GetCtrlConstants(),
                                           mpc_solver=solver)
    solver.gen = octl.gait_generator
    octl.reset()
    out = []
    for k in range(len(seq)):
        load(k)
        s = seq[k]
        for leg_ctl in (octl.swing_leg_controller, octl.stance_leg_controller):
            leg_ctl.desired_speed = [float(s.command[e, 0]), float(s.command[e, 1]), 0.0]
            leg_ctl.desired_twisting_speed = float(s.command[e, 2])
        octl.update()
        act = octl.get_action().reshape(12, 5)
        out.append((act, octl.stance_leg_controller.last_contact_forces.copy(), solver.last_schedule.copy()))
    return out


@pytest.fixture(scope="module")
def step_reference():
    gait, group = _mixed_gait(N_STEP_ENVS)
    seq = synthetic.make_state_sequence(N_STEP_ENVS, N_STEPS, GHOST, seed=synthetic.SEED + 61, env_gait=gait)
    jobs = [([s.slice(e, e + 1) for s in seq], 0, SCHEDULES[group[e]]) for e in range(N_STEP_ENVS)]
    n_proc = min(32, os.cpu_count() or 1)
    if n_proc > 1:
        with multiprocessing.get_context("fork").Pool(n_proc) as pool:
            ref = pool.map(_reference_env, jobs, chunksize=2)
    else:
        ref = [_reference_env(j) for j in jobs]
    return seq, group, ref


def _run_plan(dev, seq, group, warm_start, use_graph, contact_plan=True):
    robot = SyntheticRobotBatch(GHOST, seq[0], device=dev)
    ctl = BatchedMPCController(robot, robot.GetTimeSinceReset, warm_start=warm_start, use_graph=use_graph,
                               contact_plan=contact_plan)
    for g, name in enumerate(SCHEDULES):
        ctl.set_env_gait(schedule=name, env_ids=torch.from_numpy(np.flatnonzero(group == g)).to(dev))
    ctl.reset()
    out = []
    for k in range(len(seq)):
        robot.load(seq[k])
        ctl.command.copy_(torch.from_numpy(seq[k].command).to(dev))
        a = ctl.get_action()
        torch.cuda.synchronize()
        assert int(ctl.unverified_count()) == 0
        out.append((a.cpu().numpy().copy(), ctl.contact_forces.cpu().numpy().copy(),
                    None if ctl.mpc_contact_schedule is None else ctl.mpc_contact_schedule.cpu().numpy().copy()))
    return out


@pytest.mark.parametrize("warm_start", [True, False])
def test_planning_control_step_against_the_restated_controller(rg_lib, cuda_device, step_reference, warm_start):
    seq, group, ref = step_reference
    eager = _run_plan(cuda_device, seq, group, warm_start, use_graph=False)
    graph = _run_plan(cuda_device, seq, group, warm_start, use_graph=True)
    worst_f = worst_tau = 0.0
    changed = 0
    for k in range(N_STEPS):
        for x, y in zip(eager[k], graph[k]):                      # graph replay = eager, bitwise
            assert x.tobytes() == y.tobytes(), k
        a, f, sched = eager[k]
        for e in range(N_STEP_ENVS):
            ra, rf, rs = ref[e][k]
            assert np.array_equal(sched[e], rs), (k, e)
            changed += int(not np.all(rs == rs[0]))
            worst_f = max(worst_f, np.abs(f[e] - rf).max() / max(1.0, np.abs(rf).max()))
            ae = a[e].reshape(12, 5)
            np.testing.assert_array_equal(ae[:, [1, 2, 3]], ra[:, [1, 2, 3]])
            worst_tau = max(worst_tau, np.abs(ae[:, 4] - ra[:, 4]).max() / max(1.0, np.abs(ra[:, 4]).max()))
    assert changed > 0
    assert worst_f < REL_TOL and worst_tau < REL_TOL, (worst_f, worst_tau)
    print(f"[plan step {N_STEP_ENVS} x {N_STEPS}, warm={warm_start}] worst force {worst_f:.1e}, torque {worst_tau:.1e}; "
          f"{changed} env-steps with a changing schedule")


# ------------------------------------------------------------------------------------- 7. contact_plan=False
@pytest.mark.parametrize("n", [300, 5000])
def test_contact_plan_off_is_the_controller_without_it(rg_lib, cuda_device, n):
    seq = synthetic.make_state_sequence(n, 3, GHOST, seed=synthetic.SEED + 67)
    outs = []
    for kw in ({}, {"contact_plan": False}):
        robot = SyntheticRobotBatch(GHOST, seq[0], device=cuda_device)
        ctl = BatchedMPCController(robot, robot.GetTimeSinceReset, **kw)
        assert ctl.mpc_contact_schedule is None
        res = []
        for k in range(3):
            robot.load(seq[k])
            ctl.command.copy_(torch.from_numpy(seq[k].command).to(cuda_device))
            res.append(ctl.get_action().cpu().numpy().copy())
        outs.append(res)
    for x, y in zip(*outs):
        assert x.tobytes() == y.tobytes()
