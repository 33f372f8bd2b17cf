"""Stance QP planned over predicted footholds (rg_mpc_build_solve_footholds) and the control step that predicts them
(rg_control_step_footholds, BatchedMPCController(contact_plan=True, foothold_plan=True)).

  * random schedules and random footholds x h = 5 / 10 / 20, 4096 envs (lean kernel and fallback queue), against the
    dense per-step-B reference on a sample, with a KKT certificate on the per-step-B QP;
  * a plan whose rows are the current feet is bitwise the schedule solve: both kernel paths, with and without a per-env
    model, warm and cold; NaN in every swing-block entry changes nothing, bitwise;
  * two-kernel vs one-kernel foothold solves: bitwise for the envs the lean kernel verified, 1e-9 for the queued ones;
  * the footholds the prologue writes on both prologue mappings against the numpy rule (one float32 ulp), and its
    schedule bytes against the plan prologue's;
  * the control step against a restated oracle controller with the foothold solver on a five-schedule batch, eager and
    graph, warm and cold; a stand with zero command is the contact plan alone, bitwise."""
import dataclasses
import multiprocessing
import os

import numpy as np
import pytest
import torch

from contact_plan_reference import random_schedules
from foothold_plan_reference import (foothold_planning_solver, kkt_batch_footholds, predict_footholds, raibert_end,
                                     random_footholds, solve_batch_footholds)
from oracle import convex_mpc as cm
from oracle import kinematics, locomotion
from robot_gym import cuda as rg
from robot_gym.controllers.mpc.batched_mpc_controller import BatchedMPCController
from robot_gym.model.robots.descriptions import GAIT_SCHEDULES, GHOST, K3LSO, with_gait
from robot_gym.model.robots.synthetic_robot import SyntheticRobotBatch
from robot_gym.util import synthetic

pytestmark = pytest.mark.gpu
REL_TOL = 1e-4
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


def _solve(dev, st, horizon, schedule, footholds=None, ws=None, active_set=None, model=None):
    """(float32 forces [N,h,12], float64 forces [N,h,12], solve_info [N,4]) of one solve over a schedule and, when
    given, a foothold plan."""
    n = len(st)
    ws = ws or rg.MpcWorkspace(_params(horizon), device=dev, max_envs=n)
    h64 = torch.empty((n, horizon, 12), dtype=torch.float64, device=dev)
    inputs = [_dev(getattr(st, k), dev) for k in INPUTS]
    inputs[3] = None                                         # the contact row is not read with a schedule
    if footholds is not None:
        inputs[4] = None                                     # nor the current feet with a foothold plan
    f, hf, info = rg.mpc_build_solve(ws, *inputs, want_horizon=True, horizon_forces_f64=h64, active_set=active_set,
                                     env_model=model, contact_schedule=_dev(schedule, dev),
                                     foothold_plan=None if footholds is None else _dev(footholds, dev))
    torch.cuda.synchronize()
    hf = hf.cpu().numpy()
    np.testing.assert_array_equal(f.cpu().numpy(), hf[:, 0, :])
    return hf, h64.cpu().numpy(), info.cpu().numpy()


def _concat(states):
    return synthetic.SyntheticStates(**{f.name: np.concatenate([getattr(s, f.name) for s in states])
                                        for f in dataclasses.fields(synthetic.SyntheticStates)})


def _take(st, idx):
    return synthetic.SyntheticStates(**{f.name: getattr(st, f.name)[idx] for f in dataclasses.fields(synthetic.SyntheticStates)})


def _gait_states(n, seed, names=("trot", "pace", "bound")):
    per = -(-n // len(names))
    return _concat([synthetic.make_states(per, with_gait(GHOST, g), seed=seed + k) for k, g in enumerate(names)]).slice(0, n)


# ------------------------------------------------------------------------------------- 1. against the reference
@pytest.mark.parametrize("horizon,sample", [(5, 512), (10, 384), (20, 128)])
def test_random_footholds_against_the_reference(rg_lib, cuda_device, horizon, sample):
    n = 4096
    rng = np.random.default_rng(900 + horizon)
    st = _gait_states(n, seed=910 + horizon)
    sched = random_schedules(n, horizon, rng)
    sched[3] = 0                                                  # one all-zero schedule
    feet = random_footholds(st.foot_positions_base, horizon, rng)
    hf, h64, info = _solve(cuda_device, st, horizon, sched, feet)
    status = info[:, rg.RG_INFO_STATUS]
    assert np.all(status & rg.RG_STATUS_POLISHED), np.flatnonzero((status & rg.RG_STATUS_POLISHED) == 0)
    assert status[3] == rg.RG_STATUS_NO_STANCE | rg.RG_STATUS_POLISHED and not h64[3].any()
    swing = np.repeat(sched == 0, 3, axis=2).reshape(n, horizon, 12)
    assert np.all(hf[swing] == 0.0) and np.all(h64[swing] == 0.0)
    idx = np.unique(np.concatenate([[3], rng.choice(n, sample, replace=False)]))
    mp = cm.MpcParams(horizon=horizon)
    sub = _take(st, idx)
    ref, _ = solve_batch_footholds(mp, sub, sched[idx], feet[idx], HEIGHT)
    gpu = h64.reshape(n, -1)[idx]
    rel = np.abs(gpu - ref).max(axis=1) / np.maximum(1.0, np.abs(ref).max(axis=1))
    assert rel.max() < REL_TOL, (int(idx[rel.argmax()]), float(rel.max()))
    stance = sched[idx].any(axis=(1, 2))
    cert = kkt_batch_footholds(mp, _take(sub, np.flatnonzero(stance)), sched[idx][stance], feet[idx][stance],
                               -gpu[stance], HEIGHT)
    assert np.all(cert[:, 0] <= 1e-8 * mp.fz_max), float(cert[:, 0].max())
    assert np.all(cert[:, 1] <= 1e-6 * cert[:, 3]) and np.all(cert[:, 2] <= 1e-6 * cert[:, 3])
    print(f"[footholds h={horizon}] worst force {rel.max():.1e} rel over {len(idx)} envs, worst stationarity "
          f"{(cert[:, 1] / cert[:, 3]).max():.1e}, rounds {info[:, rg.RG_INFO_POLISH_ROUNDS].mean():.2f}, "
          f"queued {int((info[:, rg.RG_INFO_IPM_ITERS] > 0).sum())}")


# ------------------------------------------------------------------------------------- 2. held rows = the schedule solve
@pytest.mark.parametrize("horizon", [5, 10, 20])
@pytest.mark.parametrize("two_kernel", [0, 1])
@pytest.mark.parametrize("with_model", [False, True])
def test_held_rows_are_bitwise_the_schedule_solve(rg_lib, cuda_device, horizon, two_kernel, with_model):
    n = 4096                                                      # above one wave at every horizon: lean + fallback
    st = _gait_states(n, seed=170 + horizon, names=SCHEDULES)
    sched = random_schedules(n, horizon, np.random.default_rng(17 + horizon))
    held = np.repeat(st.foot_positions_base.reshape(n, 1, 12), horizon, axis=1)
    model = None
    if with_model:
        rng = np.random.default_rng(3)
        ctrl = GHOST.GetCtrlConstants()
        model = dict(mass=_dev(ctrl.MPC_BODY_MASS * rng.uniform(0.8, 1.3, n), cuda_device),
                     friction_coeffs=_dev(rng.uniform(0.3, 0.9, (n, 4)), cuda_device))
    outs = []
    for feet in (None, held):
        ws = rg.MpcWorkspace(_params(horizon, two_kernel_solve=two_kernel), device=cuda_device, max_envs=n)
        act = rg.new_active_set(n, horizon, cuda_device)
        cold = _solve(cuda_device, st, horizon, sched, feet, ws=ws, active_set=act, model=model)
        a1 = act.cpu().numpy().copy()
        warm = _solve(cuda_device, st, horizon, sched, feet, ws=ws, active_set=act, model=model)
        outs.append((cold, a1, warm, act.cpu().numpy()))
    (c0, a0, w0, b0), (c1, a1, w1, b1) = outs
    for x, y in zip(c0 + w0, c1 + w1):
        assert x.tobytes() == y.tobytes(), np.flatnonzero((x != y).reshape(n, -1).any(axis=1))[:8]
    assert np.array_equal(a0, a1) and np.array_equal(b0, b1)


def test_nan_in_swing_entries_changes_nothing(rg_lib, cuda_device):
    n, horizon = 4096, 10
    rng = np.random.default_rng(44)
    st = _gait_states(n, seed=44, names=SCHEDULES)
    sched = random_schedules(n, horizon, rng)
    feet = random_footholds(st.foot_positions_base, horizon, rng)
    poisoned = feet.copy()
    poisoned[sched == 0] = np.nan
    a = _solve(cuda_device, st, horizon, sched, feet)
    b = _solve(cuda_device, st, horizon, sched, poisoned)
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()


# ------------------------------------------------------------------------------------- 3. kernel paths
@pytest.mark.parametrize("horizon", [5, 10, 20])
def test_two_kernel_and_one_kernel_foothold_solves_agree(rg_lib, cuda_device, horizon):
    n = 4096
    rng = np.random.default_rng(51 + horizon)
    st = _gait_states(n, seed=51, names=SCHEDULES)
    sched = random_schedules(n, horizon, rng)
    feet = random_footholds(st.foot_positions_base, horizon, rng)
    res = [_solve(cuda_device, st, horizon, sched, feet,
                  ws=rg.MpcWorkspace(_params(horizon, two_kernel_solve=tk), device=cuda_device, max_envs=n))
           for tk in (0, 1)]
    assert np.all(res[0][2][:, rg.RG_INFO_STATUS] & rg.RG_STATUS_POLISHED)
    queued = res[1][2][:, rg.RG_INFO_IPM_ITERS] > 0
    assert queued.any()
    for x, y in zip(res[0][:2], res[1][:2]):
        assert x[~queued].tobytes() == y[~queued].tobytes()
        scale = np.maximum(1.0, np.abs(x[queued]).reshape(int(queued.sum()), -1).max(axis=1))
        assert (np.abs(x[queued] - y[queued]).reshape(int(queued.sum()), -1).max(axis=1) / scale).max() < 1e-9
    differing = int(((res[0][1] != res[1][1]).reshape(n, -1).any(axis=1)).sum())
    print(f"[two vs one kernel footholds h={horizon}] {int(queued.sum())} queued envs, {differing} not bitwise")


# ------------------------------------------------------------------------------------- 4. the prologue's footholds
def _random_gait(n, rng):
    stance = rng.uniform(0.1, 0.6, (n, 4))
    duty = 1.0 - rng.uniform(0.0, 0.8, (n, 4))
    duty[rng.uniform(size=(n, 4)) < 0.1] = 1.0
    phase = rng.uniform(0.0, 1.0, (n, 4))
    state = rng.integers(0, 2, (n, 4)).astype(np.int32)
    return dict(stance_duration=stance, duty_factor=duty, initial_leg_phase=phase, initial_leg_state=state)


def _ulp_close(a, b):
    """|a - b| within one float32 ulp of b, elementwise."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return np.abs(a.astype(np.float64) - b.astype(np.float64)) <= np.spacing(np.abs(b)).astype(np.float64)


@pytest.mark.parametrize("n", [6000, 40000])                     # per-(env, leg) prologue / per-env prologue
def test_prologue_footholds(rg_lib, cuda_device, n):
    horizon = 10
    rng = np.random.default_rng(n)
    st = synthetic.make_states(n, GHOST, seed=73)
    robot = SyntheticRobotBatch(GHOST, st, device=cuda_device)
    clock = {"t": torch.zeros(n, dtype=torch.float64, device=cuda_device)}
    gait = _random_gait(n, rng)
    ctls = [BatchedMPCController(robot, lambda: clock["t"], horizon=horizon, contact_plan=True, use_graph=False, **kw)
            for kw in ({}, {"foothold_plan": True})]
    cmd = torch.from_numpy(rng.uniform(-0.6, 0.6, (n, 3)).astype(np.float32)).to(cuda_device)
    for ctl in ctls:
        ctl.set_env_gait(**gait)
        ctl.command.copy_(cmd)
    rp = ctls[1].robot_params
    hips = [[rp.hip_positions[leg][a] for a in range(3)] for leg in range(4)]
    swing_height = rp.desired_height - rp.foot_clearance
    t = rng.integers(0, 5000, n) * 0.001
    clock["t"] = torch.from_numpy(t).to(cuda_device)
    for ctl in ctls:
        ctl.get_action()
    torch.cuda.synchronize()
    for ctl in ctls:
        assert int(ctl.unverified_count()) == 0
    sched = ctls[1].mpc_contact_schedule.cpu().numpy()
    assert np.array_equal(sched, ctls[0].mpc_contact_schedule.cpu().numpy())
    got = ctls[1].mpc_foothold_plan.cpu().numpy()
    vel = ctls[1].com_velocity_body.cpu().numpy()
    rate = st.base_rpy_rate.astype(np.float64)
    c = cmd.cpu().numpy()
    feet = st.foot_positions_base.reshape(n, 4, 3)
    bad = 0
    for e in range(0, n, max(1, n // 3000)):
        ends = [raibert_end(vel[e].astype(np.float64), rate[e, 2], c[e, :2].astype(np.float64), float(c[e, 2]), hips[leg],
                            gait["stance_duration"][e, leg], swing_height) for leg in range(4)]
        want = predict_footholds(sched[e], feet[e], c[e], ends, DT)
        bad += int(not _ulp_close(got[e], want).all())
    assert bad == 0, bad
    # invalid gait rows: held rows, all-stance schedule, neighbours untouched
    bad_rows = np.arange(5, n, 997)
    for ctl in ctls:
        ctl.env_duty_factor[torch.from_numpy(bad_rows).to(cuda_device), 1] = 1.5
        ctl.get_action()
    torch.cuda.synchronize()
    got2 = ctls[1].mpc_foothold_plan.cpu().numpy()
    assert np.array_equal(got2[bad_rows], np.broadcast_to(feet[bad_rows][:, None], (len(bad_rows), horizon, 4, 3)))
    assert np.array_equal(ctls[1].mpc_contact_schedule.cpu().numpy(), ctls[0].mpc_contact_schedule.cpu().numpy())


# ------------------------------------------------------------------------------------- 5. the whole control step
N_STEP_ENVS, N_STEPS = 260, 10


def _mixed_gait(n):
    group = np.arange(n) % len(SCHEDULES)
    rows = [GAIT_SCHEDULES[SCHEDULES[g]] for g in group]
    return dict(stance_duration=np.array([r["STANCE_DURATION_SECONDS"] for r in rows], dtype=np.float64),
                duty_factor=np.array([r["DUTY_FACTOR"] for r in rows], dtype=np.float64),
                initial_leg_phase=np.array([r["INIT_PHASE_FULL_CYCLE"] for r in rows], dtype=np.float64),
                initial_leg_state=np.array([[int(v) for v in r["INIT_LEG_STATE"]] for r in rows], dtype=np.int32)), group


def _reference_env(args):
    """One restated LocomotionController with the foothold planning solver, for env e over the whole sequence."""
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
    solver = foothold_planning_solver(lambda: octl._time_since_reset, DT, 10)
    octl = locomotion.build_mpc_controller(orobot, lambda: clock["t"], with_gait(GHOST, name).GetCtrlConstants(),
                                           mpc_solver=solver)
    solver.gen = octl.gait_generator
    solver.robot = orobot
    solver.swing_height = float(octl.swing_leg_controller._desired_height[2])
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
        out.append((act, octl.stance_leg_controller.last_contact_forces.copy(), solver.last_schedule.copy(),
                    solver.last_footholds.copy()))
    return out


@pytest.fixture(scope="module")
def step_reference():
    gait, group = _mixed_gait(N_STEP_ENVS)
    seq = synthetic.make_state_sequence(N_STEP_ENVS, N_STEPS, GHOST, seed=synthetic.SEED + 83, env_gait=gait)
    jobs = [([s.slice(e, e + 1) for s in seq], 0, SCHEDULES[group[e]]) for e in range(N_STEP_ENVS)]
    n_proc = min(32, os.cpu_count() or 1)
    if n_proc > 1:
        with multiprocessing.get_context("fork").Pool(n_proc) as pool:
            ref = pool.map(_reference_env, jobs, chunksize=2)
    else:
        ref = [_reference_env(j) for j in jobs]
    return seq, group, ref


def _run(dev, seq, group, warm_start, use_graph, description=GHOST, schedule_of_group=None, zero_command=False, **kw):
    robot = SyntheticRobotBatch(description, seq[0], device=dev)
    ctl = BatchedMPCController(robot, robot.GetTimeSinceReset, warm_start=warm_start, use_graph=use_graph,
                               contact_plan=True, **kw)
    for g, name in enumerate(schedule_of_group or SCHEDULES):
        ctl.set_env_gait(schedule=name, env_ids=torch.from_numpy(np.flatnonzero(group == g)).to(dev))
    ctl.reset()
    out = []
    for k in range(len(seq)):
        robot.load(seq[k])
        ctl.command.copy_(torch.zeros_like(ctl.command) if zero_command else torch.from_numpy(seq[k].command).to(dev))
        a = ctl.get_action()
        torch.cuda.synchronize()
        assert int(ctl.unverified_count()) == 0
        out.append((a.cpu().numpy().copy(), ctl.contact_forces.cpu().numpy().copy(),
                    ctl.mpc_contact_schedule.cpu().numpy().copy(),
                    None if ctl.mpc_foothold_plan is None else ctl.mpc_foothold_plan.cpu().numpy().copy()))
    return out


@pytest.mark.parametrize("warm_start", [True, False])
def test_foothold_control_step_against_the_restated_controller(rg_lib, cuda_device, step_reference, warm_start):
    seq, group, ref = step_reference
    eager = _run(cuda_device, seq, group, warm_start, use_graph=False, foothold_plan=True)
    graph = _run(cuda_device, seq, group, warm_start, use_graph=True, foothold_plan=True)
    worst_f = worst_tau = 0.0
    moved = 0
    for k in range(N_STEPS):
        for x, y in zip(eager[k], graph[k]):                      # graph replay = eager, bitwise
            assert x.tobytes() == y.tobytes(), k
        a, f, sched, feet = eager[k]
        for e in range(N_STEP_ENVS):
            ra, rf, rs, rfeet = ref[e][k]
            assert np.array_equal(sched[e], rs), (k, e)
            assert _ulp_close(feet[e], rfeet).all(), (k, e)
            moved += int(not np.array_equal(rfeet, np.broadcast_to(rfeet[0], rfeet.shape)))
            worst_f = max(worst_f, np.abs(f[e] - rf).max() / max(1.0, np.abs(rf).max()))
            ae = a[e].reshape(12, 5)
            np.testing.assert_array_equal(ae[:, [1, 2, 3]], ra[:, [1, 2, 3]])
            worst_tau = max(worst_tau, np.abs(ae[:, 4] - ra[:, 4]).max() / max(1.0, np.abs(ra[:, 4]).max()))
    assert moved > 0
    assert worst_f < REL_TOL and worst_tau < REL_TOL, (worst_f, worst_tau)
    print(f"[foothold step {N_STEP_ENVS} x {N_STEPS}, warm={warm_start}] worst force {worst_f:.1e}, torque "
          f"{worst_tau:.1e}; {moved} env-steps with moving footholds")


def test_stand_with_zero_command_is_the_contact_plan_alone(rg_lib, cuda_device):
    n = 300
    seq = synthetic.make_state_sequence(n, 3, K3LSO, seed=synthetic.SEED + 89)
    group = np.zeros(n, dtype=np.int64)
    outs = [_run(cuda_device, seq, group, True, use_graph=False, description=K3LSO, schedule_of_group=("stand",),
                 zero_command=True, **kw) for kw in ({}, {"foothold_plan": True})]
    for k, ((a0, f0, s0, _), (a1, f1, s1, feet)) in enumerate(zip(*outs)):
        assert a0.tobytes() == a1.tobytes() and f0.tobytes() == f1.tobytes() and np.array_equal(s0, s1)
        assert np.all(s1 == 1)
        held = np.broadcast_to(seq[k].foot_positions_base.reshape(n, 1, 4, 3), feet.shape)
        assert feet.tobytes() == np.ascontiguousarray(held).tobytes()


def test_foothold_plan_needs_the_contact_plan(rg_lib, cuda_device):
    st = synthetic.make_states(4, GHOST, seed=1)
    robot = SyntheticRobotBatch(GHOST, st, device=cuda_device)
    with pytest.raises(ValueError):
        BatchedMPCController(robot, robot.GetTimeSinceReset, foothold_plan=True)
