"""Per-env body and ground (rg_mpc_env_model): mass, inertia and friction coefficients per env in the stance solve
and the control step.

  * a batch mixing 8 random bodies equals 8 solves, each on a workspace set up with one body (lean + fallback kernels
    at 4096 envs, the single complete kernel at 300; h = 5, 10, 20; trot and pace);
  * 512 envs, each with its own body and friction, against the C oracle with that env's parameters (numpy oracle
    arbitrates), plus the solver-independent KKT certificate on 64 of them;
  * a model holding the workspace's own values solves what the workspace solves;
  * invalid rows get zero forces and RG_STATUS_BAD_MODEL without touching the other envs;
  * BatchedMPCController.set_env_model: eager and graph steps, in-place updates between replays, warm and cold."""
import dataclasses
import math
import os

import numpy as np
import pytest
import torch

from oracle import c_oracle, convex_mpc as cm
from robot_gym import cuda as rg
from robot_gym.controllers.mpc.batched_mpc_controller import BatchedMPCController
from robot_gym.model.robots.descriptions import GHOST, with_gait
from robot_gym.model.robots.synthetic_robot import SyntheticRobotBatch
from robot_gym.util import synthetic

pytestmark = pytest.mark.gpu
REL_TOL = 1e-4            # as tests/test_gpu_parity_full.py
RECHECK = 1e-5
CORES = os.cpu_count() or 1
INPUTS = ("com_velocity_body", "base_rpy", "base_rpy_rate", "planned_contacts", "foot_positions_base", "command")
HEIGHT = GHOST.GetCtrlConstants().MPC_BODY_HEIGHT


def _body(rng):
    """A random body and ground, drawn as test_random_parameter_sets_every_env_against_the_oracle draws them."""
    mass = float(rng.uniform(8.0, 40.0))
    a = rng.normal(size=(3, 3)) * 0.05
    inertia = np.diag(rng.uniform(0.05, 0.8, 3)) + a @ a.T                       # symmetric positive definite
    return mass, inertia.reshape(-1), rng.uniform(0.2, 1.0, 4)


def _oracle_params(horizon, mass, inertia, mu):
    return cm.MpcParams(mass=float(mass), inertia=tuple(float(x) for x in inertia), horizon=horizon,
                        friction_coeffs=tuple(float(x) for x in mu))


def _ws_params(horizon, mass=None, inertia=None, mu=None):
    ctrl = GHOST.GetCtrlConstants()
    p = rg.default_mpc_params(ctrl.MPC_BODY_MASS if mass is None else mass,
                              ctrl.MPC_BODY_INERTIA if inertia is None else [float(x) for x in inertia], HEIGHT, horizon)
    if mu is not None:
        p.friction_coeffs = tuple(float(x) for x in mu)
    return p


def _solve(ws, st, dev, model=None):
    n, h = len(st.base_rpy), ws.horizon
    t = [torch.from_numpy(np.ascontiguousarray(getattr(st, k))).to(dev) for k in INPUTS]
    h64 = torch.empty((n, h, 12), dtype=torch.float64, device=dev)
    f, _, info = rg.mpc_build_solve(ws, *t, horizon_forces_f64=h64, env_model=model)
    torch.cuda.synchronize()
    return f.cpu().numpy(), h64.cpu().numpy().reshape(n, -1), info.cpu().numpy()


def _model(dev, mass=None, inertia=None, mu=None):
    to = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)
    return dict(mass=to(mass), inertia=to(inertia), friction_coeffs=to(mu))


def _rel(a, b):
    return np.abs(a - b).max(axis=1) / np.maximum(1.0, np.abs(b).max(axis=1))


VERIFIED = rg.RG_STATUS_POLISHED | rg.RG_STATUS_NO_STANCE


@pytest.mark.parametrize("n", [4096, 300])
@pytest.mark.parametrize("schedule", ["trot", "pace"])
@pytest.mark.parametrize("horizon", [5, 10, 20])
def test_mixed_batch_equals_one_workspace_per_group(rg_lib, cuda_device, horizon, schedule, n):
    rng = np.random.default_rng(10 * horizon + len(schedule) + n)
    bodies = [_body(rng) for _ in range(8)]
    group = np.arange(n) % 8                                                     # neighbouring CTAs differ
    desc = with_gait(GHOST, schedule)
    st = synthetic.make_states(n, desc, schedule_ctrl=desc.GetCtrlConstants(), seed=500 + horizon)
    model = _model(cuda_device, *[np.stack([bodies[g][k] for g in group]) for k in range(3)])
    ws = rg.MpcWorkspace(_ws_params(horizon), device=cuda_device, max_envs=n)
    _, h_mix, info_mix = _solve(ws, st, cuda_device, model)
    status_mix = info_mix[:, rg.RG_INFO_STATUS]
    assert np.all(status_mix & VERIFIED), (horizon, schedule, n)
    for g, (mass, inertia, mu) in enumerate(bodies):
        ws_g = rg.MpcWorkspace(_ws_params(horizon, mass, inertia, mu), device=cuda_device, max_envs=n)
        _, h_g, info_g = _solve(ws_g, st, cuda_device)
        sel = group == g
        rel = _rel(h_mix[sel], h_g[sel])
        assert rel.max() < 1e-9, (g, float(rel.max()))
        assert np.array_equal(status_mix[sel] & VERIFIED, info_g[sel, rg.RG_INFO_STATUS] & VERIFIED), g


@pytest.mark.parametrize("schedule", ["trot", "pace"])
def test_every_env_with_its_own_body_against_the_oracle(rg_lib, cuda_device, schedule):
    n, horizon = 512, 10
    rng = np.random.default_rng(77 + len(schedule))
    bodies = [_body(rng) for _ in range(n)]
    desc = with_gait(GHOST, schedule)
    st = synthetic.make_states(n, desc, schedule_ctrl=desc.GetCtrlConstants(), seed=601)
    ws = rg.MpcWorkspace(_ws_params(horizon), device=cuda_device, max_envs=n)
    _, h64, info = _solve(ws, st, cuda_device, _model(cuda_device, *[np.stack([b[k] for b in bodies]) for k in range(3)]))
    status = info[:, rg.RG_INFO_STATUS]
    assert np.all(status & VERIFIED)
    ref = np.stack([c_oracle.solve_batch(_oracle_params(horizon, *bodies[i]), st.slice(i, i + 1), HEIGHT,
                                         want_horizon=True)[1].reshape(-1) for i in range(n)])
    rel = _rel(h64, ref)
    suspects = np.flatnonzero(rel > RECHECK)
    assert len(suspects) <= 8, (len(suspects), float(rel.max()))
    for i in suspects:                                                           # the numpy oracle arbitrates
        i = int(i)
        exact = cm.compute_contact_forces(_oracle_params(horizon, *bodies[i]), st.com_velocity_body[i].astype(np.float64),
                                          st.base_rpy[i].astype(np.float64), st.base_rpy_rate[i].astype(np.float64),
                                          st.planned_contacts[i], st.foot_positions_base[i].astype(np.float64),
                                          [0, 0, HEIGHT], [float(st.command[i, 0]), float(st.command[i, 1]), 0.0],
                                          [0, 0, 0], [0, 0, float(st.command[i, 2])])
        rel[i] = np.abs(h64[i] - exact).max() / max(1.0, np.abs(exact).max())
    assert rel.max() < REL_TOL, (int(rel.argmax()), float(rel.max()))
    # solver-independent: the float64 solution is a KKT point of the QP built with the env's own parameters
    for i in range(0, n, n // 64):
        if not st.planned_contacts[i].any():
            assert np.all(h64[i] == 0.0)
            continue
        mp = _oracle_params(horizon, *bodies[i])
        qp = cm.build_qp(mp, st.com_velocity_body[i].astype(np.float64), st.base_rpy[i].astype(np.float64),
                         st.base_rpy_rate[i].astype(np.float64), st.planned_contacts[i],
                         st.foot_positions_base[i].astype(np.float64), [0, 0, HEIGHT],
                         [float(st.command[i, 0]), float(st.command[i, 1]), 0.0], [0, 0, 0], [0, 0, float(st.command[i, 2])])
        cert = cm.kkt_certificate(qp.p_mat, qp.q_vec, qp.c_mat, qp.lb, qp.ub, -h64[i], act_tol=1e-8)
        qs = max(1.0, float(np.abs(qp.q_vec).max()))
        tol = 1e-6 if status[i] & rg.RG_STATUS_POLISHED else 1e-3
        assert cert["stationarity"] <= tol * qs and cert["dual_sign"] <= tol * qs, (i, cert, qs)
        assert cert["primal"] <= 1e-8 * mp.fz_max, (i, cert["primal"])


@pytest.mark.parametrize("n", [4096, 300])
def test_nominal_model_equals_no_model(rg_lib, cuda_device, n):
    p = _ws_params(10)
    ws = rg.MpcWorkspace(p, device=cuda_device, max_envs=n)
    st = synthetic.make_states(n, with_gait(GHOST, "pace"), schedule_ctrl=with_gait(GHOST, "pace").GetCtrlConstants(), seed=41)
    _, h_ref, info_ref = _solve(ws, st, cuda_device)
    full = (np.full(n, p.mass), np.tile(np.array(list(p.inertia)), (n, 1)), np.tile(np.array(list(p.friction_coeffs)), (n, 1)))
    for fields in ((0, 1, 2), (0,), (1,), (2,)):
        parts = [full[k] if k in fields else None for k in range(3)]
        _, h, info = _solve(ws, st, cuda_device, _model(cuda_device, *parts))
        assert _rel(h, h_ref).max() <= 1e-12, fields
        assert np.array_equal(info[:, rg.RG_INFO_STATUS], info_ref[:, rg.RG_INFO_STATUS]), fields


def test_bad_rows_are_isolated(rg_lib, cuda_device):
    n = 4096
    p = _ws_params(10)
    ws = rg.MpcWorkspace(p, device=cuda_device, max_envs=n)
    st = synthetic.make_states(n, GHOST, seed=43)
    rng = np.random.default_rng(5)
    mass, inertia, mu = (np.stack(x) for x in zip(*[_body(rng) for _ in range(n)]))
    good = [_model(cuda_device, mass, inertia, mu)]
    active = (rg.MpcWorkspace(p, device=cuda_device, max_envs=n), rg.new_active_set(n, 10, cuda_device))
    singular = np.array([1.0, 2, 3, 2, 4, 6, 0, 0, 1])
    bad_rows = {3: ("mass", 0.0), 10: ("inertia", np.full(9, np.nan)), 17: ("inertia", singular),
                25: ("mu", np.array([0.5, 0.5, 0.0, 0.5])), 26: ("mu", np.full(4, -0.3)), 40: ("mass", np.inf)}
    bm, bi, bmu = mass.copy(), inertia.copy(), mu.copy()
    for row, (field, value) in bad_rows.items():
        {"mass": bm, "inertia": bi, "mu": bmu}[field][row] = value
    f_ok, h_ok, info_ok = _solve(ws, st, cuda_device, good[0])
    f_bad, h_bad, info_bad = _solve(ws, st, cuda_device, _model(cuda_device, bm, bi, bmu))
    rows = np.array(sorted(bad_rows))
    others = np.setdiff1d(np.arange(n), rows)
    assert np.all(f_bad[rows] == 0) and np.all(h_bad[rows] == 0)
    assert np.all(info_bad[rows, rg.RG_INFO_STATUS] == rg.RG_STATUS_BAD_MODEL)
    assert np.array_equal(h_bad[others], h_ok[others]) and np.array_equal(info_bad[others], info_ok[others])
    # the warm-start set of a bad row is reset to UNKNOWN
    ws_w, act = active
    t = [torch.from_numpy(np.ascontiguousarray(getattr(st, k))).to(cuda_device) for k in INPUTS]
    rg.mpc_build_solve(ws_w, *t, active_set=act, env_model=good[0])
    rg.mpc_build_solve(ws_w, *t, active_set=act, env_model=_model(cuda_device, bm, bi, bmu))
    torch.cuda.synchronize()
    assert torch.all(act[torch.from_numpy(rows).to(cuda_device)] == -1)
    # the controller's setter refuses the same rows
    robot = SyntheticRobotBatch(GHOST, st.slice(0, 64), device=cuda_device)
    ctl = BatchedMPCController(robot, robot.GetTimeSinceReset)
    for kw in (dict(mass=0.0), dict(mass=math.nan), dict(inertia=np.full(9, np.nan)), dict(inertia=singular),
               dict(friction_coeffs=0.0), dict(friction_coeffs=[0.5, -0.1, 0.5, 0.5])):
        with pytest.raises(ValueError):
            ctl.set_env_model(env_ids=[5], **kw)
    assert torch.all(ctl.env_mass == p.mass) and torch.all(ctl.env_friction_coeffs == p.friction_coeffs[0])


def _run_controller(dev, seq, steps, model=None, overrides=None, warm_start=True, use_graph=None):
    robot = SyntheticRobotBatch(GHOST, seq[0], device=dev)
    ctl = BatchedMPCController(robot, robot.GetTimeSinceReset, mpc_overrides=overrides, warm_start=warm_start,
                               use_graph=use_graph)
    if model is not None:
        ctl.set_env_model(**model)
    out = []
    for k in range(steps):
        robot.load(seq[k])
        ctl.command.copy_(torch.from_numpy(seq[k].command).to(dev))
        a = ctl.get_action()
        torch.cuda.synchronize()
        assert int(ctl.unverified_count()) == 0
        out.append((a.cpu().numpy().copy(), ctl.leg_state.cpu().numpy().copy(), ctl.normalized_phase.cpu().numpy().copy(),
                    ctl.contact_forces.cpu().numpy().copy()))
    return ctl, out


def _assert_steps_match(got, ref, idx):
    for k, ((a, s, p, f), (a_r, s_r, p_r, f_r)) in enumerate(zip(got, ref)):
        assert np.array_equal(s[idx], s_r) and p[idx].tobytes() == p_r.tobytes(), k
        scale = np.maximum(1.0, np.abs(f_r).max(axis=1, keepdims=True))
        assert (np.abs(f[idx] - f_r) / scale).max() < 1e-6, k
        assert np.abs(a[idx] - a_r).max() <= 1e-5 * max(1.0, np.abs(a_r).max()), k


def _subset(seq, idx):
    return [type(s)(**{f.name: getattr(s, f.name)[idx] for f in dataclasses.fields(s)}) for s in seq]


@pytest.mark.parametrize("warm_start", [True, False])
def test_control_step_with_two_bodies_equals_two_controllers(rg_lib, cuda_device, warm_start):
    n, steps = 5000, 4                                                           # eager: above GRAPH_MAX_ENVS
    seq = synthetic.make_state_sequence(n, steps, GHOST, seed=synthetic.SEED + 21)
    rng = np.random.default_rng(8)
    bodies = [_body(rng) for _ in range(2)]
    group = np.arange(n) % 2
    model = dict(mass=np.array([bodies[g][0] for g in group]), inertia=np.stack([bodies[g][1] for g in group]),
                 friction_coeffs=np.stack([bodies[g][2] for g in group]))
    ctl, got = _run_controller(cuda_device, seq, steps, model, warm_start=warm_start)
    assert not ctl._use_graph and ctl._graph is None
    for g, (mass, inertia, mu) in enumerate(bodies):
        idx = np.flatnonzero(group == g)
        p = _ws_params(10, mass, inertia, mu)
        overrides = dict(mass=p.mass, inertia=list(p.inertia), friction_coeffs=list(p.friction_coeffs),
                         fz_max=p.fz_max, fz_min=p.fz_min)
        _, ref = _run_controller(cuda_device, _subset(seq, idx), steps, overrides=overrides, warm_start=warm_start,
                                 use_graph=False)
        _assert_steps_match(got, ref, idx)


def test_graph_replay_reads_model_values_written_in_place(rg_lib, cuda_device):
    n, steps = 512, 4
    seq = synthetic.make_state_sequence(n, steps, GHOST, seed=synthetic.SEED + 22)
    rng = np.random.default_rng(9)
    mass, inertia, mu = (np.stack(x) for x in zip(*[_body(rng) for _ in range(n)]))
    robot = SyntheticRobotBatch(GHOST, seq[0], device=cuda_device)
    ctl = BatchedMPCController(robot, robot.GetTimeSinceReset)
    assert ctl._use_graph
    ctl.set_env_model(mass=mass, inertia=inertia, friction_coeffs=mu)
    twin_robot = SyntheticRobotBatch(GHOST, seq[0], device=cuda_device)
    twin = BatchedMPCController(twin_robot, twin_robot.GetTimeSinceReset, use_graph=False)
    twin.set_env_model(mass=mass, inertia=inertia, friction_coeffs=mu)
    handle = None
    ids = torch.arange(0, n, 7, device=cuda_device)
    for k in range(steps):
        if k == 2:                                   # between two replays: new friction for some envs, in place
            new_mu = torch.full((len(ids), 4), 0.25, dtype=torch.float64, device=cuda_device)
            ctl.set_env_model(friction_coeffs=new_mu, env_ids=ids)
            twin.set_env_model(friction_coeffs=new_mu, env_ids=ids)
        for r, c in ((robot, ctl), (twin_robot, twin)):
            r.load(seq[k])
            c.command.copy_(torch.from_numpy(seq[k].command).to(cuda_device))
            c.get_action()
        torch.cuda.synchronize()
        if k == 0:
            handle = ctl._graph.value
        assert ctl._graph is not None and ctl._graph.value == handle and ctl._graph_invalidations == 0, k
        assert int(ctl.unverified_count()) == 0 and int(twin.unverified_count()) == 0
        assert torch.equal(ctl.leg_state, twin.leg_state) and torch.equal(ctl.normalized_phase, twin.normalized_phase)
        assert torch.equal(ctl.contact_forces, twin.contact_forces), k
        assert torch.equal(ctl.action, twin.action), k
    changed = ctl.env_friction_coeffs[ids]
    assert torch.all(changed == 0.25)
