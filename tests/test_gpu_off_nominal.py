"""GPU tests off the nominal state band: the stance solve, the estimator and the leg kinematics where an RL batch goes
and ``synthetic.make_states`` does not (robot_gym.util.synthetic.make_off_nominal_states).

  * every family x h in {5, 10, 20}, 256 envs, the whole horizon against the C oracle (the numpy oracle arbitrates),
    plus the solver-independent KKT certificate of every env with a stance leg;
  * the two-kernel and the one-kernel solve on one 4096-env batch of all families (the fallback queue is busy there);
  * warm starts from exact, perturbed and garbage seeds, with up to three held rows per block;
  * per-env body and ground (the model twins of both kernels) at extreme masses, inertias and friction;
  * the Riccati factorisation at the attitude-map scaling of steep pitch;
  * the moving-window estimator at windows 1 ... 64, standalone and inside the fused step (both prologue kernels);
  * IK, FK and J^T at the edge of the leg workspace, for both robots.

The reference of the solve is pinned to the numpy oracle on the same families by tests/test_off_nominal_oracle.py."""
import ctypes
import dataclasses
import math
import os

import numpy as np
import pytest
import torch

from oracle import c_oracle, convex_mpc as cm, kinematics, locomotion
from robot_gym import cuda as rg
from robot_gym.controllers.mpc.batched_kinematics import BatchedKinematics, robot_params_from_description
from robot_gym.model.robots.descriptions import GHOST, K3LSO
from robot_gym.util import synthetic

pytestmark = pytest.mark.gpu
REL_TOL = 1e-4            # forces within 1e-4 relative of the oracle optimum
RECHECK = 1e-5            # C oracle vs kernel beyond this: the numpy oracle arbitrates
CORES = os.cpu_count() or 1
HEIGHT = GHOST.GetCtrlConstants().MPC_BODY_HEIGHT
FAMILIES = synthetic.OFF_NOMINAL_FAMILIES
INPUTS = ("com_velocity_body", "base_rpy", "base_rpy_rate", "planned_contacts", "foot_positions_base", "command")


def _dev(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _params(horizon=10, **overrides):
    ctrl = GHOST.GetCtrlConstants()
    p = rg.default_mpc_params(ctrl.MPC_BODY_MASS, ctrl.MPC_BODY_INERTIA, ctrl.MPC_BODY_HEIGHT, horizon)
    for k, v in overrides.items():
        setattr(p, k, v)
    return p


def _solve(dev, st, horizon, ws=None, active_set=None, model=None, **overrides):
    """(float32 horizon forces [N,h,12], float64 horizon forces [N,h,12], solve_info [N,4]) of one solve."""
    n = len(st)
    ws = ws or rg.MpcWorkspace(_params(horizon, **overrides), device=dev, max_envs=max(1, n))
    h64 = torch.empty((n, horizon, 12), dtype=torch.float64, device=dev)
    f, hf, info = rg.mpc_build_solve(ws, *[_dev(getattr(st, k), dev) for k in INPUTS], want_horizon=True,
                                     horizon_forces_f64=h64, active_set=active_set, env_model=model)
    torch.cuda.synchronize()
    hf = hf.cpu().numpy()
    np.testing.assert_array_equal(f.cpu().numpy(), hf[:, 0, :])
    return hf, h64.cpu().numpy(), info.cpu().numpy()


def _oracle_args(st, i):
    return (st.com_velocity_body[i].astype(np.float64), st.base_rpy[i].astype(np.float64),
            st.base_rpy_rate[i].astype(np.float64), st.planned_contacts[i], st.foot_positions_base[i].astype(np.float64),
            [0, 0, HEIGHT], [float(st.command[i, 0]), float(st.command[i, 1]), 0.0], [0, 0, 0], [0, 0, float(st.command[i, 2])])


def _numpy_oracle(mp, st, i):
    return cm.compute_contact_forces(mp, *_oracle_args(st, i))


def _assert_all_envs_match(gpu, ref, st, mps, what):
    """gpu / ref: [N, m] forces over the whole horizon; ``mps``: the oracle parameters of every env.  Every env must
    agree within REL_TOL; envs where the C oracle and the kernel differ beyond RECHECK are re-solved by the numpy oracle."""
    n = len(gpu)
    scale = np.maximum(1.0, np.abs(ref).reshape(n, -1).max(axis=1))
    rel = np.abs(gpu - ref).reshape(n, -1).max(axis=1) / scale
    suspects = np.flatnonzero(rel > RECHECK)
    assert len(suspects) <= max(8, n // 200), (what, len(suspects), float(rel.max()))    # the C oracle is exact to ~1e-7
    for i in suspects:
        exact = _numpy_oracle(mps[int(i)], st, int(i))
        rel[i] = np.abs(gpu[i] - exact).max() / max(1.0, np.abs(exact).max())
    assert rel.max() < REL_TOL, (what, int(rel.argmax()), float(rel.max()))
    return float(rel.max()), len(suspects)


def _check_kkt(st, h64, info, mps, what):
    """Solver-independent certificate of the kernel's float64 solution on the dense QP of oracle.convex_mpc.build_qp:
    a verified env (RG_STATUS_POLISHED) must pass stationarity and multiplier signs at 1e-6 max(1, |q|_inf); every env
    must be primal feasible at 1e-8 fz_max (the interior point keeps the primal residual at 0).  Returns the worst
    relative stationarity of the verified envs."""
    polished = (info[:, rg.RG_INFO_STATUS] & rg.RG_STATUS_POLISHED) != 0
    worst = 0.0
    for i in range(len(st)):
        if not st.planned_contacts[i].any():
            continue
        mp = mps[i]
        qp = cm.build_qp(mp, *_oracle_args(st, i))
        cert = cm.kkt_certificate(qp.p_mat, qp.q_vec, qp.c_mat, qp.lb, qp.ub, -h64[i].reshape(-1), act_tol=1e-8)
        qs = max(1.0, float(np.abs(qp.q_vec).max()))
        assert cert["primal"] <= 1e-8 * mp.fz_max, (what, i, cert["primal"])
        if polished[i]:
            assert cert["stationarity"] <= 1e-6 * qs, (what, i, cert["stationarity"], qs)
            assert cert["dual_sign"] <= 1e-6 * qs, (what, i, cert["dual_sign"], qs)
            worst = max(worst, cert["stationarity"] / qs)
    return worst


def _check_outputs(st, hf, h64, info, what):
    """Every output finite, swing legs exactly zero over the whole horizon, no RG_STATUS_NUMERIC."""
    assert np.all(np.isfinite(hf)) and np.all(np.isfinite(h64)), what
    swing = np.repeat(st.planned_contacts[:, None, :, None] == 0, 3, axis=3)
    swing = np.broadcast_to(swing, (len(st), hf.shape[1], 4, 3)).reshape(len(st), hf.shape[1], 12)
    assert np.all(hf[swing] == 0.0) and np.all(h64[swing] == 0.0), what
    assert not np.any(info[:, rg.RG_INFO_STATUS] & rg.RG_STATUS_NUMERIC), what


def _concat(states):
    return synthetic.SyntheticStates(**{f.name: np.concatenate([getattr(s, f.name) for s in states])
                                        for f in dataclasses.fields(synthetic.SyntheticStates)})


def _all_families(n_env, seed):
    """``n_env`` envs: equal shares of every family, in family blocks."""
    per = -(-n_env // len(FAMILIES))
    return _concat([synthetic.make_off_nominal_states(per, f, GHOST, seed=seed + k) for k, f in enumerate(FAMILIES)]).slice(0, n_env)


def _summary(info):
    stance = (info[:, rg.RG_INFO_STATUS] & rg.RG_STATUS_NO_STANCE) == 0
    pol = (info[:, rg.RG_INFO_STATUS] & rg.RG_STATUS_POLISHED) != 0
    return (float(pol[stance].mean()) if stance.any() else 1.0, float(info[stance, rg.RG_INFO_POLISH_ROUNDS].mean()),
            float(info[stance, rg.RG_INFO_IPM_ITERS].mean()))


# ------------------------------------------------------------------------------------------------ a. every family
@pytest.mark.parametrize("horizon", [5, 10, 20])
@pytest.mark.parametrize("family", FAMILIES)
def test_every_family_against_the_oracle_with_kkt_certificate(rg_lib, cuda_device, family, horizon):
    n = 256
    st = synthetic.make_off_nominal_states(n, family, GHOST, seed=1000 + 10 * horizon)
    mp = cm.MpcParams(horizon=horizon)
    hf, h64, info = _solve(cuda_device, st, horizon)
    _check_outputs(st, hf, h64, info, (family, horizon))
    _, ref, _ = c_oracle.solve_batch(mp, st, HEIGHT, n_threads=CORES, want_horizon=True)
    worst, n_suspect = _assert_all_envs_match(h64.reshape(n, -1), ref.reshape(n, -1), st, [mp] * n, (family, horizon))
    stat = _check_kkt(st, h64, info, [mp] * n, (family, horizon))
    verified, rounds, ipm = _summary(info)
    print(f"[{family} h={horizon}] worst rel force error {worst:.1e} ({n_suspect} re-checked), worst KKT stationarity "
          f"(verified) {stat:.1e}, verified {verified:.3f}, mean rounds {rounds:.2f}, mean IPM iterations {ipm:.2f}")


# ------------------------------------------------------------------------------------------------ b. both kernel paths
@pytest.mark.parametrize("horizon", [5, 10, 20])
def test_two_kernel_and_one_kernel_solves_agree_off_nominal(rg_lib, cuda_device, horizon):
    """4096 envs of all families is above the one-wave threshold at every horizon (148 SMs x 24 / 7 / 5 CTAs), so
    two_kernel_solve = 1 runs the lean kernel and the fallback queue.  Envs verified by both paths agree, the queue
    is used, and three solves on one workspace are bitwise identical (the queue re-arms, the solve is deterministic)."""
    n = 4096
    st = _all_families(n, seed=2000 + horizon)
    hf1, h1, info1 = _solve(cuda_device, st, horizon, two_kernel_solve=0)
    ws2 = rg.MpcWorkspace(_params(horizon), device=cuda_device, max_envs=n)
    runs = [_solve(cuda_device, st, horizon, ws=ws2) for _ in range(3)]
    hf2, h2, info2 = runs[0]
    for hf_r, h_r, info_r in runs[1:]:
        assert hf_r.tobytes() == hf2.tobytes() and h_r.tobytes() == h2.tobytes() and np.array_equal(info_r, info2)
    both = ((info1[:, rg.RG_INFO_STATUS] & info2[:, rg.RG_INFO_STATUS]) & rg.RG_STATUS_POLISHED) != 0
    scale = np.maximum(1.0, np.abs(h1).reshape(n, -1).max(axis=1))
    gap = np.abs(h1 - h2).reshape(n, -1).max(axis=1) / scale
    assert both.any() and gap[both].max() < 1e-5, (horizon, float(gap[both].max()))
    # the lean kernel and the complete kernel run the same active-set rounds: verified envs agree bit for bit
    assert h1[both].tobytes() == h2[both].tobytes() and hf1[both].tobytes() == hf2[both].tobytes(), horizon
    stance = st.planned_contacts.any(axis=1)
    queued = stance & ((info2[:, rg.RG_INFO_STATUS] & rg.RG_STATUS_ACTIVE_SET_ONLY) == 0)
    assert queued.any()                                          # the fallback queue was used ...
    assert np.all(info2[queued, rg.RG_INFO_IPM_ITERS] > 0)       # ... and those envs went through the interior point
    print(f"[h={horizon}] {int(queued.sum())} of {n} envs queued; verified by both paths {both.mean():.3f}; "
          f"worst gap {gap[both].max():.1e}")


# ------------------------------------------------------------------------------------------------ c. warm start
@pytest.mark.parametrize("horizon", [10, 20])
def test_warm_start_off_nominal(rg_lib, cuda_device, horizon):
    """An exact seed reproduces the cold result in one round for every env with a stance leg the cold solve verified
    (an unverified env stores RG_ACTIVE_SET_UNKNOWN and is re-solved cold; an env without a stance leg takes 0 rounds); a perturbed neighbour gives the cold result; the all-rows
    garbage seed (0x3FF in every block) is repaired.  Blocks here hold up to three rows."""
    n = 2048
    st = _all_families(n, seed=3000 + horizon)
    ws = rg.MpcWorkspace(_params(horizon), device=cuda_device, max_envs=n)
    _, h_cold, info_cold = _solve(cuda_device, st, horizon, ws=ws)
    seed = rg.new_active_set(n, horizon, cuda_device)
    _, h1, info1 = _solve(cuda_device, st, horizon, ws=ws, active_set=seed)
    assert h1.tobytes() == h_cold.tobytes() and np.array_equal(info1, info_cold)      # unknown seed == cold start
    verified = (info_cold[:, rg.RG_INFO_STATUS] & rg.RG_STATUS_POLISHED) != 0
    stored = seed.cpu().numpy().astype(np.int64) & 0xFFFF
    assert np.all(stored[~verified] == 0xFFFF)
    nbits = np.array([[bin(int(v)).count("1") for v in row if v != 0xFFFF] for row in stored[verified]], dtype=object)
    assert max(max(r) for r in nbits if len(r)) == 3                                      # corners of the pyramid
    _, h2, info2 = _solve(cuda_device, st, horizon, ws=ws, active_set=seed)
    scale = lambda h: np.maximum(1.0, np.abs(h).reshape(n, -1).max(axis=1))
    gap = np.abs(h2 - h_cold).reshape(n, -1).max(axis=1) / scale(h_cold)
    assert gap[verified].max() < 1e-5, float(gap[verified].max())
    assert np.all(info2[verified, rg.RG_INFO_STATUS] & rg.RG_STATUS_POLISHED)
    # an env without a stance leg (contact pattern 0) has nothing to solve: 0 rounds, zero forces, both times
    no_stance = (info_cold[:, rg.RG_INFO_STATUS] & rg.RG_STATUS_NO_STANCE) != 0
    assert np.array_equal(no_stance, ~st.planned_contacts.any(axis=1)) and no_stance.any()
    assert np.all(info2[no_stance, rg.RG_INFO_POLISH_ROUNDS] == 0) and np.all(h2[no_stance] == 0.0)
    solved = verified & ~no_stance
    assert np.all(info2[solved, rg.RG_INFO_POLISH_ROUNDS] == 1) and np.all(info2[solved, rg.RG_INFO_IPM_ITERS] == 0)
    # a neighbouring problem (the next control step: the state drifts a little)
    rng = np.random.default_rng(horizon)
    st2 = st.slice(0, n)
    st2.com_velocity_body = (st.com_velocity_body + rng.normal(0, 0.01, st.com_velocity_body.shape)).astype(np.float32)
    st2.base_rpy = (st.base_rpy + rng.normal(0, 0.002, st.base_rpy.shape) * np.array([1, 1, 0])).astype(np.float32)
    _, h3, info3 = _solve(cuda_device, st2, horizon, ws=ws, active_set=seed)
    _, h3c, info3c = _solve(cuda_device, st2, horizon, ws=ws)
    both = ((info3[:, rg.RG_INFO_STATUS] & info3c[:, rg.RG_INFO_STATUS]) & rg.RG_STATUS_POLISHED) != 0
    gap3 = np.abs(h3 - h3c).reshape(n, -1).max(axis=1) / scale(h3c)
    assert gap3[both].max() < 1e-5, float(gap3[both].max())
    assert both.sum() >= 0.99 * ((info3c[:, rg.RG_INFO_STATUS] & rg.RG_STATUS_POLISHED) != 0).sum()
    # a garbage seed (every row of every block marked active) is repaired
    junk = torch.full((n, 4 * horizon), 0x3FF, dtype=torch.int16, device=cuda_device)
    _, h4, info4 = _solve(cuda_device, st, horizon, ws=ws, active_set=junk)
    assert np.all(info4[verified, rg.RG_INFO_STATUS] & rg.RG_STATUS_POLISHED)
    gap4 = np.abs(h4 - h_cold).reshape(n, -1).max(axis=1) / scale(h_cold)
    assert gap4[verified].max() < 1e-5, float(gap4[verified].max())
    print(f"[warm h={horizon}] cold verified {verified.mean():.3f} ({int(no_stance.sum())} without stance); neighbour "
          f"rounds warm {info3[:, rg.RG_INFO_POLISH_ROUNDS].mean():.2f} vs cold {info3c[:, rg.RG_INFO_POLISH_ROUNDS].mean():.2f}")


# ------------------------------------------------------------------------------------------------ d. per-env model
def _extreme_bodies(rng, n):
    """mass ~U(2, 80) kg; inertia R diag(lambda) R^T with R a random rotation and lambda spread 1:100 over 0.01 ... 1;
    one friction coefficient ~U(0.05, 2) per pyramid row."""
    mass = rng.uniform(2.0, 80.0, n)
    inertia = np.empty((n, 9))
    for i in range(n):
        q, r = np.linalg.qr(rng.normal(size=(3, 3)))
        q = q * np.sign(np.diag(r))
        lam = rng.permutation([0.01, 10 ** rng.uniform(-2, 0), 1.0])
        inertia[i] = (q @ np.diag(lam) @ q.T).reshape(-1)
    return mass, inertia, rng.uniform(0.05, 2.0, (n, 4))


@pytest.mark.parametrize("n,horizon", [(512, 10), (256, 20), (4096, 10)])
def test_per_env_model_at_extremes_against_the_oracle(rg_lib, cuda_device, n, horizon):
    """mpc_solve_model_kernel (below the one-wave threshold) and the lean + fallback model twins (4096 envs at h = 10):
    every env with its own body and ground against the C oracle with its own MpcParams (fz bounds follow the mass),
    the same force bar and KKT certificate as the workspace-model solve."""
    rng = np.random.default_rng(n + horizon)
    st = _all_families(n, seed=4000 + horizon)
    mass, inertia, mu = _extreme_bodies(rng, n)
    mps = [cm.MpcParams(mass=float(mass[i]), inertia=tuple(float(x) for x in inertia[i]), horizon=horizon,
                        friction_coeffs=tuple(float(x) for x in mu[i])) for i in range(n)]
    to = lambda a: _dev(a.astype(np.float64), cuda_device)
    model = dict(mass=to(mass), inertia=to(inertia), friction_coeffs=to(mu))
    hf, h64, info = _solve(cuda_device, st, horizon, model=model)
    _check_outputs(st, hf, h64, info, (n, horizon))
    assert not np.any(info[:, rg.RG_INFO_STATUS] & rg.RG_STATUS_BAD_MODEL)
    ref = np.stack([c_oracle.solve_batch(mps[i], st.slice(i, i + 1), HEIGHT, want_horizon=True)[1].reshape(-1)
                    for i in range(n)])
    worst, n_suspect = _assert_all_envs_match(h64.reshape(n, -1), ref, st, mps, (n, horizon))
    stat = _check_kkt(st, h64, info, mps, (n, horizon))
    verified, rounds, ipm = _summary(info)
    print(f"[model n={n} h={horizon}] worst rel force error {worst:.1e} ({n_suspect} re-checked), worst KKT stationarity "
          f"{stat:.1e}, verified {verified:.3f}, mean rounds {rounds:.2f}, mean IPM iterations {ipm:.2f}")


# ------------------------------------------------------------------------------------------------ e. Riccati
RICCATI_CASES = [(5, 1e-6), (5, 1e-4), (10, 1e-6), (10, 1e-4), (20, 1e-6), (20, 1e-4)]
RICCATI_INACCURATE = {(20, 1e-6)}      # see test_riccati_accuracy_at_h20_alpha_1e6


def _riccati_errors(rg_lib, cuda_device, horizon, alpha):
    """The kernel's Riccati factor / solve (rg_debug_riccati_solve) with the attitude block of the stage cost built from
    the actual T(rpy) at pitch 1.3, 1.45 and 1.5 rad (entries up to ~14), alpha in the D_t scale 1 / (2 alpha),
    all-zero, full-rank and random-rank D_t, against numpy's dense solve of the 6h x 6h system.  Every solve must
    report positive definite pivots (flag 0) and a finite result; returns (pitch, trial, relative error, kappa(Psi))
    of each system."""
    h = horizon
    j = np.arange(h)
    m = np.maximum.outer(j, j)
    c1 = (h - m).astype(float)
    c2 = np.array([[np.sum((np.arange(max(a, b) + 1, h + 1) - a - 0.5) * (np.arange(max(a, b) + 1, h + 1) - b - 0.5))
                    for b in range(h)] for a in range(h)])
    rng = np.random.default_rng(50 + horizon + round(-math.log10(alpha)))
    rg_lib.rg_debug_riccati_solve.argtypes = [ctypes.c_int] + [ctypes.c_void_p] * 8
    dt = 0.025
    out = []
    for pitch in (1.3, 1.45, 1.5):
        for trial in range(4):
            rpy = np.array([rng.uniform(-0.3, 0.3), pitch * rng.choice([-1.0, 1.0]), rng.uniform(-3, 3)])
            tm = cm.calculate_a_mat(rpy)[0:3, 6:9]
            k1 = 2 * dt ** 2 * np.array([0.5, 0.5, 0.2, 0.2, 0.2, 0.1])
            k2ang = 2 * dt ** 4 * tm.T @ np.diag([5, 5, 0.2]) @ tm
            k2lin = 2 * dt ** 4 * np.array([0.0, 0.0, 10.0])
            k2 = np.zeros((6, 6)); k2[:3, :3] = k2ang; k2[3:, 3:] = np.diag(k2lin)
            kk = np.kron(c1, np.diag(k1)) + np.kron(c2, k2)
            d = np.zeros((h, 6, 6))
            for t in range(h):
                nfree = (0, 6, None, None)[trial]
                nfree = int(rng.integers(0, 7)) if nfree is None else nfree
                bz = rng.normal(size=(6, nfree)) * np.array([5, 5, 5, .05, .05, .05])[:, None]
                d[t] = bz @ bz.T / (2 * alpha)
            b = rng.normal(size=(h, 6)) * 1e3
            psi = np.linalg.inv(kk)
            for t in range(h):
                psi[6 * t:6 * t + 6, 6 * t:6 * t + 6] += d[t]
            v_ref = np.linalg.solve(psi, b.reshape(-1))
            kappa = float(np.linalg.cond(psi))
            packed = np.array([[d[t][r, c] for r in range(6) for c in range(r + 1)] for t in range(h)])
            dev = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(cuda_device)
            k1_d, k2a_d, k2l_d, d_d, b_d = dev(k1), dev(k2ang), dev(k2lin), dev(packed), dev(b)
            v_d = torch.zeros(6 * h, dtype=torch.float64, device=cuda_device)
            flag = torch.zeros(1, dtype=torch.int32, device=cuda_device)
            p = lambda x: ctypes.c_void_p(x.data_ptr())
            rg.check(rg_lib.rg_debug_riccati_solve(h, p(k1_d), p(k2a_d), p(k2l_d), p(d_d), p(b_d), p(v_d), p(flag), None))
            torch.cuda.synchronize()
            assert int(flag.item()) == 0, (pitch, alpha, trial)
            v = v_d.cpu().numpy()
            assert np.all(np.isfinite(v)), (pitch, alpha, trial)
            out.append((pitch, trial, float(np.abs(v - v_ref).max() / np.abs(v_ref).max()), kappa))
    return out


@pytest.mark.parametrize("horizon,alpha", RICCATI_CASES)
def test_riccati_at_steep_pitch_scaling(rg_lib, cuda_device, horizon, alpha):
    """The bar is 1e-7 relative.  Where the condition number of Psi = K^-1 + blkdiag(D_t) is so large that a
    backward-stable solve in float64 -- numpy's included -- can only promise about kappa * 1e-15, that is the bound.
    At h = 20 with alpha = 1e-6 only the flag and finiteness are asserted here; its accuracy is the next test."""
    errs = _riccati_errors(rg_lib, cuda_device, horizon, alpha)
    if (horizon, alpha) not in RICCATI_INACCURATE:
        for pitch, trial, err, kappa in errs:
            assert err < max(1e-7, kappa * 1e-15), (pitch, alpha, trial, err, kappa)
    print(f"[riccati h={horizon} alpha={alpha:.0e}] worst relative error {max(e[2] for e in errs):.1e}, "
          f"largest kappa(Psi) {max(e[3] for e in errs):.1e}")


@pytest.mark.xfail(strict=True, reason="known defect: the Riccati sweep inverts Y = S + S D S by 3 x 3 cofactor blocks; "
                                       "with D_t ~ 1/(2e-6) at steep pitch Y is far worse conditioned than Psi and the "
                                       "h = 20 solve loses digits (~3e-6 relative at kappa(Psi) ~ 1e6; a backward-stable "
                                       "solve gives ~1e-9).  The solver's refinement and exact verification absorb it.")
def test_riccati_accuracy_at_h20_alpha_1e6(rg_lib, cuda_device):
    for pitch, trial, err, kappa in _riccati_errors(rg_lib, cuda_device, 20, 1e-6):
        assert err < max(1e-7, kappa * 1e-15), (pitch, trial, err, kappa)


# ------------------------------------------------------------------------------------------------ f. estimator
def _estimator_inputs(n, steps, seed):
    """World velocities with magnitudes 1e-9 ... 1e2 and random signs, and random unit attitudes, float32, per step.
    Float32 values spanning fewer than 2^29 in magnitude add up exactly in float64, which would leave the Neumaier
    correction at 0: this span makes the running sums round, so both branches produce nonzero corrections."""
    rng = np.random.default_rng(seed)
    vel = (10.0 ** rng.uniform(-9, 2, (steps, n, 3)) * rng.choice([-1.0, 1.0], (steps, n, 3))).astype(np.float32)
    quat = rng.normal(size=(steps, n, 4))
    quat = (quat / np.linalg.norm(quat, axis=2, keepdims=True)).astype(np.float32)
    return vel, quat


def _robot_ws(dev, window):
    params = robot_params_from_description(GHOST)
    params.velocity_window = window
    return rg.RobotWorkspace(params, device=dev)


def _fused_estimator_run(rg_lib, dev, window, vel, quat, reps):
    """rg_control_step over ``reps`` tiled copies of the batch with a robot workspace of window ``window``; returns the
    window sums, corrections and body velocities after every step, [steps, reps * n, 3]."""
    steps, n0 = vel.shape[:2]
    n = n0 * reps
    base = synthetic.make_states(n0, GHOST, seed=77)
    tile = lambda a: np.ascontiguousarray(np.tile(a, (reps,) + (1,) * (a.ndim - 1)))
    rws = _robot_ws(dev, window)
    mws = rg.MpcWorkspace(_params(10), device=dev, max_envs=n)
    f32, f64, i32, u8 = torch.float32, torch.float64, torch.int32, torch.uint8
    z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)
    buf = dict(time_since_reset=z((n,), f64), foot_contacts=_dev(tile(base.foot_contacts), dev),
               base_velocity_world=z((n, 3), f32), base_orientation_xyzw=z((n, 4), f32),
               base_rpy=_dev(tile(base.base_rpy), dev), base_rpy_rate=_dev(tile(base.base_rpy_rate), dev),
               foot_positions_base=_dev(tile(base.foot_positions_base), dev), motor_angles=_dev(tile(base.motor_angles), dev),
               command=_dev(tile(base.command), dev),
               vel_window=z((n, 3, window), f64), vel_window_sum=z((n, 3), f64), vel_window_corr=z((n, 3), f64),
               vel_window_count=z((n,), i32), vel_window_head=z((n,), i32),
               last_leg_state=torch.full((n, 4), -1, dtype=i32, device=dev),
               phase_switch_foot_local_position=_dev(tile(base.foot_positions_base), dev),
               swing_joint_angles=z((n, 12), f32), swing_joint_valid=z((n, 4), u8),
               desired_leg_state=z((n, 4), i32), leg_state=z((n, 4), i32), normalized_phase=z((n, 4), f64),
               mpc_contact_state=z((n, 4), u8), swing_foot_target=z((n, 12), f32), com_velocity_body=z((n, 3), f32),
               contact_forces=z((n, 12), f32), motor_torques=z((n, 12), f32), solve_info=z((n, 4), i32),
               action=z((n, 60), f32))
    s = rg.ControllerState()
    for name, t in buf.items():
        setattr(s, name, ctypes.c_void_p(t.data_ptr()))
    t0 = tile(base.time_since_reset)
    sums, corrs, vbody = [], [], []
    for k in range(steps):
        buf["time_since_reset"].copy_(_dev(t0 + 0.01 * k, dev))
        buf["base_velocity_world"].copy_(_dev(tile(vel[k]), dev))
        buf["base_orientation_xyzw"].copy_(_dev(tile(quat[k]), dev))
        rg.check(rg_lib.rg_control_step(mws.ptr, rws.ptr, n, ctypes.byref(s), rg.current_stream_ptr()))
        torch.cuda.synchronize()
        sums.append(buf["vel_window_sum"].cpu().numpy().copy())
        corrs.append(buf["vel_window_corr"].cpu().numpy().copy())
        vbody.append(buf["com_velocity_body"].cpu().numpy().copy())
    assert np.all(np.isfinite(buf["action"].cpu().numpy()))
    return np.stack(sums), np.stack(corrs), np.stack(vbody)


@pytest.mark.parametrize("window", [1, 2, 7, 20, 64])
def test_estimator_windows_bit_exact_standalone_and_fused(rg_lib, cuda_device, window):
    """rg_com_velocity_update for 3W + 5 steps: the Neumaier sum and correction of every axis (nonzero here) are
    BIT-identical to the
    oracle MovingWindowFilter (same IEEE operations in the same order, including the drop-oldest branch once the
    deque is full), the world-frame average is the float32 of the oracle's, the body frame within 5e-7 relative,
    count and head follow the deque.  Then the fused rg_control_step over the same velocities, at a batch on each side
    of kPrologueLegMaxEnvs (32768: per-(env, leg) and per-env prologue kernels), gives bitwise the same sums."""
    dev = cuda_device
    n, W = 64, window
    steps = 3 * W + 5
    vel, quat = _estimator_inputs(n, steps, seed=W)
    rws = _robot_ws(dev, W)
    f32, f64, i32 = torch.float32, torch.float64, torch.int32
    z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)
    win, wsum, wcorr, wcount, whead = z((n, 3, W), f64), z((n, 3), f64), z((n, 3), f64), z((n,), i32), z((n,), i32)
    v_body, v_world = z((n, 3), f32), z((n, 3), f32)
    filters = [[locomotion.MovingWindowFilter(W) for _ in range(3)] for _ in range(n)]
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    ref_sums, ref_corrs, ref_vbody = [], [], []
    worst_body = 0.0
    for k in range(steps):
        vel_d, quat_d = _dev(vel[k], dev), _dev(quat[k], dev)
        rg.check(rg_lib.rg_com_velocity_update(rws.ptr, n, P(vel_d), P(quat_d), P(win), P(wsum), P(wcorr), P(wcount),
                                               P(whead), P(v_body), P(v_world), None))
        torch.cuda.synchronize()
        s_np, c_np, vb, vw = wsum.cpu().numpy(), wcorr.cpu().numpy(), v_body.cpu().numpy(), v_world.cpu().numpy()
        exp_sum, exp_corr, exp_world = np.empty((n, 3)), np.empty((n, 3)), np.empty((n, 3))
        for e in range(n):
            for a in range(3):
                f = filters[e][a]
                exp_world[e, a] = f.calculate_average(float(vel[k, e, a]))
                exp_sum[e, a], exp_corr[e, a] = float(f._sum), float(f._correction)
            ref_b = locomotion.quat_rotate_inverse(quat[k, e].astype(np.float64), exp_world[e])
            worst_body = max(worst_body, float(np.abs(vb[e] - ref_b).max() / max(1.0, np.abs(ref_b).max())))
        assert s_np.tobytes() == exp_sum.tobytes() and c_np.tobytes() == exp_corr.tobytes(), (W, k)
        assert vw.tobytes() == exp_world.astype(np.float32).tobytes(), (W, k)
        assert np.array_equal(wcount.cpu().numpy(), np.full(n, min(k + 1, W))), (W, k)
        assert np.array_equal(whead.cpu().numpy(), np.full(n, (k + 1) % W)), (W, k)
        ref_sums.append(s_np.copy()); ref_corrs.append(c_np.copy()); ref_vbody.append(vb.copy())
    assert worst_body < 5e-7, (W, worst_body)
    ring = win.cpu().numpy()
    for e in range(0, n, 7):
        for a in range(3):
            dq = list(filters[e][a]._value_deque)                 # oldest first; the next write goes to head
            h = steps % W
            assert [ring[e, a, (h + i) % W] for i in range(W)] == dq, (W, e, a)
    ref_sums, ref_corrs, ref_vbody = np.stack(ref_sums), np.stack(ref_corrs), np.stack(ref_vbody)
    if W > 1:                                  # W = 1 holds one float32 sample: its sums are exact by construction
        assert np.count_nonzero(ref_corrs) > 0, W
    for reps in (1, 32768 // n + 1):
        sums, corrs, vbody = _fused_estimator_run(rg_lib, dev, W, vel, quat, reps)
        for name, got, ref in (("sum", sums, ref_sums), ("corr", corrs, ref_corrs), ("v_body", vbody, ref_vbody)):
            got = got.reshape(steps, reps, n, 3)
            for r in range(reps):
                assert got[:, r].tobytes() == ref.tobytes(), (W, reps, r, name)


@pytest.mark.parametrize("window", [0, 65])
def test_robot_setup_rejects_windows_outside_1_to_64(rg_lib, cuda_device, window):
    with pytest.raises(rg.RgCudaError, match="velocity_window"):
        _robot_ws(cuda_device, window)


# ------------------------------------------------------------------------------------------------ g. IK at the edge
def _straight_knee(chain):
    """Knee joint angle at which thigh and shank are colinear: the foot is farthest from the upper joint there."""
    from scipy.optimize import minimize_scalar
    o1 = chain.p[0] + chain.r[0] @ chain.p[1]
    dist = lambda q2: -float(np.linalg.norm(chain.fk([0.0, 0.0, q2]) - o1))
    grid = np.linspace(-math.pi, math.pi, 3601)
    q = grid[int(np.argmin([dist(g) for g in grid]))]
    return float(minimize_scalar(dist, bounds=(q - 0.01, q + 0.01), method="bounded", options=dict(xatol=1e-12)).x)


def _ik_setup(desc, dev, flip_knee=False):
    params = robot_params_from_description(desc)
    if flip_knee:
        for l in range(4):
            params.legs[l].ik_sign_knee = -params.legs[l].ik_sign_knee
    return BatchedKinematics(rg.RobotWorkspace(params, device=dev), dev)


@pytest.mark.parametrize("desc", [GHOST, K3LSO], ids=["ghost", "k3lso"])
def test_ik_fk_and_jacobian_at_the_edge_of_the_workspace(rg_lib, cuda_device, desc):
    _ik_edge_checks(rg_lib, cuda_device, desc)


def _ik_edge_checks(rg_lib, cuda_device, desc):
    """Property test, not a parity test: PyBullet's IK result for an unreachable target is an unpinned iterate.

    Near-straight knees (1e-4 ... 1e-1 rad from straight, on both sides, each side solved by the IK branch that owns
    it): FK(IK(p)) reaches p within 1e-5 m.  From 1e-2 rad on, IK(FK(q)) also returns q within 2e-5 rad plus the
    first-order effect |J^-1| |dp| of the float32 rounding dp of the target; closer to straight J is nearly singular,
    the preimage of a float32 target is not determined to that level, and reach is the claim.  Targets beyond reach (up to 1.5x the leg's reach) and inside the
    abduction cylinder (closer to the hip axis than the abduction offset): finite output; how much farther FK(IK(p))
    is from p than the oracle's damped least-squares IK seeded from the nominal pose is returned (the 1 mm bar is the
    next test; leg_ik falls back to damped least squares where its Newton clean-up cannot run).  J^T at all these poses matches the oracle Jacobian as in the nominal test.  Where the closed form
    clamps the knee straight, reach is the claim."""
    dev = cuda_device
    robot = kinematics.OracleRobot(desc)
    chains = robot._chains
    mc = desc.GetMotorConstants()
    offset, direction = np.asarray(mc.MOTOR_OFFSET, dtype=np.float64), np.asarray(mc.MOTOR_DIRECTION, dtype=np.float64)
    to_motor = lambda qj: (qj - offset) * direction
    to_joint = lambda qm: np.asarray(qm, dtype=np.float64) * direction + offset
    q0 = robot.joint_angles(desc.GetConstants().INIT_MOTOR_ANGLES)
    rng = np.random.default_rng(8)
    kin = _ik_setup(desc, dev)
    kin_flip = _ik_setup(desc, dev, flip_knee=True)
    straight = np.array([_straight_knee(chains[l]) for l in range(4)])
    own_side = np.sign((q0[2::3] - straight + math.pi) % (2 * math.pi) - math.pi)   # side of straight the calibrated branch owns
    # ---- near-straight knees
    n = 256
    delta = 10.0 ** rng.uniform(-4, -1, (n, 4))
    side = rng.choice([-1.0, 1.0], (n, 4))
    qj = np.tile(q0, (n, 1)) + rng.uniform(-0.3, 0.3, (n, 12)) * np.tile([1.0, 1.0, 0.0], 4)
    qj[:, 2::3] = straight[None] + side * delta
    qm = to_motor(qj).astype(np.float32)
    qj = to_joint(qm)                                                  # the float32 pose actually evaluated
    feet = kin.ComputeFootPositionsInBaseFrame(_dev(qm, dev))
    worst_reach = worst_q = 0.0
    near = 0
    for k_ws, branch_side in ((kin, own_side), (kin_flip, -own_side)):
        back = k_ws.ComputeMotorAnglesFromFootLocalPosition(feet).cpu().numpy()
        torch.cuda.synchronize()
        f_np = feet.cpu().numpy().astype(np.float64).reshape(n, 4, 3)
        assert np.all(np.isfinite(back))
        bj = to_joint(back)
        for i in range(n):
            for l in range(4):
                p = f_np[i, l]
                reach = float(np.linalg.norm(chains[l].fk(bj[i, 3 * l:3 * l + 3]) - p))
                assert reach < 1e-5, (i, l, reach, delta[i, l])
                worst_reach = max(worst_reach, reach)
                if side[i, l] != branch_side[l]:
                    continue                                           # the other branch's pose: reach is the claim
                if delta[i, l] < 1e-2:
                    near += 1                                          # too close to singular for a joint-angle claim
                    continue
                foot, jac = chains[l].fk(qj[i, 3 * l:3 * l + 3], with_jacobian=True)
                moved = np.linalg.norm(np.linalg.inv(jac), 2) * float(np.linalg.norm(p - foot))
                err = float(np.abs((bj[i, 3 * l:3 * l + 3] - qj[i, 3 * l:3 * l + 3] + math.pi) % (2 * math.pi) - math.pi).max())
                assert err < 2e-5 + 2 * moved, (i, l, err, moved, delta[i, l])
                worst_q = max(worst_q, err - 2 * moved)
    # ---- beyond reach and inside the abduction cylinder
    targets = np.empty((n, 4, 3))
    for l in range(4):
        ch = chains[l]
        o0 = ch.p[0]
        samples = np.array([ch.fk(q0[3 * l:3 * l + 3] + rng.uniform(-1, 1, 3)) for _ in range(400)])
        reach_max = float(np.linalg.norm(samples - o0, axis=1).max())
        # the closed form's hip-frame basis and abduction offset D (derive_ik_constants in rg_robot.cu): a target whose
        # distance from the hip axis is below |D| has no exact solution, and the IK meets rad = P1^2 + P2^2 - D^2 < 0
        e0 = ch.axis[0] / np.linalg.norm(ch.axis[0])
        a1 = ch.axis[1] / np.linalg.norm(ch.axis[1])
        e1 = ch.r[1] @ a1
        e2 = np.cross(e0, e1)
        d_abd = abs(float(ch.p[1] @ e1 + a1 @ ch.p[2] + a1 @ (ch.r[2] @ ch.toe)))
        half = n // 2
        u = rng.normal(size=(half, 3)); u /= np.linalg.norm(u, axis=1, keepdims=True)
        targets[:half, l] = o0 + u * (reach_max * rng.uniform(1.0, 1.5, half))[:, None]
        phi = rng.uniform(0, 2 * math.pi, n - half)
        rho = d_abd * rng.uniform(0.0, 0.9, n - half)
        ph = (np.outer(rng.uniform(-0.1, 0.1, n - half), e0) + np.outer(rho * np.cos(phi), e1)
              + np.outer(rho * np.sin(phi), e2))
        targets[half:, l] = o0 + ph @ ch.r[0].T
    targets32 = targets.astype(np.float32).reshape(n, 12)
    out = kin.ComputeMotorAnglesFromFootLocalPosition(_dev(targets32, dev)).cpu().numpy()
    assert np.all(np.isfinite(out))
    oj = to_joint(out)
    worst_excess = -1.0
    for i in range(0, n, 2):
        for l in range(4):
            p = targets32[i, 3 * l:3 * l + 3].astype(np.float64)
            mine = float(np.linalg.norm(chains[l].fk(oj[i, 3 * l:3 * l + 3]) - p))
            q_ref = chains[l].ik(p, q0[3 * l:3 * l + 3])
            theirs = float(np.linalg.norm(chains[l].fk(q_ref) - p))
            worst_excess = max(worst_excess, mine - theirs)
    # ---- J^T at these poses
    poses = np.concatenate([qm, out.astype(np.float32)])
    forces = rng.uniform(-60, 60, poses.shape).astype(np.float32)
    tau = kin.MapContactForceToJointTorques(_dev(forces, dev), _dev(poses, dev)).cpu().numpy()
    assert np.all(np.isfinite(tau))
    for i in range(0, len(poses), 4):
        robot.set_state(motor_angles=poses[i].astype(np.float64))
        for l in range(4):
            t = robot.MapContactForceToJointTorques(l, forces[i, 3 * l:3 * l + 3].astype(np.float64))
            ref = np.array([t[3 * l + j] for j in range(3)])
            assert np.abs(tau[i, 3 * l:3 * l + 3] - ref).max() < 1e-4 * max(1.0, np.abs(ref).max()), (i, l)
    print(f"[{'ghost' if desc is GHOST else 'k3lso'}] near-straight reach {worst_reach:.1e} m, "
          f"joint excess {worst_q:.1e} rad ({near} leg samples within 1e-2 of straight: reach only); unreachable targets: worst excess over the "
          f"oracle {worst_excess:.1e} m")
    return worst_excess


@pytest.mark.parametrize("desc", [GHOST, K3LSO], ids=["ghost", "k3lso"])
def test_ik_beyond_reach_is_within_1mm_of_damped_least_squares(rg_lib, cuda_device, desc):
    assert _ik_edge_checks(rg_lib, cuda_device, desc) <= 1e-3
