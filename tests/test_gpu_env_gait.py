"""Per-env gait (rg_gait_env_params): stance duration, duty factor, initial phase and initial state per env in the
control step's prologue.

  * every env with its own random gait: desired / measured leg states and phases bit for bit against the oracle's
    OpenloopGaitGenerator built with that env's rows, on both prologue mappings (6000 and 40000 envs);
  * 256 envs x 10 steps, each with its own gait, against one restated controller per env;
  * a batch mixing the five named schedules equals one controller per schedule (eager and graph, warm and cold);
  * rows holding the workspace's own values step exactly as no gait (each array alone and all four);
  * invalid rows hold their env in stance without touching the other envs, and set_env_gait refuses them;
  * in-place updates between graph replays need no re-capture;
  * reset(env_ids) re-arms the leg states from each env's own initial states."""
import dataclasses
import types

import numpy as np
import pytest
import torch

from oracle import c_oracle, kinematics, locomotion
from robot_gym import cuda as rg
from robot_gym.controllers.mpc.batched_mpc_controller import BatchedMPCController
from robot_gym.model.robots.descriptions import GAIT_SCHEDULES, GHOST, with_gait
from robot_gym.model.robots.synthetic_robot import SyntheticRobotBatch
from robot_gym.util import synthetic

pytestmark = pytest.mark.gpu
REL_TOL = 1e-4            # as tests/test_gpu_parity_full.py
SCHEDULES = tuple(GAIT_SCHEDULES)
KEYS = ("stance_duration", "duty_factor", "initial_leg_phase", "initial_leg_state")
SCHED_KEYS = ("STANCE_DURATION_SECONDS", "DUTY_FACTOR", "INIT_PHASE_FULL_CYCLE", "INIT_LEG_STATE")
STANCE = 1


def _schedule_row(name):
    s = GAIT_SCHEDULES[name]
    return ([float(v) for v in s["STANCE_DURATION_SECONDS"]], [float(v) for v in s["DUTY_FACTOR"]],
            [float(v) for v in s["INIT_PHASE_FULL_CYCLE"]], [int(v) for v in s["INIT_LEG_STATE"]])


def _random_gait(n, rng):
    """Every env its own valid gait: stance U(0.1, 0.6), duty U(0.2, 1] with exact 1.0s, phases U[0, 1), random
    SWING / STANCE; the first five envs hold the five named schedules."""
    stance = rng.uniform(0.1, 0.6, (n, 4))
    duty = 1.0 - rng.uniform(0.0, 0.8, (n, 4))                     # (0.2, 1]
    duty[rng.uniform(size=(n, 4)) < 0.1] = 1.0
    phase = rng.uniform(0.0, 1.0, (n, 4))
    state = rng.integers(0, 2, (n, 4)).astype(np.int32)
    for e, name in enumerate(SCHEDULES[:n]):
        stance[e], duty[e], phase[e], state[e] = _schedule_row(name)
    return dict(stance_duration=stance, duty_factor=duty, initial_leg_phase=phase, initial_leg_state=state)


def _ctrl_with(gait, e, ctrl=None):
    """A copy of GHOST's ctrl constants holding env e's gait rows."""
    c = types.SimpleNamespace(**vars(ctrl or GHOST.GetCtrlConstants()))
    for key, skey in zip(KEYS, SCHED_KEYS):
        row = gait[key][e]
        setattr(c, skey, [int(v) for v in row] if key == "initial_leg_state" else [float(v) for v in row])
    return c


class _Contacts:
    num_legs = 4

    def __init__(self):
        self.contacts = np.zeros(4, dtype=np.uint8)

    def GetFootContacts(self):
        return self.contacts


def _clock_controller(dev, st, **kw):
    """A controller whose clock is a tensor the test sets: time_since_reset equals it exactly (reset at t = 0)."""
    robot = SyntheticRobotBatch(GHOST, st, device=dev)
    clock = {"t": torch.zeros(len(st), dtype=torch.float64, device=dev)}
    ctl = BatchedMPCController(robot, lambda: clock["t"], **kw)
    return robot, clock, ctl


@pytest.mark.parametrize("n", [6000, 40000])                     # per-(env, leg) prologue / per-env prologue
def test_gait_bit_exact_against_the_oracle_generator(rg_lib, cuda_device, n):
    rng = np.random.default_rng(n)
    gait = _random_gait(n, rng)
    st = synthetic.make_states(n, GHOST, seed=71)
    robot, clock, ctl = _clock_controller(cuda_device, st)
    ctl.set_env_gait(**gait)
    gens = [locomotion.OpenloopGaitGenerator(_Contacts(), *[gait[k][e] for k in KEYS]) for e in range(n)]
    for k in range(3):
        t = rng.integers(0, 5000, n) * 0.001                       # the simulator's 1 ms grid ...
        odd = rng.uniform(size=n) < 0.5
        t[odd] = rng.uniform(0.0, 7.0, int(odd.sum()))            # ... and arbitrary doubles
        st.foot_contacts = (rng.uniform(size=(n, 4)) < 0.5).astype(np.uint8)
        robot.load(st)
        clock["t"] = torch.from_numpy(t).to(cuda_device)
        ctl.get_action()
        torch.cuda.synchronize()
        assert torch.equal(ctl.time_since_reset.cpu(), torch.from_numpy(t))
        des, sta, pha = (x.cpu().numpy() for x in (ctl.desired_leg_state, ctl.leg_state, ctl.normalized_phase))
        mpc = ctl.mpc_contact_state.cpu().numpy()
        for e in range(n):
            g = gens[e]
            g._robot.contacts = st.foot_contacts[e]
            g.update(float(t[e]))
            assert list(des[e]) == g.desired_leg_state and list(sta[e]) == g.leg_state, (k, e)
            assert pha[e].tobytes() == np.asarray(g.normalized_phase, dtype=np.float64).tobytes(), (k, e)
        assert np.array_equal(mpc, ((des == STANCE) | (des == 2)).astype(np.uint8))
        assert int(ctl.unverified_count()) == 0


def test_per_env_gait_against_the_restated_controller(rg_lib, cuda_device):
    """256 envs x 10 steps, each env with its own gait, against one restated LocomotionController per env built with
    that env's gait constants (the swing legs' Raibert foothold uses the env's stance duration)."""
    n_env, n_steps = 256, 10
    gait = _random_gait(n_env, np.random.default_rng(11))
    seq = synthetic.make_state_sequence(n_env, n_steps, GHOST, seed=synthetic.SEED + 41, env_gait=gait)
    robot = SyntheticRobotBatch(GHOST, seq[0], device=cuda_device)
    ctl = BatchedMPCController(robot, robot.GetTimeSinceReset)
    ctl.set_env_gait(**gait)
    acts, des, sta, pha, frc = [], [], [], [], []
    for k in range(n_steps):
        robot.load(seq[k])
        ctl.command.copy_(torch.from_numpy(seq[k].command).to(cuda_device))
        a = ctl.get_action()
        torch.cuda.synchronize()
        acts.append(a.cpu().numpy().copy()); des.append(ctl.desired_leg_state.cpu().numpy().copy())
        sta.append(ctl.leg_state.cpu().numpy().copy()); pha.append(ctl.normalized_phase.cpu().numpy().copy())
        frc.append(ctl.contact_forces.cpu().numpy().copy())
        assert int(ctl.unverified_count()) == 0
    worst_f = worst_q = worst_tau = 0.0
    swing_steps = 0
    for e in range(n_env):
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
        octl = locomotion.build_mpc_controller(orobot, lambda: clock["t"], _ctrl_with(gait, e),
                                               mpc_solver=c_oracle.compute_contact_forces)
        octl.reset()
        for k in range(n_steps):
            load(k)
            s = seq[k]
            for leg_ctl in (octl.swing_leg_controller, octl.stance_leg_controller):
                leg_ctl.desired_speed = [float(s.command[e, 0]), float(s.command[e, 1]), 0.0]
                leg_ctl.desired_twisting_speed = float(s.command[e, 2])
            octl.update()
            ref = octl.get_action().reshape(12, 5)
            assert list(des[k][e]) == octl.gait_generator.desired_leg_state, (e, k)
            assert list(sta[k][e]) == octl.gait_generator.leg_state, (e, k)
            assert pha[k][e].tobytes() == np.asarray(octl.gait_generator.normalized_phase, dtype=np.float64).tobytes(), (e, k)
            rf = octl.stance_leg_controller.last_contact_forces
            worst_f = max(worst_f, np.abs(frc[k][e] - rf).max() / max(1.0, np.abs(rf).max()))
            a = acts[k][e].reshape(12, 5)
            np.testing.assert_array_equal(a[:, [1, 2, 3]], ref[:, [1, 2, 3]])
            swing_steps += int((ref[:, 1] != 0).sum())
            worst_q = max(worst_q, np.abs(a[:, 0] - ref[:, 0]).max())
            worst_tau = max(worst_tau, np.abs(a[:, 4] - ref[:, 4]).max() / max(1.0, np.abs(ref[:, 4]).max()))
    assert swing_steps > 0
    assert worst_f < REL_TOL and worst_q < 5e-5 and worst_tau < REL_TOL, (worst_f, worst_q, worst_tau)
    print(f"[per-env gait 256 x 10] worst force {worst_f:.1e} rel, swing joint target {worst_q:.1e} rad, torque {worst_tau:.1e} rel")


def _subset(seq, idx):
    return [type(s)(**{f.name: getattr(s, f.name)[idx] for f in dataclasses.fields(s)}) for s in seq]


def _run(dev, seq, steps, desc=GHOST, schedules=None, warm_start=True, use_graph=None):
    robot = SyntheticRobotBatch(desc, seq[0], device=dev)
    ctl = BatchedMPCController(robot, robot.GetTimeSinceReset, warm_start=warm_start, use_graph=use_graph)
    if schedules is not None:
        for name, idx in schedules.items():
            ctl.set_env_gait(schedule=name, env_ids=torch.from_numpy(idx).to(dev))
        ctl.reset()
    out = []
    for k in range(steps):
        robot.load(seq[k])
        ctl.command.copy_(torch.from_numpy(seq[k].command).to(dev))
        a = ctl.get_action()
        torch.cuda.synchronize()
        assert int(ctl.unverified_count()) == 0
        out.append((a.cpu().numpy().copy(), ctl.desired_leg_state.cpu().numpy().copy(), ctl.leg_state.cpu().numpy().copy(),
                    ctl.normalized_phase.cpu().numpy().copy(), ctl.contact_forces.cpu().numpy().copy()))
    return ctl, out


def _assert_steps_match(got, ref, idx):
    """The tolerances of tests/test_gpu_env_model.py: states and phases bitwise, forces 1e-6 relative, actions 1e-5."""
    for k, ((a, d, s, p, f), (a_r, d_r, s_r, p_r, f_r)) in enumerate(zip(got, ref)):
        assert np.array_equal(d[idx], d_r) and np.array_equal(s[idx], s_r) and p[idx].tobytes() == p_r.tobytes(), k
        scale = np.maximum(1.0, np.abs(f_r).max(axis=1, keepdims=True))
        assert (np.abs(f[idx] - f_r) / scale).max() < 1e-6, k
        assert np.abs(a[idx] - a_r).max() <= 1e-5 * max(1.0, np.abs(a_r).max()), k


@pytest.mark.parametrize("warm_start", [True, False])
@pytest.mark.parametrize("n", [5000, 700])                       # eager (above GRAPH_MAX_ENVS) / one graph launch
def test_mixed_schedules_equal_one_controller_per_schedule(rg_lib, cuda_device, n, warm_start):
    steps = 4
    group = np.arange(n) % len(SCHEDULES)                        # interleaved env by env
    rows = [_schedule_row(SCHEDULES[g]) for g in group]
    gait = {key: np.array([r[i] for r in rows]) for i, key in enumerate(KEYS)}
    seq = synthetic.make_state_sequence(n, steps, GHOST, seed=synthetic.SEED + 43, env_gait=gait)
    schedules = {name: np.flatnonzero(group == g) for g, name in enumerate(SCHEDULES)}
    ctl, got = _run(cuda_device, seq, steps, schedules=schedules, warm_start=warm_start)
    assert ctl._use_graph == (n <= BatchedMPCController.GRAPH_MAX_ENVS)
    for name, idx in schedules.items():
        desc = with_gait(GHOST, name)
        _, ref = _run(cuda_device, _subset(seq, idx), steps, desc=desc, warm_start=warm_start, use_graph=False)
        _assert_steps_match(got, ref, idx)


def _step_twins(dev, n, gait_struct, steps=3):
    """Two controllers on the same states: one steps without a gait, the other through rg_control_step_env with the
    given rg_gait_env_params.  Returns both controllers' outputs per step."""
    seq = synthetic.make_state_sequence(n, steps, GHOST, seed=synthetic.SEED + 47)
    outs = []
    for g in (None, gait_struct):
        robot = SyntheticRobotBatch(GHOST, seq[0], device=dev)
        ctl = BatchedMPCController(robot, robot.GetTimeSinceReset, use_graph=False)
        ctl._env_gait = g                                         # the step passes this struct to rg_control_step_env
        res = []
        for k in range(steps):
            robot.load(seq[k])
            ctl.command.copy_(torch.from_numpy(seq[k].command).to(dev))
            ctl.get_action()
            torch.cuda.synchronize()
            res.append([t.cpu().clone() for t in (ctl.desired_leg_state, ctl.leg_state, ctl.normalized_phase,
                                                  ctl.mpc_contact_state, ctl.swing_foot_target, ctl.contact_forces,
                                                  ctl.action, ctl.last_leg_state)])
        outs.append(res)
    return outs


@pytest.mark.parametrize("n", [4096, 40000])                     # per-(env, leg) prologue / per-env prologue
def test_nominal_rows_equal_no_gait(rg_lib, cuda_device, n):
    c = GHOST.GetCtrlConstants()
    nominal = {key: torch.tensor([[float(v) if key != "initial_leg_state" else int(v) for v in getattr(c, skey)]] * n,
                                 dtype=torch.int32 if key == "initial_leg_state" else torch.float64, device=cuda_device)
               for key, skey in zip(KEYS, SCHED_KEYS)}
    for fields in (KEYS,) + tuple((k,) for k in KEYS):
        g = rg.GaitEnvParams()
        for key in fields:
            setattr(g, key, nominal[key].data_ptr())
        ref, got = _step_twins(cuda_device, n, g)
        for k, (a, b) in enumerate(zip(ref, got)):
            for x, y in zip(a, b):
                assert torch.equal(x, y), (fields, k)


@pytest.mark.parametrize("n", [4096, 40000])
def test_bad_rows_hold_their_env_in_stance(rg_lib, cuda_device, n):
    rng = np.random.default_rng(13)
    gait = _random_gait(n, rng)
    bad_rows = {3: ("duty_factor", 0.0), 10: ("duty_factor", 1.5), 17: ("stance_duration", -0.1),
                25: ("stance_duration", np.nan), 26: ("initial_leg_phase", 1.0), 40: ("initial_leg_state", 2)}
    seq = synthetic.make_state_sequence(n, 3, GHOST, seed=synthetic.SEED + 49, env_gait=gait)
    runs = []
    for bad in (False, True):
        robot = SyntheticRobotBatch(GHOST, seq[0], device=cuda_device)
        ctl = BatchedMPCController(robot, robot.GetTimeSinceReset, use_graph=False)
        ctl.set_env_gait(**gait)
        if bad:                                                   # written behind the setter's back
            for row, (key, value) in bad_rows.items():
                getattr(ctl, "env_" + key)[row, 2] = value
        res = []
        for k in range(3):
            robot.load(seq[k])
            ctl.command.copy_(torch.from_numpy(seq[k].command).to(cuda_device))
            ctl.get_action()
            torch.cuda.synchronize()
            res.append({name: getattr(ctl, name).cpu().clone() for name in (
                "desired_leg_state", "leg_state", "normalized_phase", "mpc_contact_state", "last_leg_state",
                "swing_joint_valid", "swing_foot_target", "contact_forces", "action", "solve_info")})
        runs.append(res)
    rows = torch.tensor(sorted(bad_rows))
    others = torch.from_numpy(np.setdiff1d(np.arange(n), rows.numpy()))
    for k, (ok, bad) in enumerate(zip(*runs)):
        assert torch.all(bad["desired_leg_state"][rows] == STANCE) and torch.all(bad["leg_state"][rows] == STANCE), k
        assert torch.all(bad["normalized_phase"][rows] == -1.0) and torch.all(bad["mpc_contact_state"][rows] == 1), k
        assert torch.all(bad["last_leg_state"][rows] == STANCE) and torch.all(bad["swing_joint_valid"][rows] == 0), k
        assert torch.all(bad["swing_foot_target"][rows] == 0), k
        for name in ok:
            assert torch.equal(bad[name][others], ok[name][others]), (k, name)
    # the setter refuses the same rows and writes nothing
    robot = SyntheticRobotBatch(GHOST, seq[0].slice(0, 64), device=cuda_device)
    ctl = BatchedMPCController(robot, robot.GetTimeSinceReset)
    ctl.set_env_gait(schedule="walk")
    before = [getattr(ctl, "env_" + key).clone() for key in KEYS]
    for key, value in bad_rows.values():
        row = [0.3, 0.6, 0.5, 1][KEYS.index(key)]
        row = [row, row, value, row]
        with pytest.raises(ValueError):
            ctl.set_env_gait(**{key: row}, env_ids=[5, 6])
    for key, b in zip(KEYS, before):
        assert torch.equal(getattr(ctl, "env_" + key), b), key


def test_graph_replay_reads_gait_values_written_in_place(rg_lib, cuda_device):
    n, steps = 512, 5
    seq = synthetic.make_state_sequence(n, steps, GHOST, seed=synthetic.SEED + 51)
    robot = SyntheticRobotBatch(GHOST, seq[0], device=cuda_device)
    ctl = BatchedMPCController(robot, robot.GetTimeSinceReset)
    assert ctl._use_graph
    ctl.set_env_gait(schedule="trot")
    twin_robot = SyntheticRobotBatch(GHOST, seq[0], device=cuda_device)
    twin = BatchedMPCController(twin_robot, twin_robot.GetTimeSinceReset, use_graph=False)
    twin.set_env_gait(schedule="trot")
    ids = torch.arange(0, n, 3, device=cuda_device)
    handle = None
    for k in range(steps):
        if k == 2:                                   # between two replays: some envs switch from trot to bound
            ctl.set_env_gait(schedule="bound", env_ids=ids)
            twin.set_env_gait(schedule="bound", env_ids=ids)
        for r, c in ((robot, ctl), (twin_robot, twin)):
            r.load(seq[k])
            c.command.copy_(torch.from_numpy(seq[k].command).to(cuda_device))
            c.get_action()
        torch.cuda.synchronize()
        if k == 0:
            handle = ctl._graph.value
        assert ctl._graph is not None and ctl._graph.value == handle and ctl._graph_invalidations == 0, k
        assert int(ctl.unverified_count()) == 0 and int(twin.unverified_count()) == 0
        for name in ("desired_leg_state", "leg_state", "normalized_phase", "contact_forces", "action"):
            assert torch.equal(getattr(ctl, name), getattr(twin, name)), (k, name)
    bound = torch.tensor(_schedule_row("bound")[3], dtype=torch.int32, device=cuda_device)
    assert torch.equal(ctl.env_initial_leg_state[ids], bound.expand(len(ids), 4))


def test_reset_rearms_each_env_from_its_own_initial_states(rg_lib, cuda_device):
    n = 64
    st = synthetic.make_states(n, GHOST, seed=53)
    robot = SyntheticRobotBatch(GHOST, st, device=cuda_device)
    ctl = BatchedMPCController(robot, robot.GetTimeSinceReset)
    init = torch.tensor([int(s) for s in GHOST.GetCtrlConstants().INIT_LEG_STATE], dtype=torch.int32, device=cuda_device)
    ctl.get_action()
    ctl.reset(torch.arange(0, 8, device=cuda_device))              # no gait: INIT_LEG_STATE, as before
    assert torch.equal(ctl.desired_leg_state[:8], init.expand(8, 4))
    states = torch.from_numpy(np.random.default_rng(4).integers(0, 2, (n, 4)).astype(np.int32)).to(cuda_device)
    ctl.set_env_gait(initial_leg_state=states)
    assert torch.equal(ctl.desired_leg_state[:8], init.expand(8, 4))   # set_env_gait itself does not reset
    ctl.get_action()
    torch.cuda.synchronize()
    stepped = ctl.desired_leg_state.clone()
    ids = torch.arange(8, n, 3, device=cuda_device)
    ctl.reset(ids)
    assert torch.equal(ctl.desired_leg_state[ids], states[ids]) and torch.equal(ctl.leg_state[ids], states[ids])
    assert torch.all(ctl.normalized_phase[ids] == 0) and torch.all(ctl.last_leg_state[ids] == -1)
    rest = torch.ones(n, dtype=torch.bool, device=cuda_device)
    rest[ids] = False
    assert torch.equal(ctl.desired_leg_state[rest], stepped[rest])
    ctl.reset()
    assert torch.equal(ctl.desired_leg_state, states) and torch.equal(ctl.leg_state, states)
