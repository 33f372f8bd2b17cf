"""Cost and effect of planning the stance QP over the gait's contact schedule (rg_mpc_build_solve_schedule,
rg_control_step_plan).

solve: the stance solve alone, h = 10, 4096 and 65536 envs whose states mix trot, pace, bound, walk and stand, each arm
  warm-started from its own previous solve of the same inputs:
    none   -- the contact row held over the horizon (rg_mpc_build_solve_warm)
    tiled  -- a schedule whose rows all equal that row: the same QPs, so the difference to `none` is the mechanism
    gait   -- each env's gait schedule at its clock (synthetic.planned_contact_schedule): the new workload
  per arm: median / p10 / p90 time, mean active-set rounds, the share of envs that ran interior-point iterations (the
  fallback queue of the two-kernel solve), the unverified count; and how often and by how much the gait schedule
  changes the first-step forces against `none`.
prologue_kernel: kernel time of the step prologue (torch.profiler, CUDA activity), plan off vs on, trot, 4096 and 65536
  envs, h = 10 and 20.
step: the warm-started control step (BatchedMPCController, one CUDA graph per step at 1 env), trot and the five-schedule
  mix, plan off / on, at 1 (5 for the mix), 4096 and 65536 envs, h = 10; and trot at 4096 envs with h = 20.
Arms are interleaved rep by rep; the L2 (126 MB) is overwritten before every timed call; CUDA events around the whole
Python call.  Prints one JSON line with the device name and power limit read in the same run.

  python tools/perf_contact_plan.py [--reps 40] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(REPO, "robot-gym_b200"), REPO]

from robot_gym import cuda as rg                                                     # noqa: E402
from robot_gym.controllers.mpc.batched_mpc_controller import BatchedMPCController   # noqa: E402
from robot_gym.model.robots.descriptions import GAIT_SCHEDULES, GHOST               # noqa: E402
from robot_gym.model.robots.synthetic_robot import SyntheticRobotBatch               # noqa: E402
from robot_gym.util import synthetic                                                 # noqa: E402

SCHEDULES = tuple(GAIT_SCHEDULES)
INPUTS = ("com_velocity_body", "base_rpy", "base_rpy_rate", "planned_contacts", "foot_positions_base", "command")


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def mixed_gait(n):
    group = np.arange(n) % len(SCHEDULES)
    rows = [GAIT_SCHEDULES[SCHEDULES[g]] for g in group]
    return group, (np.array([r["STANCE_DURATION_SECONDS"] for r in rows], dtype=np.float64),
                   np.array([r["DUTY_FACTOR"] for r in rows], dtype=np.float64),
                   np.array([r["INIT_PHASE_FULL_CYCLE"] for r in rows], dtype=np.float64),
                   np.array([[int(v) for v in r["INIT_LEG_STATE"]] for r in rows]))


def timed(fn, flush, rep):
    flush.fill_(rep & 255)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3


def stats(v):
    v = np.array(v)
    return {"median_us": float(np.median(v)), "p10_us": float(np.percentile(v, 10)), "p90_us": float(np.percentile(v, 90))}


def solve_section(dev, flush, reps):
    out = {}
    h = 10
    for n in (4096, 65536):
        group, gait = mixed_gait(n)
        st = synthetic.make_states(n, GHOST, seed=synthetic.SEED)
        # the planned contacts of each env from its own gait at its clock
        st.planned_contacts = synthetic.desired_stance(st.time_since_reset, *gait).astype(np.uint8)
        up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        inputs = [up(getattr(st, k)) for k in INPUTS]
        scheds = {"none": None,
                  "tiled": up(np.repeat(st.planned_contacts[:, None, :], h, axis=1)),
                  "gait": up(synthetic.planned_contact_schedule(st.time_since_reset, 0.025, h, *gait))}
        ctrl = GHOST.GetCtrlConstants()
        arms = {}
        for name, sched in scheds.items():
            ws = rg.MpcWorkspace(rg.default_mpc_params(ctrl.MPC_BODY_MASS, ctrl.MPC_BODY_INERTIA, ctrl.MPC_BODY_HEIGHT, h),
                                 device=dev, max_envs=n)
            act = rg.new_active_set(n, h, dev)
            forces = torch.empty((n, 12), dtype=torch.float32, device=dev)
            info = torch.empty((n, 4), dtype=torch.int32, device=dev)
            args = list(inputs)
            if sched is not None:
                args[3] = None

            def run(ws=ws, act=act, args=args, sched=sched, forces=forces, info=info):
                rg.mpc_build_solve(ws, *args, contact_forces=forces, solve_info=info, active_set=act, contact_schedule=sched)
            arms[name] = (run, forces, info)
        cold = {}
        for name, (run, forces, info) in arms.items():      # the first (cold) solve, then warm-up
            run()
            torch.cuda.synchronize()
            cold[name] = info.cpu().numpy().copy()
            for _ in range(3):
                run()
        torch.cuda.synchronize()
        times = {k: [] for k in arms}
        for rep in range(reps):
            for name, (run, _, _) in arms.items():
                times[name].append(timed(run, flush, rep))
        res = {"envs": n}
        f = {k: v[1].cpu().numpy() for k, v in arms.items()}
        for name, (_, _, info) in arms.items():
            i = info.cpu().numpy()
            c = cold[name]
            stance = (c[:, rg.RG_INFO_STATUS] & rg.RG_STATUS_NO_STANCE) == 0
            res[name] = dict(stats(times[name]),
                             cold_mean_rounds=float(c[stance, rg.RG_INFO_POLISH_ROUNDS].mean()),
                             cold_fallback_share=float((c[stance, rg.RG_INFO_IPM_ITERS] > 0).mean()),
                             warm_mean_rounds=float(i[stance, rg.RG_INFO_POLISH_ROUNDS].mean()),
                             unverified=int(((i[:, rg.RG_INFO_STATUS] & (rg.RG_STATUS_POLISHED | rg.RG_STATUS_NO_STANCE)) == 0).sum()))
        res["tiled_equals_none_bitwise"] = bool(np.array_equal(f["tiled"], f["none"]))
        scale = np.maximum(1.0, np.abs(f["none"]).max(axis=1))
        rel = np.abs(f["gait"] - f["none"]).max(axis=1) / scale
        res["first_step_force_change"] = {
            "share_changed_over_1e-6_rel": float((rel > 1e-6).mean()),
            "median_rel_of_changed": float(np.median(rel[rel > 1e-6])) if (rel > 1e-6).any() else 0.0,
            "p90_rel_of_changed": float(np.percentile(rel[rel > 1e-6], 90)) if (rel > 1e-6).any() else 0.0,
            "max_rel": float(rel.max()),
            "per_schedule_share_changed": {s: float((rel[group == g] > 1e-6).mean()) for g, s in enumerate(SCHEDULES)}}
        out[str(n)] = res
        del arms
        torch.cuda.synchronize()
    return out


def controller(n, dev, mix, plan, horizon=10):
    st = synthetic.make_states(n, GHOST, seed=synthetic.SEED + 1)
    robot = SyntheticRobotBatch(GHOST, st, device=dev)
    ctl = BatchedMPCController(robot, robot.GetTimeSinceReset, horizon=horizon, contact_plan=plan)
    if mix:
        group = np.arange(n) % len(SCHEDULES)
        for g, name in enumerate(SCHEDULES):
            ctl.set_env_gait(schedule=name, env_ids=torch.from_numpy(np.flatnonzero(group == g)).to(dev))
        ctl.reset()

    def step():
        robot.time_since_reset.add_(0.01)
        ctl.step()
    return step, ctl


def step_section(dev, flush, reps):
    out = {}
    cases = [(n, mix, 10) for n in (1, 4096, 65536) for mix in (False, True)] + [(4096, False, 20)]
    for n, mix, h in cases:
        m = max(5, n) if mix else n
        arms = {plan: controller(m, dev, mix, plan, h) for plan in (False, True)}
        for step, _ in arms.values():
            for _ in range(4):
                step()
        torch.cuda.synchronize()
        times = {k: [] for k in arms}
        for rep in range(reps):
            for plan, (step, _) in arms.items():
                times[plan].append(timed(step, flush, rep))
        key = f"{'mix' if mix else 'trot'}_{m}_h{h}"
        out[key] = {"plan_off": dict(stats(times[False]), unverified=int(arms[False][1].unverified_count())),
                    "plan_on": dict(stats(times[True]), unverified=int(arms[True][1].unverified_count()))}
        out[key]["on_over_off"] = out[key]["plan_on"]["median_us"] / out[key]["plan_off"]["median_us"]
        del arms
        torch.cuda.synchronize()
    return out


def prologue_section(dev, reps):
    """Kernel time of the control step's prologue, plan off vs on (torch.profiler, CUDA activity, a run of its own):
    4096 envs (per-(env, leg) mapping) and 65536 envs (per-env mapping), trot, h = 10 and 20."""
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for n, h in ((4096, 10), (4096, 20), (65536, 10), (65536, 20)):
        for plan in (False, True):
            step, _ = controller(n, dev, False, plan, h)
            for _ in range(4):
                step()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(reps):
                    step()
                torch.cuda.synchronize()
            times = {}
            for ev in prof.events():
                if ev.device_type == torch.autograd.DeviceType.CUDA and "step_prologue" in ev.name:
                    times.setdefault(ev.name.split("(")[0].split("::")[-1], []).append(ev.device_time)
            out[f"trot_{n}_h{h}_plan_{'on' if plan else 'off'}"] = {k: stats(v) for k, v in times.items()}
            del step
            torch.cuda.synchronize()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("perf_contact_plan.py measures the B200 kernels: no CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)           # 2x the L2
    result = {"tool": "perf_contact_plan", "device": torch.cuda.get_device_name(dev),
              "name_power_limit_max_sm_clock": power_limit(), "reps": args.reps,
              "l2": "overwritten before every timed call"}
    result["solve"] = solve_section(dev, flush, args.reps)
    result["step"] = step_section(dev, flush, args.reps)
    result["prologue_kernel"] = prologue_section(dev, args.reps)
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
