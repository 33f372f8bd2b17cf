"""Cost and effect of planning the stance QP over predicted footholds (rg_mpc_build_solve_footholds,
rg_control_step_footholds).

solve: the stance solve alone, h = 10, 4096 and 65536 envs whose gaits mix trot, pace, bound, walk and stand.  The
  inputs, the gait schedule and the predicted footholds are those of one control step of BatchedMPCController(
  contact_plan=True, foothold_plan=True) on synthetic states.  Each arm is warm-started from its own previous solve of
  the same inputs:
    schedule  -- the gait schedule alone (rg_mpc_build_solve_schedule)
    held      -- the schedule and a foothold plan whose rows are the current feet: the same QPs, so the difference to
                 `schedule` is the cost of the mechanism
    predicted -- the schedule and the predicted footholds: the new workload
  per arm: median / p10 / p90 time, mean active-set rounds, the share of envs that ran interior-point iterations (the
  fallback queue of the two-kernel solve), the unverified count; and the share of envs whose first-step forces change
  by more than 1e-6 relative against `schedule`.
step: the warm-started control step (BatchedMPCController, one CUDA graph per step at 1 env) on the five-schedule mix,
  contact plan vs contact plan + footholds, at 5, 4096 and 65536 envs, h = 10; and at 4096 envs with h = 20.
Arms are interleaved rep by rep; the L2 (126 MB) is overwritten before every timed call; CUDA events around the whole
Python call.  Prints one JSON line with the device name and power limit read in the same run.

  python tools/perf_foothold_plan.py [--reps 40] [--out FILE]
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


def mixed_controller(n, dev, horizon=10, **kw):
    st = synthetic.make_states(n, GHOST, seed=synthetic.SEED + 1)
    robot = SyntheticRobotBatch(GHOST, st, device=dev)
    ctl = BatchedMPCController(robot, robot.GetTimeSinceReset, horizon=horizon, contact_plan=True, **kw)
    group = np.arange(n) % len(SCHEDULES)
    for g, name in enumerate(SCHEDULES):
        ctl.set_env_gait(schedule=name, env_ids=torch.from_numpy(np.flatnonzero(group == g)).to(dev))
    ctl.reset()
    ctl.command.copy_(torch.from_numpy(st.command).to(dev))
    return st, robot, ctl, group


def solve_section(dev, flush, reps):
    out = {}
    h = 10
    for n in (4096, 65536):
        st, robot, ctl, group = mixed_controller(n, dev, h, foothold_plan=True)
        ctl.get_action()
        torch.cuda.synchronize()
        up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        feet = up(st.foot_positions_base)
        inputs = [ctl.com_velocity_body.clone(), up(st.base_rpy), up(st.base_rpy_rate), None, feet, ctl.command.clone()]
        sched = ctl.mpc_contact_schedule.clone()
        plans = {"schedule": None, "held": feet.view(n, 1, 12).repeat(1, h, 1).contiguous(),
                 "predicted": ctl.mpc_foothold_plan.clone()}
        del ctl, robot
        ctrl = GHOST.GetCtrlConstants()
        arms = {}
        for name, plan in plans.items():
            ws = rg.MpcWorkspace(rg.default_mpc_params(ctrl.MPC_BODY_MASS, ctrl.MPC_BODY_INERTIA, ctrl.MPC_BODY_HEIGHT, h),
                                 device=dev, max_envs=n)
            act = rg.new_active_set(n, h, dev)
            forces = torch.empty((n, 12), dtype=torch.float32, device=dev)
            info = torch.empty((n, 4), dtype=torch.int32, device=dev)

            def run(ws=ws, act=act, plan=plan, forces=forces, info=info):
                rg.mpc_build_solve(ws, *inputs, contact_forces=forces, solve_info=info, active_set=act, zero_yaw=True,
                                   contact_schedule=sched, foothold_plan=plan)
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
        res["held_over_schedule"] = res["held"]["median_us"] / res["schedule"]["median_us"]
        res["predicted_over_schedule"] = res["predicted"]["median_us"] / res["schedule"]["median_us"]
        res["held_equals_schedule_bitwise"] = bool(np.array_equal(f["held"], f["schedule"]))
        scale = np.maximum(1.0, np.abs(f["schedule"]).max(axis=1))
        rel = np.abs(f["predicted"] - f["schedule"]).max(axis=1) / scale
        res["first_step_force_change"] = {
            "share_changed_over_1e-6_rel": float((rel > 1e-6).mean()),
            "median_rel_of_changed": float(np.median(rel[rel > 1e-6])) if (rel > 1e-6).any() else 0.0,
            "max_rel": float(rel.max()),
            "per_schedule_share_changed": {s: float((rel[group == g] > 1e-6).mean()) for g, s in enumerate(SCHEDULES)}}
        out[str(n)] = res
        del arms
        torch.cuda.synchronize()
    return out


def step_section(dev, flush, reps):
    out = {}
    for n, h in ((5, 10), (4096, 10), (65536, 10), (4096, 20)):
        arms = {}
        for feet in (False, True):
            st, robot, ctl, _ = mixed_controller(n, dev, h, foothold_plan=feet)

            def step(robot=robot, ctl=ctl):
                robot.time_since_reset.add_(0.01)
                ctl.step()
            arms[feet] = (step, ctl)
        for step, _ in arms.values():
            for _ in range(4):
                step()
        torch.cuda.synchronize()
        times = {k: [] for k in arms}
        for rep in range(reps):
            for feet, (step, _) in arms.items():
                times[feet].append(timed(step, flush, rep))
        key = f"mix_{n}_h{h}"
        out[key] = {"plan": dict(stats(times[False]), unverified=int(arms[False][1].unverified_count())),
                    "plan_footholds": dict(stats(times[True]), unverified=int(arms[True][1].unverified_count()))}
        out[key]["footholds_over_plan"] = out[key]["plan_footholds"]["median_us"] / out[key]["plan"]["median_us"]
        del arms
        torch.cuda.synchronize()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("perf_foothold_plan.py measures the B200 kernels: no CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)           # 2x the L2
    result = {"tool": "perf_foothold_plan", "device": torch.cuda.get_device_name(dev),
              "name_power_limit_max_sm_clock": power_limit(), "reps": args.reps,
              "l2": "overwritten before every timed call"}
    result["solve"] = solve_section(dev, flush, args.reps)
    result["step"] = step_section(dev, flush, args.reps)
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
