"""Cost and payoff of the per-env gait (rg_gait_env_params) in the control step: h = 10, warm-started stance QPs.

Per batch size, arms interleaved rep by rep so that clock and neighbour drift hit all of them alike:
  none     -- BatchedMPCController on the trot workspace, no gait (rg_control_step: the gait-free prologue)
  nominal  -- the same controller with set_env_gait() holding the workspace's own rows (rg_control_step_env): the same
              steps, so the difference to `none` is the cost of the mechanism (112 B per env-step, the row vote)
  mixed    -- ONE controller whose envs run trot, pace, bound, walk and stand interleaved env by env
  five     -- five controllers, one per schedule, each on a fifth of the envs, stepped back to back: what a mixed batch
              took before the per-env gait.  `mixed` and `five` solve the same QPs.
Sizes: 1 env (none / nominal; one CUDA-graph launch per step), and 5 envs for mixed / five (one env per schedule,
five graphs), 4096 and 65536 envs (4095 and 65535 for mixed / five).  The clock advances 10 ms per rep, so the
gait walks through its cycle.  The L2 (126 MB) is overwritten before every timed step; each step is timed with CUDA
events around the whole Python call.  Prints one JSON line with the device name and power limit read in the same run.

  python tools/perf_env_gait.py [--reps 40] [--out FILE]
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

from robot_gym.controllers.mpc.batched_mpc_controller import BatchedMPCController   # noqa: E402
from robot_gym.model.robots.descriptions import GAIT_SCHEDULES, GHOST, with_gait    # noqa: E402
from robot_gym.model.robots.synthetic_robot import SyntheticRobotBatch               # noqa: E402
from robot_gym.util import synthetic                                                 # noqa: E402

SCHEDULES = tuple(GAIT_SCHEDULES)


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


class Arm:
    """One or more (robot, controller) pairs stepped back to back as one timed unit."""

    def __init__(self, pairs):
        self.pairs = pairs

    def step(self):
        for robot, ctl in self.pairs:
            robot.time_since_reset.add_(0.01)      # in place: the captured graphs keep their pointers
            ctl.step()

    def unverified(self):
        return int(sum(int(ctl.unverified_count()) for _, ctl in self.pairs))


def controller(desc, st, dev):
    robot = SyntheticRobotBatch(desc, st, device=dev)
    return robot, BatchedMPCController(robot, robot.GetTimeSinceReset)


def build_arms(n, dev):
    arms = {}
    st = synthetic.make_states(n, GHOST, seed=synthetic.SEED)
    arms["none"] = Arm([controller(GHOST, st, dev)])
    robot, ctl = controller(GHOST, st, dev)
    ctl.set_env_gait()
    arms["nominal"] = Arm([(robot, ctl)])
    m = max(5, n - n % 5)
    group = np.arange(m) % 5
    st = synthetic.make_states(m, GHOST, seed=synthetic.SEED + 1)
    robot, ctl = controller(GHOST, st, dev)
    for g, name in enumerate(SCHEDULES):
        ctl.set_env_gait(schedule=name, env_ids=torch.from_numpy(np.flatnonzero(group == g)).to(dev))
    ctl.reset()
    arms["mixed"] = Arm([(robot, ctl)])
    arms["five"] = Arm([controller(with_gait(GHOST, name), _rows(st, group == g), dev)
                        for g, name in enumerate(SCHEDULES)])
    return arms, m


def _rows(st, mask):
    idx = np.flatnonzero(mask)
    return type(st)(**{k: v[idx] for k, v in vars(st).items()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("perf_env_gait.py measures the B200 kernels: no CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)           # 2x the L2
    result = {"tool": "perf_env_gait", "device": torch.cuda.get_device_name(dev), "power_limit_and_max_sm_clock": power_limit(),
              "horizon": 10, "warm_start": True, "reps": args.reps, "l2": "overwritten before every timed step",
              "sizes": {}}
    for n in (1, 4096, 65536):
        arms, m = build_arms(n, dev)
        for arm in arms.values():                                           # warm-up: graphs, module load
            for _ in range(4):
                arm.step()
        torch.cuda.synchronize()
        times = {k: [] for k in arms}
        for rep in range(args.reps):
            for name, arm in arms.items():
                flush.fill_(rep & 255)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                arm.step()
                e1.record()
                e1.synchronize()
                times[name].append(e0.elapsed_time(e1) * 1e3)
        summary = {"envs_none_nominal": n, "envs_mixed_five": m}
        for name, v in times.items():
            v = np.array(v)
            summary[name] = {"median_us": float(np.median(v)), "p10_us": float(np.percentile(v, 10)),
                             "p90_us": float(np.percentile(v, 90)), "unverified_last_step": arms[name].unverified()}
        summary["nominal_over_none"] = summary["nominal"]["median_us"] / summary["none"]["median_us"]
        summary["five_over_mixed"] = summary["five"]["median_us"] / summary["mixed"]["median_us"]
        result["sizes"][str(n)] = summary
        del arms
        torch.cuda.synchronize()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
