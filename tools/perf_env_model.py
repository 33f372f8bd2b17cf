"""Cost of the per-env model (rg_mpc_env_model) in the stance solve: h = 10, trot, 4096 and 65536 envs.

Three arms, interleaved rep by rep so that clock and neighbour drift hit all of them alike:
  none     -- rg_mpc_build_solve_io (the model-free kernels)
  nominal  -- rg_mpc_build_solve_model with every env holding the workspace's own mass, inertia and friction: the
              same QPs, so the difference to `none` is the cost of the mechanism (112 B per env, one 3x3 inverse)
  random   -- every env its own body (mass 8-40 kg, SPD inertia) and friction (0.2-1.0 per row): a different workload,
              reported with its mean active-set round count, fallback-queue length and unverified envs
The L2 (126 MB) is overwritten between timed solves; each solve is timed with CUDA events.  Prints one JSON line
with the device name and power limit read in the same run.

  python tools/perf_env_model.py [--reps 30] [--out FILE]
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

from robot_gym import cuda as rg                                   # noqa: E402
from robot_gym.model.robots.descriptions import GHOST              # noqa: E402
from robot_gym.util import synthetic                               # noqa: E402

INPUTS = ("com_velocity_body", "base_rpy", "base_rpy_rate", "planned_contacts", "foot_positions_base", "command")


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("perf_env_model.py measures the B200 kernels: no CUDA device")
    dev = torch.device("cuda:0")
    ctrl = GHOST.GetCtrlConstants()
    p = rg.default_mpc_params(ctrl.MPC_BODY_MASS, ctrl.MPC_BODY_INERTIA, ctrl.MPC_BODY_HEIGHT, 10)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)           # 2x the L2
    result = {"tool": "perf_env_model", "device": torch.cuda.get_device_name(dev), "power_limit_and_max_sm_clock": power_limit(),
              "horizon": 10, "schedule": "trot", "reps": args.reps, "l2": "overwritten before every timed solve", "sizes": {}}
    for n in (4096, 65536):
        st = synthetic.make_states(n, GHOST, seed=synthetic.SEED)
        t = [torch.from_numpy(np.ascontiguousarray(getattr(st, k))).to(dev) for k in INPUTS]
        ws = rg.MpcWorkspace(p, device=dev, max_envs=n)
        f = torch.empty((n, 12), dtype=torch.float32, device=dev)
        info = torch.empty((n, 4), dtype=torch.int32, device=dev)
        f64 = torch.float64
        nominal = dict(mass=torch.full((n,), p.mass, dtype=f64, device=dev),
                       inertia=torch.tensor(list(p.inertia), dtype=f64, device=dev).repeat(n, 1),
                       friction_coeffs=torch.tensor(list(p.friction_coeffs), dtype=f64, device=dev).repeat(n, 1))
        rng = np.random.default_rng(3)
        a = rng.normal(size=(n, 3, 3)) * 0.05
        inertia = np.einsum("nij,nkj->nik", a, a) + np.stack([np.diag(d) for d in rng.uniform(0.05, 0.8, (n, 3))])
        random = dict(mass=torch.from_numpy(rng.uniform(8.0, 40.0, n)).to(dev),
                      inertia=torch.from_numpy(inertia.reshape(n, 9)).to(dev),
                      friction_coeffs=torch.from_numpy(rng.uniform(0.2, 1.0, (n, 4))).to(dev))
        arms = {"none": None, "nominal": nominal, "random": random}
        run = lambda model: rg.mpc_build_solve(ws, *t, contact_forces=f, solve_info=info, env_model=model)
        for model in arms.values():                                         # warm-up: module load, attributes
            for _ in range(3):
                run(model)
        torch.cuda.synchronize()
        times = {k: [] for k in arms}
        stats = {}
        for rep in range(args.reps):
            for name, model in arms.items():
                flush.fill_(rep & 255)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run(model)
                e1.record()
                e1.synchronize()
                times[name].append(e0.elapsed_time(e1) * 1e3)
                if rep == 0:
                    i = info.cpu().numpy()
                    status = i[:, rg.RG_INFO_STATUS]
                    stats[name] = {
                        "mean_active_set_rounds": float(i[:, rg.RG_INFO_POLISH_ROUNDS].mean()),
                        "fallback_queue": int(((status & rg.RG_STATUS_ACTIVE_SET_ONLY) == 0).sum()),
                        "unverified": int(((status & (rg.RG_STATUS_POLISHED | rg.RG_STATUS_NO_STANCE)) == 0).sum()),
                        "bad_model": int(((status & rg.RG_STATUS_BAD_MODEL) != 0).sum())}
        summary = {}
        for name, v in times.items():
            v = np.array(v)
            summary[name] = {"median_us": float(np.median(v)), "p10_us": float(np.percentile(v, 10)),
                             "p90_us": float(np.percentile(v, 90)), "solves_per_s": float(n / (np.median(v) * 1e-6)), **stats[name]}
        summary["nominal_over_none"] = summary["nominal"]["median_us"] / summary["none"]["median_us"]
        summary["random_over_none"] = summary["random"]["median_us"] / summary["none"]["median_us"]
        result["sizes"][str(n)] = summary
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
