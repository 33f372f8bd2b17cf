#!/usr/bin/env python
"""Benchmark of the batched MPC stance solve (BASELINE.json metric: MPC stance solves/sec).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle port on host cores
    python bench.py ... --dump-outputs DIR                   # also save what the last timed step computed

--dump-outputs writes the arrays the timed step hands its caller, for the whole job's batch in env order:
DIR/contact_forces.npy (float32 [envs, 12]) and DIR/solve_info.npy (the int32 [envs, 4] solve_info as
float64), 80 bytes per env (2.6 MB at 8 GPUs); the CPU arm writes its contact_forces.npy alone.  The inputs
are seeded, so two builds run with the same arguments can be compared output for output.

A "step" is one pass of rg_mpc_build_solve over one batch of synthetic robot states: BASELINE
config[1] -- 4096 envs per GPU, horizon 10, 4 legs, friction pyramid (weak scaling: every rank
solves its own contiguous 4096-env shard of one seeded, prefix-stable global batch -- rank 0 solves
the same 4096 envs at every N; the only collective is one all-gather of the 8-float rollout
statistics per timed window).  Prints ONE JSON line (rank 0).

  value        whole-job solves/s with the inputs resident in HBM (CUDA events around each step)
  e2e          the same metric through the public API from HOST buffers: pinned host -> device copy
               of the step's inputs, solve, device -> host read of the forces, all inside the timing
               (copies double-buffered on two copy streams; the solves stay serialised on one stream)
  roofline     HBM roofline of the solve kernel (algorithmic 156 B/solve; this path is NOT HBM-bound,
               the fraction is reported as it is) + roofline_fp64: executed-FLOP fraction of the
               measured FP64 FMA peak, the resource that actually binds
  cpu_baseline the oracle port (oracle/c/mpc_oracle.c, dense formulation + dense interior point + polish)
               on the host cores; reference parity is unpinned and motion_imitation/OSQP cannot run
               offline, so kind = "port"
  config5      BASELINE config[4]: 2^20 envs sharded contiguously over the N ranks (strong scaling), same kernel
  latency      p50 / p99 of one full control step (BatchedMPCController.step: gait + estimator + swing + IK + MPC +
               pack) for 1, 4096 and 65536 envs, CUDA events, cold (every QP from scratch) and warm-started
  config4      horizon {5, 10, 20} x schedule {trot, pace, bound, walk} at 65536 envs (BASELINE config[3])
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(REPO, "robot-gym_b200"))
sys.path.insert(0, REPO)

ENVS_PER_GPU = 4096
HORIZON = 10
METRIC = "mpc_stance_solves_per_sec"
UNIT = "solves/s"
ALGO_BYTES_PER_SOLVE = 156            # SURVEY.md 8(d): 108 B in + 48 B out
# algorithmic FLOPs per solve in the dense-reference formulation (SURVEY.md 8(d)):
# Hessian 3744 h^3 + gradient + Cholesky 576 h^3 + 0.033 MFLOP per solver iteration at h = 10
ALGO_FLOPS_FIXED = 4.36e6
ALGO_FLOPS_PER_ITER = 0.033e6
CONFIG5_ENVS = 1 << 20                # BASELINE config[4]


def _measured_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def _dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def _config(n_gpus, extra=None):
    cfg = {"workload": f"BASELINE config[1]: {ENVS_PER_GPU} synthetic quadruped states per GPU, batched MPC stance QP "
                       f"(horizon {HORIZON}, 4 legs, friction pyramid), ghost parameters, trot contact schedule",
           "envs_per_gpu": ENVS_PER_GPU, "global_envs": ENVS_PER_GPU * n_gpus, "horizon": HORIZON,
           "sharding": "contiguous env shards of one seeded global batch; all-gather of 8 rollout stats per window",
           "l2": "flushed between timed steps (256 MiB device memset, outside the timed interval)"}
    cfg.update(extra or {})
    return cfg


# ------------------------------------------------------------------------------------------------ CPU arm
def run_reference(args):
    """`--impl reference`: the CPU implementation of the path (oracle port; the reference's own
    motion_imitation/OSQP/PyBullet stack cannot be installed offline) on all host threads."""
    rank, world, _ = _dist_env()
    if rank != 0:
        return
    from oracle import c_oracle, convex_mpc
    from robot_gym.model.robots.descriptions import GHOST
    from robot_gym.util import synthetic
    ctrl = GHOST.GetCtrlConstants()
    cores = os.cpu_count() or 1
    n = ENVS_PER_GPU
    states = synthetic.make_states_sharded(0, n, GHOST)       # rank 0's shard of the GPU arm, whatever --gpus says
    mp = convex_mpc.MpcParams(horizon=HORIZON, mass=ctrl.MPC_BODY_MASS, inertia=tuple(ctrl.MPC_BODY_INERTIA))
    for _ in range(max(1, min(args.warmup, 2))):
        c_oracle.solve_batch(mp, states.slice(0, 512), ctrl.MPC_BODY_HEIGHT, n_threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        forces, _, _ = c_oracle.solve_batch(mp, states, ctrl.MPC_BODY_HEIGHT, n_threads=cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        _write_outputs(args.dump_outputs, {"contact_forces": forces})
    value = n * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": _config(args.gpus), "note": "CPU arm: rank 0 alone processes one 4096-env shard per step",
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{n} envs per step x {args.steps} steps, oracle/c/mpc_oracle.c (dense condensed "
                                       "build + dense Mehrotra interior point + active-set polish), one pthread per host core; "
                                       "NOT motion_imitation/OSQP (unavailable offline, parity unpinned)"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
def run_gpu(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from robot_gym import cuda as rg
    from robot_gym.controllers.mpc.batched_mpc_controller import (BatchedMPCController, gather_rollout_stats,
                                                                  reduce_rollout_stats, shard_bounds)
    from robot_gym.model.robots.descriptions import GHOST
    from robot_gym.model.robots.synthetic_robot import SyntheticRobotBatch
    from robot_gym.util import synthetic

    rank, world, local = _dist_env()
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: there is no CPU fallback for the solve kernels")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.gpus != world:
        raise RuntimeError(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch N>1 with torch.distributed.run")
    rg.load()                                  # fails loudly if librg_cuda.so is missing

    ctrl = GHOST.GetCtrlConstants()
    n_global = ENVS_PER_GPU * world
    lo, hi = shard_bounds(n_global, rank, world)
    states = synthetic.make_states_sharded(lo, hi, GHOST)              # prefix-stable: the shard does not depend on N
    n = hi - lo
    params = rg.default_mpc_params(ctrl.MPC_BODY_MASS, ctrl.MPC_BODY_INERTIA, ctrl.MPC_BODY_HEIGHT, HORIZON)
    ws = rg.MpcWorkspace(params, device=dev, max_envs=max(n, CONFIG5_ENVS // world + 1))

    host_names = ("com_velocity_body", "base_rpy", "base_rpy_rate", "planned_contacts", "foot_positions_base", "command")
    # The six input arrays live back to back in ONE pinned host allocation (and one device allocation for the
    # e2e arm), 256-byte aligned: the public API still receives six tensors (views), but a step needs one
    # host->device copy instead of six.
    arrays = {k: np.ascontiguousarray(getattr(states, k)) for k in host_names}
    offsets, total_bytes = {}, 0
    for k, a in arrays.items():
        offsets[k] = total_bytes
        total_bytes += (a.nbytes + 255) // 256 * 256
    host_pack = torch.empty(max(total_bytes, 256), dtype=torch.uint8).pin_memory()
    e2e_pack = torch.empty(max(total_bytes, 256), dtype=torch.uint8, device=dev)

    def views(pack):
        out = {}
        for k, a in arrays.items():
            flat = pack[offsets[k]:offsets[k] + a.nbytes]
            out[k] = flat.view(torch.from_numpy(a).dtype).view(a.shape)
        return out

    host = views(host_pack)
    for k, a in arrays.items():
        host[k].copy_(torch.from_numpy(a))
    e2e_in = views(e2e_pack)
    dev_in = {k: v.to(dev) for k, v in host.items()}
    forces = torch.empty((n, 12), dtype=torch.float32, device=dev)
    info = torch.empty((n, 4), dtype=torch.int32, device=dev)
    forces_host = torch.empty((n, 12), dtype=torch.float32).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def solve(inputs):
        rg.mpc_build_solve(ws, inputs["com_velocity_body"], inputs["base_rpy"], inputs["base_rpy_rate"],
                           inputs["planned_contacts"], inputs["foot_positions_base"], inputs["command"],
                           contact_forces=forces, solve_info=info)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks / throttle reasons are sampled from before the warm-up until after the e2e loop: the timed
    # regions last tens of milliseconds, shorter than one nvidia-smi sampling period
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()

    # ---- warm-up
    for _ in range(max(3, args.warmup)):
        solve(dev_in)
    barrier()

    # ---- timed: K steps, device-resident inputs, CUDA events on the launching (current) stream
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches0 = rg.launch_count()
    barrier()
    t_wall0 = time.perf_counter()
    for a, b in ev:
        flush.zero_()                       # L2 flush, outside the timed interval
        a.record()
        solve(dev_in)
        b.record()
    stats = None
    if world > 1:
        # the path's only collective: one all-gather of the small rollout-statistics vector
        s_local = _stats_vector(torch, rg, info, forces, n)
        stats = gather_rollout_stats(s_local)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = rg.launch_count() - launches0
    # the last timed step's outputs, copied now: the e2e arm below writes into the same buffers
    dump = None
    if args.dump_outputs:
        dump = {"contact_forces": _gather_rows(torch, dist, forces.clone(), world),
                "solve_info": _gather_rows(torch, dist, info.to(torch.float64), world)}
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    rank_ms = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
    if world > 1:
        dist.all_gather(rank_ms, total_ms / args.steps)           # per-rank mean step time, for the record
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    else:
        rank_ms = [total_ms / args.steps]
    rank_ms = [float(t.item()) for t in rank_ms]
    total_ms = float(total_ms.item())
    value = n_global * args.steps / (total_ms * 1e-3)

    # ---- e2e: host buffers in, host forces out, copies inside the timed region.  Every step copies its inputs from pinned
    # host memory and its forces back; the copies run on two copy streams with double-buffered device / host buffers, so the
    # step-(k+1) upload and the step-(k-1) download overlap the step-k solve.  The solves themselves stay serialised on the
    # compute stream (one batch at a time, as a control loop would issue them).
    comp = torch.cuda.current_stream()
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    packs = [e2e_pack, torch.empty_like(e2e_pack)]
    e2e_views = [views(pk) for pk in packs]
    f_dev = [forces, torch.empty_like(forces)]
    f_host = [forces_host, torch.empty_like(forces_host).pin_memory()]
    ev_up = [torch.cuda.Event() for _ in range(2)]        # upload of buffer b finished
    ev_solved = [torch.cuda.Event() for _ in range(2)]    # solve that used buffer b finished (inputs free, forces ready)
    ev_down = [torch.cuda.Event() for _ in range(2)]      # download of forces b finished (device forces b free)
    for b in range(2):
        ev_solved[b].record(comp); ev_down[b].record(comp)

    def e2e_step(k):
        b = k & 1
        s_in.wait_event(ev_solved[b])                       # the solve two steps back has read these inputs
        with torch.cuda.stream(s_in):
            packs[b].copy_(host_pack, non_blocking=True)    # pinned host -> device, this step's inputs
            ev_up[b].record(s_in)
        comp.wait_event(ev_up[b])
        comp.wait_event(ev_down[b])                         # forces b of two steps back are on the host
        i = e2e_views[b]
        rg.mpc_build_solve(ws, i["com_velocity_body"], i["base_rpy"], i["base_rpy_rate"], i["planned_contacts"],
                           i["foot_positions_base"], i["command"], contact_forces=f_dev[b], solve_info=info)
        ev_solved[b].record(comp)
        s_out.wait_event(ev_solved[b])
        with torch.cuda.stream(s_out):
            f_host[b].copy_(f_dev[b], non_blocking=True)    # device -> pinned host, this step's result
            ev_down[b].record(s_out)

    for k in range(4):
        e2e_step(k)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(comp)
    for k in range(args.steps):
        e2e_step(k)
    comp.wait_event(ev_down[0]); comp.wait_event(ev_down[1])    # the timed interval ends when the last forces are on the host
    e1.record(comp)
    barrier()
    e2e_wall = time.perf_counter() - t0
    e2e_ms = torch.tensor([max(e0.elapsed_time(e1), e2e_wall * 1e3)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = n_global * args.steps / (float(e2e_ms.item()) * 1e-3)
    # keep the GPU busy for a few sampling periods so the clock record is taken under load
    t_end = time.perf_counter() + 0.6
    while time.perf_counter() < t_end:
        solve(dev_in)
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    h2d = sum(v.numel() * v.element_size() for v in host.values()) * world      # payload (the packed copy adds < 2 KB of alignment padding)
    d2h = forces_host.numel() * forces_host.element_size() * world

    # ---- solver statistics (whole job)
    s_local = _stats_vector(torch, rg, info, forces, n)
    gathered = gather_rollout_stats(s_local) if world > 1 else s_local.unsqueeze(0)
    total = reduce_rollout_stats(gathered).cpu().numpy()
    iters_mean = float(total[1] / total[0])
    config5 = _config5(torch, dist, rg, synthetic, GHOST, ws, dev, rank, world, barrier)     # every rank takes part

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- rank 0 only: roofline numbers, FMA peaks, CPU baseline, latency and config-4 tables
    peaks, peak_kind = _measured_peaks()
    kernel_ms = statistics.mean(step_ms)          # one kernel launch per step: the step time IS the kernel time
    algo_bytes = ALGO_BYTES_PER_SOLVE * n
    achieved_gbs = algo_bytes / (kernel_ms * 1e-3) / 1e9
    traffic, executed_per_env = None, None
    prof_name = None
    for prof_name in ("r02_mpc_ncu_summary.json", "r01_mpc_ncu_summary.json"):      # newest committed capture of this kernel
        prof = os.path.join(REPO, "profiles", prof_name)
        if os.path.exists(prof):
            with open(prof) as fh:
                summary = json.load(fh)
            traffic = summary.get("dram_bytes_per_launch")
            executed_per_env = summary.get("executed_fp64_flops_per_env")
            break
    roofline = {"bound": "hbm", "achieved": achieved_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved_gbs / peaks["hbm_gbs"], "traffic": traffic, "traffic_source": f"profiles/{prof_name}",
                "peak_kind": f"of {peak_kind}", "kernel": "mpc_solve_kernel<10, lean>", "kernel_ms": kernel_ms,
                "algorithmic_bytes_per_launch": algo_bytes,
                "note": "the solve keeps the whole QP on chip: HBM is not the binding resource (see roofline_fp64); kernel_ms is "
                        "the step (lean kernel + the fallback kernel, whose queue is empty on this batch)"}
    fp64_peak = rg.measure_fma_peak(True)
    fp32_peak = rg.measure_fma_peak(False)
    polish_mean = float(total[3] / total[0])
    algo_flops = (ALGO_FLOPS_FIXED + ALGO_FLOPS_PER_ITER * (iters_mean + polish_mean)) * n
    roofline_fp64 = {"bound": "fp64 fma", "dense_equivalent_tflops": algo_flops / (kernel_ms * 1e-3) / 1e12,
                     "peak_fp64_tflops_measured": fp64_peak, "peak_fp32_tflops_measured": fp32_peak,
                     "executed_flop_per_solve_ncu": executed_per_env,
                     "executed_tflops": None if executed_per_env is None else executed_per_env * n / (kernel_ms * 1e-3) / 1e12,
                     "executed_frac_of_fp64_peak": None if executed_per_env is None else executed_per_env * n / (kernel_ms * 1e-3) / 1e12 / fp64_peak,
                     "note": "dense_equivalent_tflops = the dense-reference FLOP count (SURVEY.md 8d) over the kernel time: a rate the "
                             "reference formulation would need, NOT a utilisation (the closed-form / Woodbury / active-set kernel "
                             "executes ~14x fewer FLOPs); executed_* uses the per-solve FP64 instruction count of the committed ncu "
                             "capture: the kernel is bound by dependent-instruction latency, not by the FP64 pipe"}

    cpu = _cpu_baseline(states, ctrl)
    latency = _latency_table(torch, rg, BatchedMPCController, SyntheticRobotBatch, synthetic, GHOST, dev)
    config4 = _config4_table(torch, rg, synthetic, dev)
    control = latency.pop("_control_step", None)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": _config(world),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "roofline_fp64": roofline_fp64,
            "cpu_baseline": cpu,
            "solver": {"ipm_iters_mean": iters_mean, "ipm_iters_max": float(total[2]), "polish_rounds_mean": polish_mean,
                       "polished_fraction": float(total[4] / total[0]), "numeric_flags": float(total[6])},
            "kernel_ms_per_rank": {"min": min(rank_ms), "max": max(rank_ms), "all": rank_ms},
            "solve_latency": {"solve_p50_ms": statistics.median(step_ms), "solve_max_ms": max(step_ms), "envs": n},
            "latency": latency, "control_step": control, "config4": config4, "config5": config5,
            "wall_s_timed_region": t_wall}
    if dump is not None:
        _write_outputs(args.dump_outputs, {k: v.cpu().numpy() for k, v in dump.items()})
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def _gather_rows(torch, dist, t, world):
    """Rank shards (equal row counts) concatenated in rank order, i.e. in global env order."""
    if world == 1:
        return t
    parts = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(parts, t)
    return torch.cat(parts)


def _write_outputs(out_dir, arrays):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def _stats_vector(torch, rg, info, forces, n):
    status = info[:, rg.RG_INFO_STATUS]
    iters = info[:, rg.RG_INFO_IPM_ITERS].to(torch.float64)
    return torch.stack([
        torch.tensor(float(n), dtype=torch.float64, device=info.device), iters.sum(), iters.max(),
        info[:, rg.RG_INFO_POLISH_ROUNDS].to(torch.float64).sum(),
        ((status & rg.RG_STATUS_POLISHED) != 0).to(torch.float64).sum(),
        ((status & rg.RG_STATUS_NO_STANCE) != 0).to(torch.float64).sum(),
        ((status & rg.RG_STATUS_NUMERIC) != 0).to(torch.float64).sum(),
        forces.abs().to(torch.float64).sum()])


def _cpu_baseline(states, ctrl):
    """The oracle port timed on this box's host cores on the same 4096-env batch (bounded sample)."""
    try:
        from oracle import c_oracle, convex_mpc
        cores = os.cpu_count() or 1
        mp = convex_mpc.MpcParams(horizon=HORIZON, mass=ctrl.MPC_BODY_MASS, inertia=tuple(ctrl.MPC_BODY_INERTIA))
        c_oracle.solve_batch(mp, states.slice(0, 256), ctrl.MPC_BODY_HEIGHT, n_threads=cores)
        best = 0.0
        reps = 2
        for _ in range(reps):
            t0 = time.perf_counter()
            c_oracle.solve_batch(mp, states, ctrl.MPC_BODY_HEIGHT, n_threads=cores)
            best = max(best, len(states) / (time.perf_counter() - t0))
        return {"value": best, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"the same {len(states)}-env batch, best of {reps} passes, oracle/c/mpc_oracle.c on {cores} "
                          "pthreads (restated CPU oracle, NOT motion_imitation/OSQP which is unavailable offline)"}
    except Exception as exc:   # the baseline is a reported number, never a reason to lose the GPU measurement
        return {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {exc}"}


def _pct(values, q):
    v = sorted(values)
    return v[min(len(v) - 1, int(round(q * (len(v) - 1))))]


def _config5(torch, dist, rg, synthetic, desc, ws, dev, rank, world, barrier):
    """BASELINE config[4]: 2^20 envs sharded contiguously over the ranks (strong scaling), no collective on the data
    path.  Every rank times its shard with CUDA events; the job time is the MAX over ranks."""
    try:
        base, rem = divmod(CONFIG5_ENVS, world)
        lo = rank * base + min(rank, rem)
        hi = lo + base + (1 if rank < rem else 0)
        st = synthetic.make_states_sharded(lo, hi, desc)
        up = lambda a: torch.from_numpy(a).to(dev)
        ins = [up(getattr(st, k)) for k in ("com_velocity_body", "base_rpy", "base_rpy_rate", "planned_contacts",
                                             "foot_positions_base", "command")]
        n = hi - lo
        forces = torch.empty((n, 12), dtype=torch.float32, device=dev)
        info = torch.empty((n, 4), dtype=torch.int32, device=dev)
        reps = 3
        for _ in range(2):
            rg.mpc_build_solve(ws, *ins, contact_forces=forces, solve_info=info)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            rg.mpc_build_solve(ws, *ins, contact_forces=forces, solve_info=info)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device=dev)
        all_ms = [torch.zeros_like(ms) for _ in range(world)]
        if world > 1:
            dist.all_gather(all_ms, ms)
        else:
            all_ms = [ms]
        all_ms = [float(t.item()) for t in all_ms]
        polished = ((info[:, rg.RG_INFO_STATUS] & (rg.RG_STATUS_POLISHED | rg.RG_STATUS_NO_STANCE)) != 0).double().mean().item()
        return {"workload": "BASELINE config[4]: 2^20 synthetic envs sharded contiguously over the ranks, horizon 10, trot",
                "global_envs": CONFIG5_ENVS, "envs_per_gpu": base, "scaling": "strong", "ms": max(all_ms),
                "ms_per_rank": all_ms, "solves_per_s": CONFIG5_ENVS / (max(all_ms) * 1e-3), "reps": reps,
                "verified_fraction_rank0": polished}
    except Exception as exc:   # never lose the headline measurement to an extra
        return {"error": repr(exc)}


def _latency_table(torch, rg, Controller, RobotBatch, synthetic, desc, dev):
    """SURVEY.md 8(d) latency metric: p50 / p99 of ONE full control step (gait + estimator + swing + IK + MPC + force->torque
    + pack = BatchedMPCController.step, the public API) for 1, 4096 and 65536 envs; CUDA events on the launching stream,
    20 warm-ups, >= 200 timed steps (60 at 65536).  'cold' solves every stance QP from scratch (what the reference does);
    'warm' seeds it with the active set the env verified one step earlier (the controller's default).  The synthetic state
    source has no physics, so 'warm' is the best case of the warm start, not a rollout average."""
    out = {"unit": "ms", "what": "BatchedMPCController.step(), CUDA events, per step"}
    try:
        for n, reps in ((1, 300), (4096, 200), (65536, 60)):
            for key, warm in (("cold", False), ("warm", True)):
                robot = RobotBatch(desc, synthetic.make_states_sharded(0, n, desc), device=dev)
                ctl = Controller(robot, robot.GetTimeSinceReset, warm_start=warm)
                # the controller latched reset_time = clock at construction, which would freeze every env at gait time 0
                # (all four legs in stance, the hardest pattern): run on the states' own gait clocks (t0 ~ U(0, 0.5 s))
                ctl.reset_time.zero_()
                ctl.command.copy_(torch.from_numpy(synthetic.make_states_sharded(0, n, desc).command).to(dev))
                for _ in range(20):
                    ctl.step()
                torch.cuda.synchronize()
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
                for a, b in ev:
                    a.record()
                    ctl.step()
                    b.record()
                torch.cuda.synchronize()
                t = [a.elapsed_time(b) for a, b in ev]
                out[f"n{n}_{key}_p50_ms"] = _pct(t, 0.5)
                out[f"n{n}_{key}_p99_ms"] = _pct(t, 0.99)
                if n == 65536:
                    rounds = float(ctl.solve_info[:, rg.RG_INFO_POLISH_ROUNDS].to(torch.float64).mean())
                    out.setdefault("_control_step", {"envs": n, "launches_per_step": 4,
                                                     "workload": "BASELINE config[2]: full control step, 65536 envs, 1 GPU"})
                    out["_control_step"][key] = {"p50_ms": _pct(t, 0.5), "p99_ms": _pct(t, 0.99), "reps": reps,
                                                 "env_steps_per_s": n / (_pct(t, 0.5) * 1e-3), "active_set_rounds_mean": rounds}
                del ctl, robot
        cs = out.get("_control_step")
        if cs:
            cs["p50_ms"], cs["env_steps_per_s"] = cs["cold"]["p50_ms"], cs["cold"]["env_steps_per_s"]
    except Exception as exc:
        out["error"] = repr(exc)
    return out


def _config4_table(torch, rg, synthetic, dev):
    """BASELINE config[3]: horizon {5, 10, 20} x schedule {trot, pace, bound, walk}, 65536 envs, one GPU.  pace / bound /
    walk are builder-defined schedules in the reference's parameterisation (only trot exists in the reference)."""
    from robot_gym.model.robots.descriptions import GHOST, with_gait
    out = {"envs": 65536, "unit": "solves/s", "cells": {}}
    try:
        ctrl0 = GHOST.GetCtrlConstants()
        n = 65536
        for schedule in ("trot", "pace", "bound", "walk"):
            desc = with_gait(GHOST, schedule)
            st = synthetic.make_states_sharded(0, n, desc, schedule_ctrl=desc.GetCtrlConstants())
            up = lambda a: torch.from_numpy(a).to(dev)
            ins = [up(getattr(st, k)) for k in ("com_velocity_body", "base_rpy", "base_rpy_rate", "planned_contacts",
                                                 "foot_positions_base", "command")]
            forces = torch.empty((n, 12), dtype=torch.float32, device=dev)
            info = torch.empty((n, 4), dtype=torch.int32, device=dev)
            for horizon in (5, 10, 20):
                p = rg.default_mpc_params(ctrl0.MPC_BODY_MASS, ctrl0.MPC_BODY_INERTIA, ctrl0.MPC_BODY_HEIGHT, horizon)
                ws = rg.MpcWorkspace(p, device=dev, max_envs=n)
                rg.mpc_build_solve(ws, *ins, contact_forces=forces, solve_info=info)
                torch.cuda.synchronize()
                reps = 3 if horizon < 20 else 2
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    rg.mpc_build_solve(ws, *ins, contact_forces=forces, solve_info=info)
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / reps
                status = info[:, rg.RG_INFO_STATUS]
                out["cells"][f"h{horizon}_{schedule}"] = {
                    "ms": ms, "solves_per_s": n / (ms * 1e-3),
                    "verified": float(((status & (rg.RG_STATUS_POLISHED | rg.RG_STATUS_NO_STANCE)) != 0).double().mean()),
                    "active_set_only": float(((status & rg.RG_STATUS_ACTIVE_SET_ONLY) != 0).double().mean()),
                    "rounds_mean": float(info[:, rg.RG_INFO_POLISH_ROUNDS].double().mean()),
                    "ipm_iters_mean": float(info[:, rg.RG_INFO_IPM_ITERS].double().mean())}
                del ws
    except Exception as exc:
        out["error"] = repr(exc)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
