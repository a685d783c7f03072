#!/usr/bin/env python
"""bench.py -- dispatch LPs/sec on BASELINE.json's headline config (C2: wind+battery, 24 periods, 10 000
synthetic LMP scenarios per GPU), one JSON line on rank 0.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...        (one rank per GPU, weak scaling: 10 000 LPs per rank,
                                                            one all_gather of the objectives per step)

A "step" = one pass of the hot path over one batch: parameter rows already in HBM -> one kernel launch ->
obj/status/iters in HBM (`value`), or through the host C-ABI call with H2D / D2H inside the timed region (`e2e`).
`--impl reference` times the CPU path the reference would take for these LPs (restated LP + HiGHS in a process
pool over all host cores; CBC/IPOPT/Pyomo are not installable here, see DESIGN.md).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True                 # the benchmark writes nothing into the tree, which may be read-only

T = 24
BATCH = 10000
METRIC = "dispatch LPs/sec (24-period price-taker batch); max |obj| rel-err vs IPOPT"
ALG_BYTES_PER_LP = 8 * T + 8 + 4 + 4           # lmp row in; obj, status, iters out (SURVEY.md §8d: 208 B)
ALG_FLOP_PER_LP = 0.30e6                       # banded-IPM algorithmic FP64 flops per LP (SURVEY.md §8d)
FP64_PEAK_TFLOPS_NOMINAL = 37.0                # HGX B200 spec sheet (296 TF / 8 GPUs); no measured FP64 peak file


def workload(rank):
    from dispatches_b200 import scenarios as SC, templates as TP
    lmp, cf, W, P = SC.c2(BATCH, seed=20240101 + rank)
    rp = TP.wind_battery_rparams(T, cf, W, P)[0]
    return lmp, cf, W, P, rp


def config(n_gpus):
    return {"workload": f"C2: renewables wind+battery 24-period price-taker, {BATCH} synthetic LMP scenarios per GPU "
                        f"(seed 20240101+rank), fixed design 847 MW wind / 211.75 MW 4-h battery",
            "T": T, "batch_per_gpu": BATCH, "global_batch": BATCH * n_gpus, "parallelism": f"scenario-shard x{n_gpus}", "collective": "all_gather of the objectives per step, asynchronous: overlaps the next step's kernel (N > 1)",
            "l2": "flushed between timed steps (256 MiB write)", "template": "wind_battery_T24 (m=96, n=167, w=4)", "kernel": "dsp_ipm_stage2_wb_kernel<8,3> (4 LPs per warp, 3 periods per lane, iterate in registers, partitioned block elimination)"}


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def host_cores():
    from oracle import highs as H
    return H.host_cores()


def cpu_reference_run(lmp, cf, W, P, n_sample, procs=None):
    """The oracle loop (HiGHS dual simplex, constraints pre-built, cost vector swapped per LP) on all host cores."""
    from oracle import highs as H
    procs = procs or host_cores()
    obj, dt, procs = H.solve_batch("wind_battery", lmp[:n_sample], kwargs=dict(cf=cf, wind_mw=W, batt_mw=P), procs=procs)
    return obj, dt, procs



# ---------------------------------------------------------------------------------------------------------------
# The other BASELINE.json configs (C3 nuclear T=48 x 5000, C4 fossil surrogate T=168 x 2000, C5 design sweep 560 640 LPs):
# STRONG-scaled over the N ranks (dispatches_b200.sweep.solve_sharded: interleaved shards + one all_gather), reported in
# the `configs` block of the one JSON line, each with a seeded parity sample against the oracle and a CPU number.
CONFIG_DEFS = {
    "C3": dict(kind="nuclear", T=48, N=5000, what="nuclear_case 48-period dispatch, 5 000 LMP scenarios (seed 20240102)"),
    "C4": dict(kind="fossil_surrogate", T=168, N=2000,
               what="fossil_case USC 168-period weekly, 2 000 scenarios (seed 20240103); LP SURROGATE of the reference NLP: "
                    "structure-only, parity vs HiGHS on the surrogate, NOT vs the reference's IPOPT objective (parity unpinned)"),
    "C5": dict(kind="wind_battery", T=24, N=560640,
               what="design sweep: 64 design points x 8 760 hourly 24-h windows = 560 640 LPs, cost AND rhs batched"),
    # not a BASELINE.json config: the sweep the reference's driver really runs (run_pricetaker_wind_battery.py:37-58 solves ONE
    # full-year LP, n_time_points = 8736, per design point) -- the long-horizon stage kernel (csrc/dsp_stage2_long.cuh)
    "FY": dict(kind="wind_battery", T=8736, N=64,
               what="the reference's own sweep: 8 wind sizes x 8 battery ratios, one FULL-YEAR 8736-period LP per design point "
                    "(303 DA prices / capacity factors), long-horizon stage kernel"),
}
CPU_SAMPLE_PER_CORE = {"C3": 96, "C4": 24, "C5": 96, "FY": 1}
CPU_SAMPLE_FIXED = {"FY": [9, 27, 36, 50]}     # full-year LPs cost HiGHS ~7 s each: four fixed design points (one process each)


def config_data(name):
    """(template builder, cparams [N,Pc], rparams [N,Pr] or None, extras for the oracle or None)"""
    from dispatches_b200 import scenarios as SC, templates as TP
    if name == "C3":
        return (lambda: TP.nuclear(48)), SC.c3(5000), None, None
    if name == "C4":
        return (lambda: TP.fossil_surrogate(168)), SC.c4(2000), None, None
    if name == "FY":
        p = SC.pool()
        Tf = CONFIG_DEFS["FY"]["T"]
        lam, cf1 = p["dalmp_303"][:Tf], p["dacf_303"][:Tf]
        w = np.repeat(np.linspace(200.0, 1600.0, 8), 8)
        b = np.tile(np.linspace(0.05, 1.0, 8), 8) * w
        cf = np.tile(cf1, (64, 1))
        return (lambda: TP.wind_battery(Tf)), np.tile(lam, (64, 1)), TP.wind_battery_rparams(Tf, cf, w, b), (cf, w, b)
    lmp, cf, w, b = SC.c5()
    return (lambda: TP.wind_battery(24)), lmp, TP.wind_battery_rparams(24, cf, w, b), (cf, w, b)


def config_sample(name, cores):
    """seeded sample of a config's LP indices for the parity check / CPU baseline"""
    N = CONFIG_DEFS[name]["N"]
    if name in CPU_SAMPLE_FIXED:
        return np.array(CPU_SAMPLE_FIXED[name][:max(1, min(len(CPU_SAMPLE_FIXED[name]), cores))])
    n = int(min(N, CPU_SAMPLE_PER_CORE[name] * cores))
    return np.sort(np.random.default_rng(777).choice(N, n, replace=False))


def cpu_config_run(name, procs=None):
    """oracle objective + wall time of the seeded sample of one config (HiGHS, all host cores)"""
    from oracle import highs as H
    procs = procs or host_cores()
    _, cp, _, extra = config_data(name)
    idx = config_sample(name, procs)
    kind = CONFIG_DEFS[name]["kind"]
    if extra is not None:
        cf, w, b = extra
        ex = [(cf[i], float(w[i]), float(b[i])) for i in idx]
        obj, dt, procs = H.solve_batch(kind, cp[idx], extras=ex, procs=min(procs, idx.size))
    else:
        obj, dt, procs = H.solve_batch(kind, cp[idx], procs=procs)
    return idx, obj, dt, procs


def run_configs(world, rank, dev, reps=3, dump=None):
    """every rank: its interleaved shard of each config, timed on the device (max over ranks), one all_gather per pass;
    `dump` (a dict) receives the full obj / status / iters of each config's last timed pass"""
    import torch
    import torch.distributed as dist
    from dispatches_b200 import solver as S, sweep
    res = {}
    for name, d in CONFIG_DEFS.items():
        build_t, cp_all, rp_all, _ = config_data(name)
        N = cp_all.shape[0]
        idx = sweep.shard_indices(N, rank, world)
        sol = S.BatchLPSolver(build_t())
        cp = torch.tensor(cp_all[idx], device=dev)
        rp = torch.tensor(rp_all[idx], device=dev) if rp_all is not None else None
        del cp_all, rp_all
        out = sol.solve(cp, rp)                                   # warm-up (workspace allocation, first launch)

        def solve_fn(ix):
            o = sol.solve(cp, rp, out=out)
            return dict(obj=o.obj, status=o.status, iters=o.iters)

        full = sweep.solve_sharded(solve_fn, N)
        torch.cuda.synchronize()
        ms = []
        for _ in range(reps):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            full = sweep.solve_sharded(solve_fn, N)
            e1.record()
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms.append(float(t))
        st = full["status"].cpu().numpy(); it = full["iters"].cpu().numpy()
        best = float(np.median(ms))
        res[name] = {"workload": d["what"], "T": d["T"], "lps_total": int(N), "n_gpus": world, "scaling": "strong",
                     "ms": best, "lps": N / best * 1e3, "non_optimal": int((st != 0).sum()),
                     "iters_mean": float(it.mean()), "iters_max": int(it.max()), "launch": S.last_launch(),
                     "obj": full["obj"].cpu().numpy()}
        if dump is not None:
            dump.update({f"{name}_obj": res[name]["obj"], f"{name}_status": st, f"{name}_iters": it})
        sol.close()
        del cp, rp, out, full
        torch.cuda.empty_cache()
    return res


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    lmp, cf, W, P, rp = workload(0)
    cores = host_cores()
    per_step = int(min(BATCH, max(200, 250 * cores)))          # ~1 s of wall clock per step on all cores
    for _ in range(args.warmup):
        cpu_reference_run(lmp, cf, W, P, min(per_step, 64 * cores))
    t_tot = 0.0
    for k in range(args.steps):
        lo = (k * per_step) % max(1, BATCH - per_step + 1)
        _, dt, procs = cpu_reference_run(lmp[lo:], cf, W, P, per_step)
        t_tot += dt
    value = per_step * args.steps / t_tot
    sample = f"{per_step} LPs of the C2 batch per step, HiGHS dual simplex, {procs} processes"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "LPs/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config(args.gpus),
            "cpu_baseline": {"value": value, "unit": "LPs/s", "cores": procs, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "LPs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the C3/C4/C5 block")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed paths returned in their last step as DIR/<name>.npy (float64): C2_obj, "
                         "C2_status, C2_iters of rank 0's batch and <config>_obj / _status / _iters of every config")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    # stdout carries exactly ONE JSON line: libraries that print to fd 1 (NCCL's version banner) go to stderr instead
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    cpu = None
    import torch
    import torch.distributed as dist
    from dispatches_b200 import solver as S, templates as TP
    from dispatches_b200.csrc import build
    build.build()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the solver has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lmp, cf, W, P, rp = workload(rank)
    t = TP.wind_battery(T)
    sol = S.BatchLPSolver(t)
    cp_d = torch.tensor(lmp, device=dev)
    rp_d = torch.tensor(rp, device=dev)
    out = sol.solve(cp_d, rp_d)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    # N > 1: the one collective of the path -- an all_gather of the objectives -- is issued asynchronously and overlaps the
    # NEXT step's kernel (double-buffered results); a step's timed region is its kernel plus the wait for the previous gather
    outs = [out, sol.solve(cp_d, rp_d)] if world > 1 else [out]
    gathered = [torch.empty(BATCH * world, dtype=torch.float64, device=dev) for _ in range(2)] if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for k in range(args.warmup):
        sol.solve(cp_d, rp_d, out=outs[k % len(outs)])
        if world > 1:
            dist.all_gather_into_tensor(gathered[k % 2], outs[k % 2].obj)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(args.steps)]
    ev_tail = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    n0 = S.launch_count()
    barrier()
    t_wall0 = time.perf_counter()
    work = None
    for k in range(args.steps):
        flush.fill_(k & 0xFF)                 # L2 flush, outside the per-step event pair
        ev[k][0].record()
        sol.solve(cp_d, rp_d, out=outs[k % len(outs)])
        ev[k][2].record()                     # kernel-only stop
        if work is not None:
            work.wait()                       # gather of step k-1 (ran concurrently with this kernel)
        ev[k][1].record()
        if world > 1:
            work = dist.all_gather_into_tensor(gathered[k % 2], outs[k % 2].obj, async_op=True)
    ev_tail[0].record()
    if work is not None:
        work.wait()                           # the last gather has nothing to hide behind: its time is added to the total
    ev_tail[1].record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = S.launch_count() - n0
    out = outs[(args.steps - 1) % len(outs)]
    dump = {} if args.dump_outputs else None
    if dump is not None:                      # copied now: the passes below write into the same buffers
        dump.update(C2_obj=out.obj.cpu().numpy(), C2_status=out.status.cpu().numpy(), C2_iters=out.iters.cpu().numpy())
    step_ms = sum(a.elapsed_time(b) for a, b, _ in ev) + ev_tail[0].elapsed_time(ev_tail[1])
    kern_ms = sum(a.elapsed_time(c) for a, _, c in ev)
    tt = torch.tensor([step_ms, kern_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    step_ms, kern_ms = float(tt[0]), float(tt[1])
    # ---- e2e: the host C-ABI call (pinned staging, H2D, kernel, D2H, sync), every step
    # host buffers are page-locked (the contract's "pinned host memory"): inputs are DMA'd straight from them
    lmp_pin = S.BatchLPSolver.pinned_empty(lmp.shape); lmp_pin[:] = lmp
    rp_pin = S.BatchLPSolver.pinned_empty(rp.shape); rp_pin[:] = rp
    r_host = S.LPResult(S.BatchLPSolver.pinned_empty(BATCH), S.BatchLPSolver.pinned_empty(BATCH, np.int32),
                        S.BatchLPSolver.pinned_empty(BATCH, np.int32))
    for _ in range(2):
        sol.solve_host(lmp_pin, rp_pin, out=r_host)
    barrier()
    e2e_wall = 0.0
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()                     # the L2 flush stays outside the timed call
        t0 = time.perf_counter()
        sol.solve_host(lmp_pin, rp_pin, out=r_host)
        e2e_wall += time.perf_counter() - t0
    tt = torch.tensor([e2e_wall], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e_wall = float(tt[0])
    clocks = sampler.stop() if rank == 0 else None
    # ---- sustained: back-to-back launches for >= 2 s (no L2 flush, no host sync in between), clocks sampled under load
    sus_sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sus_sampler.start()
    n_sus = max(50, int(2.2 / max(1e-5, kern_ms * 1e-3 / args.steps)))
    es0, es1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    es0.record()
    for _ in range(n_sus):
        sol.solve(cp_d, rp_d, out=out)
    es1.record()
    torch.cuda.synchronize()
    tt = torch.tensor([es0.elapsed_time(es1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    sus_ms = float(tt[0])
    sus_clocks = sus_sampler.stop() if rank == 0 else None
    cfg_res = {} if args.no_configs else run_configs(world, rank, dev, dump=dump)
    status = out.status.cpu().numpy()
    iters = out.iters.cpu().numpy()
    stats = torch.tensor([float((status != 0).sum()), float(iters.sum()), float(iters.max())], dtype=torch.float64, device=dev)
    if world > 1:
        s2 = stats.clone()
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
        dist.all_reduce(s2, op=dist.ReduceOp.MAX)
        stats[2] = s2[2]
    stats = stats.cpu()
    if world > 1:                              # all collectives are done: every rank leaves the group together
        torch.cuda.synchronize()
        dist.destroy_process_group()
    if rank != 0:
        return
    if dump is not None:
        dump = {k: np.asarray(v, dtype=np.float64) for k, v in dump.items()}
        assert sum(a.nbytes for a in dump.values()) <= 64 << 20
        os.makedirs(args.dump_outputs, exist_ok=True)
        for k, v in dump.items():
            np.save(os.path.join(args.dump_outputs, k + ".npy"), v)
    total = BATCH * world
    value = total * args.steps / (step_ms * 1e-3)
    peaks = {}
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        peaks = json.load(open(pk))
    hbm_peak, which = (peaks.get("hbm_gbs"), "measured (MEASURED_PEAKS.json)") if peaks.get("hbm_gbs") else (6650.0, "fallback")
    kern_s = kern_ms * 1e-3 / args.steps
    ach = ALG_BYTES_PER_LP * BATCH / kern_s / 1e9
    fp64 = ALG_FLOP_PER_LP * BATCH / kern_s / 1e12
    fp64_peak = S.fp64_peak_tflops()
    if not fp64_peak > 0:
        fp64_peak = None
    # DRAM bytes per launch of the dominant kernel from the committed ncu capture (profiles/), not measured live
    traffic = None
    try:
        cur = json.load(open(ROOT / "profiles" / "current.json"))["stage_profile"]
        traffic = float(json.load(open(ROOT / "profiles" / cur))["traffic_bytes_per_launch"])
    except Exception:
        pass
    line = {"metric": METRIC, "value": value, "unit": "LPs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": config(world),
            "e2e": {"value": total * args.steps / e2e_wall, "unit": "LPs/s", "h2d_bytes_per_step": int(lmp.nbytes + rp.nbytes),
                    "d2h_bytes_per_step": int(BATCH * 16), "ms_per_step": 1e3 * e2e_wall / args.steps,
                    "api": "dsp_lp_solve_batch_host (C-ABI, host buffers)"},
            "gpu_launches": int(launches), "kernel_ms_per_step": kern_ms / args.steps,
            "roofline": {"bound": "fp64", "achieved": fp64, "peak": fp64_peak or FP64_PEAK_TFLOPS_NOMINAL, "unit": "TFLOP/s",
                         "frac": fp64 / (fp64_peak or FP64_PEAK_TFLOPS_NOMINAL), "traffic": traffic,
                         "alg_flop_per_lp": ALG_FLOP_PER_LP, "alg_bytes_per_launch": ALG_BYTES_PER_LP * BATCH,
                         "peak_source": "measured DFMA micro-benchmark on this GPU (dsp_lp_fp64_peak_tflops); MEASURED_PEAKS.json has no FP64 entry"
                                        if fp64_peak else "nominal (HGX B200 spec 296 TF / 8)",
                         "peak_tflops_nominal": FP64_PEAK_TFLOPS_NOMINAL,
                         "note": "on-chip FP64 solve: bound by FP64 issue + dependent-chain latency, not HBM or tensor cores (SURVEY.md 8d); "
                                 "achieved = algorithmic banded-IPM flops (0.30 MFLOP/LP) / kernel time",
                         "hbm": {"achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "peak_source": which}},
            "sustained": {"value": total * n_sus / (sus_ms * 1e-3), "unit": "LPs/s", "launches": n_sus, "seconds": sus_ms * 1e-3,
                          "ms_per_launch": sus_ms / n_sus, "clocks": sus_clocks,
                          "note": "back-to-back launches, no L2 flush (inputs 2 MB), device-timed, max over ranks"},
            "solver": {"non_optimal": int(stats[0]), "iters_mean": float(stats[1]) / total, "iters_max": int(stats[2]),
                       "launch": S.last_launch()},
            "clocks": clocks, "wall_s_timed_loop": t_wall}
    cfg_cpu = {}
    if not args.no_cpu_baseline:
        # CPU baseline in a fresh interpreter (no fork of this CUDA process; nothing runs before the ranks rendezvous)
        import tempfile
        with tempfile.TemporaryDirectory() as td:
            outp = os.path.join(td, "cpu.npz")
            code = ("import sys; sys.path.insert(0, %r); import numpy as np, bench; "
                    "lmp, cf, W, P, _ = bench.workload(0); c = bench.host_cores(); n = int(min(bench.BATCH, max(500, 400 * c))); "
                    "bench.cpu_reference_run(lmp, cf, W, P, min(n, 16 * c)); ref, dt, procs = bench.cpu_reference_run(lmp, cf, W, P, n); "
                    "out = dict(ref=ref, dt=dt, procs=procs, n=n)\n"
                    "for name in %r:\n"
                    "    try:\n"
                    "        idx, obj, dtc, pr = bench.cpu_config_run(name)\n"
                    "        out[name + '_idx'] = idx; out[name + '_obj'] = obj; out[name + '_dt'] = dtc; out[name + '_procs'] = pr\n"
                    "    except Exception as e:\n"
                    "        print('cpu baseline of', name, 'failed:', e, file=sys.stderr)\n"
                    "np.savez(%r, **out)") % (str(ROOT), [] if args.no_configs else list(CONFIG_DEFS), outp)
            rc = subprocess.run([sys.executable, "-B", "-c", code], capture_output=True, text=True, timeout=1500)
            if rc.returncode == 0:
                z = np.load(outp)
                cpu = dict(ref=z["ref"], dt=float(z["dt"]), procs=int(z["procs"]), n=int(z["n"]))
                for name in cfg_res:
                    if name + "_idx" in z:
                        cfg_cpu[name] = (z[name + "_idx"], z[name + "_obj"], float(z[name + "_dt"]), int(z[name + "_procs"]))
            else:
                line["cpu_baseline"] = {"error": rc.stderr[-300:]}
    if cpu is not None:
        ref, dt, procs, n_sample = cpu["ref"], cpu["dt"], cpu["procs"], cpu["n"]
        err = np.abs(r_host.obj[:n_sample] - ref) / np.maximum(1.0, np.abs(ref))
        line["cpu_baseline"] = {"value": n_sample / dt, "unit": "LPs/s", "cores": procs, "kind": "port",
                                "sample": f"first {n_sample} LPs of rank 0's batch, restated LP + HiGHS dual simplex, {procs} processes"}
        line["max_rel_err_vs_oracle"] = float(err.max())
    for name, r in cfg_res.items():
        obj = r.pop("obj")
        if name in cfg_cpu:
            idx, ref, dtc, prc = cfg_cpu[name]
            r["max_rel_err_vs_oracle"] = float(np.max(np.abs(obj[idx] - ref) / np.maximum(1.0, np.abs(ref))))
            r["parity_sample"] = (f"design points {idx.tolist()} vs restated LP + HiGHS" if name in CPU_SAMPLE_FIXED
                                  else f"{idx.size} seeded LPs (rng 777) vs restated LP + HiGHS")
            r["cpu_baseline"] = {"value": idx.size / dtc, "unit": "LPs/s", "cores": prc, "kind": "port",
                                 "sample": f"{idx.size} LPs of the config, HiGHS dual simplex, {prc} processes"}
            r["vs_cpu"] = r["lps"] / (idx.size / dtc)
        r["obj_checksum"] = float(obj.sum())
    if cfg_res:
        line["configs"] = cfg_res
    sys.stdout.flush()
    os.write(json_fd, (json.dumps(line) + "\n").encode())


if __name__ == "__main__":
    main()
