#!/usr/bin/env python
"""Headline benchmark: HMC chain-steps/s on BASELINE config c2.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1], SURVEY.md section 8(d) c2): HMCDiag, L=10
leapfrog steps, 65,536 chains PER GPU on the 1000-dim dense-precision Gaussian
(P = A A^T / D + I, A ~ N(0,1) from default_rng(0)); synthetic data, fp32
device-Philox mode.  One "step" = one sample_n(16) call: 16 draws of every chain
(1,048,576 chain-steps per GPU; 20 steps ~ 1 s of device time).  Chains shard across
ranks with no communication (weak scaling).

Prints ONE JSON line (rank 0).  `value` = chain-steps/s with the chain state
resident in HBM; `e2e` = the same metric through the public Python API with
HOST buffers (pinned host -> device copy of the chain state and device -> host
copy of every draw + log density inside the timed region, every step).
`config.secondary` carries the other BASELINE configs (c1, c3, c4 strong / weak
over the N ranks, c5, MALA on c2), each with its own roofline fraction.

`--dump-outputs DIR` writes what the last timed sample_n call of rank 0
returned, for comparing two builds output for output: DIR/draws.npy and
DIR/logp.npy (fp32, [draws, chains, ...]) for a fixed, seeded sample of chains.
The inputs depend only on the arguments, so equal arguments give equal inputs.
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

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

D = 1000
L = 10
EPS = 0.1            # eps*L = 1.0 < pi/sqrt(lambda_max): no fixed-length-HMC resonance on c2
                     # (eps = 0.2 gives accept 0.9 but omega*T crosses pi -> non-ergodic modes)
CHAINS_PER_GPU = 65536
METRIC = "hmc_chain_steps_per_s"
UNIT = "chain-steps/s"


def c2_precision():
    import numpy as np
    rng = np.random.default_rng(0)
    A = rng.normal(size=(D, D))
    return A @ A.T / D + np.eye(D)


# --------------------------------------------------------------------------------
# CPU baseline: the reference algorithm on host cores
# --------------------------------------------------------------------------------
def _cpu_chain_worker(args):
    """One chain of HMCDiag on c2 for n draws; returns seconds.  Uses the
    unmodified reference when baseline/_ref holds it, else the oracle port."""
    n, seed, use_ref = args
    import numpy as np
    try:
        from threadpoolctl import threadpool_limits
        ctx = threadpool_limits(limits=1)
    except Exception:  # pragma: no cover
        import contextlib
        ctx = contextlib.nullcontext()
    with ctx:
        from oracle.models import DensePrecGauss
        model = DensePrecGauss(c2_precision())
        rng = np.random.default_rng(seed)
        th0 = rng.normal(size=D)
        if use_ref:
            from oracle.record import load_reference
            bkref = load_reference()
            s = bkref.HMCDiag(model, EPS, L, init=th0, seed=seed)
            s.sample()
            t0 = time.perf_counter()
            for _ in range(n):
                s.sample()
            return time.perf_counter() - t0
        from oracle import samplers as osm
        zs, us = rng.standard_normal((n, D)), rng.random(n)
        osm.hmc_diag(model, th0, zs[:1], us[:1], EPS, L)
        t0 = time.perf_counter()
        osm.hmc_diag(model, th0, zs, us, EPS, L)
        return time.perf_counter() - t0


def _ref_on_box() -> bool:
    return os.path.isfile(os.path.join(ROOT, "baseline", "_ref", "bayes_kit", "hmc.py"))


def cpu_baseline_single(target_s=12.0):
    """1 core, bounded sample: 1 chain x n draws of the c2 workload."""
    use_ref = _ref_on_box()
    t = _cpu_chain_worker((20, 0, use_ref))
    n = max(20, int(target_s / max(t / 20, 1e-6)))
    t = _cpu_chain_worker((n, 1, use_ref))
    return {"value": n / t, "unit": UNIT, "cores": 1, "kind": "reference" if use_ref else "port",
            "sample": f"1 chain x {n} draws of HMCDiag(L={L}, eps={EPS}) on the {D}-dim dense-precision "
                      f"Gaussian, 1 BLAS thread; rate is per chain-step"}


def run_reference_arm(args):
    """--impl reference: the reference's CPU path on all host cores.  One step =
    every worker process advances one chain by `draws` draws."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    use_ref = _ref_on_box()
    t1 = _cpu_chain_worker((10, 0, use_ref)) / 10
    draws = max(5, int(3.0 / t1))             # ~3 s of work per worker per step
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        for w in range(args.warmup):
            pool.map(_cpu_chain_worker, [(max(2, draws // 10), 100 + c, use_ref) for c in range(cores)])
        t0 = time.perf_counter()
        for k in range(args.steps):
            pool.map(_cpu_chain_worker, [(draws, 1000 * k + c, use_ref) for c in range(cores)])
        dt = time.perf_counter() - t0
    value = cores * draws * args.steps / dt
    sample = (f"{cores} processes x 1 chain x {draws} draws per step of HMCDiag(L={L}, eps={EPS}) on the "
              f"{D}-dim dense-precision Gaussian (1 BLAS thread per process)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": f"c2: HMCDiag L={L} eps={EPS}, {D}-dim dense-precision Gaussian, "
                                   f"chains run independently on host cores"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores,
                             "kind": "reference" if use_ref else "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# --------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.p, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 9 for n, v in zip(names, r[5:9]) if v.startswith("Active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# --------------------------------------------------------------------------------
DRAWS_PER_STEP = 16   # one step = one sample_n(16) call for every chain: 20 steps ~ 1 s of device time
DUMP_BYTES = 32 << 20  # --dump-outputs budget: a whole step's draws are 4 GB at the default size


def dump_outputs(out_dir, draws, logp):
    """Save draws [n, C, D] and logp [n, C] of one sample_n call, restricted to a seeded sample of chains."""
    import numpy as np
    import torch
    n, C, D = draws.shape
    k = min(C, max(1, DUMP_BYTES // (n * (D + 1) * 4)))
    idx = np.sort(np.random.default_rng(0).choice(C, size=k, replace=False))
    sel = torch.as_tensor(idx, device=draws.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "draws.npy"), draws[:, sel].cpu().numpy())
    np.save(os.path.join(out_dir, "logp.npy"), logp[:, sel].cpu().numpy())


def bind_to_gpu_numa(local):
    """Run this rank (and first-touch its pinned buffers) on the cores next to its GPU."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cores = [64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1]
        allowed = sorted(set(cores) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
        return len(allowed)
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chains", type=int, default=CHAINS_PER_GPU, help="chains per GPU")
    ap.add_argument("--draws-per-step", type=int, default=DRAWS_PER_STEP)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the c1 / c3 / c4 / c5 / MALA legs")
    ap.add_argument("--e2e-chunk", type=int, default=0, help="chains per sample_host chunk (0: library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's draws and log densities here")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the CUDA path; the reference arm has nothing to dump")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference_arm(args)
    for v in ("BK_TC_DEBUG", "BK_DISABLE_TC", "BK_FORCE_GENERIC", "BK_HLR_DEBUG", "BK_ESS", "BK_ACF", "BK_LIB", "BK_TC_FUSE", "BK_TC_PAIR", "BK_SEP_WIDE", "BK_SMC_LAYOUT", "BK_SMC_OCC", "BK_ACF_RFFT", "BK_TC_TURN", "BK_HLR_FUSE", "BK_SEP_LAYOUT", "BK_HLR_PDL"):   # diagnostic switches of the library (for some of them "0" is the diagnostic value)
        if os.environ.get(v, "") != "":
            raise SystemExit(f"{v} is set: refusing to benchmark a diagnostic configuration")

    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    n_cores = bind_to_gpu_numa(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import bayes_kit_b200 as bk
    from bayes_kit_b200 import _lib
    lib = _lib.lib()

    C, n = args.chains, args.draws_per_step
    model = bk.DensePrecGauss(c2_precision(), dtype=torch.float32, device=dev)
    # theta0 ~ N(0, I) per chain (the reference's default init, hmc.py:27); global chain ids
    sampler = bk.HMCDiag(model, EPS, L, chains=C, seed=0, chain_offset=rank * C)

    t_start = time.perf_counter()

    def stage(msg):
        if os.environ.get("BENCH_VERBOSE", "0") == "1":
            print(f"[bench rank {rank} +{time.perf_counter() - t_start:7.2f}s] {msg}", file=sys.stderr, flush=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def rank_max(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    # ---- device-resident throughput ------------------------------------------------
    stage("model + sampler ready")
    for _ in range(args.warmup):
        sampler.sample_n(n)
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    lib.bk_profile_enable(1)
    launches0 = lib.bk_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        # every draw streams ~1.6 GB of chain state (>> L2) and a step writes a fresh 16 x 262 MB draw block;
        # the previous step's block is released first, so every step reuses the same cached allocation
        last = None
        last = sampler.sample_n(n)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = lib.bk_launch_count() - launches0
    lib.bk_profile_enable(0)
    gms, gn = _lib.f64(0), _lib.u64(0)
    lib.bk_profile_read(_lib.PROF_GRAD, gms, gn)
    sms_, sn = _lib.f64(0), _lib.u64(0)
    lib.bk_profile_read(_lib.PROF_STEP, sms_, sn)
    accept = float(sampler.last_accept.float().mean())
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    del last
    ms_max = rank_max(ms)
    value = world * C * n * args.steps / (ms_max * 1e-3)
    stage(f"device-resident done: {ms:.1f} ms")

    # ---- end to end through the public API with host buffers --------------------------
    # One step = the call a user of the reference makes for n draws of every chain, host arrays in and out
    # (hmc.py:55-63 returns host arrays): the chain state is uploaded from pinned host memory (the previous
    # step's last draw), all n draws + log densities come back into pinned host memory.
    host_draws = torch.empty(n, C, D, dtype=torch.float32, pin_memory=True)
    host_lp = torch.empty(n, C, dtype=torch.float32, pin_memory=True)
    host_draws[n - 1].copy_(sampler.theta)
    e2e_steps = args.steps

    def e2e_step():
        # next step's input = this step's last draw, read in place from the pinned result buffer (a chunk's
        # rows are uploaded before that chunk's draws are written back, so the aliasing is safe)
        sampler.sample_host_n(n, host_draws[n - 1], out=(host_draws, host_lp), chunk_chains=args.e2e_chunk or None)

    stage("pinned buffers ready")
    for _ in range(2):
        e2e_step()
    barrier()
    stage("e2e warm-up done")
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = rank_max(time.perf_counter() - t0)
    e2e_value = world * C * n * e2e_steps / e2e_s
    # the box's copy floor for exactly these bytes: all ranks copy one step's D2H volume at the same time
    # (pinned, one stream per rank) -- the e2e step cannot finish faster than this on this box
    dsrc = torch.empty(C, D, dtype=torch.float32, device=dev)
    barrier()
    t0 = time.perf_counter()
    for _ in range(2):
        for t in range(n):
            host_draws[t].copy_(dsrc, non_blocking=True)
    barrier()
    floor_s = rank_max((time.perf_counter() - t0) / 2)
    del dsrc
    stage(f"e2e done: {e2e_s:.2f} s, floor {floor_s:.3f} s")

    # ---- secondary workloads (all ranks take part in the sharded ones) ------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_bw = peaks.get("hbm_gbs") or 6650.0               # fallback: B200_PROFILING.md
    peak_tf = peaks.get("bf16_tflops_sustained") or 1400.0
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    secondary = {}
    if not args.no_secondary:
        del host_draws
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        import bench_legs as legs
        torch.cuda.empty_cache()
        for name, fn in (("c4_strong", lambda: legs.leg_c4(rank, world, peak_bw, weak=False)),
                         ("c4_weak", lambda: legs.leg_c4(rank, world, peak_bw, weak=True)),
                         ("c3", lambda: legs.leg_c3(rank, world, peak_tf))):
            if name == "c4_weak" and world == 1:
                continue
            stage(f"leg {name} ...")
            try:
                secondary[name] = fn()
            except Exception as e:      # a failed leg must not lose the headline
                secondary[name] = {"error": repr(e)}
                stage(f"leg {name} FAILED: {e!r}")
            torch.cuda.empty_cache()
        stage("sharded legs done")
        if rank == 0:
            for name, fn in (("c1", lambda: legs.leg_c1(peak_bw)), ("c2_mala", lambda: legs.leg_c2_mala(peak_bw, peak_tf)),
                             ("c5", lambda: legs.leg_c5(peak_bw))):
                stage(f"leg {name} ...")
                try:
                    secondary[name] = fn()
                except Exception as e:
                    secondary[name] = {"error": repr(e)}
                    stage(f"leg {name} FAILED: {e!r}")
                torch.cuda.empty_cache()
            stage("rank-0 legs done")

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- min-ESS/s (BASELINE metric): ESS per chain-step from a side run of the same
    # sampler on 2048 chains x 200 draws (device diagnostics, Geyer IMSE like ess.py:52-69),
    # scaled by the measured chain-steps/s.  Anti-correlated chains give ESS > n (or an
    # IAT <= 0): those are counted as n draws (conservative).
    n_side, c_side = 200, 2048
    side = bk.HMCDiag(model, EPS, L, chains=c_side, seed=1)
    side.sample_n(50, keep_draws=False)
    dr, _ = side.sample_n(n_side)
    e = bk.ess(dr, draws_first=True)                     # [chains, params]
    e = torch.where((e <= 0) | (e > n_side), torch.full_like(e, float(n_side)), e)
    ess_per_step = float(e.mean(0).min()) / n_side       # min over parameters
    del dr, e, side

    # ---- roofline of the dominant kernel -----------------------------------------------
    # k_dense_tc in STEP mode (gradient GEMM + fused leapfrog update): L-1 of the L
    # gradient launches of a draw and ~2/3 of its time.  It is HBM-bound: SURVEY 8(d)
    # c2 "HBM side" = 4*D*s bytes per chain per leapfrog step (theta, rho round trip).
    # one persistent STEP launch fuses the interior leapfrog steps of a draw (L-1 of them at c2); algorithmic
    # bytes per launch = 16 B per chain-dim-step x the steps that launch ran
    n_draws_timed = n * args.steps
    steps_per_launch = (L - 1) * n_draws_timed / max(sn.value, 1)
    bytes_per_launch = 4.0 * D * 4 * C * steps_per_launch   # 16 KB per chain-leapfrog-step
    s_avg_ms = sms_.value / max(sn.value, 1)
    g_avg_ms = gms.value / max(gn.value, 1)
    achieved = bytes_per_launch / (s_avg_ms * 1e-3) / 1e9 if sn.value else None
    # DRAM bytes of one launch from the committed ncu --set full capture of this kernel (never a constant typed
    # into this file): profiles/ncu_traffic.json, written by scripts/summarize_ncu.py from the .ncu-rep
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["k_dense_tc_step"]
        if C == tj["chains"] and abs(steps_per_launch - tj["leapfrog_steps_per_launch"]) < 1e-9:
            traffic, traffic_src = tj["dram_bytes_per_launch"], tj["source"]
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak_bw, "unit": "GB/s",
                "frac": (achieved / peak_bw) if achieved else None,
                "traffic": traffic, "traffic_source": traffic_src,
                "kernel": "k_dense_tc STEP mode (tcgen05 gradient GEMM + fused leapfrog epilogue, "
                          "persistent over the interior leapfrog steps of a draw)",
                "leapfrog_steps_per_launch": steps_per_launch,
                "launches_timed": int(sn.value), "avg_launch_ms": s_avg_ms,
                "share_of_step": sms_.value / ms if ms else None, "peak_source": peak_src,
                "whole_step": {  # every kernel of a draw, on the algorithmic bytes of the whole draw:
                    # 16 B x C x D per interior leapfrog step + GRAD operand/gradient (10 B) + the row kernels of a
                    # sample_n(n) call: one begin (18 B), n - 1 turns (end + begin fused, 22 B), one end (24 B)
                    "bytes_per_draw": (16.0 * (L - 1) + 10 + (18 + 24 + 22 * (n - 1)) / n) * C * D,
                    "achieved": (16.0 * (L - 1) + 10 + (18 + 24 + 22 * (n - 1)) / n) * C * D * n_draws_timed / (ms * 1e-3) / 1e9,
                    "frac": (16.0 * (L - 1) + 10 + (18 + 24 + 22 * (n - 1)) / n) * C * D * n_draws_timed / (ms * 1e-3) / 1e9 / peak_bw},
                "tensor_side": {  # the endpoint gradient (3-pass bf16 split) is tensor-bound
                    "kernel": "k_dense_tc GRAD mode", "flops_per_launch": 3 * 2.0 * C * D * D,
                    "avg_launch_ms": g_avg_ms, "launches_timed": int(gn.value),
                    "achieved_tflops": (3 * 2.0 * C * D * D / (g_avg_ms * 1e-3) / 1e12) if gn.value else None,
                    "peak_tflops": peak_tf,
                    "frac": (3 * 2.0 * C * D * D / (g_avg_ms * 1e-3) / 1e12 / peak_tf) if gn.value else None,
                    "share_of_step": gms.value / ms if ms else None}}

    cpu = None if args.no_cpu_baseline else cpu_baseline_single()
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"c2: HMCDiag L={L} eps={EPS}, {C} chains/GPU x {D}-dim dense-precision "
                               f"Gaussian (P=AA^T/D+I, seed 0), device Philox; one step = sample_n({n}): "
                               f"{n} draws of every chain",
                   "chains_per_gpu": C, "dims": D, "leapfrog_steps": L, "draws_per_step": n,
                   "chain_steps_per_step": world * C * n, "ms_per_draw": ms_max / args.steps / n,
                   "timed_region_s": ms_max * 1e-3, "accept_rate": accept,
                   "grad_evals_per_s": value * L, "min_ess_per_s": value * ess_per_step,
                   "ess_per_chain_step_min_param": ess_per_step,
                   "l2": "inputs larger than L2 (>= 1.5 GB of chain state streamed per draw)",
                   "cpu_cores_bound_to_gpu_numa": n_cores,
                   "secondary": secondary},
        "roofline": roofline, "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": C * D * 4,
                "d2h_bytes_per_step": n * (C * D * 4 + C * 4), "steps": e2e_steps,
                "ms_per_step": 1e3 * e2e_s / e2e_steps,
                "api": f"HMCDiag.sample_host_n({n}, theta_host, out=(draws_host, logp_host))",
                # this box's D2H copy time for one step's draws with all ranks copying at once
                "d2h_copy_floor_ms": 1e3 * floor_s,
                "floor_frac": floor_s / (e2e_s / e2e_steps)},
        "gpu_launches": int(launches), "clocks": clk,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
