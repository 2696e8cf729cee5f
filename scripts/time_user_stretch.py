"""Stretcher on user-written CUDA models (CudaModel): what the fused one-thread-per-walker half-step kernel
bk_user_stretch buys over the three-launch engine (k_stretch_propose, bk_user_eval, k_stretch_accept; ensemble.cu).
One GPU run, JSON to argv[1].

    python scripts/time_user_stretch.py profiles/r3_time_user_stretch.json

Records the card name and power limit; NVRTC compile + load time of a first and of a cached bk_stretch_cuda_prepare at
D = 24; per point (fp32, a = 2; D in {2, 8, 16, 32}; a banana padded with standard normals and a diagonal Gaussian
written as a user model; 2^20 walkers (throughput) and the default 2 * D walkers (launch-bound, how most users run it))
the median over 7 timed calls, after 2 warm-up calls, of ms per sweep, each call SWEEPS sample() calls between two
CUDA events, with the fused kernel and the three-launch engine (BK_FORCE_GENERIC=1) alternated call by call;
walker-moves/s, the accept rate over the timed sweeps, and the registers, stack frame and spills of bk_user_stretch
from ptxas."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from _user_cuda import BANANA, DIAG, card, ptxas_report  # noqa: E402

SWEEPS = 20


def regs(log):
    r = ptxas_report(log).get("bk_user_stretch")
    if r is None:
        return None
    return {k: r[k] for k in ("registers", "stack_frame_bytes", "spill_store_bytes", "spill_load_bytes")}


def main(out_path):
    import ctypes as C

    import numpy as np
    import torch

    import bayes_kit_b200 as bk
    from bayes_kit_b200 import _lib as L

    lib = L.lib()
    smi = card()
    big = 1 << 20
    res = {"gpu": smi, "dtype": "float32", "a": 2.0, "sweeps_per_call": SWEEPS, "compile_s": {}, "points": []}

    # NVRTC compile + load of the Stretcher program: the first prepare of a model library, then a cached one
    os.environ["BK_FORCE_GENERIC"] = "0"
    m24 = bk.CudaModel(BANANA, 24, params=[0.5])
    log = C.create_string_buffer(1 << 20)
    t0 = time.perf_counter()
    L.check(lib.bk_stretch_cuda_prepare(m24.handle, log, len(log)))
    t1 = time.perf_counter()
    L.check(lib.bk_stretch_cuda_prepare(m24.handle, log, len(log)))
    t2 = time.perf_counter()
    res["compile_s"] = {"first_prepare": t1 - t0, "cached_prepare": t2 - t1, "D": 24,
                        "ptxas": regs(log.value.decode())}

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(s, generic, acc):
        os.environ["BK_FORCE_GENERIC"] = "1" if generic else "0"
        e0.record()
        for _ in range(SWEEPS):
            s.sample()
        e1.record()
        torch.cuda.synchronize()
        if acc is not None:
            acc.append(float(s.last_accept.float().mean()))
        return e0.elapsed_time(e1) / SWEEPS

    def summary(W, per_sweep, acc):
        ms = float(np.median(per_sweep))
        return {"ms_per_sweep": ms, "ms_per_sweep_all": per_sweep, "walker_moves_per_s": W / (ms * 1e-3),
                "accept": float(np.mean(acc))}

    def compare(model, W):
        """fused and three-launch Stretchers of the same walkers, alternated call by call"""
        os.environ["BK_FORCE_GENERIC"] = "0"
        fu = bk.Stretcher(model, walkers=W, seed=1)
        ge = bk.Stretcher(model, walkers=W, seed=1)
        for _ in range(2):
            timed(fu, False, None)
            timed(ge, True, None)
        wf, wg, af, ag = [], [], [], []
        for _ in range(7):
            wf.append(timed(fu, False, af))
            wg.append(timed(ge, True, ag))
        out = {"walkers": W, "fused": summary(W, wf, af), "generic": summary(W, wg, ag), "ptxas": regs(fu.compile_log)}
        out["fused_over_generic"] = out["generic"]["ms_per_sweep"] / out["fused"]["ms_per_sweep"]
        del fu, ge
        torch.cuda.empty_cache()
        return out

    rng = np.random.default_rng(0)
    for D in (2, 8, 16, 32):
        ban = bk.CudaModel(BANANA, D, params=[0.5])
        mu, pr = rng.normal(size=D), rng.uniform(0.5, 3.0, D)
        diag = bk.CudaModel(DIAG, D, params=np.concatenate([mu, pr]))
        for W in (big, 2 * D):
            pt = {"D": D, "walkers": W, "banana": compare(ban, W), "diag_user": compare(diag, W)}
            res["points"].append(pt)
            print(json.dumps({"D": D, "W": W,
                              "banana": [pt["banana"]["fused"]["ms_per_sweep"], pt["banana"]["generic"]["ms_per_sweep"],
                                         pt["banana"]["fused_over_generic"]],
                              "diag_user": [pt["diag_user"]["fused"]["ms_per_sweep"],
                                            pt["diag_user"]["generic"]["ms_per_sweep"],
                                            pt["diag_user"]["fused_over_generic"]],
                              "ptxas": pt["banana"]["ptxas"]}), flush=True)
    os.environ["BK_FORCE_GENERIC"] = "0"
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": smi, "compile_s": res["compile_s"]}))


if __name__ == "__main__":
    main(sys.argv[1])
