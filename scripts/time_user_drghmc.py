"""DrGhmcDiag on user-written CUDA models (CudaModel): what the fused one-thread-per-chain kernel bk_user_drghmc buys
over the lockstep engine (drghmc_generic.cu), with the built-in DiagGauss plugin through its own fused kernel
(k_drghmc) beside them for scale.  One GPU run, JSON to argv[1].

    python scripts/time_user_drghmc.py profiles/r3_time_user_drghmc.json

Records the card name and power limit; NVRTC compile + load time of a first and of a cached bk_drghmc_cuda_prepare at
D = 24; per point (2^20 fp32 chains, 10 draws per call, keep_draws=False, damping 0.5, K in {2, 3} with step sizes
(0.4, 0.2, 0.1) and counts (4, 8, 16) cut to K; D in {2, 8, 16, 32}; a banana padded with standard normals and a
diagonal Gaussian written as a user model) the median wall time of 7 calls after 2 warm-up calls by CUDA events, with
the fused kernel and the lockstep engine (BK_FORCE_GENERIC=1) alternated call by call, chain-draws/s, the accept rate,
the mean number of uniforms a draw consumed (last_n_uniform: 2 per attempt, 1 for a retry stop), and the registers,
stack frame and spills of bk_user_drghmc from ptxas."""
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BANANA = """
__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* params) {
    const bk_real b = params[0], half = 0.5, two = 2;
    const bk_real u = x[1] - b * x[0] * x[0];
    bk_real lp = -half * (x[0] * x[0]) - half * (u * u);
    g[0] = -x[0] + two * b * x[0] * u;
    g[1] = -u;
    for (int e = 2; e < BK_DIMS; ++e) { lp -= half * (x[e] * x[e]); g[e] = -x[e]; }
    return lp;
}
"""
DIAG = """
__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) {
        const bk_real d = x[e] - p[e];
        const bk_real pd = p[BK_DIMS + e] * d;
        s += d * pd;
        g[e] = -pd;
    }
    return bk_real(-0.5) * s;
}
"""
SIZES, COUNTS, DAMPING = (0.4, 0.2, 0.1), (4, 8, 16), 0.5


def regs(log):
    m = re.search(r"Function properties for bk_user_drghmc\n.*?(\d+) bytes stack frame, (\d+) bytes spill stores, "
                  r"(\d+) bytes spill loads\n.*?Used (\d+) registers", log, re.S)
    if not m:
        return None
    return {"registers": int(m.group(4)), "stack_frame_bytes": int(m.group(1)), "spill_store_bytes": int(m.group(2)),
            "spill_load_bytes": int(m.group(3))}


def main(out_path):
    sys.path.insert(0, ROOT)
    import ctypes as C

    import numpy as np
    import torch

    import bayes_kit_b200 as bk
    from bayes_kit_b200 import _lib as L

    lib = L.lib()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    Cn, n = 1 << 20, 10
    res = {"gpu": smi, "chains": Cn, "draws_per_call": n, "dtype": "float32", "keep_draws": False,
           "step_sizes": SIZES, "step_counts": COUNTS, "damping": DAMPING, "compile_s": {}, "points": []}

    # NVRTC compile + load of the DrGHMC program: the first prepare of a model library, then a cached one
    os.environ["BK_FORCE_GENERIC"] = "0"
    m24 = bk.CudaModel(BANANA, 24, params=[0.5])
    log = C.create_string_buffer(1 << 20)
    t0 = time.perf_counter()
    L.check(lib.bk_drghmc_cuda_prepare(m24.handle, log, len(log)))
    t1 = time.perf_counter()
    L.check(lib.bk_drghmc_cuda_prepare(m24.handle, log, len(log)))
    t2 = time.perf_counter()
    res["compile_s"] = {"first_prepare": t1 - t0, "cached_prepare": t2 - t1, "D": 24,
                        "ptxas": regs(log.value.decode())}

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(s, generic):
        os.environ["BK_FORCE_GENERIC"] = "1" if generic else "0"
        e0.record()
        s.sample_n(n, keep_draws=False)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def summary(s, walls):
        wall = float(np.median(walls))
        return {"wall_ms": wall, "walls_ms": walls, "chain_draws_per_s": Cn * n / (wall * 1e-3),
                "accept": float(s.last_accept.float().mean()),
                "mean_n_uniform": float(s.last_n_uniform.float().mean())}

    def compare(model, K):
        """fused and lockstep samplers of the same chains, alternated call by call"""
        os.environ["BK_FORCE_GENERIC"] = "0"
        fu = bk.DrGhmcDiag(model, K, list(SIZES[:K]), list(COUNTS[:K]), DAMPING, chains=Cn, seed=1)
        os.environ["BK_FORCE_GENERIC"] = "1"
        ls = bk.DrGhmcDiag(model, K, list(SIZES[:K]), list(COUNTS[:K]), DAMPING, chains=Cn, seed=1)
        for _ in range(2):
            timed(fu, False)
            timed(ls, True)
        wf, wl = [], []
        for _ in range(7):
            wf.append(timed(fu, False))
            wl.append(timed(ls, True))
        out = {"fused": summary(fu, wf), "lockstep": summary(ls, wl), "ptxas": regs(fu.compile_log)}
        out["fused_over_lockstep"] = out["lockstep"]["wall_ms"] / out["fused"]["wall_ms"]
        del fu, ls
        torch.cuda.empty_cache()
        return out

    def builtin(model, K):
        os.environ["BK_FORCE_GENERIC"] = "0"
        s = bk.DrGhmcDiag(model, K, list(SIZES[:K]), list(COUNTS[:K]), DAMPING, chains=Cn, seed=1)
        for _ in range(2):
            timed(s, False)
        out = summary(s, [timed(s, False) for _ in range(7)])
        del s
        torch.cuda.empty_cache()
        return out

    rng = np.random.default_rng(0)
    for D in (2, 8, 16, 32):
        ban = bk.CudaModel(BANANA, D, params=[0.5])
        mu, pr = rng.normal(size=D), rng.uniform(0.5, 3.0, D)
        diag_u = bk.CudaModel(DIAG, D, params=np.concatenate([mu, pr]))
        diag_b = bk.DiagGauss(mu, pr)
        for K in (2, 3):
            pt = {"D": D, "K": K, "banana": compare(ban, K), "diag_user": compare(diag_u, K),
                  "diag_builtin_k_drghmc": builtin(diag_b, K)}
            res["points"].append(pt)
            print(json.dumps({"D": D, "K": K,
                              "banana": [pt["banana"]["fused"]["chain_draws_per_s"],
                                         pt["banana"]["lockstep"]["chain_draws_per_s"],
                                         pt["banana"]["fused_over_lockstep"]],
                              "diag_user": [pt["diag_user"]["fused"]["chain_draws_per_s"],
                                            pt["diag_user"]["lockstep"]["chain_draws_per_s"],
                                            pt["diag_user"]["fused_over_lockstep"]],
                              "diag_builtin": pt["diag_builtin_k_drghmc"]["chain_draws_per_s"],
                              "ptxas": pt["banana"]["ptxas"]}), flush=True)
    os.environ["BK_FORCE_GENERIC"] = "0"
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": smi, "compile_s": res["compile_s"]}))


if __name__ == "__main__":
    main(sys.argv[1])
