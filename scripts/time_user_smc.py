"""TemperedLikelihoodSMC on a user-written model (CudaPriorLikModel) against the built-in plugin.  One GPU run, JSON to
argv[1].

    python scripts/time_user_smc.py profiles/r3_time_user_smc.json

Workload: the c4 shape (M = 10^6 particles, N = 100 temperatures, systematic resampling, fp32, seed 1) on GaussPriorLik
(m0 = 0, p0 = 1, pl = 4, mu ~ N(0, I)), written as a CudaPriorLikModel and as the built-in plugin, at D in
{2, 8, 16, 32, 50} with the RW (scale 0.2), MALA (epsilon 0.05) and HMC (stepsize 0.1, L = 5) moves.  Per point:
ms per temperature from CUDA events around run() (which ends in a synchronise), median of 5 runs after one warm-up
run.  Also records the card name and power limit, the NVRTC compile + load time of a first and of a cached create,
and the registers / spill bytes of bk_user_smc_* per D from the compile log."""
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

GPL = """
__device__ bk_real quad(const bk_real* x, bk_real* g, const bk_real* m, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) {
        const bk_real d = x[e] - m[e], pd = p[e] * d;
        s += pd * d;
        g[e] = -pd;
    }
    return bk_real(-0.5) * s;
}
__device__ bk_real log_prior_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    return quad(x, g, p + 2 * BK_DIMS, p + 3 * BK_DIMS);
}
__device__ bk_real log_likelihood_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    return quad(x, g, p, p + BK_DIMS);
}
"""

KERNELS = {"rw": 0.2, "mala": 0.05, "hmc": 0.1}
DIMS = (2, 8, 16, 32, 50)
M, N, SEED, REPS = 1_000_000, 100, 1, 5


def regs(log):
    out = {}
    for k in ("bk_user_smc_rw", "bk_user_smc_mala", "bk_user_smc_hmc", "bk_user_eval_pl"):
        m = re.search(rf"Function properties for {k}\n.*?(\d+) bytes spill stores, (\d+) bytes spill loads\n"
                      rf".*?Used (\d+) registers", log, re.S)
        if m:
            out[k] = {"registers": int(m.group(3)), "spill_store_bytes": int(m.group(1)),
                      "spill_load_bytes": int(m.group(2))}
    return out


def main(out_path):
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch

    import bayes_kit_b200 as bk

    assert torch.cuda.is_available(), "time_user_smc.py needs a CUDA device"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": smi, "M": M, "N": N, "resample": "systematic", "dtype": "float32", "seed": SEED,
           "kernels": {"rw": {"scale": 0.2}, "mala": {"epsilon": 0.05}, "hmc": {"stepsize": 0.1, "steps": 5}},
           "runs_per_point": REPS, "compile_s": {}, "points": []}

    def params(D):
        g = np.random.default_rng(D)
        return np.zeros(D), np.ones(D), g.normal(size=D), 4 * np.ones(D)

    m0, p0, mu, pl = params(24)
    t0 = time.perf_counter()
    bk.CudaPriorLikModel(GPL, 24, params=np.concatenate([mu, pl, m0, p0]))
    t1 = time.perf_counter()
    bk.CudaPriorLikModel(GPL, 24, params=np.concatenate([mu, pl, m0, p0]))
    t2 = time.perf_counter()
    res["compile_s"] = {"first_create": t1 - t0, "cached_create": t2 - t1, "D": 24}

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def measure(model, D, kind):
        th0 = torch.randn(M, D, device="cuda", generator=torch.Generator(device="cuda").manual_seed(SEED))
        kern = {"rw": lambda: bk.metropolis_kernel(0.2), "mala": lambda: bk.mala_kernel(0.05),
                "hmc": lambda: bk.hmc_kernel(0.1, 5)}[kind]()
        times = []
        for rep in range(REPS + 1):
            smc = bk.TemperedLikelihoodSMC(model, M, N, th0, kern, resample="systematic", seed=SEED)
            torch.cuda.synchronize()
            e0.record()
            smc.run()
            e1.record()
            torch.cuda.synchronize()
            if rep > 0:                 # the first run warms up
                times.append(e0.elapsed_time(e1) / N)
            acc = float(smc.last_accept.float().mean())
            del smc
        return {"ms_per_temperature": float(np.median(times)), "spread_ms": [min(times), max(times)],
                "last_accept": acc}

    for D in DIMS:
        m0, p0, mu, pl = params(D)
        user = bk.CudaPriorLikModel(GPL, D, params=np.concatenate([mu, pl, m0, p0]))
        built = bk.GaussPriorLik(m0, p0, mu, pl)
        pt = {"D": D, "ptxas": regs(user.compile_log)}
        for kind in KERNELS:
            u, b = measure(user, D, kind), measure(built, D, kind)
            pt[kind] = {"user": u, "builtin": b, "user_over_builtin": u["ms_per_temperature"] / b["ms_per_temperature"]}
        res["points"].append(pt)
        print(json.dumps({"D": D, **{k: (pt[k]["user"]["ms_per_temperature"], pt[k]["builtin"]["ms_per_temperature"])
                                     for k in KERNELS}}), flush=True)
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": smi, "compile_s": res["compile_s"]}))


if __name__ == "__main__":
    main(sys.argv[1])
