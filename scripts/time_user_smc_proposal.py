"""TemperedLikelihoodSMC with a user-written proposal as the move (proposal_kernel, bk_user_smc_mhp) against the
built-in random-walk move of the same user model (metropolis_kernel, bk_user_smc_rw).  One GPU run, JSON to argv[1].

    python scripts/time_user_smc_proposal.py profiles/r3_time_user_smc_proposal.json

Workload: the c4 shape (M = 10^6 particles, N = 100 temperatures, systematic resampling, fp32, seed 1) on GaussPriorLik
(m0 = 0, p0 = 1, pl = 4, mu ~ N(0, I)) written as a CudaPriorLikModel, at D in {2, 8, 16, 32, 50}: the random walk
restated as a CudaProposal (scale 0.2, no transition density) against metropolis_kernel(0.2).  Both read the same
Philox words and do the same arithmetic, so the two runs give the same particles.  One more row: the log-normal walk
(s = 0.4, with its Hastings term) on a Gamma x Poisson model at D = 16, against metropolis_kernel(0.2) on that model.
Per point: ms per temperature from CUDA events around run() (which ends in a synchronise), median of 5 runs after one
warm-up run, the two kernels alternating.  Also records the card name and power limit, the time of a first (NVRTC
compile + load) and of a cached bk_smc_cuda_prepare, and the registers / spill bytes of bk_user_smc_mhp and
bk_user_smc_rw from the compile logs."""
import ctypes as C
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

# Gamma(a, rate b) priors x Poisson likelihoods, params = [a, b, n, S (D)]
GAMMA_POIS = """
__device__ bk_real log_prior_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) {
        if (!(x[e] > 0)) return log(bk_real(0));
        s += (p[0] - 1) * log(x[e]) - p[1] * x[e];
        g[e] = (p[0] - 1) / x[e] - p[1];
    }
    return s;
}
__device__ bk_real log_likelihood_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) {
        if (!(x[e] > 0)) return log(bk_real(0));
        s += p[3 + e] * log(x[e]) - p[2] * x[e];
        g[e] = p[3 + e] / x[e] - p[2];
    }
    return s;
}
"""

WALK = """
__device__ void propose(const bk_real* theta, bk_real* q, const bk_real* z, const bk_real* u, const bk_real* p) {
    for (int e = 0; e < BK_DIMS; ++e) q[e] = theta[e] + p[0] * z[e];
}
"""

LOGNORMAL = """
__device__ void propose(const bk_real* theta, bk_real* q, const bk_real* z, const bk_real* u, const bk_real* p) {
    for (int e = 0; e < BK_DIMS; ++e) q[e] = theta[e] * exp(p[0] * z[e]);
}
__device__ bk_real transition_log_density(const bk_real* to, const bk_real* from, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) {
        const bk_real d = (log(to[e]) - log(from[e])) / p[0];
        s += bk_real(-0.5) * (d * d) - log(to[e]);
    }
    return s;
}
"""

DIMS = (2, 8, 16, 32, 50)
M, N, SEED, REPS, SCALE = 1_000_000, 100, 1, 5, 0.2


def regs(log, kernels):
    out = {}
    for k in kernels:
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
    from bayes_kit_b200 import _lib as L

    assert torch.cuda.is_available(), "time_user_smc_proposal.py needs a CUDA device"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": smi, "M": M, "N": N, "resample": "systematic", "dtype": "float32", "seed": SEED,
           "walk": {"scale": SCALE}, "lognormal": {"s": 0.4, "D": 16}, "runs_per_point": REPS, "prepare_s": {},
           "points": []}

    def gpl(D):
        g = np.random.default_rng(D)
        m0, p0, mu, pl = np.zeros(D), np.ones(D), g.normal(size=D), 4 * np.ones(D)
        return bk.CudaPriorLikModel(GPL, D, params=np.concatenate([mu, pl, m0, p0]))

    # first (NVRTC compile + load) and cached prepare of one (model, proposal) pair
    model, prop = gpl(24), bk.CudaProposal(WALK, 24, params=[SCALE], transition=False)
    log = C.create_string_buffer(1 << 20)
    t0 = time.perf_counter()
    L.check(L.lib().bk_smc_cuda_prepare(model.handle, prop.handle, log, len(log)))
    t1 = time.perf_counter()
    L.check(L.lib().bk_smc_cuda_prepare(model.handle, prop.handle, log, len(log)))
    t2 = time.perf_counter()
    res["prepare_s"] = {"first": t1 - t0, "cached": t2 - t1, "D": 24}

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def measure(model, D, kernels, init):
        """kernels: {name: kernel}; the runs alternate between them."""
        th0 = init(D)
        times = {k: [] for k in kernels}
        out = {}
        for rep in range(REPS + 1):
            for name, kern in kernels.items():
                smc = bk.TemperedLikelihoodSMC(model, M, N, th0, kern, resample="systematic", seed=SEED)
                torch.cuda.synchronize()
                e0.record()
                smc.run()
                e1.record()
                torch.cuda.synchronize()
                if rep > 0:                 # the first run warms up
                    times[name].append(e0.elapsed_time(e1) / N)
                out[name] = {"last_accept": float(smc.last_accept.float().mean()), "thetas": smc.thetas.clone()}
                del smc
        for name in kernels:
            t = times[name]
            out[name].update({"ms_per_temperature": float(np.median(t)), "spread_ms": [min(t), max(t)]})
        return out

    normal = lambda D: torch.randn(M, D, device="cuda", generator=torch.Generator(device="cuda").manual_seed(SEED))
    for D in DIMS:
        model = gpl(D)
        kern = bk.proposal_kernel(bk.CudaProposal(WALK, D, params=[SCALE], transition=False))
        smc = bk.TemperedLikelihoodSMC(model, 4, 1, torch.zeros(4, D, device="cuda"), kern)
        pt = {"D": D, "model": "gauss_prior_lik", "ptxas": {**regs(smc.compile_log, ["bk_user_smc_mhp"]),
                                                             **regs(model.compile_log, ["bk_user_smc_rw"])}}
        r = measure(model, D, {"proposal_walk": kern, "metropolis_kernel": bk.metropolis_kernel(SCALE)}, normal)
        pt["same_particles"] = bool(torch.equal(r["proposal_walk"].pop("thetas"), r["metropolis_kernel"].pop("thetas")))
        pt.update(r)
        pt["proposal_over_rw"] = r["proposal_walk"]["ms_per_temperature"] / r["metropolis_kernel"]["ms_per_temperature"]
        res["points"].append(pt)
        print(json.dumps({"D": D, "ms": [r[k]["ms_per_temperature"] for k in r], "ratio": pt["proposal_over_rw"],
                          "same": pt["same_particles"]}), flush=True)
        torch.cuda.empty_cache()

    D = 16
    a, b, n = 2.0, 1.0, 4.0
    S = np.random.default_rng(16).integers(1, 10, D).astype(np.float64)
    model = bk.CudaPriorLikModel(GAMMA_POIS, D, params=np.concatenate([[a, b, n], S]))
    kern = bk.proposal_kernel(bk.CudaProposal(LOGNORMAL, D, params=[0.4], transition=True))
    smc = bk.TemperedLikelihoodSMC(model, 4, 1, torch.ones(4, D, device="cuda"), kern)
    gamma = lambda D: torch.distributions.Gamma(torch.full((D,), a, device="cuda"), torch.full((D,), b, device="cuda")
                                                ).sample((M,))
    torch.manual_seed(SEED)
    r = measure(model, D, {"lognormal": kern, "metropolis_kernel": bk.metropolis_kernel(SCALE)}, gamma)
    for k in r:
        r[k].pop("thetas")
    pt = {"D": D, "model": "gamma_poisson", "ptxas": {**regs(smc.compile_log, ["bk_user_smc_mhp"]),
                                                       **regs(model.compile_log, ["bk_user_smc_rw"])}, **r,
          "proposal_over_rw": r["lognormal"]["ms_per_temperature"] / r["metropolis_kernel"]["ms_per_temperature"]}
    res["points"].append(pt)
    print(json.dumps({"D": D, "gamma_poisson": [r[k]["ms_per_temperature"] for k in r]}), flush=True)

    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": smi, "prepare_s": res["prepare_s"]}))


if __name__ == "__main__":
    main(sys.argv[1])
