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
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from _user_cuda import GAMMA_POIS, GPL, LOGNORMAL_NO_HELPER, WALK, card, ptxas_report  # noqa: E402

DIMS = (2, 8, 16, 32, 50)
M, N, SEED, REPS, SCALE = 1_000_000, 100, 1, 5, 0.2


def regs(log, kernels):
    rep = ptxas_report(log)
    return {k: {f: rep[k][f] for f in ("registers", "spill_store_bytes", "spill_load_bytes")}
            for k in kernels if k in rep}


def main(out_path):
    import numpy as np
    import torch

    import bayes_kit_b200 as bk
    from bayes_kit_b200 import _lib as L

    assert torch.cuda.is_available(), "time_user_smc_proposal.py needs a CUDA device"
    smi = card()
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
    kern = bk.proposal_kernel(bk.CudaProposal(LOGNORMAL_NO_HELPER, D, params=[0.4], transition=True))
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
