"""TemperedLikelihoodSMC with several MCMC moves per temperature (moves=k).  One GPU run, JSON to argv[1] (default
profiles/r3_time_smc_moves.json).

    python scripts/time_smc_moves.py profiles/r3_time_smc_moves.json

Workload: the c4 shape (M = 10^6 fp32 particles, D = 50, N = 100 temperatures, systematic resampling, seed 1) on
GaussPriorLik (m0 = 0, p0 = 1, pl = 4, mu ~ N(0, I); posterior N(0.8 mu, 0.2 I)), as the built-in plugin and restated as
a CudaPriorLikModel, with moves in {1, 2, 5, 10} and the RW (scale 0.2), MALA (epsilon 0.05) and HMC (stepsize 0.1,
L = 5) kernels.  Per configuration: ms per temperature from CUDA events around run() (which ends in a synchronise),
the median of 5 runs after one warm-up run, the configurations alternating within each round; the marginal cost of an
extra move (t_k - t_1) / (k - 1) next to t_1; and, from the last run, the max-abs error of the final particles' mean
against 0.8 mu and the number of distinct particles the last resampling kept.  Also records the card name and power
limit, and the ptxas report of the user model's multi-move kernels."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from _user_cuda import GPL, card, ptxas_report  # noqa: E402

M, D, N, SEED, REPS = 1_000_000, 50, 100, 1, 5
MOVES = (1, 2, 5, 10)
KERNELS = {"rw": (0.2,), "mala": (0.05,), "hmc": (0.1, 5)}


def main(out_path):
    import numpy as np
    import torch

    import bayes_kit_b200 as bk

    assert torch.cuda.is_available(), "time_smc_moves.py needs a CUDA device"
    g = np.random.default_rng(D)
    m0, p0, mu, pl = np.zeros(D), np.ones(D), g.normal(size=D), 4 * np.ones(D)
    th0 = torch.from_numpy(np.random.default_rng(SEED).normal(size=(M, D))).float().cuda()
    models = {"builtin": bk.GaussPriorLik(m0, p0, mu, pl, dtype=torch.float32),
              "user": bk.CudaPriorLikModel(GPL, D, params=np.concatenate([mu, pl, m0, p0]), dtype=torch.float32)}
    make_kernel = {"rw": bk.metropolis_kernel, "mala": bk.mala_kernel, "hmc": bk.hmc_kernel}
    res = {"gpu": card(), "M": M, "D": D, "N": N, "resample": "systematic", "dtype": "float32", "seed": SEED,
           "kernels": {"rw": {"scale": 0.2}, "mala": {"epsilon": 0.05}, "hmc": {"stepsize": 0.1, "steps": 5}},
           "moves": list(MOVES), "runs_per_point": REPS, "ptxas": {}, "points": []}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    configs = [(mn, kn, k) for mn in models for kn in KERNELS for k in MOVES]
    smcs, times, last = {}, {c: [] for c in configs}, {}
    for c in configs:
        mn, kn, k = c
        smcs[c] = bk.TemperedLikelihoodSMC(models[mn], M, N, th0, make_kernel[kn](*KERNELS[kn]),
                                           resample="systematic", seed=SEED, moves=k)
        if mn == "user" and k > 1 and smcs[c].compile_log:
            res["ptxas"].setdefault(kn, {k2: {f: v[f] for f in ("registers", "spill_store_bytes", "spill_load_bytes")}
                                         for k2, v in ptxas_report(smcs[c].compile_log).items()})

    def one(c):
        s = smcs[c]
        s.thetas = th0
        s._pending = False
        e0.record()
        s.run()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / N, s

    for c in configs:   # warm-up
        one(c)
    for _ in range(REPS):   # alternate the configurations within every round
        for c in configs:
            t, s = one(c)
            times[c].append(t)
            last[c] = s
    for c in configs:
        mn, kn, k = c
        s = last[c]
        mean = s.thetas.double().mean(0).cpu().numpy()
        t = float(np.median(times[c]))
        t1 = float(np.median(times[(mn, kn, 1)]))
        res["points"].append({"model": mn, "kernel": kn, "moves": k, "ms_per_temperature": t,
                              "runs_ms": times[c], "ms_per_extra_move": (t - t1) / (k - 1) if k > 1 else None,
                              "ms_per_temperature_moves_1": t1,
                              "posterior_mean_max_abs_err": float(np.abs(mean - 0.8 * mu).max()),
                              "unique_particles": int(torch.unique(s.last_indices).numel()),
                              "mean_accepted_moves_last_step": float(s.last_accept.float().mean())})
        p = res["points"][-1]
        print(f"{mn:8s} {kn:5s} moves={k:3d}  {t:8.3f} ms/temp  +{p['ms_per_extra_move'] or 0:7.3f} ms/move  "
              f"err={p['posterior_mean_max_abs_err']:.3f}  unique={p['unique_particles']}", flush=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(res["gpu"])


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_time_smc_moves.json"))
