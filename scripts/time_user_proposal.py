"""User-written CUDA proposals (CudaProposal): what a run-time compiled proposal costs against the built-in Gaussian
random walk doing the same work.  One GPU run, JSON to argv[1].

    python scripts/time_user_proposal.py profiles/r3_time_user_proposal.json

Records the card name and power limit; NVRTC compile time of a first and of a cached CudaProposal create and of the
fused model + proposal program (first and cached sampler construction); registers and spills of bk_user_mhp and
bk_user_propose from ptxas.  Timed (fp32, 2^20 chains, 10 draws per call, keep_draws=False, median of 7 calls after 2
warm-up calls, CUDA events around each call):
  (a) a user model (banana padded with standard normals) at D = 2, 8, 16, 32: Metropolis with a CudaProposal that
      restates the random walk (fused bk_user_mhp) against GaussianRW (fused bk_user_mh);
  (b) the same at D = 64 (three-launch path against the generic engine), and the built-in DiagGauss at D = 100 and
      DensePrecGauss at D = 1000 with the restated walk (three launches per draw) against GaussianRW on the generic
      engine (BK_FORCE_GENERIC=1, timed in a child process);
  (c) the log-normal walk and the independence sampler at D = 16 on the banana (fused)."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from _user_cuda import BANANA, INDEP, LOGNORMAL_NO_HELPER, RW, card, ptxas_report  # noqa: E402

C_ = 1 << 20
N_DRAWS, WARM, REPS = 10, 2, 7

def timed(sampler):
    import torch
    for _ in range(WARM):
        sampler.sample_n(N_DRAWS, keep_draws=False)
    ms = []
    for _ in range(REPS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        sampler.sample_n(N_DRAWS, keep_draws=False)
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    ms.sort()
    med = ms[len(ms) // 2]
    return {"median_ms": med, "min_ms": ms[0], "max_ms": ms[-1],
            "chain_draws_per_s": C_ * N_DRAWS / (med * 1e-3)}


def builtin(bk, kind, D):
    import numpy as np
    from oracle.models import DensePrecGauss
    rng = np.random.default_rng(0)
    if kind == "diag":
        return bk.DiagGauss(rng.normal(size=D), rng.uniform(0.5, 3.0, D))
    return bk.DensePrecGauss(DensePrecGauss.c2_precision(D, 0))


def child():
    """GaussianRW on the generic engine (BK_FORCE_GENERIC=1 in the environment) for the built-in plugins."""
    import bayes_kit_b200 as bk
    out = {}
    for kind, D in (("diag", 100), ("dense", 1000)):
        s = bk.Metropolis(builtin(bk, kind, D), bk.GaussianRW(1.0 / D ** 0.5), chains=C_, seed=1)
        out[f"{kind}_D{D}"] = timed(s)
        del s
    print("CHILD_JSON " + json.dumps(out))


def regs(log, kernel):
    """(registers, spill stores, spill loads) of `kernel` in a ptxas report."""
    r = ptxas_report(log).get(kernel)
    return None if r is None else {"registers": r["registers"], "spill_stores": r["spill_store_bytes"],
                                   "spill_loads": r["spill_load_bytes"]}


def main(out_path):
    import numpy as np
    import torch

    import bayes_kit_b200 as bk

    smi = card()
    res = {"gpu": smi, "chains": C_, "draws_per_call": N_DRAWS, "dtype": "float32",
           "timing": f"median of {REPS} calls after {WARM} warm-up calls, CUDA events", "compile": {}, "ptxas": {},
           "a_fused": {}, "b_three_launch": {}, "c_asymmetric": {}}
    t0 = time.perf_counter()
    prop = bk.CudaProposal(RW, 16, params=[0.3])
    res["compile"]["proposal_first_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    bk.CudaProposal(RW, 16, params=[0.3])
    res["compile"]["proposal_cached_s"] = time.perf_counter() - t0
    res["ptxas"]["bk_user_propose_D16"] = regs(prop.compile_log, "bk_user_propose")
    model = bk.CudaModel(BANANA, 16, params=[0.5])
    t0 = time.perf_counter()
    s = bk.Metropolis(model, prop, chains=8, seed=1)
    res["compile"]["fused_program_first_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    bk.Metropolis(model, prop, chains=8, seed=1)
    res["compile"]["fused_program_cached_s"] = time.perf_counter() - t0
    del s

    # (a) fused, and (b) the banana above the fused threshold
    for D in (2, 8, 16, 32, 64):
        model = bk.CudaModel(BANANA, D, params=[0.5])
        scale = 2.4 / np.sqrt(D)
        prop = bk.CudaProposal(RW, D, params=[scale])
        s = bk.Metropolis(model, prop, chains=C_, seed=1)
        mine = timed(s)
        if D <= 32:
            res["ptxas"][f"bk_user_mhp_D{D}"] = regs(s.compile_log, "bk_user_mhp")
            res["ptxas"][f"bk_user_mh_D{D}"] = regs(model.compile_log, "bk_user_mh")
        del s
        s = bk.Metropolis(model, bk.GaussianRW(scale), chains=C_, seed=1)
        ref = timed(s)
        del s
        key = "a_fused" if D <= 32 else "b_three_launch"
        res[key][f"banana_D{D}"] = {"cuda_proposal": mine, "gaussian_rw": ref,
                                    "ratio": mine["median_ms"] / ref["median_ms"]}
        torch.cuda.empty_cache()
    res["ptxas"]["bk_user_propose_D64"] = regs(prop.compile_log, "bk_user_propose")

    # (b) built-in plugins: three launches per draw against the generic engine (child process)
    env = dict(os.environ, BK_FORCE_GENERIC="1")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child"], capture_output=True, text=True, env=env)
    line = [l for l in r.stdout.splitlines() if l.startswith("CHILD_JSON ")]
    if not line:
        raise RuntimeError(f"child failed:\n{r.stdout}\n{r.stderr}")
    gen = json.loads(line[0][len("CHILD_JSON "):])
    for kind, D in (("diag", 100), ("dense", 1000)):
        prop = bk.CudaProposal(RW, D, params=[1.0 / D ** 0.5])
        s = bk.Metropolis(builtin(bk, kind, D), prop, chains=C_, seed=1)
        mine = timed(s)
        del s
        ref = gen[f"{kind}_D{D}"]
        res["b_three_launch"][f"{kind}_D{D}"] = {"cuda_proposal": mine, "gaussian_rw_generic": ref,
                                                 "ratio": mine["median_ms"] / ref["median_ms"]}
        res["ptxas"][f"bk_user_propose_D{D}"] = regs(prop.compile_log, "bk_user_propose")
        torch.cuda.empty_cache()

    # (c) asymmetric proposals, fused, D = 16
    D = 16
    model = bk.CudaModel(BANANA, D, params=[0.5])
    init = torch.rand(C_, D, device="cuda") + 0.5
    p = bk.CudaProposal(LOGNORMAL_NO_HELPER, D, params=[0.3])
    s = bk.MetropolisHastings(model, p, p.transition_lp, init=init, seed=1)
    res["c_asymmetric"]["lognormal_D16"] = timed(s)
    res["ptxas"]["bk_user_mhp_lognormal_D16"] = regs(s.compile_log, "bk_user_mhp")
    del s
    p = bk.CudaProposal(INDEP, D, params=np.concatenate([np.zeros(D), np.ones(D)]))
    s = bk.MetropolisHastings(model, p, p.transition_lp, chains=C_, seed=1)
    res["c_asymmetric"]["independence_D16"] = timed(s)
    res["ptxas"]["bk_user_mhp_independence_D16"] = regs(s.compile_log, "bk_user_mhp")
    del s

    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    if sys.argv[1:] == ["--child"]:
        child()
    else:
        main(sys.argv[1] if len(sys.argv) > 1 else "profiles/r3_time_user_proposal.json")
