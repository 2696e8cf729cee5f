"""Gradient proposals (CudaProposal(gradient=True)): what a run-time compiled proposal that reads the model's gradient
costs against bk.MALA doing the same work.  One GPU run, JSON to argv[1].

    python scripts/time_user_grad_proposal.py profiles/r3_time_user_grad_proposal.json

Records the card name and power limit, and the registers and spill stores ptxas reports for every kernel of a
gradient proposal (bk_user_mhp_grad, bk_user_propose_grad, bk_user_dh_grad).  Timed (fp32, 2^20 chains, 10 draws per
call, keep_draws=False, CUDA events around each call; the two sides alternate call by call, median of 7 calls each
after 2 warm-up calls each):
  (a) MALA restated as a gradient proposal against bk.MALA on a user model (banana padded with standard normals):
      fused bk_user_mhp_grad against fused bk_user_mala at D = 2, 8, 16, 32; the four-launch path against the generic
      engine's MALA at D = 40, 64 (BK_FORCE_GENERIC=1 for both sides: MALA would otherwise run the wide kernel);
  (b) the same on the built-in DiagGauss plugin at D = 100 (generic engine on both sides);
  (c) the Barker proposal (one uniform per coordinate, so D <= 64) at the same D on the banana."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from _user_cuda import BANANA, BARKER, MALA_G, card, ptxas_report  # noqa: E402

C_ = 1 << 20
N_DRAWS, WARM, REPS = 10, 2, 7


def _call_ms(sampler):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    sampler.sample_n(N_DRAWS, keep_draws=False)
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def _summary(ms):
    ms = sorted(ms)
    med = ms[len(ms) // 2]
    return {"median_ms": med, "min_ms": ms[0], "max_ms": ms[-1], "chain_draws_per_s": C_ * N_DRAWS / (med * 1e-3)}


def timed(*samplers):
    """the samplers timed call by call in turn"""
    for s in samplers:
        for _ in range(WARM):
            s.sample_n(N_DRAWS, keep_draws=False)
    ms = [[] for _ in samplers]
    for _ in range(REPS):
        for k, s in enumerate(samplers):
            ms[k].append(_call_ms(s))
    return [_summary(m) for m in ms]


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
           "timing": f"two sides alternating call by call; median of {REPS} calls each after {WARM} warm-up calls "
                     "each, CUDA events", "ptxas": {}, "a_mala_user": {}, "b_mala_diag": {}, "c_barker": {}}

    def mala_params(eps):
        return [eps, float(np.sqrt(2 * eps)), -0.25 / eps]

    for D in (2, 8, 16, 32, 40, 64):
        generic = D > 32
        os.environ["BK_FORCE_GENERIC"] = "1" if generic else "0"
        model = bk.CudaModel(BANANA, D, params=[0.5])
        eps = 0.6 / D ** (1 / 3)
        prop = bk.CudaProposal(MALA_G, D, params=mala_params(eps), gradient=True)
        g = bk.MetropolisHastings(model, prop, prop.transition_lp, chains=C_, seed=1)
        m = bk.MALA(model, eps, chains=C_, seed=1)
        tg, tm = timed(g, m)
        res["a_mala_user"][f"D{D}"] = {"engine": "four launches / generic" if generic else
                                       "bk_user_mhp_grad / bk_user_mala", "grad_proposal": tg, "mala": tm,
                                       "ratio": tg["median_ms"] / tm["median_ms"]}
        if generic:
            res["ptxas"][f"bk_user_propose_grad_mala_D{D}"] = regs(prop.compile_log, "bk_user_propose_grad")
            res["ptxas"][f"bk_user_dh_grad_mala_D{D}"] = regs(prop.compile_log, "bk_user_dh_grad")
        else:
            res["ptxas"][f"bk_user_mhp_grad_mala_D{D}"] = regs(g.compile_log, "bk_user_mhp_grad")
        del g, m
        bp = bk.CudaProposal(BARKER, D, params=[1.6 / D ** (1 / 6)], uniforms=D, gradient=True)
        b = bk.MetropolisHastings(model, bp, bp.transition_lp, chains=C_, seed=1)
        (tb,) = timed(b)
        res["c_barker"][f"D{D}"] = {"engine": "four launches" if generic else "bk_user_mhp_grad", "time": tb,
                                    "accept_rate": float(b.last_accept.float().mean())}
        if generic:
            res["ptxas"][f"bk_user_propose_grad_barker_D{D}"] = regs(bp.compile_log, "bk_user_propose_grad")
            res["ptxas"][f"bk_user_dh_grad_barker_D{D}"] = regs(bp.compile_log, "bk_user_dh_grad")
        else:
            res["ptxas"][f"bk_user_mhp_grad_barker_D{D}"] = regs(b.compile_log, "bk_user_mhp_grad")
        del b, model
        torch.cuda.empty_cache()

    os.environ["BK_FORCE_GENERIC"] = "1"
    D = 100
    rng = np.random.default_rng(0)
    model = bk.DiagGauss(rng.normal(size=D), rng.uniform(0.5, 3.0, D))
    eps = 0.1
    prop = bk.CudaProposal(MALA_G, D, params=mala_params(eps), gradient=True)
    g = bk.MetropolisHastings(model, prop, prop.transition_lp, chains=C_, seed=1)
    m = bk.MALA(model, eps, chains=C_, seed=1)
    tg, tm = timed(g, m)
    res["b_mala_diag"][f"D{D}"] = {"engine": "four launches / generic", "grad_proposal": tg, "mala": tm,
                                   "ratio": tg["median_ms"] / tm["median_ms"]}
    res["ptxas"][f"bk_user_propose_grad_mala_D{D}"] = regs(prop.compile_log, "bk_user_propose_grad")
    res["ptxas"][f"bk_user_dh_grad_mala_D{D}"] = regs(prop.compile_log, "bk_user_dh_grad")
    os.environ["BK_FORCE_GENERIC"] = "0"

    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "profiles/r3_time_user_grad_proposal.json")
