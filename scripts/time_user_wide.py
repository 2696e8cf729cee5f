"""User-written CUDA models past the register-resident kernels (32 < D <= 256): what the wide kernels (trajectory in
shared memory, one warp of 32 chains per CTA) buy over the generic engine.  One GPU run, JSON to argv[1].

    python scripts/time_user_wide.py profiles/r3_time_user_wide.json

Records the card name and power limit; NVRTC prepare time of the wide program, first and cached; for HMCDiag
(L = 10), MALA and RW-Metropolis with 2^20 fp32 chains and 10 draws per call, at D in {48, 64, 96, 128, 192, 256},
for a banana padded with standard normals and for a diagonal Gaussian, both written as user models: the wide kernel
and BK_FORCE_GENERIC=1 alternated call by call on two samplers of the same chains (median of 7 timed calls after 2
warm-up calls each, CUDA events), the accept rates of both, and ptxas's registers, shared memory and spills of the
three wide kernels; and one point at 4096 chains, a size bound by launches and the host.  Where the library's
USER_WIDE_MAX_D is below 256 the script links a variant with BK_USER_WIDE_MAX_D = 256 in a temporary directory
(the default build is left alone)."""
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(os.path.dirname(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from _user_cuda import BANANA, DIAG, WIDE_MAX_D, build_variant, card, ptxas_report  # noqa: E402

MAX_D = 256
DIMS = (48, 64, 96, 128, 192, 256)


def main(out_path):
    tmp = tempfile.mkdtemp(prefix="bk_user_wide_")
    if WIDE_MAX_D < MAX_D:
        os.environ["BK_LIB"] = build_variant(tmp, f"BK_USER_WIDE_MAX_D={MAX_D}")
    import ctypes as C

    import numpy as np
    import torch

    import bayes_kit_b200 as bk
    from bayes_kit_b200 import _lib as L

    lib = L.lib()
    smi = card()
    Cn, n, Lsteps = 1 << 20, 10, 10
    res = {"gpu": smi, "chains": Cn, "hmc_steps_L": Lsteps, "draws_per_call": n, "dtype": "float32",
           "library_wide_max_d": WIDE_MAX_D, "timed_calls": 7, "warmup_calls": 2, "points": []}
    os.environ["BK_FORCE_GENERIC"] = "0"

    # NVRTC: the first prepare compiles and loads the wide program, the second finds it in the cache
    m = bk.CudaModel(BANANA, 72, params=[0.5])
    log = C.create_string_buffer(1 << 20)
    t0 = time.perf_counter()
    L.check(lib.bk_user_wide_prepare(m.handle, log, len(log)))
    t1 = time.perf_counter()
    L.check(lib.bk_user_wide_prepare(m.handle, log, len(log)))
    t2 = time.perf_counter()
    res["prepare_s"] = {"first": t1 - t0, "cached": t2 - t1, "D": 72}

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def makers(D):
        return {"hmc": lambda mod, C_: bk.HMCDiag(mod, 0.1, Lsteps, chains=C_, seed=1),
                "mala": lambda mod, C_: bk.MALA(mod, 0.05, chains=C_, seed=1),
                "mh": lambda mod, C_: bk.Metropolis(mod, bk.GaussianRW(1.5 / D ** 0.5), chains=C_, seed=1)}

    def call(s, generic):
        os.environ["BK_FORCE_GENERIC"] = "1" if generic else "0"
        e0.record()
        s.sample_n(n)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def measure(make, model, C_):
        os.environ["BK_FORCE_GENERIC"] = "0"
        w = make(model, C_)
        g = make(model, C_)
        log = w.compile_log
        walls = {"wide": [], "generic": []}
        for k in range(9):   # alternate the engines call by call: 2 warm-ups, then 7 timed
            tw, tg = call(w, False), call(g, True)
            if k >= 2:
                walls["wide"].append(tw)
                walls["generic"].append(tg)
        out = {}
        for eng, s in (("wide", w), ("generic", g)):
            wall = float(np.median(walls[eng]))
            out[eng] = {"wall_ms": wall, "chain_draws_per_s": C_ * n / (wall * 1e-3),
                        "accept": float(s.last_accept.float().mean())}
        out["wide_over_generic"] = out["wide"]["chain_draws_per_s"] / out["generic"]["chain_draws_per_s"]
        del w, g
        torch.cuda.empty_cache()
        return out, log

    rng = np.random.default_rng(0)
    for D in DIMS:
        mu, pr = rng.normal(size=D), rng.uniform(0.5, 3.0, D)
        models = {"banana": bk.CudaModel(BANANA, D, params=[0.5]),
                  "diag": bk.CudaModel(DIAG, D, params=np.concatenate([mu, pr]))}
        pt = {"D": D, "smem_bytes_per_cta": {"hmc": 3 * 32 * (D | 1) * 4, "mala": 3 * 32 * (D | 1) * 4,
                                             "mh": 2 * 32 * (D | 1) * 4}}
        for mname, mod in models.items():
            for sname, make in makers(D).items():
                r, log = measure(make, mod, Cn)
                pt[f"{mname}_{sname}"] = r
                if sname == "hmc":
                    pt[f"ptxas_{mname}"] = ptxas_report(log)
                print(json.dumps({"D": D, "model": mname, "sampler": sname,
                                  "wide": r["wide"]["chain_draws_per_s"], "generic": r["generic"]["chain_draws_per_s"],
                                  "ratio": r["wide_over_generic"], "acc": (r["wide"]["accept"],
                                                                           r["generic"]["accept"])}), flush=True)
        res["points"].append(pt)

    # a size bound by launches and the host
    small = {"chains": 4096, "D": 64}
    mod = bk.CudaModel(BANANA, 64, params=[0.5])
    for sname, make in makers(64).items():
        small[sname], _ = measure(make, mod, 4096)
    res["small"] = small
    print(json.dumps({"small": {k: v["wide_over_generic"] for k, v in small.items() if isinstance(v, dict)}}))

    os.environ["BK_FORCE_GENERIC"] = "0"
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": smi, "prepare_s": res["prepare_s"]}))


if __name__ == "__main__":
    main(sys.argv[1])
