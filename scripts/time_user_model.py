"""User-written CUDA models (CudaModel): what the fused one-thread-per-chain kernels buy over the generic engine, and
what the run-time compiled path costs against the hand-tuned built-in plugin.  One GPU run, JSON to argv[1].

    python scripts/time_user_model.py profiles/r3_time_user_model.json

Records the card name and power limit; NVRTC compile time of a first and of a cached create; HMCDiag L = 10
chain-steps/s with 2^20 fp32 chains at D in {2, 8, 16, 32, 64} for a banana padded with standard normals (fused vs
BK_FORCE_GENERIC=1) and for a diagonal Gaussian written as a user model (fused, generic) and as the built-in DiagGauss
plugin (its own fused kernel); registers and spills of the fused kernels per D from ptxas.  To measure the fused
kernels above the library's dispatch threshold, the script links a variant of the library in a temporary directory
with BK_USER_FUSED_MAX_D = 64 (the default build is left alone).  Per point: median of 7 timed calls after 2 warm-up
calls; wall time by CUDA events, kernel time by bk_profile_read (fused: BK_PROF_SAMPLER; generic: the model
evaluations, BK_PROF_GRAD) in separate calls."""
import glob
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "bayes-kit_b200")
MAX_D = 64


def build_variant(tmp):
    sys.path.insert(0, PKG)
    import build as b
    b.build()
    nvcc = b.NVCC
    obj = os.path.join(tmp, "user_model.o")
    subprocess.run([nvcc, *b.FLAGS, f"-DBK_USER_FUSED_MAX_D={MAX_D}", "-c", os.path.join(b.CSRC, "user_model.cu"),
                    "-o", obj], check=True)
    objs = [o for o in glob.glob(os.path.join(b.OBJ, "*.o")) if not o.endswith("user_model.o")] + [obj]
    lib = os.path.join(tmp, "libbk_b200.so")
    subprocess.run([nvcc, "-shared", "-o", lib, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart",
                    "static", "-Xcompiler", "-fPIC", "-ldl"], check=True)
    return lib


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


def main(out_path):
    tmp = tempfile.mkdtemp(prefix="bk_user_time_")
    os.environ["BK_LIB"] = build_variant(tmp)
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch

    import bayes_kit_b200 as bk
    from bayes_kit_b200 import _lib as L

    lib = L.lib()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": smi, "chains": 1 << 20, "steps_L": 10, "draws_per_call": 10, "dtype": "float32",
           "fused_max_d_of_variant": MAX_D, "compile_s": {}, "points": []}

    # NVRTC compile: first create (compile + load) and a cached create of the same (source, D, dtype)
    t0 = time.perf_counter()
    bk.CudaModel(BANANA, 24, params=[0.5])
    t1 = time.perf_counter()
    bk.CudaModel(BANANA, 24, params=[0.5])
    t2 = time.perf_counter()
    res["compile_s"] = {"first_create": t1 - t0, "cached_create": t2 - t1, "D": 24}

    C, n, Lsteps, eps = 1 << 20, 10, 10, 0.1
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fv, nl = L.f64(0), L.u64(0)

    def measure(model, generic):
        os.environ["BK_FORCE_GENERIC"] = "1" if generic else "0"
        s = bk.HMCDiag(model, eps, Lsteps, chains=C, seed=1)
        for _ in range(2):
            s.sample_n(n)
        walls = []
        for _ in range(7):
            e0.record()
            s.sample_n(n)
            e1.record()
            torch.cuda.synchronize()
            walls.append(e0.elapsed_time(e1))
        tag = L.PROF_GRAD if generic else L.PROF_SAMPLER
        lib.bk_profile_read(tag, fv, nl)
        lib.bk_profile_enable(1)
        kern = []
        for _ in range(5):
            s.sample_n(n)
            torch.cuda.synchronize()
            lib.bk_profile_read(tag, fv, nl)
            kern.append(fv.value)
        lib.bk_profile_enable(0)
        acc = float(s.last_accept.float().mean())
        del s
        torch.cuda.empty_cache()
        wall = float(np.median(walls))
        return {"wall_ms": wall, "kernel_ms": float(np.median(kern)), "chain_steps_per_s": C * n / (wall * 1e-3),
                "accept": acc}

    def regs(log):
        out = {}
        for k in ("bk_user_hmc", "bk_user_mala", "bk_user_mh", "bk_user_eval"):
            m = re.search(rf"Function properties for {k}\n.*?(\d+) bytes spill stores, (\d+) bytes spill loads\n"
                          rf".*?Used (\d+) registers", log, re.S)
            if m:
                out[k] = {"registers": int(m.group(3)), "spill_store_bytes": int(m.group(1)),
                          "spill_load_bytes": int(m.group(2))}
        return out

    rng = np.random.default_rng(0)
    for D in (2, 8, 16, 32, 64):
        ban = bk.CudaModel(BANANA, D, params=[0.5])
        mu, pr = rng.normal(size=D), rng.uniform(0.5, 3.0, D)
        diag_u = bk.CudaModel(DIAG, D, params=np.concatenate([mu, pr]))
        diag_b = bk.DiagGauss(mu, pr)
        pt = {"D": D, "banana_fused": measure(ban, False), "banana_generic": measure(ban, True),
              "diag_user_fused": measure(diag_u, False), "diag_user_generic": measure(diag_u, True),
              "diag_builtin_fused": measure(diag_b, False),
              "ptxas_banana": regs(ban.compile_log), "ptxas_diag": regs(diag_u.compile_log)}
        pt["banana_fused_over_generic"] = (pt["banana_fused"]["chain_steps_per_s"] /
                                           pt["banana_generic"]["chain_steps_per_s"])
        res["points"].append(pt)
        print(json.dumps({k: (v["chain_steps_per_s"] if isinstance(v, dict) and "wall_ms" in v else v)
                          for k, v in pt.items() if not k.startswith("ptxas")}), flush=True)
    os.environ["BK_FORCE_GENERIC"] = "0"
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": smi, "compile_s": res["compile_s"]}))


if __name__ == "__main__":
    main(sys.argv[1])
