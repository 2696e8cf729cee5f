"""What the tests and timing scripts of user-written CUDA programs share: the CUDA sources of models and proposals, their
NumPy twins, the test helpers, and an NVRTC harness that compiles a program's text the way user_model.cu does (a
model's program cannot be created without a device, so the host tests compile its text here instead).

Imports without a GPU: nothing here touches a device until it is called."""
import ctypes as C
import glob
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from _dev import np_

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "bayes-kit_b200")
CSRC = os.path.join(PKG, "csrc")
HEADER = os.path.join(ROOT, "include", "bk.h")


def _define(path, name):
    with open(path) as f:
        return int(re.search(rf"#define {name} (\d+)", f.read()).group(1))


FUSED_MAX_D = _define(os.path.join(CSRC, "model.h"), "BK_USER_FUSED_MAX_D")
WIDE_MAX_D = _define(os.path.join(CSRC, "model.h"), "BK_USER_WIDE_MAX_D")
SMC_MAX_WORLD = _define(HEADER, "BK_SMC_MAX_WORLD")
SMC_MAILBOX_BYTES = _define(HEADER, "BK_SMC_MAILBOX_BYTES")
# BK_PROGRAM_* (user_kernels.cuh)
PROGRAM_MODEL, PROGRAM_PROPOSAL, PROGRAM_MODEL_PROPOSAL, PROGRAM_DRGHMC, PROGRAM_STRETCH, PROGRAM_WIDE = range(1, 7)

# ---- models -----------------------------------------------------------------------------------------------------------
# banana: x0 ~ N(0, 1), x1 - b x0^2 ~ N(0, 1), every further coordinate N(0, 1); params = [b]
BANANA = """
__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* params) {
    const bk_real b = params[0], half = 0.5, two = 2;
    const bk_real u = x[1] - b * x[0] * x[0];
    bk_real lp = -half * (x[0] * x[0]) - half * (u * u);
    g[0] = -x[0] + two * b * x[0] * u;
    g[1] = -u;
    for (int e = 2; e < BK_DIMS; ++e) {
        lp -= half * (x[e] * x[e]);
        g[e] = -x[e];
    }
    return lp;
}
"""

# the banana, also defined at D = 1 (then a standard normal); params = [b]
BANANA_1 = """
__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* params) {
#if BK_DIMS == 1
    g[0] = -x[0];
    return bk_real(-0.5) * (x[0] * x[0]);
#else
    const bk_real b = params[0], half = 0.5, two = 2;
    const bk_real u = x[1] - b * x[0] * x[0];
    bk_real lp = -half * (x[0] * x[0]) - half * (u * u);
    g[0] = -x[0] + two * b * x[0] * u;
    g[1] = -u;
    for (int e = 2; e < BK_DIMS; ++e) {
        lp -= half * (x[e] * x[e]);
        g[e] = -x[e];
    }
    return lp;
#endif
}
"""

# diagonal Gaussian, params = [mu (D), prec (D)]: the built-in DiagGauss restated
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

# a standard normal
PLAIN = """
__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) { s += x[e] * x[e]; g[e] = -x[e]; }
    return bk_real(-0.5) * s;
}
"""

# prior N(0, I), likelihood N(1, I)
PRIOR_LIK = """
__device__ bk_real log_prior_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) { s += x[e] * x[e]; g[e] = -x[e]; }
    return bk_real(-0.5) * s;
}
__device__ bk_real log_likelihood_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) { const bk_real d = x[e] - 1; s += d * d; g[e] = -d; }
    return bk_real(-0.5) * s;
}
"""

# prior N(0, I), likelihood N(1, diag(1 / w)) with weights params = [w (D)]
PRIOR_LIK_WEIGHTED = """
__device__ bk_real log_prior_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) { s += x[e] * x[e]; g[e] = -x[e]; }
    return bk_real(-0.5) * s;
}
__device__ bk_real log_likelihood_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) { const bk_real d = x[e] - 1; s += p[e] * d * d; g[e] = -p[e] * d; }
    return bk_real(-0.5) * s;
}
"""

# GaussPriorLik restated: params = [mu (D), pl (D), m0 (D), p0 (D)]
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

# the reference's beta-binomial on the logit scale restated: params = [alpha, beta, x, N, log C(N, x), log B(alpha, beta)]
BINOM = """
__device__ void logs(bk_real th, bk_real& lp1, bk_real& l1m, bk_real& p) {
    const bk_real e = exp(-fabs(th)), l = log1p(e);
    lp1 = th >= 0 ? -l : th - l;
    l1m = th >= 0 ? -th - l : -l;
    p = th >= 0 ? bk_real(1) / (1 + e) : e / (1 + e);
}
__device__ bk_real log_prior_gradient(const bk_real* x, bk_real* g, const bk_real* q) {
    bk_real lp1, l1m, p;
    logs(x[0], lp1, l1m, p);
    g[0] = q[0] - (q[0] + q[1]) * p;
    return (q[0] * lp1 + q[1] * l1m) - q[5];
}
__device__ bk_real log_likelihood_gradient(const bk_real* x, bk_real* g, const bk_real* q) {
    bk_real lp1, l1m, p;
    logs(x[0], lp1, l1m, p);
    g[0] = q[2] - q[3] * p;
    return (q[4] + q[2] * lp1) + (q[3] - q[2]) * l1m;
}
"""

# no built-in counterpart: prior N(0, tau^2 I), likelihood 1/2 N(x; mu, s^2 I) + 1/2 N(x; -mu, s^2 I) (up to its
# normalising constant), a bimodal posterior.  params = [mu (D), 1 / s^2, 1 / tau^2]
MIXTURE_MODEL = """
__device__ bk_real log_prior_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    const bk_real p0 = p[BK_DIMS + 1];
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) { s += x[e] * x[e]; g[e] = -p0 * x[e]; }
    return bk_real(-0.5) * p0 * s;
}
__device__ bk_real log_likelihood_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    const bk_real* mu = p;
    const bk_real pl = p[BK_DIMS];
    bk_real sa = 0, sb = 0;
    for (int e = 0; e < BK_DIMS; ++e) {
        const bk_real da = x[e] - mu[e], db = x[e] + mu[e];
        sa += da * da;
        sb += db * db;
    }
    const bk_real a = bk_real(-0.5) * pl * sa, b = bk_real(-0.5) * pl * sb;
    const bk_real m = a > b ? a : b;
    const bk_real ea = exp(a - m), eb = exp(b - m), z = ea + eb;
    const bk_real wa = ea / z, wb = eb / z;
    for (int e = 0; e < BK_DIMS; ++e) g[e] = -pl * (wa * (x[e] - mu[e]) + wb * (x[e] + mu[e]));
    return m + log(bk_real(0.5) * z);
}
"""
MIX_MU = np.array([1.5, -1.5, 1.5, -1.5])
MIX_S, MIX_TAU = 0.5, 2.0

# independent Gamma(a, rate b) priors and Poisson likelihoods on positive rates: coordinate e saw S_e events in
# n intervals.  params = [a, b, n, S (D)]; the tempered posterior at t is Gamma(a + t S_e, b + t n).
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

# ---- proposals --------------------------------------------------------------------------------------------------------
# the Gaussian random walk restated, params = [scale]
RW = """
__device__ void propose(const bk_real* theta, bk_real* q, const bk_real* z, const bk_real* u, const bk_real* p) {
    for (int e = 0; e < BK_DIMS; ++e) q[e] = theta[e] + p[0] * z[e];
}
__device__ bk_real transition_log_density(const bk_real* to, const bk_real* from, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) { const bk_real d = to[e] - from[e]; s += d * d; }
    return bk_real(-0.5) * s / (p[0] * p[0]);
}
"""

# the random walk without its transition density, params = [scale]
WALK = """
__device__ void propose(const bk_real* theta, bk_real* q, const bk_real* z, const bk_real* u, const bk_real* p) {
    for (int e = 0; e < BK_DIMS; ++e) q[e] = theta[e] + p[0] * z[e];
}
"""

# independence sampler N(m, diag s^2), params = [m (D), s (D)]
INDEP = """
__device__ void propose(const bk_real* theta, bk_real* q, const bk_real* z, const bk_real* u, const bk_real* p) {
    for (int e = 0; e < BK_DIMS; ++e) q[e] = p[e] + p[BK_DIMS + e] * z[e];
}
__device__ bk_real transition_log_density(const bk_real* to, const bk_real* from, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) {
        const bk_real d = (to[e] - p[e]) / p[BK_DIMS + e];
        s += bk_real(-0.5) * (d * d) - log(p[BK_DIMS + e]);
    }
    return s;
}
"""

# multiplicative (log-normal) walk for positive parameters, params = [s]; the Jacobian -log(to) makes it asymmetric.
# Its helper `sq` may share a model's helper's name: each source is compiled in a namespace of its own.
LOGNORMAL = """
__device__ bk_real sq(bk_real x) { return x * x; }
__device__ void propose(const bk_real* theta, bk_real* q, const bk_real* z, const bk_real* u, const bk_real* p) {
    for (int e = 0; e < BK_DIMS; ++e) q[e] = theta[e] * exp(p[0] * z[e]);
}
__device__ bk_real transition_log_density(const bk_real* to, const bk_real* from, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) {
        const bk_real d = (log(to[e]) - log(from[e])) / p[0];
        s += bk_real(-0.5) * sq(d) - log(to[e]);
    }
    return s;
}
"""

# the log-normal walk with the square written out (the text the timing scripts measure)
LOGNORMAL_NO_HELPER = """
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

# random-scan single-site walk: u[0] picks the coordinate, z[0] is the step; params = [s]
RSCAN = """
__device__ void propose(const bk_real* theta, bk_real* q, const bk_real* z, const bk_real* u, const bk_real* p) {
    for (int e = 0; e < BK_DIMS; ++e) q[e] = theta[e];
    int j = (int)(u[0] * BK_DIMS);
    if (j > BK_DIMS - 1) j = BK_DIMS - 1;
    q[j] = theta[j] + p[0] * z[0];
}
__device__ bk_real transition_log_density(const bk_real* to, const bk_real* from, const bk_real* p) { return 0; }
"""

# a two-scale mixture walk with an extra small jitter: 2 D normals (more than D, so the stream skips the accept block)
# and two uniforms; params = [s1, s2, w]
MIXTURE_WALK = """
__device__ void propose(const bk_real* theta, bk_real* q, const bk_real* z, const bk_real* u, const bk_real* p) {
    const bk_real s = (u[0] < p[2] ? p[0] : p[1]) * (bk_real(0.5) + u[1]);
    for (int e = 0; e < BK_DIMS; ++e) q[e] = theta[e] + s * z[e] + bk_real(0.01) * z[BK_DIMS + e];
}
"""

# MALA as a gradient proposal, params = [eps, sqrt(2 eps), -1 / (4 eps)]
MALA_G = """
__device__ void propose(const bk_real* th, const bk_real* g, bk_real* q, const bk_real* z, const bk_real* u,
                        const bk_real* p) {
    for (int e = 0; e < BK_DIMS; ++e) q[e] = th[e] + p[0] * g[e] + p[1] * z[e];
}
__device__ bk_real transition_log_density(const bk_real* to, const bk_real* from, const bk_real* gf,
                                          const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) { const bk_real d = to[e] - from[e] - p[0] * gf[e]; s += d * d; }
    return p[2] * s;
}
"""

# the Barker proposal (Livingstone & Zanella 2022), params = [sigma]: w_e = sigma z_e, kept with probability
# 1 / (1 + exp(-w_e g_e)) and flipped otherwise (u_e, one uniform per coordinate)
BARKER = """
__device__ bk_real softplus(bk_real x) { return x > 0 ? x + log1p(exp(-x)) : log1p(exp(x)); }
__device__ void propose(const bk_real* th, const bk_real* g, bk_real* q, const bk_real* z, const bk_real* u,
                        const bk_real* p) {
    for (int e = 0; e < BK_DIMS; ++e) {
        const bk_real w = p[0] * z[e];
        const bk_real keep = 1 / (1 + exp(-w * g[e]));
        q[e] = th[e] + (u[e] < keep ? w : -w);
    }
}
__device__ bk_real transition_log_density(const bk_real* to, const bk_real* from, const bk_real* gf,
                                          const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) {
        const bk_real w = to[e] - from[e], r = w / p[0];
        s -= bk_real(0.5) * r * r + softplus(-w * gf[e]);
    }
    return s;
}
"""


# ---- NumPy twins ------------------------------------------------------------------------------------------------------
class NpBanana:
    """NumPy twin of BANANA, and of BANANA_1 at D = 1.  dot: the tail of log p summed by np.dot instead of coordinate
    by coordinate (a different rounding order)."""

    def __init__(self, D, b, dot=False):
        self.D, self.b, self.dot = D, b, dot

    def dims(self):
        return self.D

    def log_density_gradient(self, x):
        x = np.asarray(x, dtype=np.float64)
        if self.D == 1:
            return -0.5 * x[0] * x[0], -x.copy()
        u = x[1] - self.b * x[0] * x[0]
        lp = -0.5 * (x[0] * x[0]) - 0.5 * (u * u)
        if self.dot:
            lp -= 0.5 * float(np.dot(x[2:], x[2:]))
        else:
            for e in range(2, self.D):
                lp -= 0.5 * (x[e] * x[e])
        g = -x.copy()
        g[0] = -x[0] + 2 * self.b * x[0] * u
        g[1] = -u
        return lp, g

    def log_density(self, x):
        return self.log_density_gradient(x)[0]


# non-centred eight schools: theta = (mu, log tau, eta[8]); y_j ~ N(mu + tau eta_j, sigma_j), eta ~ N(0, 1),
# mu ~ N(0, 5^2), log tau ~ N(1, 1); params = [y (8), sigma (8)]
SCHOOLS_Y = np.array([28.0, 8.0, -3.0, 7.0, -1.0, 1.0, 18.0, 12.0])
SCHOOLS_SIGMA = np.array([15.0, 10.0, 16.0, 11.0, 9.0, 11.0, 10.0, 18.0])


class NpSchools:
    def dims(self):
        return 10

    def log_density_gradient(self, th):
        th = np.asarray(th, dtype=np.float64)
        mu, lt = th[0], th[1]
        tau = np.exp(lt)
        lp = -0.5 * (mu * mu) / 25 - 0.5 * ((lt - 1) * (lt - 1))
        g = np.empty(10)
        gmu, glt = -mu / 25, -(lt - 1)
        for j in range(8):
            eta = th[2 + j]
            d = SCHOOLS_Y[j] - mu - tau * eta
            r = d / (SCHOOLS_SIGMA[j] * SCHOOLS_SIGMA[j])
            lp += -0.5 * (eta * eta) - 0.5 * (d * r)
            gmu += r
            glt += r * tau * eta
            g[2 + j] = -eta + r * tau
        g[0], g[1] = gmu, glt
        return lp, g

    def log_density(self, th):
        return self.log_density_gradient(th)[0]


class NpPriorLik:
    """NumPy twin of PRIOR_LIK_WEIGHTED."""

    def __init__(self, w):
        self.w = np.asarray(w, dtype=np.float64)

    def dims(self):
        return self.w.size

    def log_density_gradient(self, x):
        x = np.asarray(x, dtype=np.float64)
        d = x - 1
        return -0.5 * float(x @ x) - 0.5 * float(self.w @ (d * d)), -x - self.w * d

    def log_density(self, x):
        return self.log_density_gradient(x)[0]


class Mixture:
    """NumPy twin of MIXTURE_MODEL."""

    def __init__(self, mu, s, tau):
        self.mu, self.pl, self.p0 = np.asarray(mu, dtype=np.float64), 1.0 / s ** 2, 1.0 / tau ** 2

    def params(self):
        return np.concatenate([self.mu, [self.pl, self.p0]])

    def dims(self):
        return self.mu.shape[0]

    def log_prior(self, x):
        return -0.5 * self.p0 * float(np.sum(x * x))

    def log_prior_gradient(self, x):
        return -self.p0 * x

    def _ab(self, x):
        return -0.5 * self.pl * float(np.sum((x - self.mu) ** 2)), -0.5 * self.pl * float(np.sum((x + self.mu) ** 2))

    def log_likelihood(self, x):
        a, b = self._ab(x)
        m = max(a, b)
        return m + math.log(0.5 * (math.exp(a - m) + math.exp(b - m)))

    def log_likelihood_gradient(self, x):
        a, b = self._ab(x)
        m = max(a, b)
        ea, eb = math.exp(a - m), math.exp(b - m)
        wa, wb = ea / (ea + eb), eb / (ea + eb)
        return -self.pl * (wa * (x - self.mu) + wb * (x + self.mu))

    def log_density(self, x):
        return self.log_likelihood(x) + self.log_prior(x)


class GammaPois:
    """NumPy twin of GAMMA_POIS."""

    def __init__(self, a, b, n, S):
        self.a, self.b, self.n, self.S = float(a), float(b), float(n), np.asarray(S, dtype=np.float64)

    def params(self):
        return np.concatenate([[self.a, self.b, self.n], self.S])

    def log_prior(self, x):
        s = 0.0
        for e in range(x.shape[0]):
            if not x[e] > 0:
                return -math.inf
            s += (self.a - 1) * math.log(x[e]) - self.b * x[e]
        return s

    def log_likelihood(self, x):
        s = 0.0
        for e in range(x.shape[0]):
            if not x[e] > 0:
                return -math.inf
            s += self.S[e] * math.log(x[e]) - self.n * x[e]
        return s


def np_indep(m, s):
    def propose(th, z, u):
        return m + s * z

    def tld(to, frm):
        acc = 0.0
        for e in range(to.shape[0]):
            d = (to[e] - m[e]) / s[e]
            acc += -0.5 * (d * d) - np.log(s[e])
        return acc
    return propose, tld


def np_lognormal(s):
    def propose(th, z, u):
        return th * np.exp(s * z)

    def tld(to, frm):
        acc = 0.0
        for e in range(to.shape[0]):
            d = (np.log(to[e]) - np.log(frm[e])) / s
            acc += -0.5 * (d * d) - np.log(to[e])
        return acc
    return propose, tld


def np_rscan(s):
    def propose(th, z, u):
        D = th.shape[0]
        q = th.copy()
        j = min(int(u[0] * D), D - 1)
        q[j] = th[j] + s * z[0]
        return q
    return propose, (lambda to, frm: 0.0)


def np_mixture_walk(s1, s2, w):
    """NumPy twin of MIXTURE_WALK (2 D normals, 2 uniforms, no transition)."""
    def propose(th, z, u):
        D = th.shape[0]
        s = (s1 if u[0] < w else s2) * (0.5 + u[1])
        return th + s * z[:D] + 0.01 * z[D:]
    return propose


# ---- test helpers -----------------------------------------------------------------------------------------------------
def banana(bk, D, b=0.5, dtype=torch.float64, dot=False):
    return bk.CudaModel(BANANA, D, params=[b], dtype=dtype), NpBanana(D, b, dot)


def diag_params(D, seed=3):
    rng = np.random.default_rng(seed)
    return rng.normal(size=D), rng.uniform(0.5, 3.0, D)


def gpl(bk, m0, p0, mu, pl, dtype=torch.float64):
    return bk.CudaPriorLikModel(GPL, len(mu), params=np.concatenate([mu, pl, m0, p0]), dtype=dtype)


def binom(bk, a, b, x, n, dtype=torch.float64):
    lch = math.lgamma(n + 1) - math.lgamma(x + 1) - math.lgamma(n - x + 1)
    lbe = math.lgamma(a) + math.lgamma(b) - math.lgamma(a + b)
    return bk.CudaPriorLikModel(BINOM, 1, params=[a, b, x, n, lch, lbe], dtype=dtype)


def user_twin(bk, z):
    """The CUDA restatement of a golden fixture's built-in SMC model."""
    kind = str(z["model_kind"])
    if kind == "gpl":
        return gpl(bk, z["model_m0"], z["model_p0"], z["model_mu"], z["model_pl"])
    a, b, x, n = z["model_abxn"]
    return binom(bk, float(a), float(b), int(x), int(n))


def streams_uniforms_first(C, D, n, seed, n_uniform=1):
    """(start points, normals, uniforms), the uniforms drawn first"""
    rng = np.random.default_rng(seed)
    u = rng.random((n, C)) if n_uniform == 1 else rng.random((n, C, n_uniform))
    return rng.normal(size=(C, D)) * 0.7, rng.standard_normal((n, C, D)), u


def streams_uniforms_last(C, D, n, seed):
    """(start points, normals, uniforms), the uniforms drawn last"""
    rng = np.random.default_rng(seed)
    return rng.normal(size=(C, D)) * 0.7, rng.standard_normal((n, C, D)), rng.random((n, C))


def check(d, l, a, want):
    wd, wl, wa = want
    assert np.array_equal(np_(a).astype(bool), wa)
    np.testing.assert_allclose(np_(d), wd, rtol=1e-10, atol=1e-10)
    np.testing.assert_allclose(np_(l), wl, rtol=1e-10, atol=1e-10)


def same(a, b, da, db, la, lb):
    assert torch.equal(a.last_accept, b.last_accept)
    assert 0 < float(a.last_accept.float().mean()) < 1
    np.testing.assert_allclose(np_(da), np_(db), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(np_(la), np_(lb), rtol=1e-12, atol=1e-12)


def run_split(s, zs, us, k):
    """the n draws in two calls (the first evaluates the cache, the second starts from it)"""
    d1, l1 = s.sample_n(k, normals=zs[:k], uniforms=us[:k])
    a1 = s.last_accept.clone()
    d2, l2 = s.sample_n(len(zs) - k, normals=zs[k:], uniforms=us[k:])
    return torch.cat([d1, d2]), torch.cat([l1, l2]), torch.cat([a1, s.last_accept])


def philox_streams(bk, seed, chain_offset, C_, D, nz, nu, n, draw0):
    """The proposal's Philox streams rebuilt outside the sampler: normals from bk_init_normal over enough element blocks
    (the accept block's columns dropped), uniforms and the accept uniform from the NumPy restatement."""
    from bayes_kit_b200 import _lib as L
    from bayes_kit_b200._util import stream_ptr
    from oracle import philox as ph
    from oracle import proposals as opr
    blocks = opr.proposal_blocks(D, nz)
    cols = [4 * b + i for b in blocks for i in range(4)][:nz]
    Dp = 4 * (max(blocks) + 1)
    Z = torch.empty(n, C_, nz, dtype=torch.float64, device="cuda")
    U = np.empty((n, C_, 1 + nu))
    ch = np.uint64(chain_offset) + np.arange(C_, dtype=np.uint64)
    for t in range(n):
        full = torch.empty(C_, Dp, dtype=torch.float64, device="cuda")
        L.check(L.lib().bk_init_normal(full.data_ptr(), C_, Dp, L.BK_F64, seed, chain_offset, draw0 + t, stream_ptr()))
        Z[t] = full[:, cols]
        U[t, :, 0] = ph.accept_uniform(seed, ch, draw0 + t, D, np.float64)
        U[t, :, 1:] = opr.proposal_uniforms(seed, chain_offset, draw0 + t, C_, nu)
    return Z, U


def run_fake(bk, world, make, T, streams):
    """make(group) -> smc for that rank; streams(n, lo, hi, smc) -> (normals, acc_u, res_u) or Nones.
    Returns (indices [T, M], thetas [M, D], ranks).  (The FakeWorld harness of test_gpu_sharded_smc.py.)"""
    fw = bk.peer.FakeWorld(world)
    ranks = [make(fw.rank(r)) for r in range(world)]
    all_idx = []
    for n in range(1, T + 1):
        for s in ranks:
            z, au, _ = streams(n, s._lo, s._hi, s)
            s._move(n, z, au)
        for ph in (1, 2):
            for s in ranks:
                _, _, ru = streams(n, s._lo, s._hi, s)
                s._resample(n, ru, ph)
        torch.cuda.synchronize()
        all_idx.append(np.concatenate([np_(s.last_indices) for s in ranks]))
    th = np.concatenate([np_(s.thetas) for s in ranks])
    for s in ranks:
        s._check()
    return np.stack(all_idx), th, ranks


# ---- NVRTC harness ----------------------------------------------------------------------------------------------------
def nvrtc():
    """libnvrtc.so.12 as the library finds it, or None"""
    from bayes_kit_b200.models import _load_nvrtc
    _load_nvrtc()
    try:
        return C.CDLL("libnvrtc.so.12")
    except OSError:
        return None


def __getattr__(name):
    # needs_nvrtc is made on first use: finding NVRTC imports bayes_kit_b200, which fixes the library's path (BK_LIB),
    # and the timing scripts import this module before they point BK_LIB at a variant build
    if name == "needs_nvrtc":
        return pytest.mark.skipif(nvrtc() is None, reason="NVRTC (libnvrtc.so.12) cannot be loaded")
    raise AttributeError(name)


def _read(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def compile_program(kind, D, f64, model=None, proposal=None, prior_lik=False, normals=0, uniforms=0, transition=0,
                    gradient=False):
    """(ok, log) of NVRTC compiling the program of `kind` as user_model.cu does: program_text() and compile()."""
    smc = prior_lik and not gradient and kind in (PROGRAM_MODEL, PROGRAM_MODEL_PROPOSAL)
    text = ("typedef unsigned int uint32_t;\ntypedef unsigned long long uint64_t;\n"
            "typedef int int32_t;\ntypedef long long int64_t;\n")
    text += '#line 1 "bk_device_rng.cuh"\n' + _read("device_rng.cuh")
    text += "\ntypedef double bk_real;\n" if f64 else "\ntypedef float bk_real;\n"
    if model is not None:
        text += '#line 1 "model.cu"\n' + model
        if smc:
            text += '\n#line 1 "bk_smc_mailbox.cuh"\n' + _read("smc_mailbox.cuh")
    if proposal is not None:
        text += '\nnamespace bk_proposal {\n#line 1 "proposal.cu"\n' + proposal + "\n}  // namespace bk_proposal\n"
    text += '\n#line 1 "bk_user_kernels.cuh"\n' + _read("user_kernels.cuh")
    opts = ["-arch=sm_100a", "-std=c++17", f"-DBK_PROGRAM={kind}", f"-DBK_DIMS={D}",
            f"-DBK_USER_FUSED_MAX_D={FUSED_MAX_D}", "--ptxas-options=-v"]
    if f64:
        opts.append("--fmad=false")
    if prior_lik:
        opts.append("-DBK_PRIOR_LIK=1")
    if smc:
        opts += ["-DBK_SMC_KERNELS=1", f"-DBK_SMC_MAX_WORLD={SMC_MAX_WORLD}",
                 f"-DBK_SMC_MAILBOX_BYTES={SMC_MAILBOX_BYTES}"]
    opts += {PROGRAM_DRGHMC: ["-DBK_DRGHMC=1"], PROGRAM_STRETCH: ["-DBK_STRETCH=1"],
             PROGRAM_WIDE: ["-DBK_WIDE=1"]}.get(kind, [])
    if proposal is not None:
        opts += [f"-DBK_PROPOSAL_NORMALS={normals}", f"-DBK_PROPOSAL_UNIFORMS={uniforms}",
                 f"-DBK_PROPOSAL_TRANSITION={transition}"]
        if gradient:
            opts.append("-DBK_PROPOSAL_GRADIENT=1")
    nv = nvrtc()
    prog = C.c_void_p()
    name = b"proposal.cu" if kind == PROGRAM_PROPOSAL else b"model.cu"
    assert nv.nvrtcCreateProgram(C.byref(prog), text.encode(), name, 0, None, None) == 0
    arr = (C.c_char_p * len(opts))(*[o.encode() for o in opts])
    rc = nv.nvrtcCompileProgram(prog, len(opts), arr)
    n = C.c_size_t(0)
    nv.nvrtcGetProgramLogSize(prog, C.byref(n))
    buf = C.create_string_buffer(n.value)
    nv.nvrtcGetProgramLog(prog, buf)
    nv.nvrtcDestroyProgram(C.byref(prog))
    return rc == 0, buf.value.decode()


def entries(log):
    """the kernels ptxas reports, sorted"""
    return sorted(re.findall(r"Compiling entry function '(\w+)'", log))


def ptxas_report(log):
    """kernel -> its registers, stack frame, spill stores and spill loads (bytes) in a ptxas report, and the rest of
    ptxas's "Used ... registers" line"""
    out = {}
    for k in entries(log):
        m = re.search(rf"Function properties for {k}\n.*?(\d+) bytes stack frame, (\d+) bytes spill stores, "
                      rf"(\d+) bytes spill loads\n.*?Used (\d+) registers(.*?)\n", log, re.S)
        if m:
            out[k] = {"registers": int(m.group(4)), "stack_frame_bytes": int(m.group(1)),
                      "spill_store_bytes": int(m.group(2)), "spill_load_bytes": int(m.group(3)),
                      "ptxas_line": m.group(5).strip()}
    return out


# ---- timing scripts ---------------------------------------------------------------------------------------------------
def card():
    """name and power limit of GPU 0, as nvidia-smi reports them"""
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()


def build_variant(tmp, define):
    """The library linked in `tmp` with user_model.cu compiled under -D`define` (the default build is left alone);
    returns its path, for BK_LIB."""
    sys.path.insert(0, PKG)
    import build as b
    b.build()
    obj = os.path.join(tmp, "user_model.o")
    subprocess.run([b.NVCC, *b.FLAGS, f"-D{define}", "-c", os.path.join(b.CSRC, "user_model.cu"), "-o", obj],
                   check=True)
    objs = [o for o in glob.glob(os.path.join(b.OBJ, "*.o")) if not o.endswith("user_model.o")] + [obj]
    lib = os.path.join(tmp, "libbk_b200.so")
    subprocess.run([b.NVCC, "-shared", "-o", lib, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart",
                    "static", "-Xcompiler", "-fPIC", "-ldl"], check=True)
    return lib
