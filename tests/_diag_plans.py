"""Python restatement of the transform-size and pass-plan rules of fft_autocorr.cu (rfft_size / rfft_plan,
fft_size / fft_plan) and of the pass bookkeeping of k_ess_stream (ess_stream.cu).  The GPU tests choose their
series lengths with it; tests/test_diagnostics_plan_host.py checks it against the C++ itself."""
from __future__ import annotations

RF_MAX_M = 11264          # RF_MAX_M_CONST: largest half-length transform kept in shared memory
RADIX_PASS_MAX_LOG2 = 5   # fft_plan: radix-32 passes, the remainder last
ES_L = 32                 # k_ess_stream: lags per pass
ES_MAX_K0 = 736           # k_ess_stream: last first-lag of a pass served by the shared-memory ring


def rfft_size(N: int) -> int:
    """Smallest S = c 2^a >= 2N - 1 (c in {1, 3, 5}, S even) with S / 2 <= RF_MAX_M; 0 when there is none."""
    best = 0
    for c in (1, 3, 5):
        S = 2 * c
        while S // 2 <= RF_MAX_M:
            if S >= 2 * N - 1:
                if not best or S < best:
                    best = S
                break
            S *= 2
    return best


def rfft_plan(M: int):
    """Forward passes of the M-point transform as (radix, m) pairs, m = block length after the pass."""
    rest, plan = M, []

    def push(r):
        nonlocal rest
        rest //= r
        plan.append((r, rest))

    if rest % 5 == 0:
        push(5)
    elif rest % 3 == 0:
        push(3)
    while rest % 16 == 0 and rest > 16:
        push(16)
    while rest > 1:
        if rest % 16 == 0:
            push(16)
        elif rest % 8 == 0:
            push(8)
        elif rest % 4 == 0:
            push(4)
        else:
            push(2)
    return tuple(plan)


def rf_lin(r: int, m: int) -> bool:
    """rf_pass_r: the pass addresses the skewed line at a constant stride."""
    return m >= 8 or r * m <= 8


def rfft_passes(M: int):
    """{(radix, m, lin)} of every pass of M's plan."""
    return {(r, m, rf_lin(r, m)) for r, m in rfft_plan(M)}


def fft_size(N: int) -> int:
    S = 1
    while S < 2 * N - 1:
        S <<= 1
    return S


def fft_plan(S: int):
    """log2 of the radix of each forward pass of the global-scratch transform."""
    m = S.bit_length() - 1
    assert 1 << m == S
    plan = []
    while m > 0:
        r = min(m, RADIX_PASS_MAX_LOG2)
        plan.append(r)
        m -= r
    return tuple(plan)


def rfft_lengths(n_max: int = 10241):
    """{M: [N, ...]} of every N in 2..n_max that the shared-memory transform serves."""
    by_m = {}
    for N in range(2, n_max + 1):
        S = rfft_size(N)
        if S:
            by_m.setdefault(S // 2, []).append(N)
    return by_m


def ess_last_k0(end_pos: int, N: int) -> int:
    """First lag of the last pass k_ess_stream runs for a series whose Geyer truncation (oracle end_pos_pairs) is
    at end_pos: the pass holding pair end_pos / 2 -- or, with no negative pair, the pass reaching pair N // 2."""
    e = min(end_pos // 2, N // 2)
    return ES_L * (e // (ES_L // 2))


def ess_regime(end_pos: int, N: int) -> str:
    k0 = ess_last_k0(end_pos, N)
    if k0 == 0:
        return "first-pass"
    return "multi-pass" if k0 <= ES_MAX_K0 else "far-lag"
