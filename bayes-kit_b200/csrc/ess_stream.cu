// Streaming Geyer IAT / ESS (iat.py:46-135, ess.py:5-69): one WARP per series, no
// block-level synchronisation, the series is never staged whole.
//
// ess/iat only consume autocorrelations up to the first negative pair
// (iat.py:37-43) -- a dozen lags for a mixing chain -- so lags are produced 32 at a
// time (a pass costs about the same for 16 or 32 lags, and 32 finish 90 % of AR(1)-like
// chains in one pass).  A pass streams the series once in 256-draw chunks through a
// small per-warp shared-memory ring (4 chunks, fp64): lane l owns draws 8l..8l+7 of the
// chunk and a 40-value window behind them, i.e. an 8 x 32 register tile of
//        S_k = sum_t y_t y_{t+k}          (256 DFMA per 24 128-bit shared loads)
// with every global load issued one chunk ahead of its use.  The autocorrelation of
// autocorr.py:27-32 (zero-padded FFT, padding >= 2N-1, so circular == linear) is
// exactly  acor_k = sum_t (x_t - mean)(x_{t+k} - mean) / var / N.  The first pass
// does not know the mean yet: it centres on a provisional value c (32 samples spread
// over the series) and corrects afterwards with y = x - c, m = mean(y):
//        sum (y_t - m)(y_{t+k} - m) = S_k - m (2T - head_k - tail_k) + (N - k) m^2
// (T = sum y, head_k / tail_k = sums of the first / last k values; fp64 throughout,
// |m| << sd so there is no cancellation).  Later passes centre on the exact mean.
#include "diag.h"

namespace bk {

constexpr int ES_WARPS = 8;      // series per block
constexpr int ES_TT = 8;         // consecutive draws per lane (register tile rows)
constexpr int ES_CH = 32 * ES_TT;  // draws per chunk
constexpr int ES_L = 32;         // lags per pass (register tile columns)
constexpr int ES_RING = 4;       // chunks in the ring
constexpr int ES_POS = ES_RING * ES_CH;
// two unused slots after every ES_TT values: lanes are ES_TT values apart, the 16-byte skew
// spreads a quarter-warp's 128-bit loads over all 32 banks
__host__ __device__ constexpr int rsk(int p) { return p + ((p / ES_TT) << 1); }
constexpr int ES_RING_DOUBLES = rsk(ES_POS);
// the window of chunk i ends at position CH i + CH + k0 + L - 2, which must stay inside the ring
constexpr int ES_MAX_K0 = (((ES_RING - 1) * ES_CH - ES_L + 1) / ES_L) * ES_L;

__device__ __forceinline__ void cp_async_elem(float* dst, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src)
                 : "memory");
}
__device__ __forceinline__ void cp_async_elem(double* dst, const double* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src)
                 : "memory");
}

__device__ __forceinline__ void cp_async_16(void* dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src)
                 : "memory");
}

__device__ __forceinline__ void ring_ld8(const double* __restrict__ ring, int pos, double* v) {
    const double2* p = reinterpret_cast<const double2*>(ring + rsk(pos & (ES_POS - 1)));
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const double2 x = p[i];
        v[2 * i] = x.x;
        v[2 * i + 1] = x.y;
    }
}

template <typename TI>   // element type of the draws (fp32 or fp64); all arithmetic is fp64
__global__ void __launch_bounds__(ES_WARPS * 32, 2) k_ess_stream(SeriesView v, int estimator,
                                                              double* __restrict__ iat_out,
                                                              double* __restrict__ ess_out) {
    extern __shared__ __align__(16) double ring_all[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double* ring = ring_all + warp * ES_RING_DOUBLES;
    TI* stage = reinterpret_cast<TI*>(ring_all + ES_WARPS * ES_RING_DOUBLES) + warp * (2 * ES_CH);
    const int64_t N = v.N;
    const int64_t n_pairs = N / 2;
    const double dn = (double)N;

    for (int64_t s = (int64_t)blockIdx.x * ES_WARPS + warp; s < v.n_series; s += (int64_t)gridDim.x * ES_WARPS) {
        const TI* __restrict__ xs = reinterpret_cast<const TI*>(v.x) + (s / v.n_inner) * v.ostride +
                                    (s % v.n_inner) * v.istride;
        const int64_t ds = v.dstride;
        const bool vec = sizeof(TI) == 4 && ds == 1 && (reinterpret_cast<uintptr_t>(xs) & 15) == 0;
        // provisional centre from 32 draws spread over the series
        double c = warp_sum((double)xs[(((int64_t)lane * N) >> 5) * ds]) * (1.0 / 32.0);
        double total = 0, low = 0, inv_vn = 0;
        bool done = false;
        for (int64_t k0 = 0; !done; k0 += ES_L) {
            double S;   // lane j: sum_t d_t d_{t+k0+j} with d = x - mean
            if (k0 <= ES_MAX_K0) {
                const int ahead = (int)((ES_CH + k0 + ES_L - 2) / ES_CH);  // chunks the window reaches beyond its own
                const int64_t n_a = (N - k0 + ES_CH - 1) / ES_CH;          // chunks with any t + k0 < N
                // chunk j: global -> per-warp staging slot j & 1 with cp.async (no registers held, so the
                // copy really is in flight during a whole chunk of FMAs), then staging -> ring, centred fp64
                // fp32 draws, unit stride, 16-byte aligned series (vec, warp-uniform): a lane stages ITS 8 consecutive
                // draws with two 16-byte copies and moves them into the ring with four 128-bit stores -- a quarter of
                // the copy / address instructions of the element-wise path (which serves every other layout)
                auto issue = [&](int64_t j) {
                    TI* dst = stage + (j & 1) * ES_CH;
                    if (vec) {
                        const int64_t e0 = j * ES_CH + ES_TT * lane;
#pragma unroll
                        for (int h = 0; h < ES_TT / 4; ++h) {
                            if (e0 + 4 * h + 3 < N) {
                                cp_async_16(dst + ES_TT * lane + 4 * h, xs + e0 + 4 * h);
                            } else {
#pragma unroll
                                for (int i = 0; i < 4; ++i)
                                    if (e0 + 4 * h + i < N) cp_async_elem(dst + ES_TT * lane + 4 * h + i, xs + e0 + 4 * h + i);
                            }
                        }
                    } else {
#pragma unroll
                        for (int u = 0; u < ES_TT; ++u) {
                            const int64_t e = j * ES_CH + lane + 32 * u;
                            if (e < N) cp_async_elem(dst + lane + 32 * u, xs + e * ds);
                        }
                    }
                    asm volatile("cp.async.commit_group;" ::: "memory");
                };
                auto stash = [&](int64_t j) {
                    const TI* src = stage + (j & 1) * ES_CH;
                    if (vec) {
                        const int64_t e0 = j * ES_CH + ES_TT * lane;
                        const int pos = (int)((j & (ES_RING - 1)) * ES_CH) + ES_TT * lane;
                        double2* out2 = reinterpret_cast<double2*>(ring + rsk(pos));   // 8 consecutive, 16-byte aligned
                        double dv[ES_TT];
#pragma unroll
                        for (int i = 0; i < ES_TT; ++i) dv[i] = e0 + i < N ? (double)src[ES_TT * lane + i] - c : 0.0;
#pragma unroll
                        for (int i = 0; i < ES_TT / 2; ++i) out2[i] = make_double2(dv[2 * i], dv[2 * i + 1]);
                    } else {
#pragma unroll
                        for (int u = 0; u < ES_TT; ++u) {
                            const int64_t e = j * ES_CH + lane + 32 * u;
                            ring[rsk((int)((j & (ES_RING - 1)) * ES_CH) + lane + 32 * u)] =
                                e < N ? (double)src[lane + 32 * u] - c : 0.0;
                        }
                    }
                };
                for (int64_t j = 0; j <= ahead; ++j) {
                    issue(j);
                    asm volatile("cp.async.wait_group 0;" ::: "memory");
                    __syncwarp();
                    stash(j);
                    __syncwarp();
                }
                issue(ahead + 1);
                __syncwarp();
                double acc[ES_L];
#pragma unroll
                for (int j = 0; j < ES_L; ++j) acc[j] = 0;
                double tsum = 0;
                for (int64_t i = 0; i < n_a; ++i) {
                    issue(i + ahead + 2);                                 // two chunks in flight during the FMAs
                    const int base = (int)((i & (ES_RING - 1)) * ES_CH) + ES_TT * lane;
                    double a[ES_TT], w[ES_TT + ES_L];
#pragma unroll
                    for (int b = 0; b < ES_TT / 8; ++b) ring_ld8(ring, base + 8 * b, a + 8 * b);
#pragma unroll
                    for (int b = 0; b < (ES_TT + ES_L) / 8; ++b) ring_ld8(ring, base + (int)k0 + 8 * b, w + 8 * b);
#pragma unroll
                    for (int ii = 0; ii < ES_TT; ++ii) {
                        tsum += a[ii];
#pragma unroll
                        for (int j = 0; j < ES_L; ++j) acc[j] = fma(a[ii], w[ii + j], acc[j]);
                    }
                    asm volatile("cp.async.wait_group 1;" ::: "memory");  // chunk i + ahead + 1 has landed
                    __syncwarp();                                         // ... and chunk i is consumed: refill its slot
                    stash(i + ahead + 1);
                    __syncwarp();
                }
                asm volatile("cp.async.wait_group 0;" ::: "memory");
                __syncwarp();
                // transposing butterfly: lane j (mod ES_L) ends with the warp total of acc[j]
                static_assert(ES_L == 16 || ES_L == 32, "lane <-> lag mapping");
                if constexpr (ES_L == 16) {
#pragma unroll
                    for (int j = 0; j < ES_L; ++j) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 16);
                }
#pragma unroll
                for (int h = ES_L / 2; h >= 1; h >>= 1) {
                    const bool up = (lane & h) != 0;
#pragma unroll
                    for (int j = 0; j < h; ++j) {
                        const double send = up ? acc[j] : acc[j + h];
                        const double keep = up ? acc[j + h] : acc[j];
                        acc[j] = keep + __shfl_xor_sync(0xffffffffu, send, h);
                    }
                }
                S = acc[0];
                if (k0 == 0) {
                    // exact centring after the fact (header comment)
                    const double T = warp_sum(tsum);
                    const double m = T / dn;
                    double head = 0, tail = 0;
                    for (int t = 0; t < (lane & (ES_L - 1)); ++t) {
                        if (t < N) head += (double)xs[t * ds] - c;
                        if (N - 1 - t >= 0) tail += (double)xs[(N - 1 - t) * ds] - c;
                    }
                    const double nk = dn - (double)(lane & (ES_L - 1));
                    S = S - m * (2.0 * T - head - tail) + (nk > 0 ? nk : 0.0) * m * m;
                    c += m;                                               // later passes centre on the mean itself
                }
            } else {
                // far lags (IAT in the hundreds): plain strided sums from global memory
                S = 0;
                for (int j = 0; j < ES_L; ++j) {
                    const int64_t k = k0 + j;
                    double p = 0;
                    for (int64_t t = lane; t + k < N; t += 32)
                        p = fma((double)xs[t * ds] - c, (double)xs[(t + k) * ds] - c, p);
                    p = warp_sum(p);
                    if ((lane & (ES_L - 1)) == j) S = p;
                }
            }
            if (k0 == 0) {
                const double var = __shfl_sync(0xffffffffu, S, 0) / dn;    // ddof = 0 (autocorr.py:27)
                inv_vn = 1.0 / (var * dn);                                // acor = S_k / var / N (autocorr.py:32)
            }
            // Geyer truncation over this pass's 16 pairs, in order (iat.py:37-43, 127-135)
            const double pr = (S + __shfl_down_sync(0xffffffffu, S, 1)) * inv_vn;   // even lanes: a pair sum
#pragma unroll 1
            for (int j = 0; j < ES_L / 2; ++j) {
                const int64_t pj = k0 / 2 + j;
                if (pj >= n_pairs) { done = true; break; }
                const double pair = __shfl_sync(0xffffffffu, pr, 2 * j);
                if (estimator == BK_IAT_IPSE) {
                    if (pair < 0) { done = true; break; }
                    total += pair;
                } else if (pj == 0) {
                    low = pair; total = pair;
                    if (pair < 0) { done = true; break; }
                } else {
                    if (pair < 0) { done = true; break; }
                    low = fmin(low, pair);
                    total += low;
                }
            }
        }
        if (lane == 0) {
            const double iat = 2.0 * total - 1.0;
            if (iat_out) iat_out[s] = iat;
            if (ess_out) ess_out[s] = dn / iat;
        }
    }
}

// [series, draws] copy of a block of series whose draws are strided in memory (the samplers'
// [draws, chains, params] layout: neighbouring series are neighbouring words, one series' draws are
// a whole row apart).  32 x 32 tiles through shared memory: reads coalesced along the series axis,
// writes along the draw axis.  A warp walking ONE such series would use 4 bytes of every 32-byte
// sector it touches and a new page per draw.
// grid.x: 32-series tiles; grid.y: 32-draw tiles tt0, tt0 + 1, ... (gridDim.y is at most 65,535: longer series take
// several launches, see ess_stream_launch).
constexpr int64_t ES_GATHER_MAX_TY = 65535;
template <typename TI>
__global__ void __launch_bounds__(256) k_gather_series(SeriesView v, int64_t s0, int64_t ns, int64_t tt0,
                                                       TI* __restrict__ out) {
    __shared__ TI tile[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t sb = (int64_t)blockIdx.x * 32, tb = (tt0 + blockIdx.y) * 32;
    const TI* x = reinterpret_cast<const TI*>(v.x);
    {
        const int64_t s = s0 + sb + tx;
        if (sb + tx < ns) {
            const int64_t base = (s / v.n_inner) * v.ostride + (s % v.n_inner) * v.istride;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int64_t t = tb + ty + 8 * k;
                if (t < v.N) tile[ty + 8 * k][tx] = x[base + t * v.dstride];
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int64_t sl = sb + ty + 8 * k, t = tb + tx;
        if (sl < ns && t < v.N) out[sl * v.N + t] = tile[tx][ty + 8 * k];
    }
}

size_t ess_stream_ws_bytes(const SeriesView& v) {
    if (v.dstride == 1 || v.n_series == 0) return 0;
    const size_t esz = v.dtype == BK_F64 ? 8 : 4;
    const int64_t ns = v.n_series < 65536 ? v.n_series : 65536;
    return (size_t)ns * v.N * esz + 256;
}

static int ess_stream_launch_direct(const SeriesView& v, int estimator, double* iat, double* ess, cudaStream_t st);

// strided draws + scratch available: gather blocks of series into [series, draws] form first
int ess_stream_launch(const SeriesView& v, int estimator, double* iat, double* ess, void* ws, size_t ws_bytes,
                      cudaStream_t st) {
    const size_t esz = v.dtype == BK_F64 ? 8 : 4;
    const int64_t fit = ws ? (int64_t)((ws_bytes > 256 ? ws_bytes - 256 : 0) / ((size_t)v.N * esz)) : 0;
    if (v.dstride == 1 || fit < 32 || v.n_series < 64) return ess_stream_launch_direct(v, estimator, iat, ess, st);
    int64_t chunk = fit < v.n_series ? fit : v.n_series;
    if (chunk < v.n_series) chunk = chunk / 32 * 32;       // full 32-series tiles except at the very end
    void* buf = reinterpret_cast<void*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
    for (int64_t s0 = 0; s0 < v.n_series; s0 += chunk) {
        const int64_t ns = v.n_series - s0 < chunk ? v.n_series - s0 : chunk;
        const int64_t n_tt = (v.N + 31) / 32;
        for (int64_t tt0 = 0; tt0 < n_tt; tt0 += ES_GATHER_MAX_TY) {
            const int64_t ny = n_tt - tt0 < ES_GATHER_MAX_TY ? n_tt - tt0 : ES_GATHER_MAX_TY;
            dim3 grid((unsigned)((ns + 31) / 32), (unsigned)ny);
            if (v.dtype == BK_F64) k_gather_series<double><<<grid, 256, 0, st>>>(v, s0, ns, tt0, (double*)buf);
            else k_gather_series<float><<<grid, 256, 0, st>>>(v, s0, ns, tt0, (float*)buf);
            BK_LAUNCH_CHECK();
        }
        const SeriesView sv{buf, v.dtype, ns, v.N, 1, v.N, 0, 1};
        int rc = ess_stream_launch_direct(sv, estimator, iat ? iat + s0 : nullptr, ess ? ess + s0 : nullptr, st);
        if (rc) return rc;
    }
    return BK_OK;
}

static int ess_stream_launch_direct(const SeriesView& v, int estimator, double* iat, double* ess, cudaStream_t st) {
    // rings + 2 staging chunks per warp
    const size_t esz = v.dtype == BK_F64 ? 8 : 4;
    const size_t smem = (size_t)ES_WARPS * (ES_RING_DOUBLES * sizeof(double) + 2 * ES_CH * esz);
    static bool attr = false;
    if (!attr) {
        const int mx = ES_WARPS * (ES_RING_DOUBLES + 2 * ES_CH) * (int)sizeof(double);
        BK_CUDA(cudaFuncSetAttribute(k_ess_stream<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
        BK_CUDA(cudaFuncSetAttribute(k_ess_stream<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
        attr = true;
    }
    const int64_t want = (v.n_series + ES_WARPS - 1) / ES_WARPS;
    const unsigned blocks = (unsigned)(want < 148 * 2 ? want : 148 * 2);
    if (v.dtype == BK_F64) k_ess_stream<double><<<blocks, ES_WARPS * 32, smem, st>>>(v, estimator, iat, ess);
    else k_ess_stream<float><<<blocks, ES_WARPS * 32, smem, st>>>(v, estimator, iat, ess);
    BK_LAUNCH_CHECK();
    return BK_OK;
}

}  // namespace bk
