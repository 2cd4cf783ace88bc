// vw_varlen.cu -- single-level MODWT over a packed batch of rows of DIFFERENT lengths
// (MODWTTransform.forwardBatch / inverseBatch with mixed lengths, CORE/modwt/MODWTTransform.java:486-559): row b is
// x[off[b] .. off[b+1]) of one packed buffer and its coefficients sit at the same packed positions.
//
// CTAs tile the PACKED index space, not the rows, so 10^5 rows of 3 samples and 16 rows of 2^20 samples spread the same
// way.  A CTA stages its tile plus an (l-1)-sample halo of the input(s) into shared memory with 8-byte cp.async (rows
// start anywhere: nothing here assumes more than 8-byte alignment), finds the rows its tile covers (one warp-wide
// 32-ary search in the device copy of the offsets, then the tile's offsets in shared memory), and gives each thread
// groups of kR consecutive outputs:
//   - a group inside one row whose taps all stay inside that row reads the staged window, each staged sample loaded
//     once per group (the fast path; every output of a long row but the first / last l-1);
//   - every other output computes the true ext() index of its own row (SURVEY.md Appendix B): periodic wrap, zero
//     skip or half-sample mirror, multi-wrap included when n < l (coif5 on a row of 3 samples).
// Analysis and SYMMETRIC synthesis (t - l) stage the halo on the left, PERIODIC / ZERO_PADDING synthesis (t + l) on
// the right.  EXACT: products and sums rounded separately, taps ascending, synthesis pair-added
// (sum += h*V + g*W, CORE/modwt/MODWTTransform.java:246-295) -- bit-identical to the JVM.  Outputs go back through
// shared memory so the global stores are coalesced.
#include <cuda_pipeline.h>

#include <algorithm>

#include "vw_internal.cuh"

namespace {

constexpr int kThreads = 256;
#ifndef VW_VARLEN_R
#define VW_VARLEN_R 4
#endif
constexpr int kR = VW_VARLEN_R;                    // consecutive outputs per thread and group
constexpr int kMinBlocks = kR >= 8 ? 3 : 4;        // CTAs per SM the register budget is cut for (R = 8: 3 CTAs, measured slower)
constexpr int kIter = 1;                           // groups per thread
constexpr int kTile = kThreads * kR * kIter;       // outputs per CTA

__device__ __forceinline__ int64_t ext_periodic(int64_t i, int64_t n) {
    if (i < 0) { i += n; if (i < 0) { i %= n; if (i < 0) i += n; } }
    else if (i >= n) { i -= n; if (i >= n) i %= n; }
    return i;
}
// CORE/util/MathUtils.java:30-51
__device__ __forceinline__ int64_t ext_mirror(int64_t i, int64_t n) {
    if (i >= 0 && i < n) return i;
    const int64_t p = 2 * n;
    i %= p; if (i < 0) i += p;
    return i < n ? i : p - 1 - i;
}
// row-local index of a tap; false when the term is skipped (ZERO_PADDING)
__device__ __forceinline__ bool ext_index(int64_t &i, int64_t n, int mode) {
    if (mode == VW_PERIODIC) { i = ext_periodic(i, n); return true; }
    if (mode == VW_SYMMETRIC) { i = ext_mirror(i, n); return true; }
    return i >= 0 && i < n;
}

template <bool EXACT>
__device__ __forceinline__ double mac(double acc, double a, double b) {
    if (EXACT) return __dadd_rn(acc, __dmul_rn(a, b));
    return fma(a, b, acc);
}
template <bool EXACT>
__device__ __forceinline__ double mac2(double acc, double h, double a, double g, double c) {
    if (EXACT) return __dadd_rn(acc, __dadd_rn(__dmul_rn(h, a), __dmul_rn(g, c)));
    return fma(h, a, fma(g, c, acc));
}

// largest r in [0, batch) with off[r] - obase <= key (off strictly increasing, off[0] - obase == 0 <= key): one warp,
// 32 probes per step -- four dependent loads for 10^6 rows
__device__ int64_t find_row(const int64_t *__restrict__ off, int64_t batch, int64_t obase, int64_t key, int lane) {
    int64_t lo = 0, hi = batch;
    while (hi - lo > 1) {
        const int64_t step = (hi - lo + 31) / 32;
        const int64_t q = lo + (int64_t)lane * step;
        const bool ok = q < hi && __ldg(off + q) - obase <= key;
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        lo += (int64_t)(31 - __clz(m)) * step;   // lane 0 probes lo itself: m != 0
        hi = min(hi, lo + step);
    }
    return lo;
}

// s[i] = g[wb + i] for i < wlen, zeros outside [0, total); 8-byte cp.async (any row alignment)
__device__ __forceinline__ void stage(double *s, const double *__restrict__ g, int64_t wb, int wlen, int64_t total) {
    for (int i = threadIdx.x; i < wlen; i += kThreads) {
        const int64_t q = wb + i;
        if (q >= 0 && q < total) __pipeline_memcpy_async(s + i, g + q, 8);
        else s[i] = 0.0;
    }
    __pipeline_commit();
}

// rows of the tile [tile0, tend) -> s_off[0 .. nr] (offsets relative to the packed buffer), returns nr
__device__ __forceinline__ int tile_rows(const int64_t *__restrict__ off, int64_t batch, int64_t obase, int64_t tile0,
                                         int64_t tend, int64_t *s_off, int64_t *s_r) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp < 2) {
        const int64_t r = find_row(off, batch, obase, warp ? tend - 1 : tile0, lane);
        if (lane == 0) s_r[warp] = r;
    }
    __syncthreads();
    const int64_t r0 = s_r[0];
    const int nr = (int)(s_r[1] - r0 + 1);
    for (int i = threadIdx.x; i <= nr; i += kThreads) s_off[i] = __ldg(off + r0 + i) - obase;
    return nr;
}

// row (index into s_off) holding packed position p, searching from row `lo` on
__device__ __forceinline__ int row_at(const int64_t *s_off, int lo, int nr, int64_t p) {
    int hi = nr;   // s_off[hi] > p
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (s_off[mid] <= p) lo = mid; else hi = mid;
    }
    return lo;
}

// L > 0: compile-time filter length; L == 0: any l <= VW_MAX_FILTER_TAPS
template <int L, bool EXACT>
__global__ void __launch_bounds__(kThreads, kMinBlocks)
k_varlen_analysis(const double *__restrict__ x, const int64_t *__restrict__ off, int64_t batch, int64_t obase, int64_t total,
                  const __grid_constant__ VwFilt f, int l, int mode, double *__restrict__ w, double *__restrict__ v) {
    extern __shared__ double smem[];
    __shared__ int64_t s_r[2];
    const int LL = L ? L : l, halo = LL - 1;
    double *sx = smem;                                        // x[tile0 - halo, tile0 + kTile)
    int64_t *s_off = (int64_t *)(smem + kTile + halo);       // kTile + 1 entries
    const int64_t tile0 = (int64_t)blockIdx.x * kTile, tend = min(tile0 + kTile, total), wb = tile0 - halo;
    stage(sx, x, wb, kTile + halo, total);
    const int nr = tile_rows(off, batch, obase, tile0, tend, s_off, s_r);
    __pipeline_wait_prior(0);
    __syncthreads();

    double ov[kIter][kR], ow[kIter][kR];
    int r = 0;
#pragma unroll
    for (int it = 0; it < kIter; it++) {
        const int64_t p0 = tile0 + (int64_t)(it * kThreads + threadIdx.x) * kR;
#pragma unroll
        for (int j = 0; j < kR; j++) ov[it][j] = ow[it][j] = 0.0;
        if (p0 >= tend) continue;
        r = row_at(s_off, r, nr, p0);
        const int base = (int)(p0 - wb);                      // x[p0] in sx
        if (p0 - halo >= s_off[r] && p0 + kR <= s_off[r + 1]) {
            if (L) {
                // staged sample m = x[p0 - (L-1) + m] feeds output j through tap k = L-1+j-m; m descending = taps ascending
#pragma unroll
                for (int m = L - 1 + kR - 1; m >= 0; m--) {
                    const double xv = sx[base - (L - 1) + m];
#pragma unroll
                    for (int j = 0; j < kR; j++) {
                        const int k = L - 1 + j - m;
                        if (k >= 0 && k < L) {
                            ov[it][j] = mac<EXACT>(ov[it][j], xv, f.h[k]);
                            ow[it][j] = mac<EXACT>(ow[it][j], xv, f.g[k]);
                        }
                    }
                }
            } else {
#pragma unroll
                for (int j = 0; j < kR; j++)
                    for (int k = 0; k < LL; k++) {
                        const double xv = sx[base + j - k];
                        ov[it][j] = mac<EXACT>(ov[it][j], xv, f.h[k]);
                        ow[it][j] = mac<EXACT>(ow[it][j], xv, f.g[k]);
                    }
            }
        } else {
#pragma unroll
            for (int j = 0; j < kR; j++) {
                const int64_t p = p0 + j;
                if (p >= tend) continue;
                while (p >= s_off[r + 1]) r++;
                const int64_t s = s_off[r], n = s_off[r + 1] - s, t = p - s;
                double a = 0.0, c = 0.0;
                if (t >= halo) {
                    for (int k = 0; k < LL; k++) {
                        const double xv = sx[base + j - k];
                        a = mac<EXACT>(a, xv, f.h[k]);
                        c = mac<EXACT>(c, xv, f.g[k]);
                    }
                } else {
                    for (int k = 0; k < LL; k++) {
                        int64_t i = t - k;
                        if (!ext_index(i, n, mode)) continue;
                        const int64_t q = s + i;
                        const double xv = (q >= wb && q < tile0 + kTile) ? sx[q - wb] : __ldg(x + q);
                        a = mac<EXACT>(a, xv, f.h[k]);
                        c = mac<EXACT>(c, xv, f.g[k]);
                    }
                }
                ov[it][j] = a;
                ow[it][j] = c;
            }
        }
    }
    __syncthreads();   // window and offsets are dead: they hold the outputs now
    double *sv = sx, *sw = (double *)s_off;
#pragma unroll
    for (int it = 0; it < kIter; it++)
#pragma unroll
        for (int j = 0; j < kR; j++) {
            const int i = (it * kThreads + threadIdx.x) * kR + j;
            if (tile0 + i < tend) { sv[i] = ov[it][j]; sw[i] = ow[it][j]; }
        }
    __syncthreads();
    for (int i = threadIdx.x; i < tend - tile0; i += kThreads) {
        v[tile0 + i] = sv[i];
        w[tile0 + i] = sw[i];
    }
}

// MINUS: taps at t - k (SYMMETRIC, the single-signal inverse's rule); else t + k (PERIODIC / ZERO_PADDING)
template <int L, bool EXACT, bool MINUS>
__global__ void __launch_bounds__(kThreads, kMinBlocks)
k_varlen_synthesis(const double *__restrict__ v, const double *__restrict__ w, const int64_t *__restrict__ off, int64_t batch,
                   int64_t obase, int64_t total, const __grid_constant__ VwFilt f, int l, int mode, double *__restrict__ out) {
    extern __shared__ double smem[];
    __shared__ int64_t s_r[2];
    const int LL = L ? L : l, halo = LL - 1, wlen = kTile + halo;
    double *sv = smem, *sw = smem + wlen;
    int64_t *s_off = (int64_t *)(smem + 2 * wlen);
    const int64_t tile0 = (int64_t)blockIdx.x * kTile, tend = min(tile0 + kTile, total), wb = MINUS ? tile0 - halo : tile0;
    stage(sv, v, wb, wlen, total);
    stage(sw, w, wb, wlen, total);
    const int nr = tile_rows(off, batch, obase, tile0, tend, s_off, s_r);
    __pipeline_wait_prior(0);
    __syncthreads();

    double ox[kIter][kR];
    int r = 0;
#pragma unroll
    for (int it = 0; it < kIter; it++) {
        const int64_t p0 = tile0 + (int64_t)(it * kThreads + threadIdx.x) * kR;
#pragma unroll
        for (int j = 0; j < kR; j++) ox[it][j] = 0.0;
        if (p0 >= tend) continue;
        r = row_at(s_off, r, nr, p0);
        const int base = (int)(p0 - wb);
        const bool inside = MINUS ? (p0 - halo >= s_off[r] && p0 + kR <= s_off[r + 1])
                                  : (p0 + kR - 1 + halo < s_off[r + 1]);
        if (inside) {
            if (L) {
                // MINUS: sample m = [p0 - (L-1) + m] feeds output j through k = L-1+j-m (m descending = k ascending);
                // PLUS:  sample m = [p0 + m] feeds output j through k = m - j (m ascending = k ascending)
#pragma unroll
                for (int mm = 0; mm < L - 1 + kR; mm++) {
                    const int m = MINUS ? L - 1 + kR - 1 - mm : mm;
                    const int q = MINUS ? base - (L - 1) + m : base + m;
                    const double a = sv[q], c = sw[q];
#pragma unroll
                    for (int j = 0; j < kR; j++) {
                        const int k = MINUS ? L - 1 + j - m : m - j;
                        if (k >= 0 && k < L) ox[it][j] = mac2<EXACT>(ox[it][j], f.h[k], a, f.g[k], c);
                    }
                }
            } else {
#pragma unroll
                for (int j = 0; j < kR; j++)
                    for (int k = 0; k < LL; k++) {
                        const int q = MINUS ? base + j - k : base + j + k;
                        ox[it][j] = mac2<EXACT>(ox[it][j], f.h[k], sv[q], f.g[k], sw[q]);
                    }
            }
        } else {
#pragma unroll
            for (int j = 0; j < kR; j++) {
                const int64_t p = p0 + j;
                if (p >= tend) continue;
                while (p >= s_off[r + 1]) r++;
                const int64_t s = s_off[r], n = s_off[r + 1] - s, t = p - s;
                double acc = 0.0;
                if (MINUS ? t >= halo : t + halo < n) {
                    for (int k = 0; k < LL; k++) {
                        const int q = MINUS ? base + j - k : base + j + k;
                        acc = mac2<EXACT>(acc, f.h[k], sv[q], f.g[k], sw[q]);
                    }
                } else {
                    for (int k = 0; k < LL; k++) {
                        int64_t i = MINUS ? t - k : t + k;
                        if (!ext_index(i, n, mode)) continue;
                        const int64_t q = s + i;
                        const bool st = q >= wb && q < wb + wlen;
                        const double a = st ? sv[q - wb] : __ldg(v + q), c = st ? sw[q - wb] : __ldg(w + q);
                        acc = mac2<EXACT>(acc, f.h[k], a, f.g[k], c);
                    }
                }
                ox[it][j] = acc;
            }
        }
    }
    __syncthreads();
    double *so = sv;
#pragma unroll
    for (int it = 0; it < kIter; it++)
#pragma unroll
        for (int j = 0; j < kR; j++) {
            const int i = (it * kThreads + threadIdx.x) * kR + j;
            if (tile0 + i < tend) so[i] = ox[it][j];
        }
    __syncthreads();
    for (int i = threadIdx.x; i < tend - tile0; i += kThreads) out[tile0 + i] = so[i];
}

// lowest packed index of a NaN / Inf in a[0, n) and b[0, n) (b may be null): each thread stops at its first hit
__global__ void __launch_bounds__(256)
k_first_nonfinite(const double *__restrict__ a, const double *__restrict__ b, int64_t n, unsigned long long *first) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        if (!isfinite(a[i]) || (b && !isfinite(b[i]))) { atomicMin(first, (unsigned long long)i); break; }
}

unsigned tiles(int64_t total) { return (unsigned)((total + kTile - 1) / kTile); }

int set_smem(vw_ctx *ctx, const void *kernel, size_t bytes) {
    if (bytes <= 48 * 1024) return VW_OK;
    return vw_cuda_check(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes),
                         "cudaFuncSetAttribute(varlen smem)");
}

}  // namespace

// the compile-time filter lengths of the tile kernels (vw_fused.cu VW_DISPATCH_L), 0 = any length
#define VW_VARLEN_DISPATCH(CALL)      \
    switch (l) {                      \
        case 2: CALL(2); break;       \
        case 4: CALL(4); break;       \
        case 6: CALL(6); break;       \
        case 8: CALL(8); break;       \
        case 10: CALL(10); break;     \
        case 12: CALL(12); break;     \
        case 16: CALL(16); break;     \
        case 18: CALL(18); break;     \
        case 20: CALL(20); break;     \
        case 30: CALL(30); break;     \
        default: CALL(0); break;      \
    }

int vw_launch_varlen_analysis(vw_ctx *ctx, const double *x, const int64_t *off_dev, int64_t batch, int64_t obase, int64_t total,
                              const VwFilt &f, int l, int mode, double *w, double *v, bool exact) {
    if (total <= 0) return VW_OK;
    const size_t smem = (size_t)(kTile + l - 1 + kTile + 1) * 8;
    int rc = VW_OK;
#define VW_VA(LC)                                                                                                     \
    {                                                                                                                 \
        auto kern = exact ? k_varlen_analysis<LC, true> : k_varlen_analysis<LC, false>;                               \
        if ((rc = set_smem(ctx, (const void *)kern, smem))) return rc;                                                \
        kern<<<tiles(total), kThreads, smem, ctx->stream>>>(x, off_dev, batch, obase, total, f, l, mode, w, v);       \
    }
    VW_VARLEN_DISPATCH(VW_VA)
#undef VW_VA
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "varlen analysis launch");
}

int vw_launch_varlen_synthesis(vw_ctx *ctx, const double *v, const double *w, const int64_t *off_dev, int64_t batch, int64_t obase,
                               int64_t total, const VwFilt &f, int l, int mode, double *out, bool exact) {
    if (total <= 0) return VW_OK;
    const size_t smem = (size_t)(2 * (kTile + l - 1) + kTile + 1) * 8;
    const bool minus = mode == VW_SYMMETRIC;
    int rc = VW_OK;
#define VW_VS(LC)                                                                                                     \
    {                                                                                                                 \
        auto kern = exact ? (minus ? k_varlen_synthesis<LC, true, true> : k_varlen_synthesis<LC, true, false>)        \
                          : (minus ? k_varlen_synthesis<LC, false, true> : k_varlen_synthesis<LC, false, false>);     \
        if ((rc = set_smem(ctx, (const void *)kern, smem))) return rc;                                                \
        kern<<<tiles(total), kThreads, smem, ctx->stream>>>(v, w, off_dev, batch, obase, total, f, l, mode, out);     \
    }
    VW_VARLEN_DISPATCH(VW_VS)
#undef VW_VS
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "varlen synthesis launch");
}

int vw_launch_first_nonfinite(vw_ctx *ctx, const double *a, const double *b, int64_t n, unsigned long long *first_dev) {
    if (n <= 0) return VW_OK;
    const int64_t blocks = std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 8);
    k_first_nonfinite<<<(unsigned)blocks, 256, 0, ctx->stream>>>(a, b, n, first_dev);
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "finite check launch");
}
