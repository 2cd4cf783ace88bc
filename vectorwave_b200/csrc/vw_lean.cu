// vw_lean.cu -- the tile kernels of the common case, written for issue slots.
//
// ncu on the general tile kernels (profiles/r02_where_the_time_goes.md) showed them ISSUE-bound, not HBM- or FP64-bound:
// 4096 x 4096 db4 J = 4 executed 147 M warp instructions of which 41 M were DFMA; removing every global store changed the
// time by 4 %.  The general kernels pay for their generality in integer work: runtime filter length, partial items,
// generic (shared-or-global) store pointers, 64-bit pointer walks, per-level integer divisions, 64-bit tile index
// arithmetic.  The kernels here take only the case the benchmark configs are made of --
//   bulk-copy-aligned rows, PERIODIC / ZERO_PADDING / span boundary, compile-time filter length with the taps in uniform
//   registers (L <= 12, or a quadrature-mirror pair up to 20), full detail mask (the synthesis thresholds W tiles on load) --
// and spend one integer instruction per shared-memory access: shared memory is addressed by 32-bit element offsets into
// one `extern __shared__ double[]`, every item is a full item (tile buffers carry slack behind the tile, so items that
// overshoot the tile end compute on garbage that nothing valid ever reads), per-level geometry comes from the host in
// the kernel parameters, and the tile / row of a CTA come from a 2-D grid instead of a division.
// Same tiling, staging and numerics (same summation order) as vw_fused.cu, whose kernels keep every other case.
//
// Reference semantics: CORE/modwt/MultiLevelMODWTTransform.java:244-251,710-757 (analysis cascade), :554-601 (synthesis
// cascade, PERIODIC / ZERO_PADDING), boundary rules CORE/internal/ScalarOps.java:700-723,790-808.
#include <algorithm>

#include "vw_internal.cuh"
#include "vw_tma.cuh"

namespace {

constexpr int kR = 9;          // outputs per item (odd: the strided LDS.64 pattern is bank-conflict free at every power-of-two dilation)
constexpr int kMaxLev = 6;     // levels per launch

extern __shared__ __align__(128) double lean_smem[];

struct LeanFwd {
    const double *x; long long ldx;
    double *w; long long ldw, lsw;
    double *v; long long ldv;
    long long n_in, t0, n_out;
    int tile, htot, pbuf, nlev, log2d0, mode, tiles_per_row, use_stage, stage_all, pf_dist, batch;
    int ra[kMaxLev];      // first tile-buffer index computed at each level (a multiple of 2d below htot)
    int items[kMaxLev];   // items (chunks x phases) of each level
    double h[VW_LEAN_MAX_L], g[VW_LEAN_MAX_L];
};

struct LeanInv {
    const double *v; long long ldv;
    const double *w; long long ldw, lsw;
    double *out; long long ldo;
    long long n_in, n_out;
    int tile, htot, pbuf, nlev, log2d0, mode, tiles_per_row, pf_dist, pf_mask, batch;
    const double *thr; int thr_per_row, thr_soft;   // SWT denoise: threshold every W tile as it lands (nullptr: off)
    int ext[kMaxLev];     // input extent of each level of the group beyond the owned samples: Tt + ext[lev]
    double h[VW_LEAN_MAX_L], g[VW_LEAN_MAX_L];
    int thr_lstride;         // level lev of the group reads thr[lev * thr_lstride]; 0: one table for every level
};

template <int L, bool QMF>
__device__ __forceinline__ double tap_g(const double (&h)[VW_LEAN_MAX_L], const double (&g)[VW_LEAN_MAX_L], int k) {
    return QMF ? ((k & 1) ? -h[L - 1 - k] : h[L - 1 - k]) : g[k];
}

// Shared memory by 32-bit shared-window ADDRESS (byte address with the window base already folded in): one integer
// instruction per access.  Through a C++ pointer the compiler re-adds the base of `lean_smem` to the offset at every
// access (two IMADs per LDS / STS in the SASS).  "memory" clobber, not volatile: the accesses keep their order relative
// to barriers and to each other, the FMAs around them schedule freely.
__device__ __forceinline__ double lds_a(uint32_t addr) {
    double v;
    asm("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts_a(uint32_t addr, double v) {
    asm volatile("st.shared.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}

// ------------------------------------------------------------------------------------------------
// analysis
// ------------------------------------------------------------------------------------------------
// shared memory (doubles): [buf0: pbuf][buf1: pbuf][stg0: tile][stg1: tile] (stg only when use_stage), then one mbarrier.
// Detail rows of dilation 1 / 2 always leave through a staging buffer and ONE bulk store (8-byte global stores at those
// strides would be partial-sector writes).  With stage_all (groups that start at level 1, where the two staging buffers
// exist anyway) every level does: levels alternate between the buffers, thread 0 makes sure the store issued two levels
// earlier has read its buffer before anybody rewrites it -- two instructions per coefficient instead of three to five
// for a strided 64-bit global store, and HBM only ever sees whole contiguous rows.
template <int L, bool QMF>
__global__ void __launch_bounds__(256, L <= 12 ? 3 : 2) k_lean_analysis(const __grid_constant__ LeanFwd a) {
    const int T = a.tile, HT = a.htot, PB = a.pbuf;
    uint64_t *bar = reinterpret_cast<uint64_t *>(lean_smem + 2 * PB + (a.use_stage ? 2 * T : 0));
    const int tid = threadIdx.x;
    const int tile = blockIdx.x;
    const long long b = blockIdx.y + (long long)blockIdx.z * gridDim.y;   // batches beyond 32768 rows spill into grid.z
    if (b >= a.batch) return;
    const long long g0 = a.t0 + (long long)tile * T;            // first owned position (input coordinates)
    const long long rem = a.t0 + a.n_out - g0;
    const int Tt = (int)(rem < T ? rem : T);                     // owned samples of this tile
    const int PP = HT + Tt;                                      // valid extent of the tile buffers

    if (tid == 0) { mbar_init(bar, 1); mbar_fence_init(); }
    __syncthreads();
    // PERIODIC rows are staged by thread 0 alone (bulk copies only): the other warps skip the address arithmetic
    if (a.mode != VW_PERIODIC || tid == 0) stage_tile(lean_smem, a.x + b * a.ldx, g0 - HT, PP, a.n_in, a.mode, true, bar, false);
    if (a.pf_dist > 0 && tid == 32) {
        // the CTA that will inherit this slot: its input tile goes to L2 now (see vw_fused.cu)
        const unsigned lin = (unsigned)b * (unsigned)a.tiles_per_row + blockIdx.x + (unsigned)a.pf_dist;
        const unsigned fb = lin / (unsigned)a.tiles_per_row;
        if ((int)fb < a.batch) {
            const unsigned ft = lin - fb * (unsigned)a.tiles_per_row;
            prefetch_l2_span(a.x + (long long)fb * a.ldx, a.t0 + (long long)ft * T - HT, T + HT, a.n_in);
        }
    }
    mbar_wait(bar, 0);
    if (a.mode != VW_PERIODIC) __syncthreads();   // hand-filled samples of the open ends

    const uint32_t sbase = smem_u32(lean_smem);
    uint32_t cur8 = sbase, nxt8 = sbase + PB * 8;   // shared-window addresses of the ping-pong buffers
    const uint32_t stg8 = sbase + 2 * PB * 8;
    for (int lev = 0; lev < a.nlev; lev++) {
        const int ld2 = a.log2d0 + lev;
        const int d8 = 8 << ld2;
        const uint32_t ostg8 = stg8 + (lev & 1) * T * 8;
        const bool staged = a.stage_all || (a.use_stage && ld2 < 2);
        const int ra = a.ra[lev];
        const int items = a.items[lev];
        for (int wi = tid; wi < items; wi += (int)blockDim.x) {
            const int c = wi >> ld2, ph = wi & ((1 << ld2) - 1);
            const int base = ra + ((c * kR) << ld2) + ph;
            double ah[kR], ag[kR];
#pragma unroll
            for (int r = 0; r < kR; r++) { ah[r] = 0.0; ag[r] = 0.0; }
            {
                uint32_t p = cur8 + base * 8 + (kR - 1) * d8;
#pragma unroll
                for (int m = kR - 1; m >= -(L - 1); m--) {   // descending m => ascending tap index per output
                    const double xv = lds_a(p);
                    p -= d8;
#pragma unroll
                    for (int r = 0; r < kR; r++) {
                        const int k = r - m;
                        if (k >= 0 && k < L) {
                            ah[r] = fma(a.h[k], xv, ah[r]);
                            ag[r] = fma(tap_g<L, QMF>(a.h, a.g, k), xv, ag[r]);
                        }
                    }
                }
            }
            // V_lev: unconditional (overshoot lands in the slack behind the tile)
            {
                uint32_t q = nxt8 + base * 8;
#pragma unroll
                for (int r = 0; r < kR; r++) { sts_a(q, ah[r]); q += d8; }
            }
            // W_lev: owned outputs only, tile indices [HT, HT + T) (a ragged last tile stages a little garbage behind
            // its Tt samples; the bulk store moves Tt)
            const int rel = base - HT;
            if (staged) {
                uint32_t q = ostg8 + rel * 8;
                if (rel >= 0 && rel + (kR - 1) * (d8 >> 3) < T) {
#pragma unroll
                    for (int r = 0; r < kR; r++) { sts_a(q, ag[r]); q += d8; }
                } else {
                    int pos = rel;
#pragma unroll
                    for (int r = 0; r < kR; r++) { if (pos >= 0 && pos < T) sts_a(q, ag[r]); q += d8; pos += d8 >> 3; }
                }
            } else {
                // dilation >= 4: lanes hold consecutive samples, every warp store writes whole 32-byte sectors
                char *wq = reinterpret_cast<char *>(a.w + (long long)lev * a.lsw + b * a.ldw + (g0 - a.t0) + rel);
                if (rel >= 0 && rel + (kR - 1) * (d8 >> 3) < Tt) {
#pragma unroll
                    for (int r = 0; r < kR; r++) { *reinterpret_cast<double *>(wq) = ag[r]; wq += d8; }
                } else {
                    int pos = rel;
#pragma unroll
                    for (int r = 0; r < kR; r++) { if (pos >= 0 && pos < Tt) *reinterpret_cast<double *>(wq) = ag[r]; wq += d8; pos += d8 >> 3; }
                }
            }
        }
        if (staged || lev + 1 == a.nlev) fence_async_smem();   // generic-proxy writes a bulk store is about to read
        // stage_all: the buffer the NEXT level stages into was handed to a bulk store one level ago -- it must have been read
        if (a.stage_all && tid == 0) bulk_wait_read<0>();
        __syncthreads();
        if (staged && tid == 0) {
            bulk_s2g(a.w + (long long)lev * a.lsw + b * a.ldw + (g0 - a.t0), lean_smem + ((ostg8 - sbase) >> 3), (uint32_t)Tt * 8u);
            bulk_commit();
        }
        // SYMMETRIC: V_lev at positions < 0 is the mirror of V_lev itself (ScalarOps.java:818-835 applied per level); only
        // the first tile(s) of a row hold such positions
        if (a.mode == VW_SYMMETRIC && lev + 1 < a.nlev && g0 - HT < 0) {
            const int neg = (int)(HT - g0);                     // tile indices [0, neg) are positions < 0
            double *vn = lean_smem + ((nxt8 - sbase) >> 3);
            for (int i = ra + tid; i < neg; i += (int)blockDim.x) vn[i] = vn[2 * neg - 1 - i];   // position p -> -1 - p
            __syncthreads();
        }
        const uint32_t t = cur8; cur8 = nxt8; nxt8 = t;
    }
    if (tid == 0) {
        bulk_s2g(a.v + b * a.ldv + (g0 - a.t0), lean_smem + ((cur8 - sbase) >> 3) + HT, (uint32_t)Tt * 8u);
        bulk_commit();
        bulk_wait_read<0>();
    }
}

// ------------------------------------------------------------------------------------------------
// synthesis (index rule t + k*d: PERIODIC, ZERO_PADDING, span)
// ------------------------------------------------------------------------------------------------
// shared memory (doubles): [bufA: pbuf][bufB: pbuf][W0: pbuf][W1: pbuf], then three mbarriers (V, W0, W1)
template <int L, bool QMF>
__global__ void __launch_bounds__(256, L <= 12 ? 3 : 2) k_lean_synthesis(const __grid_constant__ LeanInv a) {
    const int T = a.tile, PB = a.pbuf;
    uint64_t *bars = reinterpret_cast<uint64_t *>(lean_smem + 4 * PB);
    const int tid = threadIdx.x;
    const int tile = blockIdx.x;
    const long long b = blockIdx.y + (long long)blockIdx.z * gridDim.y;   // batches beyond 32768 rows spill into grid.z
    if (b >= a.batch) return;
    const long long g0 = (long long)tile * T;
    const long long rem = a.n_out - g0;
    const int Tt = (int)(rem < T ? rem : T);

    if (tid == 0) {
        mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_init(&bars[2], 1);
        mbar_fence_init();
    }
    __syncthreads();
    const int top = a.nlev - 1;
    // bulk copies move 16-byte units: extents are even by construction (Tt even, ext even)
    const bool stager = a.mode != VW_PERIODIC || tid == 0;   // PERIODIC: thread 0 alone issues the bulk copies
    if (stager) stage_tile(lean_smem, a.v + b * a.ldv, g0, Tt + a.ext[top], a.n_in, a.mode, true, &bars[0], false);
    auto stage_w = [&](int lev, int slot) {
        if (stager)
            stage_tile(lean_smem + (2 + slot) * PB, a.w + (long long)lev * a.lsw + b * a.ldw, g0, Tt + a.ext[lev], a.n_in, a.mode,
                       true, &bars[1 + slot], false);
    };
    stage_w(top, top & 1);
    if (tid == 32) {
        // L2 prefetches (fire and forget; they put more bytes in flight than the one-level-ahead bulk copies can):
        // bit 0: V and top-level W tile of the CTA that will inherit this slot; bit 1: this tile's own lower W levels, which
        // the bulk copies below fetch one level at a time; bit 2: the successor's lower W levels as well
        if ((a.pf_mask & 2) && top > 0)
            for (int lev = top - 1; lev >= 0; lev--)
                prefetch_l2_span(a.w + (long long)lev * a.lsw + b * a.ldw, g0, Tt + a.ext[lev], a.n_in);
        if (a.pf_dist > 0 && (a.pf_mask & 5)) {
            const unsigned lin = (unsigned)b * (unsigned)a.tiles_per_row + blockIdx.x + (unsigned)a.pf_dist;
            const unsigned fb = lin / (unsigned)a.tiles_per_row;
            if ((int)fb < a.batch) {
                const long long fg = (long long)(lin - fb * (unsigned)a.tiles_per_row) * T;
                if (a.pf_mask & 1) {
                    prefetch_l2_span(a.v + (long long)fb * a.ldv, fg, T + a.htot, a.n_in);
                    prefetch_l2_span(a.w + (long long)top * a.lsw + (long long)fb * a.ldw, fg, T + a.htot, a.n_in);
                }
                if (a.pf_mask & 4)
                    for (int lev = top - 1; lev >= 0; lev--)
                        prefetch_l2_span(a.w + (long long)lev * a.lsw + (long long)fb * a.ldw, fg, T + a.ext[lev], a.n_in);
            }
        }
    }
    mbar_wait(&bars[0], 0);
    uint32_t wphase0 = 0, wphase1 = 0;

    const uint32_t sbase = smem_u32(lean_smem);
    uint32_t cur8 = sbase, nxt8 = sbase + PB * 8;
    for (int lev = top; lev >= 0; lev--) {
        const int slot = lev & 1;
        if (lev > 0) stage_w(lev - 1, slot ^ 1);   // the next level's details land while this one computes
        if (slot) { mbar_wait(&bars[2], wphase1); wphase1 ^= 1; }
        else { mbar_wait(&bars[1], wphase0); wphase0 ^= 1; }
        // hand-filled samples (zero padding) of this level's tiles were written before the previous level's closing
        // barrier; only the first level's were written just now
        if (lev == top && a.mode != VW_PERIODIC) __syncthreads();
        if (a.thr) {
            // MutableMultiLevelMODWTResult.applyThresholdToArray (:97-118) on the landed tile: W is thresholded exactly once
            // on its way from HBM to the FMAs, the thresholded coefficients never exist in memory
            const double lam = __ldg(a.thr + (a.thr_per_row ? b : 0) + lev * a.thr_lstride);
            const bool nonneg = !(lam < 0.0);
            double2 *w2 = reinterpret_cast<double2 *>(lean_smem + (2 + slot) * PB);
            const int n2 = (Tt + a.ext[lev]) >> 1;                  // extents are even
            for (int i = tid; i < n2; i += (int)blockDim.x) {
                double2 q = w2[i];
                q.x = nonneg ? vw_threshold_nonneg(q.x, lam, a.thr_soft) : vw_threshold_value(q.x, lam, a.thr_soft);
                q.y = nonneg ? vw_threshold_nonneg(q.y, lam, a.thr_soft) : vw_threshold_value(q.y, lam, a.thr_soft);
                w2[i] = q;
            }
            __syncthreads();
        }
        const uint32_t wof8 = sbase + (2 + slot) * PB * 8;
        const int ld2 = a.log2d0 + lev;
        const int d8 = 8 << ld2;
        const int M = Tt + (lev > 0 ? a.ext[lev - 1] : 0);      // outputs of this level
        const int Q = (M + (1 << ld2) - 1) >> ld2;
        const int items = ((Q + kR - 1) / kR) << ld2;
        for (int wi = tid; wi < items; wi += (int)blockDim.x) {
            const int c = wi >> ld2, ph = wi & ((1 << ld2) - 1);
            const int base8 = (((c * kR) << ld2) + ph) * 8;
            double acc[kR];
#pragma unroll
            for (int r = 0; r < kR; r++) acc[r] = 0.0;
            // all H taps, then all G taps (MultiLevelMODWTTransform.java:578-589); overshoot outputs read slack
            {
                uint32_t p = cur8 + base8;
#pragma unroll
                for (int m = 0; m <= kR + L - 2; m++) {
                    const double xv = lds_a(p);
                    p += d8;
#pragma unroll
                    for (int r = 0; r < kR; r++) {
                        const int k = m - r;
                        if (k >= 0 && k < L) acc[r] = fma(a.h[k], xv, acc[r]);
                    }
                }
            }
            {
                uint32_t p = wof8 + base8;
#pragma unroll
                for (int m = 0; m <= kR + L - 2; m++) {
                    const double xw = lds_a(p);
                    p += d8;
#pragma unroll
                    for (int r = 0; r < kR; r++) {
                        const int k = m - r;
                        if (k >= 0 && k < L) acc[r] = fma(tap_g<L, QMF>(a.h, a.g, k), xw, acc[r]);
                    }
                }
            }
            uint32_t q = nxt8 + base8;
#pragma unroll
            for (int r = 0; r < kR; r++) { sts_a(q, acc[r]); q += d8; }
        }
        fence_async_smem();   // order this level's generic-proxy traffic before later bulk copies touch the buffers
        __syncthreads();
        const uint32_t t = cur8; cur8 = nxt8; nxt8 = t;
    }
    if (tid == 0) {
        bulk_s2g(a.out + b * a.ldo + g0, lean_smem + ((cur8 - sbase) >> 3), (uint32_t)Tt * 8u);
        bulk_commit();
        bulk_wait_read<0>();
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// process-wide high-water mark of the opt-in dynamic shared memory per (device, kernel); see set_smem in vw_fused.cu
int raise_smem(vw_ctx *ctx, const void *func, size_t bytes) {
    struct Entry { int device; const void *func; size_t bytes; };
    static std::mutex mu;
    static std::vector<Entry> marks;
    std::lock_guard<std::mutex> lk(mu);
    Entry *hit = nullptr;
    for (auto &e : marks)
        if (e.device == ctx->device && e.func == func) { hit = &e; break; }
    if (hit && hit->bytes >= bytes) return VW_OK;
    int rc = vw_cuda_check(ctx, cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes),
                           "cudaFuncSetAttribute(max dynamic smem)");
    if (rc) return rc;
    if (hit) hit->bytes = bytes;
    else marks.push_back({ctx->device, func, bytes});
    return VW_OK;
}

int resident_distance(vw_ctx *ctx, const void *func, int nthreads, size_t smem, unsigned grid) {
    if (ctx->opt_l2pf <= 0) return 0;
    int per_sm = 0;
    for (const auto &e : ctx->occ_cache)
        if (e.func == func && e.nthreads == nthreads && e.smem == smem) per_sm = e.per_sm;
    if (!per_sm) {
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, func, nthreads, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
        ctx->occ_cache.push_back({func, nthreads, smem, per_sm});
    }
    const long long resident = (long long)per_sm * ctx->sm_count;
    if ((long long)grid <= resident) return 0;
    return (int)std::min<long long>(resident, 1 << 30);
}

#define VW_LEAN_DISPATCH(L, Q, CALL)                                  \
    switch (L) {                                                      \
        case 2: CALL(2, false); break;                                \
        case 4: CALL(4, false); break;                                \
        case 6: CALL(6, false); break;                                \
        case 8: CALL(8, false); break;                                \
        case 10: CALL(10, false); break;                              \
        case 12: CALL(12, false); break;                              \
        case 16: CALL(16, true); break;                               \
        case 18: CALL(18, true); break;                               \
        case 20: CALL(20, true); break;                               \
        default: return VW_EUNSUPPORTED;                              \
    }

bool lean_filter_ok(int l, bool qmf) {
    if (l == 2 || l == 4 || l == 6 || l == 8 || l == 10 || l == 12) return true;
    return qmf && (l == 16 || l == 18 || l == 20);
}

}  // namespace

// geometry (tile, halo) was chosen by the caller in vw_fused.cu; returns VW_EUNSUPPORTED when the shape is not the lean case
int vw_lean_forward(vw_ctx *ctx, const VwFusedFwd &p, const VwFilt32 &f, int64_t tile, int64_t htot, int64_t hexact,
                    bool use_stage, int nthreads) {
    const bool qmf = vw_is_qmf(f.h, f.g, p.l);
    if (!lean_filter_ok(p.l, qmf) || p.nlevels > kMaxLev) return VW_EUNSUPPORTED;
    if (p.mode == VW_SYMMETRIC && (p.n_in < htot || tile < htot)) return VW_EUNSUPPORTED;   // the mirror patch needs its sources inside the tile
    if (!(ctx->opt_lean & (p.l <= 12 ? 1 : 2))) return VW_EUNSUPPORTED;
    const int64_t tiles_per_row = (p.n_out + tile - 1) / tile;
    if (tiles_per_row > 0x7fffffff || tiles_per_row * p.batch > 0x7fffffffll) return VW_EUNSUPPORTED;
    LeanFwd a;
    a.x = p.x; a.ldx = p.ldx; a.w = p.w; a.ldw = p.ldw; a.lsw = p.lsw; a.v = p.v; a.ldv = p.ldv;
    a.n_in = p.n_in; a.t0 = p.t0; a.n_out = p.n_out; a.batch = (int)p.batch;
    a.tile = (int)tile; a.htot = (int)htot; a.nlev = p.nlevels; a.log2d0 = p.first_level - 1; a.mode = p.mode;
    a.tiles_per_row = (int)tiles_per_row; a.use_stage = use_stage;
    a.stage_all = use_stage && p.l <= 12;   // short filters are issue-bound: see the kernel comment
    const int64_t d0 = 1ll << (p.first_level - 1);
    const int64_t dmax = d0 << (p.nlevels - 1);
    const int64_t pbuf = ((tile + htot + kR * dmax) + 1) & ~1ll;   // slack: an item overshoots its level's range by < R*d
    a.pbuf = (int)pbuf;
    int64_t lo = htot - hexact;
    for (int i = 0; i < p.nlevels; i++) {
        const int64_t d = d0 << i;
        lo += (int64_t)(p.l - 1) * d;                               // first index where V of this level is defined
        const int64_t ra = i + 1 == p.nlevels ? htot : lo;          // the last level needs no halo outputs
        const int64_t q = (htot + tile - ra + d - 1) / d;
        a.ra[i] = (int)ra;
        a.items[i] = (int)(((q + kR - 1) / kR) * d);
    }
    for (int k = 0; k < VW_LEAN_MAX_L; k++) { a.h[k] = k < p.l ? f.h[k] : 0.0; a.g[k] = k < p.l ? f.g[k] : 0.0; }
    const size_t smem = (size_t)(2 * pbuf + (use_stage ? 2 * tile : 0)) * 8 + 64;
    if (smem > ctx->smem_optin - 1024) return VW_EUNSUPPORTED;
    const unsigned gy = (unsigned)std::min<int64_t>(p.batch, 32768);
    const dim3 grid((unsigned)tiles_per_row, gy, (unsigned)((p.batch + gy - 1) / gy));
    int rc = VW_OK;
#define VW_CALL(LL, QQ)                                                                                          \
    do {                                                                                                         \
        const void *fn = (const void *)k_lean_analysis<LL, QQ>;                                                  \
        if ((rc = raise_smem(ctx, fn, smem))) return rc;                                                         \
        a.pf_dist = resident_distance(ctx, fn, nthreads, smem, (unsigned)(tiles_per_row * p.batch));             \
        k_lean_analysis<LL, QQ><<<grid, nthreads, smem, ctx->stream>>>(a);                                       \
    } while (0)
    VW_LEAN_DISPATCH(p.l, qmf, VW_CALL)
#undef VW_CALL
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "lean analysis launch");
}

int vw_lean_inverse(vw_ctx *ctx, const VwFusedInv &p, const VwFilt32 &f, int64_t tile, int64_t htot, int nthreads) {
    const bool qmf = vw_is_qmf(f.h, f.g, p.l);
    const uint64_t full_mask = p.nlevels >= 64 ? ~0ull : ((1ull << p.nlevels) - 1);
    if (!lean_filter_ok(p.l, qmf) || p.nlevels > kMaxLev || p.mode == VW_SYMMETRIC || p.has_align || !p.v ||
        (p.detail_mask & full_mask) != full_mask || (tile & 1))
        return VW_EUNSUPPORTED;
    if (!(ctx->opt_lean & (p.l <= 12 ? 1 : 2))) return VW_EUNSUPPORTED;
    const int64_t tiles_per_row = (p.n_out + tile - 1) / tile;
    if (tiles_per_row > 0x7fffffff || tiles_per_row * p.batch > 0x7fffffffll) return VW_EUNSUPPORTED;
    LeanInv a;
    a.v = p.v; a.ldv = p.ldv; a.w = p.w; a.ldw = p.ldw; a.lsw = p.lsw; a.out = p.out; a.ldo = p.ldo;
    a.n_in = p.n_in; a.n_out = p.n_out; a.batch = (int)p.batch;
    a.tile = (int)tile; a.htot = (int)htot; a.nlev = p.nlevels; a.log2d0 = p.first_level - 1; a.mode = p.mode;
    a.tiles_per_row = (int)tiles_per_row;
    a.pf_mask = (int)ctx->opt_l2pf;
    a.thr = p.thr_dev; a.thr_per_row = p.thr_per_row; a.thr_soft = p.thr_soft; a.thr_lstride = p.thr_lstride;
    const int64_t d0 = 1ll << (p.first_level - 1);
    const int64_t dmax = d0 << (p.nlevels - 1);
    for (int i = 0; i < p.nlevels; i++) {
        const int64_t e = (int64_t)(p.l - 1) * d0 * ((1ll << (i + 1)) - 1);
        a.ext[i] = (int)((e + 1) & ~1ll);
    }
    const int64_t pbuf = ((tile + htot + kR * dmax) + 1) & ~1ll;   // slack: overshoot outputs (and what they read) stay inside the buffers
    a.pbuf = (int)pbuf;
    for (int k = 0; k < VW_LEAN_MAX_L; k++) { a.h[k] = k < p.l ? f.h[k] : 0.0; a.g[k] = k < p.l ? f.g[k] : 0.0; }
    const size_t smem = (size_t)(4 * pbuf) * 8 + 64;
    if (smem > ctx->smem_optin - 1024) return VW_EUNSUPPORTED;
    const unsigned gy = (unsigned)std::min<int64_t>(p.batch, 32768);
    const dim3 grid((unsigned)tiles_per_row, gy, (unsigned)((p.batch + gy - 1) / gy));
    int rc = VW_OK;
#define VW_CALL(LL, QQ)                                                                                          \
    do {                                                                                                         \
        const void *fn = (const void *)k_lean_synthesis<LL, QQ>;                                                 \
        if ((rc = raise_smem(ctx, fn, smem))) return rc;                                                         \
        a.pf_dist = resident_distance(ctx, fn, nthreads, smem, (unsigned)(tiles_per_row * p.batch));             \
        k_lean_synthesis<LL, QQ><<<grid, nthreads, smem, ctx->stream>>>(a);                                      \
    } while (0)
    VW_LEAN_DISPATCH(p.l, qmf, VW_CALL)
#undef VW_CALL
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "lean synthesis launch");
}
