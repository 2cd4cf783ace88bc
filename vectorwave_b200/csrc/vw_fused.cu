// vw_fused.cu -- the hot path: fused multi-level MODWT analysis / synthesis tile kernels for sm_100a.
//
// One CTA owns a tile of T output samples of one signal.  The tile plus the dilated halo the fused
// levels need ((L-1)*2^(first-1)*(2^nlev-1) samples on the left for analysis, on the right for
// synthesis) is staged into shared memory with TMA bulk copies (cp.async.bulk, one per contiguous
// piece: a periodic wrap is two pieces landing on one mbarrier); zero padding and the symmetric mirror
// are patched in shared memory.  Each level is an a-trous FIR over the resident tile: a thread produces
// R outputs of one dilation phase (positions base + r*d), sliding one shared-memory load over up to
// min(R,L) outputs x 2 filters of FP64 FMAs whose tap operands come straight from the constant bank.
// R is odd, which makes the strided LDS.64 pattern bank-conflict free for every power-of-two dilation.
// V_j stays in shared memory (ping-pong) for the next level; W_j leaves through a staging buffer and a
// TMA bulk store (dilation < 4) or as coalesced 256-byte-per-warp stores (dilation >= 4, where lanes
// hold consecutive samples).  Tensor cores are not used: a 2-30 tap dilated filter is not a contraction.
//
// Reference semantics (what is computed): CORE/modwt/MultiLevelMODWTTransform.java:244-251,710-757
// (analysis cascade), :554-601 (synthesis cascade, PERIODIC / ZERO_PADDING), with the boundary rules of
// CORE/internal/ScalarOps.java:700-723,790-808,818-835 and CORE/util/MathUtils.java:30-51.
#include <math.h>

#include <algorithm>
#include <vector>

#include "vw_internal.cuh"
#include "vw_tma.cuh"

namespace {

#ifndef VW_MERGED_MAXL
#define VW_MERGED_MAXL 8   // filters up to this length run the analysis halo and owned outputs as one item range
#endif
#ifndef VW_LB4_MAXL
#define VW_LB4_MAXL 0   // filters up to this length are compiled for 4 CTAs of 256 threads per SM (64 registers)
#endif
#ifndef VW_KR
#define VW_KR 9
#endif
#ifndef VW_FENCE_MIN
#define VW_FENCE_MIN 0
#endif
#ifndef VW_EXP_NOSTORE
#define VW_EXP_NOSTORE 0   // 1 (developer builds, WRONG results): the analysis tile kernel skips its global stores -- compute-only timing
#endif
#ifndef VW_STAGE_W
#define VW_STAGE_W 1   // 0 (developer builds): detail rows of dilation 1 / 2 leave straight from registers instead of smem + bulk store
#endif
constexpr int kR = VW_KR;          // outputs per thread item (odd => conflict-free strided LDS.64)
constexpr int kThreads = 256;  // maximum threads per CTA (launch bound); the launch may use fewer

// ------------------------------------------------------------------------------------------------
// inner products
// ------------------------------------------------------------------------------------------------
// analysis: out[i_r] = sum_k f[k] * in[i_r - k*d],  i_r = base + r*d.  One load feeds up to min(R,L) outputs x 2
// filters.  `top` points at in[base + (R-1)*d]; the window is walked downwards with one pointer step per load.
// FULL == false: only the first `nvalid` outputs exist; loads that would only feed the others are skipped.
template <int L, int R, bool WITH_G, bool FULL, bool QMF>
__device__ __forceinline__ void analysis_item(const double *__restrict__ top, int d, int nvalid, const VwFilt32 &f,
                                              double (&ah)[R], double (&ag)[R]) {
#pragma unroll
    for (int r = 0; r < R; r++) { ah[r] = 0.0; ag[r] = 0.0; }
    const double *p = top;
#pragma unroll
    for (int m = R - 1; m >= -(L - 1); m--) {  // descending m => ascending tap index per output
        double xv;
        if (FULL || m <= 0) xv = *p;
        else xv = m < nvalid ? *p : 0.0;
        p -= d;
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int k = r - m;
            if (k >= 0 && k < L) {
                ah[r] = fma(f.h[k], xv, ah[r]);
                if (WITH_G) ag[r] = fma(vw_tap_g<L, QMF>(f, k), xv, ag[r]);
            }
        }
    }
}

// synthesis: acc[i_r] += sum_k taps[k] * in[i_r + k*d]; `bot` points at in[base]; G selects the high-pass taps
template <int L, int R, bool FULL, bool G, bool QMF>
__device__ __forceinline__ void synthesis_item(const double *__restrict__ bot, int d, int nvalid, const VwFilt32 &f,
                                               double (&acc)[R]) {
    const double *p = bot;
#pragma unroll
    for (int m = 0; m <= R + L - 2; m++) {  // ascending m => ascending tap index per output
        double xv;
        if (FULL || m < L) xv = *p;
        else xv = m < nvalid + L - 1 ? *p : 0.0;
        p += d;
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int k = m - r;
            if (k >= 0 && k < L) acc[r] = fma(G ? vw_tap_g<L, QMF>(f, k) : f.h[k], xv, acc[r]);
        }
    }
}

// ---- long filters: taps from shared memory -------------------------------------------------------------------
// sm_100 ptxas feeds DFMA tap operands from uniform registers only (no constant-bank operand), and there are 63 of
// them: from 16 taps on (32 doubles = 64 URs) it spills them to vector registers and refills with R2UR between the
// DFMAs.  Long filters instead keep (h[k], g[k]) pairs at the front of shared memory; the item loops fetch the one
// pair that enters the R-wide tap window per input step with a broadcast LDS.128 (volatile asm keeps the load at its
// step instead of hoisted out of the item loop into 2L live registers).
template <int L> struct smem_taps { static constexpr bool value = L >= 16; };
constexpr int kTapBytes = VW_FUSED_MAX_L * 16;   // tap pairs live at the front of dynamic shared memory
__device__ __forceinline__ void lds_tap_pair(uint32_t addr, double &h, double &g) {
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(h), "=d"(g) : "r"(addr));
}
__device__ __forceinline__ void lds_tap_one(uint32_t addr, double &h) {
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(h) : "r"(addr));
}

// analysis, step s = 0 .. R+L-2 reads in[top - s*d]; output r meets tap k = r - (R-1) + s, so tap s enters at step s
template <int L, int R, bool WITH_G, bool FULL>
__device__ __forceinline__ void analysis_item_st(const double *__restrict__ top, int d, int nvalid, uint32_t taps,
                                                 double (&ah)[R], double (&ag)[R]) {
#pragma unroll
    for (int r = 0; r < R; r++) { ah[r] = 0.0; ag[r] = 0.0; }
    double th[L], tg[L];
    const double *p = top;
#pragma unroll
    for (int s = 0; s <= R + L - 2; s++) {
        const int m = R - 1 - s;
        double xv;
        if (FULL || m <= 0) xv = *p;
        else xv = m < nvalid ? *p : 0.0;
        p -= d;
        if (s < L) {
            if (WITH_G) lds_tap_pair(taps + 16u * s, th[s], tg[s]);
            else lds_tap_one(taps + 16u * s, th[s]);
        }
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int k = r - m;
            if (k >= 0 && k < L) {
                ah[r] = fma(th[k], xv, ah[r]);
                if (WITH_G) ag[r] = fma(tg[k], xv, ag[r]);
            }
        }
    }
}

// synthesis, both streams in one walk: step m reads V[bot_v + m*d] and W[bot_w + m*d]; output r meets tap k = m - r
template <int L, int R, bool FULL, bool HAVE_W>
__device__ __forceinline__ void synthesis_item_st(const double *__restrict__ bv, const double *__restrict__ bw, int d,
                                                  int nvalid, uint32_t taps, double (&acc)[R]) {
    double th[L], tg[L];
    const double *pv = bv, *pw = bw;
#pragma unroll
    for (int m = 0; m <= R + L - 2; m++) {
        double xv, xw = 0.0;
        if (FULL || m < L) { xv = *pv; if (HAVE_W) xw = *pw; }
        else {
            const bool live = m < nvalid + L - 1;
            xv = live ? *pv : 0.0;
            if (HAVE_W) xw = live ? *pw : 0.0;
        }
        pv += d; pw += d;
        if (m < L) {
            if (HAVE_W) lds_tap_pair(taps + 16u * m, th[m], tg[m]);
            else lds_tap_one(taps + 16u * m, th[m]);
        }
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int k = m - r;
            if (k >= 0 && k < L) {
                acc[r] = fma(th[k], xv, acc[r]);
                if (HAVE_W) acc[r] = fma(tg[k], xw, acc[r]);
            }
        }
    }
}

// runtime-L variants (filter lengths without a specialisation, L <= 32)
template <int R, bool WITH_G>
__device__ __forceinline__ void analysis_item_dyn(const double *__restrict__ in, int base, int d, int hi_clamp, int L,
                                                  const VwFilt32 &f, double (&ah)[R], double (&ag)[R]) {
#pragma unroll
    for (int r = 0; r < R; r++) { ah[r] = 0.0; ag[r] = 0.0; }
    for (int k = 0; k < L; k++) {
        const double hk = f.h[k], gk = f.g[k];
#pragma unroll
        for (int r = 0; r < R; r++) {
            int idx = base + (r - k) * d;
            idx = idx < hi_clamp ? idx : hi_clamp;
            const double xv = in[idx];
            ah[r] = fma(hk, xv, ah[r]);
            if (WITH_G) ag[r] = fma(gk, xv, ag[r]);
        }
    }
}
template <int R>
__device__ __forceinline__ void synthesis_item_dyn(const double *__restrict__ in, int base, int d, int hi_clamp, int L,
                                                   const double (&taps)[VW_FUSED_MAX_L], double (&acc)[R]) {
    for (int k = 0; k < L; k++) {
        const double tk = taps[k];
#pragma unroll
        for (int r = 0; r < R; r++) {
            int idx = base + (r + k) * d;
            idx = idx < hi_clamp ? idx : hi_clamp;
            acc[r] = fma(tk, in[idx], acc[r]);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// kernel parameters
// ------------------------------------------------------------------------------------------------
// Developer instrumentation (make EXTRA=-DVW_PHASE_CLOCKS): thread 0 of every analysis CTA stamps %globaltimer (ns) at its
// phase boundaries -- [0] start, [1] input tile landed, [2 + lev] level done, [7] last bulk store read out -- plus the SM
// id in [6]; tools/phase_clocks.py reads the log through vw_debug_phase_log and reports where a tile's lifetime goes.
#ifdef VW_PHASE_CLOCKS
constexpr int kPhaseSlots = 8, kPhaseCtas = 16384;
__device__ unsigned long long g_phase_log[kPhaseCtas * kPhaseSlots];
__device__ __forceinline__ void phase_stamp(int slot) {
    if (threadIdx.x == 0 && blockIdx.x < kPhaseCtas) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        g_phase_log[blockIdx.x * kPhaseSlots + slot] = t;
    }
}
__device__ __forceinline__ void phase_smid() {
    if (threadIdx.x == 0 && blockIdx.x < kPhaseCtas) {
        unsigned int s;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(s));
        g_phase_log[blockIdx.x * kPhaseSlots + 6] = s;
    }
}
// synthesis log, 16 words per CTA: [0] start, [1] V tile landed, level k of the launch (k = 0 first computed): [2 + 2k] its
// W tile landed, [3 + 2k] level done; [10] SM id, [11] output bulk store read out
constexpr int kPhaseSlotsInv = 16;
__device__ unsigned long long g_phase_log_inv[kPhaseCtas * kPhaseSlotsInv];
__device__ __forceinline__ void phase_stamp_inv(int slot) {
    if (threadIdx.x == 0 && blockIdx.x < kPhaseCtas) {
        unsigned long long t;
        if (slot == 10) { unsigned int s; asm volatile("mov.u32 %0, %%smid;" : "=r"(s)); t = s; }
        else asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        g_phase_log_inv[blockIdx.x * kPhaseSlotsInv + slot] = t;
    }
}
#define VW_PHASE(slot) phase_stamp(slot)
#define VW_PHASE_INV(slot) phase_stamp_inv(slot)
#else
#define VW_PHASE(slot) ((void)0)
#define VW_PHASE_INV(slot) ((void)0)
#endif

struct FwdArgs {
    const double *x; long long ldx;
    double *w; long long ldw, lsw;
    double *v; long long ldv;
    long long n_in, t0, n_out, batch;
    int tile, htot, slack, nlev, log2d0, mode, tiles_per_row, use_tma, use_stage, lrt;
    int pf_dist;   // > 0: prefetch into L2 the input tile of the CTA `pf_dist` launches ahead (the one that takes this CTA's slot)
    VwFilt32 f;
};

struct InvArgs {
    const double *v; long long ldv;
    const double *w; long long ldw, lsw;
    double *out; long long ldo;
    unsigned long long detail_mask;
    long long n_in, n_out, batch;
    int tile, htot, nlev, log2d0, mode, tiles_per_row, use_tma, lrt;
    int pf_dist;   // as in FwdArgs: V and top-level W tiles of a future CTA
    const double *thr; int thr_per_row, thr_soft;
    long long off_v, off_w;   // stream offsets of an aligned single-level stage (SYMMETRIC sigma/tau); 0 otherwise
    VwFilt32 f;               // taps of a sigma = -1 stream arrive reversed
    int thr_lstride;          // level lev of the group reads thr[lev * thr_lstride]; 0: one table for every level
};

// ------------------------------------------------------------------------------------------------
// fused analysis
// ------------------------------------------------------------------------------------------------
// shared memory: [tap pairs: 512 B][bufA: P][bufB: P][S0: T][S1: T] doubles (S only when use_stage), then one mbarrier
template <int L, bool QMF>
__global__ void __launch_bounds__(kThreads, (L > 0 && L <= VW_LB4_MAXL) ? 4 : ((L > 0 && L <= 12) ? 3 : 2)) k_fused_analysis(const __grid_constant__ FwdArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int LR = L > 0 ? L : a.lrt;  // runtime filter length
    const int T = a.tile, HT = a.htot, P = T + HT;
    constexpr bool ST = smem_taps<L>::value && !QMF;   // a quadrature-mirror pair fits the uniform registers
    constexpr bool kMergedHalo = L > 0 && L <= VW_MERGED_MAXL;
    const uint32_t taps = smem_u32(smem_raw);
    if (ST && threadIdx.x < L) reinterpret_cast<double2 *>(smem_raw)[threadIdx.x] = make_double2(a.f.h[threadIdx.x], a.f.g[threadIdx.x]);
    double *buf0 = reinterpret_cast<double *>(smem_raw + kTapBytes);
    double *buf1 = buf0 + P;
    double *stg0 = buf1 + P;
    double *stg1 = stg0 + (a.use_stage ? T : 0);
    uint64_t *bar = reinterpret_cast<uint64_t *>(stg1 + (a.use_stage ? T : 0));

    const int tid = threadIdx.x;
    const long long b = blockIdx.x / a.tiles_per_row;
    const int tile = blockIdx.x % a.tiles_per_row;
    const long long g0 = a.t0 + (long long)tile * T;            // first owned position (input coordinates)
    long long rem = a.t0 + a.n_out - g0;
    const int Tt = (int)(rem < T ? rem : T);                     // owned samples in this tile
    const int PP = HT + Tt;                                      // valid extent of the tile buffers
    const double *xrow = a.x + b * a.ldx;

    VW_PHASE(0);
#ifdef VW_PHASE_CLOCKS
    phase_smid();
#endif
    if (a.use_tma && tid == 0) { mbar_init(bar, 1); mbar_fence_init(); }
    __syncthreads();
    stage_tile(buf0, xrow, g0 - HT, PP, a.n_in, a.mode, a.use_tma, bar, false);
    if (a.pf_dist > 0 && tid == 32) {
        const long long fb = ((long long)blockIdx.x + a.pf_dist) / a.tiles_per_row;
        if (fb < a.batch) {
            const int ft = (int)(((long long)blockIdx.x + a.pf_dist) % a.tiles_per_row);
            prefetch_l2_span(a.x + fb * a.ldx, a.t0 + (long long)ft * T - HT, P, a.n_in);
        }
    }
    if (a.use_tma) mbar_wait(bar, 0);
    __syncthreads();
    VW_PHASE(1);


    double *cur = buf0, *nxt = buf1;
    int lo_prev = 0;
#if VW_EXP_NOSTORE
    const bool do_store = a.nlev > 64;   // never true; opaque to the compiler
#else
    constexpr bool do_store = true;
#endif
    for (int lev = 0; lev < a.nlev; lev++) {
        const int ld2 = a.log2d0 + lev;
        const int d = 1 << ld2;
        const int H = (LR - 1) << ld2;
        const bool last = lev + 1 == a.nlev;
        const int lo_cur = (lev == 0 ? a.slack : lo_prev) + H;   // first index where V_lev is defined
        const bool staged = a.use_stage && d < 4;
        double *stg = (lev & 1) ? stg1 : stg0;
        double *wrow = a.w + (long long)lev * a.lsw + b * a.ldw + (g0 - a.t0);  // W_lev[owned region]

        // Short filters (compile-time, L <= VW_MERGED_MAXL): ONE item range [lo_cur, PP) instead of a halo pass followed
        // by an owned pass, so no warp runs two items back to back before the level barrier.  Halo outputs compute their
        // (discarded) detail FMAs too; HT - lo_cur is a multiple of 2d, so phases and store alignment are unchanged.
        // Measured (A/B on one box, full GPU suite green on the merged build): db4 4096 x 4096 J = 4 analysis 0.196 ->
        // 0.186 ms, haar 0.137 -> 0.134; with 16 taps the halo is 10-45 % of the tile and the wasted detail FMAs cost more
        // than the barrier wait (sym8 1.72 -> 1.88 ms, db8 4.87 -> 5.4), hence the length cut-off.
        if (kMergedHalo) {
            const int ra = last ? HT : lo_cur, rb = PP;
            const int M = rb - ra;
            const int qh = (HT - ra) >> ld2;                   // outputs q < qh of every phase lie in the halo: no W
            const int Q = (M + d - 1) >> ld2;
            const int items = ((Q + kR - 1) / kR) << ld2;
            for (int wi = tid; wi < items; wi += (int)blockDim.x) {
                const int c = wi >> ld2, ph = wi & (d - 1);
                const int base = ra + ((c * kR) << ld2) + ph;
                if (base >= rb) continue;
                const int nvalid = min(kR, (rb - base + d - 1) >> ld2);
                const bool full = nvalid == kR;
                const int rlo = qh - c * kR;                   // outputs r < rlo are halo
                const double *top = cur + base + ((kR - 1) << ld2);
                double ah[kR], ag[kR];
                if (L > 0) {
                    constexpr int LL = L > 0 ? L : 2;
                    if (ST) {
                        if (full) analysis_item_st<LL, kR, true, true>(top, d, nvalid, taps, ah, ag);
                        else analysis_item_st<LL, kR, true, false>(top, d, nvalid, taps, ah, ag);
                    } else {
                        if (full) analysis_item<LL, kR, true, true, QMF>(top, d, nvalid, a.f, ah, ag);
                        else analysis_item<LL, kR, true, false, QMF>(top, d, nvalid, a.f, ah, ag);
                    }
                } else {
                    analysis_item_dyn<kR, true>(cur, base, d, PP - 1, LR, a.f, ah, ag);
                }
                double *q = nxt + base;
                double *wq = (staged ? stg : wrow) + (base - HT);   // never dereferenced below r = rlo
#pragma unroll
                for (int r = 0; r < kR; r++) {
                    if (full || r < nvalid) { *q = ah[r]; if (r >= rlo && (staged || do_store)) *wq = ag[r]; }
                    q += d; wq += d;
                }
            }
        } else {
        // part 0: halo region [lo_cur, HT) -- approximation only (not needed after the last level)
        // part 1: owned region [HT, PP) -- approximation and detail
        for (int part = last ? 1 : 0; part < 2; part++) {
            const int ra = part == 0 ? lo_cur : HT, rb = part == 0 ? HT : PP;
            const int M = rb - ra;
            if (M <= 0) continue;
            const int Q = (M + d - 1) >> ld2;                  // samples per phase (max)
            const int items = ((Q + kR - 1) / kR) << ld2;      // chunks x phases
            for (int wi = tid; wi < items; wi += (int)blockDim.x) {
                const int c = wi >> ld2, ph = wi & (d - 1);
                const int base = ra + ((c * kR) << ld2) + ph;
                if (base >= rb) continue;
                const int nvalid = min(kR, (rb - base + d - 1) >> ld2);
                const bool full = nvalid == kR;
                const double *top = cur + base + ((kR - 1) << ld2);
                double ah[kR], ag[kR];
                if (L > 0) {
                    constexpr int LL = L > 0 ? L : 2;
                    if (ST) {
                        if (part == 0) {
                            if (full) analysis_item_st<LL, kR, false, true>(top, d, nvalid, taps, ah, ag);
                            else analysis_item_st<LL, kR, false, false>(top, d, nvalid, taps, ah, ag);
                        } else {
                            if (full) analysis_item_st<LL, kR, true, true>(top, d, nvalid, taps, ah, ag);
                            else analysis_item_st<LL, kR, true, false>(top, d, nvalid, taps, ah, ag);
                        }
                    } else if (part == 0) {
                        if (full) analysis_item<LL, kR, false, true, QMF>(top, d, nvalid, a.f, ah, ag);
                        else analysis_item<LL, kR, false, false, QMF>(top, d, nvalid, a.f, ah, ag);
                    } else {
                        if (full) analysis_item<LL, kR, true, true, QMF>(top, d, nvalid, a.f, ah, ag);
                        else analysis_item<LL, kR, true, false, QMF>(top, d, nvalid, a.f, ah, ag);
                    }
                } else {
                    if (part == 0) analysis_item_dyn<kR, false>(cur, base, d, PP - 1, LR, a.f, ah, ag);
                    else analysis_item_dyn<kR, true>(cur, base, d, PP - 1, LR, a.f, ah, ag);
                }
                double *q = nxt + base;
                if (part == 0) {
#pragma unroll
                    for (int r = 0; r < kR; r++) { if (full || r < nvalid) *q = ah[r]; q += d; }
                } else {
                    if (staged) {
                        double *wq = stg + (base - HT);
#pragma unroll
                        for (int r = 0; r < kR; r++) {
                            if (full || r < nvalid) { *q = ah[r]; *wq = ag[r]; }
                            q += d; wq += d;
                        }
                    } else {
                        double *wq = wrow + (base - HT);
#pragma unroll
                        for (int r = 0; r < kR; r++) {
                            if (full || r < nvalid) { *q = ah[r]; *wq = ag[r]; }
                            q += d; wq += d;
                        }
                    }
                }
            }
        }
        }
#if VW_FENCE_MIN   // developer builds: only the levels whose outputs a bulk store reads (staged W, the final V) need the proxy fence
        if (staged || last) fence_async_smem();
#else
        fence_async_smem();   // generic-proxy writes of nxt / stg must be visible to the bulk-store (async) proxy
#endif
        __syncthreads();
        // SYMMETRIC: V_lev at positions < 0 is the mirror of V_lev itself (ScalarOps.java:818-835 applied per level)
        if (a.mode == VW_SYMMETRIC && !last && g0 - HT < 0) {
            const int neg = (int)(HT - g0);                     // tile indices [0, neg) are positions < 0
            for (int i = lo_cur + tid; i < neg; i += (int)blockDim.x) {
                const long long pos = g0 - HT + i;              // negative
                nxt[i] = nxt[(int)((-1 - pos) - (g0 - HT))];
            }
            __syncthreads();
        }
        if (staged) {
            // a group has at most two staged levels (dilation 1 and 2) and each owns a staging buffer, so nothing is ever
            // written twice: no wait, no barrier -- the bulk store drains while the next level computes
            if (a.use_tma) {
                if (tid == 0 && do_store) {
                    bulk_s2g(wrow, stg, (uint32_t)Tt * 8u);
                    bulk_commit();
                }
            } else {
                for (int i = tid; i < Tt; i += (int)blockDim.x) wrow[i] = stg[i];
            }
        }
        double *t = cur; cur = nxt; nxt = t;
        lo_prev = lo_cur;
        if (lev < 4) VW_PHASE(2 + lev);
    }
    // V after the last level sits in cur[HT .. HT+Tt)
    double *vrow = a.v + b * a.ldv + (g0 - a.t0);
    if (a.use_tma) {
        if (tid == 0 && do_store) {
            bulk_s2g(vrow, cur + HT, (uint32_t)Tt * 8u);
            bulk_commit();
            bulk_wait_read<0>();
        }
    } else {
        for (int i = tid; i < Tt; i += (int)blockDim.x) vrow[i] = cur[HT + i];
    }
    VW_PHASE(7);
}

// MutableMultiLevelMODWTResult.applyThresholdToArray fused into the synthesis load (:97-118): one pass over a landed W tile
// in shared memory, 16-byte accesses.  Out of line and register-light on purpose: the kernel's register count is the maximum
// over its call graph, and an unrolled inlined pass pushed the short-filter kernels from 56 to 80 registers, which cost the
// plain inverse an occupancy step (haar 0.153 -> 0.217 ms).
__device__ __noinline__ void threshold_tile(double *wbuf, int tot, bool aligned16, const double *lam_ptr, int soft) {
    const double lam = __ldg(lam_ptr);
    const bool nonneg = !(lam < 0.0);
    auto thr1 = [&](double c) { return nonneg ? vw_threshold_nonneg(c, lam, soft) : vw_threshold_value(c, lam, soft); };
    double2 *w2 = reinterpret_cast<double2 *>(wbuf);
    const int tid = threadIdx.x, nt = (int)blockDim.x;
    const int n2 = aligned16 ? tot >> 1 : 0;       // odd buffer pitch (no bulk copies): scalar loop below
    for (int i = tid; i < n2; i += nt) {
        const double2 q = w2[i];
        w2[i] = make_double2(thr1(q.x), thr1(q.y));
    }
    for (int i = 2 * n2 + tid; i < tot; i += nt) wbuf[i] = thr1(wbuf[i]);
}

// ------------------------------------------------------------------------------------------------
// fused synthesis (index rule t + k*d: PERIODIC, ZERO_PADDING, linear span)
// ------------------------------------------------------------------------------------------------
// shared memory: [tap pairs: 512 B][bufA: P][bufB: P][W0: P][W1: P] doubles, then three mbarriers (V, W0, W1)
template <int L, bool QMF>
__global__ void __launch_bounds__(kThreads, (L > 0 && L <= VW_LB4_MAXL) ? 4 : ((L > 0 && L <= 12) ? 3 : 2)) k_fused_synthesis(const __grid_constant__ InvArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int LR = L > 0 ? L : a.lrt;
    const int T = a.tile, HT = a.htot, P = T + HT;
    constexpr bool ST = smem_taps<L>::value && !QMF;   // a quadrature-mirror pair fits the uniform registers
    const uint32_t taps = smem_u32(smem_raw);
    if (ST && threadIdx.x < L) reinterpret_cast<double2 *>(smem_raw)[threadIdx.x] = make_double2(a.f.h[threadIdx.x], a.f.g[threadIdx.x]);
    double *buf0 = reinterpret_cast<double *>(smem_raw + kTapBytes);
    double *buf1 = buf0 + P;
    double *wb0 = buf1 + P, *wb1 = buf1 + 2 * P;
    uint64_t *bars = reinterpret_cast<uint64_t *>(buf1 + 3 * P);  // [0]=V, [1]=W0, [2]=W1

    const int tid = threadIdx.x;
    const long long b = blockIdx.x / a.tiles_per_row;
    const int tile = blockIdx.x % a.tiles_per_row;
    const long long g0 = (long long)tile * T;
    long long rem = a.n_out - g0;
    const int Tt = (int)(rem < T ? rem : T);

    VW_PHASE_INV(0);
    VW_PHASE_INV(10);
    if (a.use_tma && tid == 0) {
        mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_init(&bars[2], 1);
        mbar_fence_init();
    }
    __syncthreads();

    // extent of level j's inputs: Tt + sum of H over the group's levels <= j
    auto extent = [&](int lev) {  // lev = index inside the group, 0 = finest
        return Tt + (int)(((long long)(LR - 1) << a.log2d0) * ((1ll << (lev + 1)) - 1));
    };
    const int top = a.nlev - 1;
    const double *vrow = a.v ? a.v + b * a.ldv : nullptr;
    auto stage_count = [&](int lev) { int e = extent(lev); return a.use_tma ? ((e + 1) & ~1) : e; };  // bulk copies move 16-byte units
    // aligned single-level stages read V from g0 + off_v and W from g0 + off_w; staging starts on an even position
    // (bulk copies move 16-byte units) and the item loops skip the parity sample
    const int par_v = (int)((g0 + a.off_v) & 1), par_w = (int)((g0 + a.off_w) & 1);
    stage_tile(buf0, vrow, g0 + a.off_v - par_v, stage_count(top) + 2 * par_v, a.n_in, a.mode, a.use_tma, &bars[0], vrow == nullptr);
    auto stage_w = [&](int lev, int slot) {
        const bool have = (a.detail_mask >> lev) & 1ull;
        const double *wrow = have ? a.w + (long long)lev * a.lsw + b * a.ldw : nullptr;
        stage_tile(slot ? wb1 : wb0, wrow, g0 + a.off_w - par_w, stage_count(lev) + 2 * par_w, a.n_in, a.mode, a.use_tma,
                   &bars[1 + slot], !have);
    };
    stage_w(top, top & 1);
    if (a.pf_dist > 0 && tid == 32) {
        const long long fb = ((long long)blockIdx.x + a.pf_dist) / a.tiles_per_row;
        if (fb < a.batch) {
            const long long fg = (long long)(((long long)blockIdx.x + a.pf_dist) % a.tiles_per_row) * T;
            if (a.v) prefetch_l2_span(a.v + fb * a.ldv, fg + a.off_v, P, a.n_in);
            if ((a.detail_mask >> top) & 1ull) prefetch_l2_span(a.w + (long long)top * a.lsw + fb * a.ldw, fg + a.off_w, P, a.n_in);
        }
    }
    if (a.use_tma) mbar_wait(&bars[0], 0);
    VW_PHASE_INV(1);
    uint32_t wphase0 = 0, wphase1 = 0;

    double *cur = buf0, *nxt = buf1;
    for (int lev = top; lev >= 0; lev--) {
        const int slot = lev & 1;
        if (lev > 0) stage_w(lev - 1, slot ^ 1);   // prefetch the next level's details while this one computes
        if (a.use_tma) {
            if (slot) { mbar_wait(&bars[2], wphase1); wphase1 ^= 1; }
            else { mbar_wait(&bars[1], wphase0); wphase0 ^= 1; }
        }
        // hand-patched samples (padding, mirrors) of this level's tiles were written before the previous level's closing
        // barrier; only the first level's were written just now.  Every thread polls the mbarrier itself for the bulk part.
        if (lev == top || !a.use_tma) __syncthreads();
        if (top - lev < 4) VW_PHASE_INV(2 + 2 * (top - lev));
        const bool have_w = (a.detail_mask >> lev) & 1ull;
        double *wt = (slot ? wb1 : wb0) + par_w;
        const double *cv = cur + (lev == top ? par_v : 0);
        const int in_ext = extent(lev);
        if (a.thr && have_w) {
            threshold_tile(slot ? wb1 : wb0, in_ext + par_w, (P & 1) == 0, a.thr + (a.thr_per_row ? b : 0) + lev * a.thr_lstride, a.thr_soft);
            __syncthreads();
        }
        const int ld2 = a.log2d0 + lev;
        const int d = 1 << ld2;
        const int M = lev > 0 ? extent(lev - 1) : Tt;           // outputs of this level
        const int Q = (M + d - 1) >> ld2;
        const int items = ((Q + kR - 1) / kR) << ld2;
        for (int wi = tid; wi < items; wi += (int)blockDim.x) {
            const int c = wi >> ld2, ph = wi & (d - 1);
            const int base = ((c * kR) << ld2) + ph;
            if (base >= M) continue;
            const int nvalid = min(kR, (M - base + d - 1) >> ld2);
            const bool full = nvalid == kR;
            double acc[kR];
#pragma unroll
            for (int r = 0; r < kR; r++) acc[r] = 0.0;
            if (L > 0) {
                constexpr int LL = L > 0 ? L : 2;
                if (ST) {
                    if (full) {
                        if (have_w) synthesis_item_st<LL, kR, true, true>(cv + base, wt + base, d, nvalid, taps, acc);
                        else synthesis_item_st<LL, kR, true, false>(cv + base, wt + base, d, nvalid, taps, acc);
                    } else {
                        if (have_w) synthesis_item_st<LL, kR, false, true>(cv + base, wt + base, d, nvalid, taps, acc);
                        else synthesis_item_st<LL, kR, false, false>(cv + base, wt + base, d, nvalid, taps, acc);
                    }
                } else if (full) {
                    synthesis_item<LL, kR, true, false, QMF>(cv + base, d, nvalid, a.f, acc);
                    if (have_w) synthesis_item<LL, kR, true, true, QMF>(wt + base, d, nvalid, a.f, acc);
                } else {
                    synthesis_item<LL, kR, false, false, QMF>(cv + base, d, nvalid, a.f, acc);
                    if (have_w) synthesis_item<LL, kR, false, true, QMF>(wt + base, d, nvalid, a.f, acc);
                }
            } else {
                synthesis_item_dyn<kR>(cv, base, d, in_ext - 1, LR, a.f.h, acc);
                if (have_w) synthesis_item_dyn<kR>(wt, base, d, in_ext - 1, LR, a.f.g, acc);
            }
            double *q = nxt + base;
#pragma unroll
            for (int r = 0; r < kR; r++) { if (full || r < nvalid) *q = acc[r]; q += d; }
        }
        fence_async_smem();   // order this level's generic-proxy traffic before later bulk copies touch the buffers
        __syncthreads();
        if (top - lev < 4) VW_PHASE_INV(3 + 2 * (top - lev));
        double *t = cur; cur = nxt; nxt = t;
    }
    double *orow = a.out + b * a.ldo + g0;
    if (a.use_tma) {
        if (tid == 0) {
            bulk_s2g(orow, cur, (uint32_t)Tt * 8u);
            bulk_commit();
            bulk_wait_read<0>();
        }
    } else {
        for (int i = tid; i < Tt; i += (int)blockDim.x) orow[i] = cur[i];
    }
    VW_PHASE_INV(11);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// opt-in dynamic shared memory.  cudaFuncAttributeMaxDynamicSharedMemorySize is per function per DEVICE and absolute, and
// several contexts may live on one device (one per host thread): the high-water mark is therefore process-global per
// (device, function), under its own mutex, and only ever raised -- a ctx launching a smaller tile never lowers it
// under another ctx's feet.
template <typename K>
int set_smem(vw_ctx *ctx, K kernel, size_t bytes) {
    struct Entry { int device; const void *func; size_t bytes; };
    static std::mutex mu;
    static std::vector<Entry> marks;
    const void *func = (const void *)kernel;
    std::lock_guard<std::mutex> lk(mu);
    Entry *hit = nullptr;
    for (auto &e : marks)
        if (e.device == ctx->device && e.func == func) { hit = &e; break; }
    if (hit && hit->bytes >= bytes) return VW_OK;
    int rc = vw_cuda_check(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes),
                           "cudaFuncSetAttribute(max dynamic smem)");
    if (rc) return rc;
    if (hit) hit->bytes = bytes;
    else marks.push_back({ctx->device, func, bytes});
    return VW_OK;
}

// from 16 taps on a quadrature-mirror pair (every orthogonal wavelet) takes the uniform-register QMF build
#define VW_DISPATCH_L(L, Q, CALL)                                     \
    switch (L) {                                                      \
        case 2: CALL(2, false); break;                                \
        case 4: CALL(4, false); break;                                \
        case 6: CALL(6, false); break;                                \
        case 8: CALL(8, false); break;                                \
        case 10: CALL(10, false); break;                              \
        case 12: CALL(12, false); break;                              \
        case 16: if (Q) CALL(16, true); else CALL(16, false); break;  \
        case 18: if (Q) CALL(18, true); else CALL(18, false); break;  \
        case 20: if (Q) CALL(20, true); else CALL(20, false); break;  \
        case 30: if (Q) CALL(30, true); else CALL(30, false); break;  \
        default: CALL(0, false); break;                               \
    }

}  // namespace

namespace {

// Threads per CTA.  Long filters run register-heavy item loops (2 CTAs of 256 threads per SM at most): 128-thread CTAs
// put 4 independent tiles on an SM instead, whose load / compute / store phases overlap far better (coif5 fused
// levels: 1.76 -> 1.3 ms per level; sym8 / db8 +3..5 %); short filters keep 256.
// The 16..20-tap synthesis (four buffers per tile, at most 3 tiles per SM) does best in between: 192 threads
// (db8 J = 6 N = 2^20 inverse 6.32 -> 5.95 ms; 128 and 256 are both slower).
// Single-level synthesis stages (the aligned SYMMETRIC ones) keep 128 (db8 SYMMETRIC inverse 7.05 vs 7.26 ms).
// Lean short filters (vw_lean.cu, <= 12 taps): 128-thread CTAs on ~1024-sample tiles whenever the halo is small next to
// the tile -- six independent tiles per SM interleave their load / compute / store phases better than three of twice
// the size (4096 x 4096 J = 4: db4 forward 0.137 -> 0.129 ms, haar inverse 0.124 -> 0.120).
bool lean_small_tiles(const vw_ctx *ctx, int l, int64_t htot) {
    return ctx->plan_lean_ok && (ctx->opt_lean & 1) && ctx->opt_lean_small && l <= 12 && !(l & 1) && htot * 8 <= 1024;
}
int launch_threads(const vw_ctx *ctx, int l, bool fwd, int nlev, int64_t htot = -1) {
    if (ctx->opt_threads > 0) return (int)std::min<int64_t>(std::max<int64_t>(ctx->opt_threads, 32), kThreads) & ~31;
    if (htot >= 0 && lean_small_tiles(ctx, l, htot)) return 128;
    if (l >= 16 && l < 24 && !fwd && nlev >= 2) return 192;
    return l >= 16 ? 128 : kThreads;
}

// How many launches ahead a CTA prefetches (L2) the input tile of the CTA that will take over its slot: the number of
// CTAs resident at once.  0 = off (everything resident, no bulk path, or vw_set_option("l2pf", 0)).
int prefetch_distance(vw_ctx *ctx, const void *func, int nthreads, size_t smem, bool use_tma, unsigned grid) {
    if (ctx->opt_l2pf <= 0 || !use_tma) return 0;
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

int64_t even_up(int64_t v) { return (v + 1) & ~1ll; }
int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// `slack`: doubles behind every tile buffer of the lean kernels (vw_lean.cu: items overshoot their range by < R * d)
size_t smem_bytes(bool fwd, int64_t tile, int64_t htot, bool use_stage, int64_t slack = 0) {
    if (fwd) return (size_t)((2 * (tile + htot + slack) + (use_stage ? 2 * tile : 0)) * 8 + 64 + kTapBytes);
    return (size_t)(4 * (tile + htot + slack) * 8 + 64 + kTapBytes);
}
// does the planner have to budget for the lean kernels' slack?  (quadrature-mirror pairs are assumed from 16 taps on)
int64_t lean_slack(const vw_ctx *ctx, int l, int first, int nf) {
    const bool lean = (l <= 12 && !(l & 1) && (ctx->opt_lean & 1)) || ((l == 16 || l == 18 || l == 20) && (ctx->opt_lean & 2));
    return lean && ctx->plan_lean_ok && nf <= 6 ? (int64_t)kR * ((int64_t)1 << (first - 1 + nf - 1)) : 0;
}

// modelled cycles per owned sample (per SM) of one fused group at tile t; INFINITY when it cannot run
double tile_cost(const vw_ctx *ctx, bool fwd, int l, int first, int nf, int64_t t) {
    const int64_t d0 = 1ll << (first - 1);
    const int64_t hexact = (int64_t)(l - 1) * d0 * ((1ll << nf) - 1);
    const int64_t htot = even_up(hexact);
    const int nthreads = launch_threads(ctx, l, fwd, nf, htot);
    const bool use_stage = fwd && d0 < 4 && VW_STAGE_W;
    const size_t smem = smem_bytes(fwd, t, htot, use_stage, lean_slack(ctx, l, first, nf));
    if (smem > ctx->smem_optin - 1024) return INFINITY;
    const int regs = lean_slack(ctx, l, first, nf) > 0 ? 85 : (l <= VW_LB4_MAXL ? 64 : (l <= 12 ? 85 : 128));
    int64_t ctas = std::min<int64_t>((int64_t)(228 * 1024) / (int64_t)(smem + 1024), 65536 / (regs * nthreads));
    ctas = std::min<int64_t>(ctas, 8);
    if (ctas < 1) return INFINITY;
    double dfma = 0.0, bytes = 0.0;
    int64_t hsum = 0;
    for (int i = 0; i < nf; i++) {
        const int64_t d = d0 << i, H = (int64_t)(l - 1) * d;
        hsum += H;
        if (fwd) {
            const int64_t hrem = i + 1 == nf ? 0 : hexact - hsum;  // halo region still needed by later levels
            const int64_t items_h = hrem > 0 ? ceil_div(ceil_div(hrem, d), kR) * d : 0;
            const int64_t items_o = ceil_div(ceil_div(t, d), kR) * d;
            dfma += (double)(ceil_div(items_h, nthreads) * nthreads) * kR * l;
            dfma += (double)(ceil_div(items_o, nthreads) * nthreads) * 2.0 * kR * l;
        } else {
            const int64_t m = t + (hsum - H);                       // outputs of level i: owned + halo of the levels below
            const int64_t items = ceil_div(ceil_div(m, d), kR) * d;
            dfma += (double)(ceil_div(items, nthreads) * nthreads) * 2.0 * kR * l;
            bytes += 8.0 * (double)(t + hsum);                      // W_i tile with its halo
        }
    }
    if (fwd) bytes = 8.0 * (double)(t + htot) + 8.0 * (double)t * (nf + 1);
    else bytes += 8.0 * (double)(t + htot) + 8.0 * (double)t;
    // FP64 pipe: 64 DFMA/clk/SM.  Taps in uniform registers (l <= 12) reach ~80 % of it inside the item loops; taps in
    // vector registers (l >= 16, three register operands per DFMA) top out at 52/clk (tools/dfma_probe.cu), ~62 % net
    const double c = dfma / 64.0 / (l < 24 ? 0.80 : 0.62);   // (calibrated on coif5; shorter filters are not FP64-bound)
    const double m = bytes / 22.5 / 0.85;         // HBM fair share per SM per clock at 6.55 TB/s, 1.965 GHz
    const double fixed = 3000.0 + 700.0 * nf;     // load latency, barriers, drain: hidden only across resident CTAs
    const double time = std::max(std::max(c, m), (c + m + fixed) / (double)ctas);
    return time / (double)t;
}

double group_cost(const vw_ctx *ctx, bool fwd, int l, int first, int nf, int64_t n, int64_t *best_tile) {
    const int64_t d0 = 1ll << (first - 1);
    const int64_t hexact = (int64_t)(l - 1) * d0 * ((1ll << nf) - 1);
    const int64_t htot = even_up(hexact);
    *best_tile = -1;
    if (l < 2 || l > VW_FUSED_MAX_L || hexact > n || htot > 24576 || first + nf - 1 > 30) return INFINITY;
    double best = INFINITY;
    const int64_t tmin = std::max<int64_t>(512, fwd ? even_up(htot) : 512);
    const int64_t ncap = even_up(n);
    if (ctx->opt_tile > 0) {
        int64_t t = std::max<int64_t>(even_up(ctx->opt_tile), fwd ? htot : 2);
        *best_tile = std::min(t, ncap);
        return tile_cost(ctx, fwd, l, first, nf, *best_tile);
    }
    if (lean_small_tiles(ctx, l, htot) && n >= 1024) {
        const int64_t nt = ceil_div(n, 1024);
        *best_tile = std::max<int64_t>(even_up(ceil_div(n, nt)), fwd ? htot : 2);
        return tile_cost(ctx, fwd, l, first, nf, *best_tile);
    }
    // the launch equalises tiles over the row (ceil(n / ntiles)), so cost the tile that will really run
    int64_t last_bal = -1;
    for (int64_t t = tmin; t <= 28672; t += 256) {
        const int64_t tt = std::min(t, ncap);
        const int64_t nt = ceil_div(n, tt);
        int64_t bal = even_up(ceil_div(n, nt));
        if (fwd && bal < htot) bal = tt;
        if (bal != last_bal) {
            last_bal = bal;
            const double c = tile_cost(ctx, fwd, l, first, nf, bal);
            if (c == INFINITY) { if (bal >= tt) break; else continue; }
            // clearly cheaper, or a tie with a larger tile up to one full round of items (256 threads x 9): the model is
            // flat where HBM dominates, the machine is not (haar, n = 4096: tile 2048 runs 9 % faster than 1366)
            if (c < best * 0.985 || (c <= best * 1.0001 && bal <= 2304)) { best = std::min(best, c); *best_tile = bal; }
        }
        if (tt == ncap) break;
    }
    return best;
}

}  // namespace

int vw_plan_levels(const vw_ctx *ctx, bool forward, int l, int levels, int64_t n, std::vector<VwPlanGroup> &out) {
    for (const auto &e : ctx->plan_cache)
        if (e.forward == forward && e.lean_ok == ctx->plan_lean_ok && e.l == l && e.levels == levels && e.n == n) { out = e.groups; return VW_OK; }
    out.clear();
    // FP64-bound filters (l >= 24) gain nothing from sharing a launch -- the halo recompute only adds FMAs (measured on coif5)
    // 16-20 taps are FP64-pipe bound in the analysis: two levels per launch keep the halo recompute small (sym8 J = 8 forward
    // 1.62 -> 1.57 ms, db8 J = 6 4.58 -> 4.39); the synthesis of those filters prefers three (db8 J = 6 N = 2^20 inverse: 1-3 | 4-5 |
    // 6 column 5.1-5.6 ms vs 1-4 | 5-6 5.7-5.8 ms, tools/gpu_r2_plans.sh), shorter filters four
    const int cap = ctx->opt_fuse > 0 ? (int)std::min<int64_t>(ctx->opt_fuse, 6) : (l >= 24 ? 1 : (l >= 16 ? (forward ? 2 : 3) : 4));
    const double kGeneric = 60.0;  // per-level kernels: one thread per output through L1/L2
    std::vector<double> best(levels + 1, INFINITY);
    std::vector<VwPlanGroup> pick(levels + 1);
    best[0] = 0.0;
    for (int done = 0; done < levels; done++) {
        if (best[done] == INFINITY) continue;
        // two column levels per pass: the lattice pair kernels (vw_column.cu) exist for 30 taps (both directions); a pair the kernels decline at
        // run time (a table that fits no lattice, SYMMETRIC) is run level by level by the cascade drivers
        // ... and, for 16-20-tap quadrature-mirror pairs, in direct form (synthesis from dilation 8 on, analysis from 16 on: the
        // analysis tile groups of two levels are cheaper than a pair until the halo recompute of levels 7-8 sets in)
        const bool pair16 = (l == 16 || l == 18 || l == 20) && (ctx->opt_lattice & (forward ? 8 : 4)) &&
                            done + 1 >= (ctx->opt_colmin > 0 ? (int)ctx->opt_colmin : (forward ? 5 : 4));
        const bool pair_len = ctx->opt_poly != 0 &&
                              ((l == 30 && (ctx->opt_lattice & 2) && done + 1 >= vw_column_min_level(ctx, l, forward)) || pair16);
        for (int nf = 1; nf <= std::max(cap, pair_len ? 2 : 1) && done + nf <= levels; nf++) {
            int64_t tile;
            double c = nf <= cap ? group_cost(ctx, forward, l, done + 1, nf, n, &tile) : INFINITY;
            if (nf > cap) tile = -1;
            if (nf == 2 && pair_len && (int64_t)3 * (l - 1) * (1ll << done) <= n) {
                const double dfma = l == 30 ? 2.0 * (l + 3) : 4.0 * l;                              // lattice / direct form, two levels
                const double cpair = std::max(dfma / 64.0 / 0.80, 32.0 / 22.5 / 0.80) + 0.1;        // two levels: 32 B/sample
                if (cpair < c) { c = cpair; tile = -2; }
            }
            if (nf == 1 && done + 1 >= vw_column_min_level(ctx, l, forward) && ctx->opt_poly != 0) {
                // deep single level (dilation >= 32): the column kernel streams 24 B/sample with no halo recompute
                bool has = l == 2 || l == 4 || l == 6 || l == 8 || l == 10 || l == 12 || l == 16 || l == 18 || l == 20 || l == 30;
                const double ccol = std::max(2.0 * l / 64.0 / 0.70, 24.0 / 22.5 / 0.80) + 0.1;
                if (has && (ccol < c || ctx->opt_poly == 2)) { c = ctx->opt_poly == 2 ? 0.01 : ccol; tile = -2; }   // poly = 2: force (diagnostics)
            }
            if (c == INFINITY) { if (nf > 1) continue; c = kGeneric; tile = -1; }
            if (best[done] + c < best[done + nf]) {
                best[done + nf] = best[done] + c;
                pick[done + nf] = VwPlanGroup{done + 1, nf, tile, c};
            }
        }
    }
    for (int at = levels; at > 0; at -= pick[at].nlev) out.push_back(pick[at]);
    std::reverse(out.begin(), out.end());   // ascending levels; the inverse walks it backwards
    if (ctx->plan_cache.size() >= 32) ctx->plan_cache.erase(ctx->plan_cache.begin());
    ctx->plan_cache.push_back({forward, ctx->plan_lean_ok, l, levels, n, out});
    return VW_OK;
}

int vw_fused_forward(vw_ctx *ctx, const VwFusedFwd &p, const VwFilt &f) {
    if (p.l < 2 || p.l > VW_FUSED_MAX_L || p.nlevels < 1 || p.batch < 1 || p.n_out < 1) return VW_EUNSUPPORTED;
    const int64_t d0 = 1ll << (p.first_level - 1);
    const int64_t hexact = (int64_t)(p.l - 1) * d0 * ((1ll << p.nlevels) - 1);
    const int64_t htot = (hexact + 1) & ~1ll;
    if (hexact > p.n_in || htot > 24576) return VW_EUNSUPPORTED;
    if (p.first_level + p.nlevels - 1 > 30) return VW_EUNSUPPORTED;
    const bool use_stage = d0 < 4 && VW_STAGE_W;
    const bool use_tma = aligned16(p.x) && aligned16(p.w) && aligned16(p.v) && !(p.ldx & 1) && !(p.ldw & 1) &&
                         !(p.lsw & 1) && !(p.ldv & 1) && !(p.n_in & 1) && !(p.t0 & 1) && !(p.n_out & 1);
    const size_t smem_cap = ctx->smem_optin - 1024;
    int64_t tile = p.tile;
    if (tile <= 0 && group_cost(ctx, true, p.l, p.first_level, p.nlevels, p.n_out, &tile) == INFINITY) return VW_EUNSUPPORTED;
    if (tile < htot) tile = htot;            // the symmetric mirror patch needs its sources inside the tile
    tile = even_up(tile);
    auto smem_for = [&](int64_t t) { return smem_bytes(true, t, htot, use_stage); };
    if (smem_for(tile) > smem_cap) return VW_EUNSUPPORTED;
    if (ctx->opt_tile <= 0) {  // equal tiles: ceil(n_out / ntiles), even
        int64_t nt = (p.n_out + tile - 1) / tile;
        int64_t bal = (((p.n_out + nt - 1) / nt) + 1) & ~1ll;
        if (bal >= htot) tile = bal;
    }
    if (tile > p.n_out) tile = (p.n_out + 1) & ~1ll;
    if (p.mode == VW_SYMMETRIC && (p.n_in < htot || tile < htot)) return VW_EUNSUPPORTED;
    const int64_t tiles_per_row = (p.n_out + tile - 1) / tile;
    if (tiles_per_row * p.batch > 0x7fffffffll) return VW_EUNSUPPORTED;

    FwdArgs a;
    a.x = p.x; a.ldx = p.ldx; a.w = p.w; a.ldw = p.ldw; a.lsw = p.lsw; a.v = p.v; a.ldv = p.ldv;
    a.n_in = p.n_in; a.t0 = p.t0; a.n_out = p.n_out; a.batch = p.batch;
    a.tile = (int)tile; a.htot = (int)htot; a.slack = (int)(htot - hexact); a.nlev = p.nlevels;
    a.log2d0 = p.first_level - 1; a.mode = p.mode; a.tiles_per_row = (int)tiles_per_row;
    a.use_tma = use_tma; a.use_stage = use_stage; a.lrt = p.l;
    for (int k = 0; k < VW_FUSED_MAX_L; k++) { a.f.h[k] = k < p.l ? f.h[k] : 0.0; a.f.g[k] = k < p.l ? f.g[k] : 0.0; }
    if (use_tma && ctx->opt_lean && ctx->plan_lean_ok) {   // the common case runs on the issue-lean kernels (vw_lean.cu)
        const int rcl = vw_lean_forward(ctx, p, a.f, tile, htot, hexact, use_stage, launch_threads(ctx, p.l, true, p.nlevels, htot));
        if (rcl != VW_EUNSUPPORTED) return rcl;
    }
    const size_t smem = smem_for(tile);
    const unsigned grid = (unsigned)(tiles_per_row * p.batch);
    const int nthreads = launch_threads(ctx, p.l, true, p.nlevels, htot);
    int rc = VW_OK;
    const bool qmf = vw_is_qmf(a.f.h, a.f.g, p.l);
#define VW_FWD_CALL(LL, QQ)                                                                \
    do {                                                                                   \
        if ((rc = set_smem(ctx, k_fused_analysis<LL, QQ>, smem))) return rc;               \
        a.pf_dist = prefetch_distance(ctx, (const void *)k_fused_analysis<LL, QQ>, nthreads, smem, use_tma, grid); \
        k_fused_analysis<LL, QQ><<<grid, nthreads, smem, ctx->stream>>>(a);                \
    } while (0)
    VW_DISPATCH_L(p.l, qmf, VW_FWD_CALL)
#undef VW_FWD_CALL
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "fused analysis launch");
}

int vw_fused_inverse(vw_ctx *ctx, const VwFusedInv &p, const VwFilt &f) {
    if (p.l < 2 || p.l > VW_FUSED_MAX_L || p.nlevels < 1 || p.batch < 1 || p.n_out < 1) return VW_EUNSUPPORTED;
    const bool aligned_stage = p.has_align;   // general (sigma, tau) alignment: one level per launch
    if (aligned_stage && p.nlevels != 1) return VW_EUNSUPPORTED;
    if (p.mode == VW_SYMMETRIC && !aligned_stage) return VW_EUNSUPPORTED;
    const int64_t d0 = 1ll << (p.first_level - 1);
    const int64_t hexact = (int64_t)(p.l - 1) * d0 * ((1ll << p.nlevels) - 1);
    const int64_t htot = ((hexact + 1) & ~1ll) + (aligned_stage ? 4 : 0);   // room for the parity sample of odd stream offsets
    if (hexact > p.n_in || htot > 12288) return VW_EUNSUPPORTED;
    if (p.first_level + p.nlevels - 1 > 30) return VW_EUNSUPPORTED;
    if (p.thr_dev && p.thr_lstride * p.nlevels > 0x7fffffffll) return VW_EUNSUPPORTED;   // the kernels index levels in 32 bits
    const bool use_tma = (!p.v || aligned16(p.v)) && aligned16(p.w) && aligned16(p.out) && !(p.ldv & 1) && !(p.ldw & 1) &&
                         !(p.lsw & 1) && !(p.ldo & 1) && !(p.n_in & 1) && !(p.n_out & 1);
    const size_t smem_cap = ctx->smem_optin - 1024;
    int64_t tile = p.tile;
    if (tile <= 0 && group_cost(ctx, false, p.l, p.first_level, p.nlevels, p.n_out, &tile) == INFINITY) return VW_EUNSUPPORTED;
    tile = even_up(tile);
    auto smem_for = [&](int64_t t) { return smem_bytes(false, t, htot, false); };
    if (smem_for(tile) > smem_cap) return VW_EUNSUPPORTED;
    if (ctx->opt_tile <= 0) {
        int64_t nt = (p.n_out + tile - 1) / tile;
        tile = (((p.n_out + nt - 1) / nt) + 1) & ~1ll;
    }
    if (tile > p.n_out) tile = (p.n_out + 1) & ~1ll;
    const int64_t tiles_per_row = (p.n_out + tile - 1) / tile;
    if (tiles_per_row * p.batch > 0x7fffffffll) return VW_EUNSUPPORTED;

    InvArgs a;
    a.v = p.v; a.ldv = p.ldv; a.w = p.w; a.ldw = p.ldw; a.lsw = p.lsw; a.out = p.out; a.ldo = p.ldo;
    a.detail_mask = p.detail_mask; a.n_in = p.n_in; a.n_out = p.n_out; a.batch = p.batch;
    a.tile = (int)tile; a.htot = (int)htot; a.nlev = p.nlevels; a.log2d0 = p.first_level - 1; a.mode = p.mode;
    a.tiles_per_row = (int)tiles_per_row; a.use_tma = use_tma; a.lrt = p.l;
    a.thr = p.thr_dev; a.thr_per_row = p.thr_per_row; a.thr_soft = p.thr_soft; a.thr_lstride = p.thr_lstride;
    a.off_v = a.off_w = 0;
    bool rev_h = false, rev_g = false;
    if (aligned_stage) {
        // sigma=+1: sum_k f[k] S[t - tau + k d];  sigma=-1: sum_k f[k] S[t + tau - k d] = sum_k' f[L-1-k'] S[t + tau - (L-1) d + k' d]
        rev_h = p.align.sigma_h < 0; rev_g = p.align.sigma_g < 0;
        a.off_v = rev_h ? (int64_t)p.align.tau_h - (int64_t)(p.l - 1) * d0 : -(int64_t)p.align.tau_h;
        a.off_w = rev_g ? (int64_t)p.align.tau_g - (int64_t)(p.l - 1) * d0 : -(int64_t)p.align.tau_g;
    }
    for (int k = 0; k < VW_FUSED_MAX_L; k++) {
        a.f.h[k] = k < p.l ? (rev_h ? f.h[p.l - 1 - k] : f.h[k]) : 0.0;
        a.f.g[k] = k < p.l ? (rev_g ? f.g[p.l - 1 - k] : f.g[k]) : 0.0;
    }
    if (use_tma && ctx->opt_lean && ctx->plan_lean_ok && !aligned_stage) {
        const int rcl = vw_lean_inverse(ctx, p, a.f, tile, htot, launch_threads(ctx, p.l, false, p.nlevels, htot));
        if (rcl != VW_EUNSUPPORTED) return rcl;
    }
    const size_t smem = smem_for(tile);
    const unsigned grid = (unsigned)(tiles_per_row * p.batch);
    const int nthreads = launch_threads(ctx, p.l, false, p.nlevels, htot);
    int rc = VW_OK;
    const bool qmf = vw_is_qmf(a.f.h, a.f.g, p.l);   // on the arrays as the kernel sees them (reversed streams differ)
#define VW_INV_CALL(LL, QQ)                                                                \
    do {                                                                                   \
        if ((rc = set_smem(ctx, k_fused_synthesis<LL, QQ>, smem))) return rc;              \
        a.pf_dist = prefetch_distance(ctx, (const void *)k_fused_synthesis<LL, QQ>, nthreads, smem, use_tma, grid); \
        k_fused_synthesis<LL, QQ><<<grid, nthreads, smem, ctx->stream>>>(a);               \
    } while (0)
    VW_DISPATCH_L(p.l, qmf, VW_INV_CALL)
#undef VW_INV_CALL
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "fused synthesis launch");
}

#ifdef VW_PHASE_CLOCKS
// developer builds only: copies the phase log of the last analysis launch (count = CTAs x 8 words) to the host
extern "C" __attribute__((visibility("default"))) int vw_debug_phase_log(unsigned long long *out, int ctas) {
    if (ctas > kPhaseCtas) ctas = kPhaseCtas;
    cudaDeviceSynchronize();
    return (int)cudaMemcpyFromSymbol(out, g_phase_log, sizeof(unsigned long long) * (size_t)ctas * kPhaseSlots);
}
extern "C" __attribute__((visibility("default"))) int vw_debug_phase_log_inv(unsigned long long *out, int ctas) {
    if (ctas > kPhaseCtas) ctas = kPhaseCtas;
    cudaDeviceSynchronize();
    return (int)cudaMemcpyFromSymbol(out, g_phase_log_inv, sizeof(unsigned long long) * (size_t)ctas * kPhaseSlotsInv);
}
#endif
