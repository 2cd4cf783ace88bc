// vw_column.cu -- single-level MODWT kernels for DEEP levels (dilation d >= 32), where the dilated halo
// (L-1)*d no longer fits beside a tile in shared memory.
//
// At dilation d the transform splits into d independent "columns" (positions p = q*d + phi share phi): level j on
// the signal is the undilated filter on each column.  A thread owns one column phi and walks a chunk of rows q
// with a register-resident sliding window: per block of R rows it loads R new samples (lanes hold consecutive
// phi, so every warp load / store is one contiguous 256-byte segment), produces R outputs x 2 filters of FP64 FMAs
// with constant-bank taps, then shifts the last L-1 samples down.  Every input is read once (plus L-1 warm-up rows
// per chunk), every output written once: 24 B/sample/level, no shared memory, no recompute.
//
// Analysis:   V_j[p] = sum_k hs[k] X[ext(p - k d)],  W_j[p] likewise with gs       (ScalarOps.java:700-723,790-835)
// Synthesis:  out[p] = sum_k hs[k] V[ext(p + sh (k d - th))] + sum_k gs[k] W[ext(p + sg (k d - tg))]
//             (MultiLevelMODWTTransform.java:554-645; sigma = -1 streams are run with reversed taps)
#include <mutex>
#include <vector>

#include "vw_internal.cuh"

namespace {

constexpr int kCR = 72;        // granularity of rows_per_chunk: a multiple of every col_rows<L>::value (the lattice kernels pass their own)
#ifndef VW_COL_RA
#define VW_COL_RA 10
#endif
#ifndef VW_COL_RS
#define VW_COL_RS 10
#endif
template <int L> struct col_rows { static constexpr int value = L >= 24 ? VW_COL_RA : 9; };       // analysis
// synthesis keeps L-1+R running sums: long filters take R = 10 at two CTAs per SM (254 registers, no spills) -- fewer
// window shifts per FMA beat the third CTA (measured on coif5)
template <int L> struct col_rows_syn { static constexpr int value = L >= 24 ? VW_COL_RS : (L >= 16 ? 8 : 9); };
constexpr int kCThreads = 128;

// Tap delivery.  sm_100 ptxas never folds a constant-bank operand into DFMA: taps go through uniform registers, and
// there are only 63 of them.  Up to 12 taps (24 doubles = 48 URs) that is free; from 16 taps on ptxas spills URs to
// vector registers and refills them with R2UR between the DFMAs (measured: DFMA < 45 % of issued instructions for
// coif5).  Long filters therefore keep (h[k], g[k]) pairs in shared memory and fetch one pair per tap step with a
// broadcast LDS.128 (volatile, so the loads stay inside the loop instead of being hoisted into 120 live registers):
// 1 LDS per 2R DFMAs.
template <int L> struct col_smem_taps { static constexpr bool value = L >= 16; };          // analysis
template <int L> struct col_smem_taps_syn { static constexpr bool value = L >= 12; };      // synthesis
__device__ __forceinline__ void lds_tap_pair(uint32_t addr, double &h, double &g) {
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(h), "=d"(g) : "r"(addr));
}

// one wrap is the common case (halo shorter than the row): a 64-bit % is a ~100-instruction call
__device__ __forceinline__ int64_t wrap_mod(int64_t i, int64_t n) {
    if (i >= n && i < 2 * n) return i - n;
    if (i < 0 && i >= -n) return i + n;
    i %= n;
    return i < 0 ? i + n : i;
}
// EDGE == false: the caller has proven pos is inside [0, n) (interior chunks, the overwhelming majority)
template <bool EDGE>
__device__ __forceinline__ double ext_load(const double *__restrict__ row, int64_t pos, int64_t n, int mode) {
    if (!EDGE) return __ldg(row + pos);
    if (pos >= 0 && pos < n) return __ldg(row + pos);
    if (mode == VW_PERIODIC) return __ldg(row + wrap_mod(pos, n));
    if (mode == VW_SYMMETRIC) { int64_t m = wrap_mod(pos, 2 * n); return __ldg(row + (m < n ? m : 2 * n - 1 - m)); }
    return 0.0;
}

struct ColArgs {
    const double *x; long long ldx;          // analysis input / synthesis V (may be null => zeros)
    const double *w_in; long long ldw_in;    // synthesis W (may be null => zeros)
    double *v; long long ldv;                // analysis V out / synthesis out
    double *w; long long ldw;                // analysis W out
    long long n_in, t0, n_out, batch, d;     // outputs cover positions [t0, t0+n_out) of the input coordinate system
    long long off_h, off_g;                  // synthesis stream offsets (see below)
    int rows_per_chunk, chunks, mode;
    const double *thr; int thr_per_row, thr_soft;   // synthesis: threshold W on load (SWT denoise); thr == nullptr: off
    VwFilt32 f;                              // synthesis: taps already reversed for sigma = -1 streams
};

// Issue-slot budget (measured with tools/dfma_probe.cu on B200): a DFMA occupies the FP64 pipe for 2 cycles but one issue
// slot; ALU-pipe integer instructions (IADD3, ISETP, LEA, LOP3) cost TWO issue slots each, FMA-pipe ones (IMAD, IMAD.WIDE,
// IMAD.MOV) one.  At 60 DFMAs per sample (coif5) every integer instruction in the row loop shows up in the run time, so
// the loops below keep one 64-bit byte pointer per stream that is bumped once per block, reach row r through
// `ptr + d * (8 r)` (a single IMAD.WIDE with a 32-bit d), and use unpredicated loads / stores whenever a whole block
// is in range.
// Prefetch load that stays where it is written: NVVM otherwise sinks the next block's loads below the FMA block to
// save registers, which leaves no time to cover the HBM latency (measured: 12 % of warp time on the first use).
__device__ __forceinline__ double ldg_early(const double *p) {
    double v;
    asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ const double *row_ptr(const char *base, int d, int r) {
    return reinterpret_cast<const double *>(base + (long long)d * (long long)(8 * r));
}
__device__ __forceinline__ double *row_ptr(char *base, int d, int r) {
    return reinterpret_cast<double *>(base + (long long)d * (long long)(8 * r));
}

// ---- analysis ------------------------------------------------------------------------------------------------
template <int L, bool QMF>
__global__ void __launch_bounds__(kCThreads, (L >= 16) ? 3 : 4) k_column_analysis(const __grid_constant__ ColArgs a) {
    constexpr int R = col_rows<L>::value;
    constexpr bool ST = col_smem_taps<L>::value && !QMF;   // quadrature-mirror pairs fit the uniform registers: no LDS taps
    __shared__ double2 s_taps[ST ? L : 1];
    if (ST) {
        if (threadIdx.x < L) s_taps[threadIdx.x] = make_double2(a.f.h[threadIdx.x], a.f.g[threadIdx.x]);
        __syncthreads();
    }
    const uint32_t taps_addr = (uint32_t)__cvta_generic_to_shared(s_taps);
    // flattened (chunk, column) index, column fastest: 32 | d keeps every warp inside one chunk => coalesced rows
    const long long gid = (long long)blockIdx.x * kCThreads + threadIdx.x;
    const int d = (int)a.d;                   // host guarantees d <= 2^30
    const long long chunk = gid / a.d;
    const int col = (int)(gid - chunk * a.d);  // phase phi in [0, d); d is any integer (SoA batches: 2^(j-1) * batch)
    if (chunk >= a.chunks) return;
    for (long long b = blockIdx.y; b < a.batch; b += gridDim.y) {
        // rows of this column inside the output range: positions t0 + col + q*d < t0 + n_out
        const long long rows = (a.n_out - col + a.d - 1) / a.d;
        const long long q0 = chunk * a.rows_per_chunk;
        long long left64 = rows - q0;
        if (left64 <= 0) continue;
        int left = (int)(left64 < a.rows_per_chunk ? left64 : a.rows_per_chunk);   // rows this thread still owes
        const long long p = a.t0 + col + q0 * a.d;        // input-coordinate position of the chunk's first row
        const double *x = a.x + b * a.ldx;
        const char *xp = reinterpret_cast<const char *>(x + p);                      // current block, row 0
        char *vp = reinterpret_cast<char *>(a.v + b * a.ldv + (p - a.t0));
        char *wp = reinterpret_cast<char *>(a.w + b * a.ldw + (p - a.t0));
        // seq[0 .. L-2] = the L-1 rows before the block (oldest first), seq[L-1 + r] = the block's new rows
        double seq[L - 1 + R];
        if (p - (long long)(L - 1) * a.d >= 0) {
#pragma unroll
            for (int i = 0; i < L - 1; i++) seq[i] = __ldg(row_ptr(xp, d, -(L - 1 - i)));
        } else {
#pragma unroll
            for (int i = 0; i < L - 1; i++) seq[i] = ext_load<true>(x, p - (long long)(L - 1 - i) * a.d, a.n_in, a.mode);
        }
        // software pipeline: the next block's rows are in flight while this block's FMAs run (output rows lie inside [0, n_in))
        double nxt[R];
        if (left >= R) {
#pragma unroll
            for (int r = 0; r < R; r++) nxt[r] = __ldg(row_ptr(xp, d, r));
        } else {
#pragma unroll
            for (int r = 0; r < R; r++) nxt[r] = r < left ? __ldg(row_ptr(xp, d, r)) : 0.0;
        }
        while (left > 0) {
#pragma unroll
            for (int r = 0; r < R; r++) seq[L - 1 + r] = nxt[r];
            if (left >= 2 * R) {
#pragma unroll
                for (int r = 0; r < R; r++) nxt[r] = ldg_early(row_ptr(xp, d, R + r));
            } else if (left > R) {
#pragma unroll
                for (int r = 0; r < R; r++) nxt[r] = R + r < left ? __ldg(row_ptr(xp, d, R + r)) : 0.0;
            }
            double ah[R], ag[R];
#pragma unroll
            for (int r = 0; r < R; r++) { ah[r] = 0.0; ag[r] = 0.0; }
            if (ST) {
                // out[r] = sum_k f[k] seq[L-1+r-k], tap-outer: one broadcast LDS.128 feeds 2R DFMAs, taps ascending
#pragma unroll
                for (int k = 0; k < L; k++) {
                    double hk, gk;
                    lds_tap_pair(taps_addr + 16u * k, hk, gk);
#pragma unroll
                    for (int r = 0; r < R; r++) {
                        const double xv = seq[L - 1 + r - k];
                        ah[r] = fma(hk, xv, ah[r]);
                        ag[r] = fma(gk, xv, ag[r]);
                    }
                }
            } else {
                // walk seq downwards so every output meets its taps in ascending order; taps live in uniform registers
#pragma unroll
                for (int m = R - 1; m >= -(L - 1); m--) {
                    const double xv = seq[L - 1 + m];
#pragma unroll
                    for (int r = 0; r < R; r++) {
                        const int k = r - m;
                        if (k >= 0 && k < L) { ah[r] = fma(a.f.h[k], xv, ah[r]); ag[r] = fma(vw_tap_g<L, QMF>(a.f, k), xv, ag[r]); }
                    }
                }
            }
            if (left >= R) {
#pragma unroll
                for (int r = 0; r < R; r++) { *row_ptr(vp, d, r) = ah[r]; *row_ptr(wp, d, r) = ag[r]; }
            } else {
#pragma unroll
                for (int r = 0; r < R; r++)
                    if (r < left) { *row_ptr(vp, d, r) = ah[r]; *row_ptr(wp, d, r) = ag[r]; }
            }
#pragma unroll
            for (int i = 0; i < L - 1; i++) seq[i] = seq[i + R];   // slide: keep the last L-1 rows
            const long long step = (long long)d * (8 * R);
            xp += step; vp += step; wp += step;
            left -= R;
        }
    }
}

// ---- synthesis -----------------------------------------------------------------------------------------------
// out[o] = sum_k th[k] V[pos(o+k) + off_h] + sum_k tg[k] W[pos(o+k) + off_g],  pos(m) = t0 + col + m d
// with (taps, off) = (f, -tau) for sigma=+1 and (reversed f, tau - (L-1) d) for sigma=-1.
// Transposed FIR: the thread keeps the L-1 unfinished output sums instead of two L-1 deep input windows (half the
// registers): input row m adds th[k] V_m + tg[k] W_m to output m-k; an output is complete after input row o+L-1.
// A chunk of `nout` output rows consumes nout + L-1 input rows; block i reads input rows [iR, iR+R) and completes
// output rows [iR-(L-1), iR-(L-1)+R).
template <int L, bool EDGE, bool QMF>
__device__ __forceinline__ void col_synth_chunk(const ColArgs &a, const double *__restrict__ v, const double *__restrict__ w,
                                                char *op, int d, int nout, long long pin, uint32_t taps_addr, bool thr_on,
                                                double lam) {
    constexpr int R = col_rows_syn<L>::value;
    const bool thr_nonneg = !(lam < 0.0);
    // acc[j] <-> output row  m0 - (L-1) + j ; rows below 0 are never emitted
    double acc[L - 1 + R];
#pragma unroll
    for (int j = 0; j < L - 1 + R; j++) acc[j] = 0.0;
    int in_left = nout + (L - 1);                 // input rows still to consume
    int lead = L - 1;                             // output rows of the current block that precede the chunk (not emitted)
    const char *vp = v ? reinterpret_cast<const char *>(v + pin + a.off_h) : nullptr;   // only dereferenced when !EDGE
    const char *wp = w ? reinterpret_cast<const char *>(w + pin + a.off_g) : nullptr;
    auto load_block = [&](int first, int avail, double (&nv)[R], double (&nw)[R]) {
        // rows first .. first+R-1 relative to the current block start; `avail` = rows still in range counted from `first`
        if (!EDGE && avail >= R) {
#pragma unroll
            for (int r = 0; r < R; r++) {
                nv[r] = v ? ldg_early(row_ptr(vp, d, first + r)) : 0.0;
                nw[r] = w ? ldg_early(row_ptr(wp, d, first + r)) : 0.0;
            }
        } else {
#pragma unroll
            for (int r = 0; r < R; r++) {
                const bool live = r < avail;
                if (EDGE) {
                    const long long pos = pin + (long long)(first + r) * a.d;
                    nv[r] = (live && v) ? ext_load<true>(v, pos + a.off_h, a.n_in, a.mode) : 0.0;
                    nw[r] = (live && w) ? ext_load<true>(w, pos + a.off_g, a.n_in, a.mode) : 0.0;
                } else {
                    nv[r] = (live && v) ? __ldg(row_ptr(vp, d, first + r)) : 0.0;
                    nw[r] = (live && w) ? __ldg(row_ptr(wp, d, first + r)) : 0.0;
                }
            }
        }
    };
    // software pipeline: block i+1's rows are in flight while block i's FMAs run
    double nv[R], nw[R];
    load_block(0, in_left, nv, nw);
    while (in_left > 0) {
        double cv[R], cw[R];
#pragma unroll
        for (int r = 0; r < R; r++) { cv[r] = nv[r]; cw[r] = thr_on ? (thr_nonneg ? vw_threshold_nonneg(nw[r], lam, a.thr_soft) : vw_threshold_value(nw[r], lam, a.thr_soft)) : nw[r]; }
        if (in_left > R) load_block(R, in_left - R, nv, nw);
        if (col_smem_taps_syn<L>::value && !QMF) {
#pragma unroll
            for (int k = 0; k < L; k++) {
                double hk, gk;
                lds_tap_pair(taps_addr + 16u * k, hk, gk);
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const int j = r + L - 1 - k;
                    acc[j] = fma(hk, cv[r], acc[j]);
                    acc[j] = fma(gk, cw[r], acc[j]);
                }
            }
        } else {
#pragma unroll
            for (int r = 0; r < R; r++) {
#pragma unroll
                for (int k = 0; k < L; k++) {
                    const int j = r + L - 1 - k;
                    acc[j] = fma(a.f.h[k], cv[r], acc[j]);
                    acc[j] = fma(vw_tap_g<L, QMF>(a.f, k), cw[r], acc[j]);
                }
            }
        }
        // outputs j in [0, R) are complete: chunk rows  m0-(L-1)+j; op points at chunk row m0-(L-1) (may precede the chunk)
        // (row j of the block is chunk row m0-(L-1)+j: inside the chunk iff lead <= j < in_left)
        if (lead <= 0 && in_left >= R) {
#pragma unroll
            for (int j = 0; j < R; j++) *row_ptr(op, d, j) = acc[j];
        } else {
#pragma unroll
            for (int j = 0; j < R; j++)
                if (j >= lead && j < in_left) *row_ptr(op, d, j) = acc[j];
        }
#pragma unroll
        for (int j = 0; j < L - 1; j++) acc[j] = acc[j + R];
#pragma unroll
        for (int j = L - 1; j < L - 1 + R; j++) acc[j] = 0.0;
        const long long step = (long long)d * (8 * R);
        if (!EDGE) { if (vp) vp += step; if (wp) wp += step; }
        pin += (long long)R * a.d;
        op += step;
        in_left -= R;
        lead -= R;
    }
}

#ifndef VW_COL_CS
#define VW_COL_CS 2
#endif
template <int L, bool QMF>
__global__ void __launch_bounds__(kCThreads, (L >= 24) ? VW_COL_CS : ((L >= 16) ? 3 : 4)) k_column_synthesis(const __grid_constant__ ColArgs a) {
    constexpr bool ST = col_smem_taps_syn<L>::value && !QMF;
    __shared__ double2 s_taps[ST ? L : 1];
    if (ST) {
        if (threadIdx.x < L) s_taps[threadIdx.x] = make_double2(a.f.h[threadIdx.x], a.f.g[threadIdx.x]);
        __syncthreads();
    }
    const uint32_t taps_addr = (uint32_t)__cvta_generic_to_shared(s_taps);
    const long long gid = (long long)blockIdx.x * kCThreads + threadIdx.x;
    const int d = (int)a.d;
    const long long chunk = gid / a.d;
    const int col = (int)(gid - chunk * a.d);   // any integer dilation (SoA batches run at 2^(j-1) * batch)
    if (chunk >= a.chunks) return;
    for (long long b = blockIdx.y; b < a.batch; b += gridDim.y) {
        const double *v = a.x ? a.x + b * a.ldx : nullptr;
        const double *w = a.w_in ? a.w_in + b * a.ldw_in : nullptr;
        const long long rows = (a.n_out - col + a.d - 1) / a.d;
        const long long o_start = chunk * a.rows_per_chunk;
        const long long left64 = rows - o_start;
        if (left64 <= 0) continue;
        const int nout = (int)(left64 < a.rows_per_chunk ? left64 : a.rows_per_chunk);
        const long long pin0 = a.t0 + col + o_start * a.d;  // position of input row o_start (before stream offsets)
        // the first block's outputs are chunk rows -(L-1) .. : start the output pointer there (never dereferenced below row 0)
        char *op = reinterpret_cast<char *>(a.v + b * a.ldv + col + o_start * a.d) - (long long)d * (8 * (L - 1));
        const long long lo_off = a.off_h < a.off_g ? a.off_h : a.off_g, hi_off = a.off_h < a.off_g ? a.off_g : a.off_h;
        const long long last_pos = pin0 + (long long)(nout + L - 2) * a.d;
        const bool thr_on = a.thr != nullptr && w != nullptr;
        const double lam = thr_on ? a.thr[a.thr_per_row ? b : 0] : 0.0;
        if (pin0 + lo_off >= 0 && last_pos + hi_off < a.n_in) col_synth_chunk<L, false, QMF>(a, v, w, op, d, nout, pin0, taps_addr, thr_on, lam);
        else col_synth_chunk<L, true, QMF>(a, v, w, op, d, nout, pin0, taps_addr, thr_on, lam);
    }
}

// ---- lattice form (long quadrature-mirror pairs whose taps fit a paraunitary lattice: vw_lattice.cu) -------------
// Same thread / chunk / column geometry and the same loads and stores as the direct kernels above; only the arithmetic
// differs.  Per column the undilated sequence u[q] goes through  E(z) = S_{K-1} Lam ... S_1 Lam B  (Lam delays the second
// channel by TWO rows: the undecimated transform is two interleaved decimated ones, rows of equal parity share a delay
// line): per row one 2 x 2 product and K-1 stages of two FMAs give V[q] and W[q] together -- L + 2 FP64 instructions per
// sample where the direct form spends 2L, which moves coif5 from the FP64 roof to the HBM roof (24 B/sample).  State per
// thread: 2 (K-1) delayed values + the previous input row -- the size of the direct form's L-1 window, but nothing shifts:
// with R even every delay slot is a fixed register of the unrolled body.
struct ColLat { double b[4]; double t[VW_LATTICE_MAX_K - 1]; };

constexpr int kLR = 10;   // rows per block (even)

template <int K>
__global__ void __launch_bounds__(kCThreads, 3) k_column_analysis_lat(const __grid_constant__ ColArgs a, const __grid_constant__ ColLat c) {
    constexpr int L = 2 * K, R = kLR;
    constexpr int LEAD = ((L - 1 + R - 1) / R) * R;   // warm-up rows before the chunk: whole blocks, nothing of them is stored
    static_assert(R % 2 == 0 && LEAD % 2 == 0, "row parity must be a compile-time property of the unrolled body");
    const long long gid = (long long)blockIdx.x * kCThreads + threadIdx.x;
    const int d = (int)a.d;
    const long long chunk = gid / a.d;
    const int col = (int)(gid - chunk * a.d);
    if (chunk >= a.chunks) return;
    for (long long b = blockIdx.y; b < a.batch; b += gridDim.y) {
        const long long rows = (a.n_out - col + a.d - 1) / a.d;
        const long long q0 = chunk * a.rows_per_chunk;
        const long long left64 = rows - q0;
        if (left64 <= 0) continue;
        const int left = (int)(left64 < a.rows_per_chunk ? left64 : a.rows_per_chunk);
        const long long p = a.t0 + col + q0 * a.d;            // position of the chunk's first output row
        const long long p_lead = p - (long long)LEAD * a.d;   // position of the first warm-up row
        const double *x = a.x + b * a.ldx;
        const bool lead_plain = p_lead >= 0;                   // warm-up rows inside the row: plain loads
        const long long step = (long long)d * (8 * R);
        // all three pointers address row 0 of the CURRENT block; v / w are not dereferenced during the warm-up
        const char *xp = reinterpret_cast<const char *>(x + p) - (long long)d * (8 * LEAD);
        char *vp = reinterpret_cast<char *>(a.v + b * a.ldv + (p - a.t0)) - (long long)d * (8 * LEAD);
        char *wp = reinterpret_cast<char *>(a.w + b * a.ldw + (p - a.t0)) - (long long)d * (8 * LEAD);
        double dl[K - 1][2];
#pragma unroll
        for (int k = 0; k < K - 1; k++) { dl[k][0] = 0.0; dl[k][1] = 0.0; }
        double uprev = 0.0;     // the row before the first warm-up row: nothing that is stored depends on it
        int lead = LEAD;        // warm-up rows still ahead (counted from the current block)
        int todo = left;        // output rows still owed once the warm-up is over
        double nxt[R];
        if (lead_plain) {
#pragma unroll
            for (int r = 0; r < R; r++) nxt[r] = __ldg(row_ptr(xp, d, r));
        } else {
#pragma unroll
            for (int r = 0; r < R; r++) nxt[r] = ext_load<true>(x, p_lead + (long long)r * a.d, a.n_in, a.mode);
        }
        while (todo > 0) {
            double cur[R];
#pragma unroll
            for (int r = 0; r < R; r++) cur[r] = nxt[r];
            // next block: still warm-up (maybe outside the row), or output rows (always inside [0, n_in))
            const int avail = lead > 0 ? todo + lead - R : todo - R;     // rows that exist from the next block's row 0 on
            if (lead > R && !lead_plain) {
                const long long pn = p - (long long)(lead - R) * a.d;
#pragma unroll
                for (int r = 0; r < R; r++) nxt[r] = ext_load<true>(x, pn + (long long)r * a.d, a.n_in, a.mode);
            } else if (avail >= R) {
#pragma unroll
                for (int r = 0; r < R; r++) nxt[r] = ldg_early(row_ptr(xp, d, R + r));
            } else if (avail > 0) {
#pragma unroll
                for (int r = 0; r < R; r++) nxt[r] = r < avail ? __ldg(row_ptr(xp, d, R + r)) : 0.0;
            }
            double ah[R], ag[R];
#pragma unroll
            for (int r = 0; r < R; r++) {
                const double xv = cur[r];
                double aa = fma(c.b[1], uprev, c.b[0] * xv);
                double bb = fma(c.b[3], uprev, c.b[2] * xv);
                uprev = xv;
#pragma unroll
                for (int k = 0; k < K - 1; k++) {
                    const double bd = dl[k][r & 1];
                    dl[k][r & 1] = bb;
                    const double an = fma(c.t[k], bd, aa);
                    bb = fma(-c.t[k], aa, bd);
                    aa = an;
                }
                ah[r] = aa; ag[r] = bb;
            }
            if (lead <= 0) {
                if (todo >= R) {
#pragma unroll
                    for (int r = 0; r < R; r++) { *row_ptr(vp, d, r) = ah[r]; *row_ptr(wp, d, r) = ag[r]; }
                } else {
#pragma unroll
                    for (int r = 0; r < R; r++)
                        if (r < todo) { *row_ptr(vp, d, r) = ah[r]; *row_ptr(wp, d, r) = ag[r]; }
                }
                todo -= R;
            }
            lead -= R;
            xp += step; vp += step; wp += step;
        }
    }
}

// out[o] = y0(o + L - 2) + y1(o + L - 1) with  y(m) = B^T D S_1^T D ... D S_{K-1}^T [V'[m]; W'[m]]  (D delays the FIRST channel by
// two rows): the transposed cascade.  Input row m completes output row m - (L-1), exactly like the transposed direct form
// above, so the chunk bookkeeping (lead, in_left, the output pointer that starts L-1 rows early) is shared with it.
template <int K, bool EDGE, bool THR>
__device__ __forceinline__ void col_synth_chunk_lat(const ColArgs &a, const ColLat &c, const double *__restrict__ v,
                                                    const double *__restrict__ w, char *op, int d, int nout, long long pin,
                                                    double lam) {
    constexpr int L = 2 * K, R = kLR;
    static_assert(R % 2 == 0, "row parity must be a compile-time property of the unrolled body");
    const bool thr_nonneg = !(lam < 0.0);
    double dl[K - 1][2];
#pragma unroll
    for (int k = 0; k < K - 1; k++) { dl[k][0] = 0.0; dl[k][1] = 0.0; }
    double y0prev = 0.0;
    int in_left = nout + (L - 1);
    int lead = L - 1;
    const char *vp = v ? reinterpret_cast<const char *>(v + pin + a.off_h) : nullptr;
    const char *wp = w ? reinterpret_cast<const char *>(w + pin + a.off_g) : nullptr;
    auto load_block = [&](int first, int avail, double (&nv)[R], double (&nw)[R]) {
        if (!EDGE && avail >= R) {
#pragma unroll
            for (int r = 0; r < R; r++) {
                nv[r] = v ? ldg_early(row_ptr(vp, d, first + r)) : 0.0;
                nw[r] = w ? ldg_early(row_ptr(wp, d, first + r)) : 0.0;
            }
        } else {
#pragma unroll
            for (int r = 0; r < R; r++) {
                const bool live = r < avail;
                if (EDGE) {
                    const long long pos = pin + (long long)(first + r) * a.d;
                    nv[r] = (live && v) ? ext_load<true>(v, pos + a.off_h, a.n_in, a.mode) : 0.0;
                    nw[r] = (live && w) ? ext_load<true>(w, pos + a.off_g, a.n_in, a.mode) : 0.0;
                } else {
                    nv[r] = (live && v) ? __ldg(row_ptr(vp, d, first + r)) : 0.0;
                    nw[r] = (live && w) ? __ldg(row_ptr(wp, d, first + r)) : 0.0;
                }
            }
        }
    };
    double nv[R], nw[R];
    load_block(0, in_left, nv, nw);
    while (in_left > 0) {
        double cv[R], cw[R];
#pragma unroll
        for (int r = 0; r < R; r++) { cv[r] = nv[r]; cw[r] = THR ? (thr_nonneg ? vw_threshold_nonneg(nw[r], lam, a.thr_soft) : vw_threshold_value(nw[r], lam, a.thr_soft)) : nw[r]; }
        if (in_left > R) load_block(R, in_left - R, nv, nw);
        double o[R];
#pragma unroll
        for (int r = 0; r < R; r++) {
            double aa = cv[r], bb = cw[r];
#pragma unroll
            for (int k = K - 2; k >= 0; k--) {
                const double an = fma(-c.t[k], bb, aa);
                bb = fma(c.t[k], aa, bb);
                aa = dl[k][r & 1];
                dl[k][r & 1] = an;
            }
            const double y0 = fma(c.b[2], bb, c.b[0] * aa);
            const double y1 = fma(c.b[3], bb, c.b[1] * aa);
            o[r] = y0prev + y1;
            y0prev = y0;
        }
        if (lead <= 0 && in_left >= R) {
#pragma unroll
            for (int j = 0; j < R; j++) *row_ptr(op, d, j) = o[j];
        } else {
#pragma unroll
            for (int j = 0; j < R; j++)
                if (j >= lead && j < in_left) *row_ptr(op, d, j) = o[j];
        }
        const long long step = (long long)d * (8 * R);
        if (!EDGE) { if (vp) vp += step; if (wp) wp += step; }
        pin += (long long)R * a.d;
        op += step;
        in_left -= R;
        lead -= R;
    }
}

template <int K>
__global__ void __launch_bounds__(kCThreads, 3) k_column_synthesis_lat(const __grid_constant__ ColArgs a, const __grid_constant__ ColLat c) {
    constexpr int L = 2 * K;
    const long long gid = (long long)blockIdx.x * kCThreads + threadIdx.x;
    const int d = (int)a.d;
    const long long chunk = gid / a.d;
    const int col = (int)(gid - chunk * a.d);
    if (chunk >= a.chunks) return;
    for (long long b = blockIdx.y; b < a.batch; b += gridDim.y) {
        const double *v = a.x ? a.x + b * a.ldx : nullptr;
        const double *w = a.w_in ? a.w_in + b * a.ldw_in : nullptr;
        const long long rows = (a.n_out - col + a.d - 1) / a.d;
        const long long o_start = chunk * a.rows_per_chunk;
        const long long left64 = rows - o_start;
        if (left64 <= 0) continue;
        const int nout = (int)(left64 < a.rows_per_chunk ? left64 : a.rows_per_chunk);
        const long long pin0 = a.t0 + col + o_start * a.d;
        char *op = reinterpret_cast<char *>(a.v + b * a.ldv + col + o_start * a.d) - (long long)d * (8 * (L - 1));
        const long long lo_off = a.off_h < a.off_g ? a.off_h : a.off_g, hi_off = a.off_h < a.off_g ? a.off_g : a.off_h;
        const long long last_pos = pin0 + (long long)(nout + L - 2) * a.d;
        const bool thr_on = a.thr != nullptr && w != nullptr;
        const double lam = thr_on ? a.thr[a.thr_per_row ? b : 0] : 0.0;
        const bool inside = pin0 + lo_off >= 0 && last_pos + hi_off < a.n_in;
        if (thr_on) {
            if (inside) col_synth_chunk_lat<K, false, true>(a, c, v, w, op, d, nout, pin0, lam);
            else col_synth_chunk_lat<K, true, true>(a, c, v, w, op, d, nout, pin0, lam);
        } else {
            if (inside) col_synth_chunk_lat<K, false, false>(a, c, v, w, op, d, nout, pin0, lam);
            else col_synth_chunk_lat<K, true, false>(a, c, v, w, op, d, nout, pin0, lam);
        }
    }
}

// ---- two levels per pass ------------------------------------------------------------------------------------------
// With the lattice the column kernels stream at the HBM roof, so the next lever is bytes.  Level j+1 at dilation 2d is,
// inside one level-j column (rows q <-> positions col + q d), a filter over every SECOND row: the even rows are the
// level-(j+1) column col, the odd rows the column col + d.  And the level-j lattice itself only chains rows of equal parity
// (its delays are two rows); the parities meet in the 2 x 2 base product alone.  So a PAIR of lanes takes one level-j column
// -- the even lane its even rows, the odd lane the odd rows -- and each lane runs level j on its own rows (delay lines one
// slot deep), then level j+1 on the V_j it has just produced (two slots), everything in registers; the one value per row
// that crosses parities (analysis: the neighbouring input row; synthesis: the second output channel) moves by a lane
// shuffle.  V_j never exists in memory: the analysis reads V_{j-1} and writes W_j, W_{j+1}, V_{j+1} (32 B per sample for two
// levels instead of 48), the synthesis reads V_{j+1}, W_{j+1}, W_j and writes V_{j-1}.  State per lane: 3 (K-1) + 2 doubles.
// Valid where V_j outside the row is what the cascade computes from the extended input: PERIODIC, ZERO_PADDING, span calls --
// not SYMMETRIC (V_j is re-mirrored per level, ScalarOps.java:818-835), which keeps one level per pass.
template <class P>
struct ColPairT {
    const double *x; long long ldx;       // analysis: V_{j-1};  synthesis: V_{j+1}
    const double *wa; long long ldwa;     // synthesis: W_{j+1}
    const double *wb; long long ldwb;     // synthesis: W_j
    double *o0; long long ldo0;           // analysis: V_{j+1};  synthesis: V_{j-1}
    double *o1; long long ldo1;           // analysis: W_j
    double *o2; long long ldo2;           // analysis: W_{j+1}
    long long n_in, t0, n_out, batch, d;  // d = dilation of level j; a lane walks positions c2 + i * 2d, c2 in [0, 2d)
    int rows_per_chunk, chunks, mode;     // chunks of a lane's own rows (level-(j+1) rows); the kernels spread the boundaries evenly
                                          // themselves and ignore rows_per_chunk
    const double *thr; int thr_per_row, thr_soft;
    P c;                                  // the arithmetic core's coefficients (lattice, or the low-pass taps of a quadrature-mirror pair)
    long long thr_lstride;                // synthesis: W_j reads thr[0], W_{j+1} reads thr[thr_lstride] (0: one table for both)
};
typedef ColPairT<ColLat> ColPair;

#ifndef VW_PAIR_CTAS
#define VW_PAIR_CTAS 3
#endif
#ifndef VW_PAIR_R
#define VW_PAIR_R 8
#endif
// Measured on config #4 (tools/gpu_r2_pairab.sh, gpu_r2_ring.sh).  With the input rows prefetched into registers (one block of
// 8 rows ahead) the kernels needed ~250 registers: 2 CTAs/SM beat 3 CTAs/SM with spills (forward 10.1 vs 10.7 ms, inverse 10.4
// vs 13.5), 8 rows per block beat 4 and 16, a prefetch.global.L2 32 / 64 rows ahead changed nothing repeatable.  With the rows
// in a shared-memory ring filled by cp.async (below) the same kernels fit 168 registers without spills worth the name: 3 CTAs/SM
// with a ring of 2 blocks beat 2 CTAs/SM with a ring of 4 (config #4 14.0 vs 13.5-14.0 GSamples/s, its 2^25-sample spans 11.9 vs
// 11.5, sym8 J = 8 inverse 1.81 vs 2.10 ms).
constexpr int kPR = VW_PAIR_R;    // own rows per block (even: the level-(j+1) delay slots are compile-time registers)

__device__ __forceinline__ double shfl_partner(unsigned mask, double v) {
    return __shfl_xor_sync(mask, v, 1);
}

// Input rows of the pair kernels travel through a per-lane ring in shared memory, filled by 8-byte cp.async: ncu showed the
// pairs read-latency bound (long_scoreboard 1.3-3.2 warps per issue at 8 warps/SM) with a register prefetch of one block (8
// rows) -- all the ~250 registers allowed.  The ring holds kPD blocks per stream and costs no registers (which is what lets a
// third CTA onto the SM): rows are requested (kPD-1) blocks before they are used.  Slot [row mod (kPD*R)][thread]: a lane only
// ever touches its own column of the ring, so neither barriers nor bank conflicts; rows outside the signal (wrap, zero padding)
// are written with plain stores.
#ifndef VW_PAIR_DEPTH
#define VW_PAIR_DEPTH 2
#endif
constexpr int kPD = VW_PAIR_DEPTH;
extern __shared__ __align__(16) double pair_ring[];
__device__ __forceinline__ void cp_async8(uint32_t dst, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void sts64(uint32_t dst, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(dst), "d"(v) : "memory"); }
__device__ __forceinline__ double lds64(uint32_t src) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(src) : "memory");
    return v;
}

// Analysis pair: one skeleton (lanes, chunks, ring prefetch, stores), two arithmetic cores -- the lattice (long filters whose
// table fits one) and the direct form (16-20-tap quadrature-mirror pairs).  A core turns own input row xv (plus what the
// partner lane holds) into W_j, V_{j+1}, W_{j+1} of that row; LOOKBACK = own rows of history behind an output row.
struct DirTaps { double h[VW_LEAN_MAX_L]; };     // low-pass taps of a quadrature-mirror pair; g[k] = (-1)^k h[L-1-k]

template <int K> struct LatAnaCore {
    typedef ColLat Params;
    static constexpr int L = 2 * K;
    // V_{j+1} at own row i needs V_j at own rows i-(L-1) .. i, each of which needs L-1 level-j rows = L/2 own rows more
    static constexpr int LOOKBACK = L - 1 + L / 2;
    static constexpr int CTAS = VW_PAIR_CTAS;
    double dl1[K - 1], dl2[K - 1][2], xprev, vprev;
    __device__ __forceinline__ void init() {
#pragma unroll
        for (int k = 0; k < K - 1; k++) { dl1[k] = 0.0; dl2[k][0] = dl2[k][1] = 0.0; }
        xprev = vprev = 0.0;
    }
    __device__ __forceinline__ void row(const Params &c, int r, int rho, unsigned mask, double xv, double &w1, double &v2, double &w2) {
        // the neighbouring level-j row: the even lane needs the odd lane's PREVIOUS row, the odd lane the even lane's current one
        const double un = shfl_partner(mask, rho ? xprev : xv);
        xprev = xv;
        double aa = fma(c.b[1], un, c.b[0] * xv);
        double bb = fma(c.b[3], un, c.b[2] * xv);
#pragma unroll
        for (int k = 0; k < K - 1; k++) {
            const double bd = dl1[k];
            dl1[k] = bb;
            const double an = fma(c.t[k], bd, aa);
            bb = fma(-c.t[k], aa, bd);
            aa = an;
        }
        w1 = bb;
        double a2 = fma(c.b[1], vprev, c.b[0] * aa);
        double b2 = fma(c.b[3], vprev, c.b[2] * aa);
        vprev = aa;
#pragma unroll
        for (int k = 0; k < K - 1; k++) {
            const double bd = dl2[k][r & 1];
            dl2[k][r & 1] = b2;
            const double an = fma(c.t[k], bd, a2);
            b2 = fma(-c.t[k], a2, bd);
            a2 = an;
        }
        v2 = a2; w2 = b2;
    }
    __device__ __forceinline__ void end_block() {}
};

// Direct form.  col[]: the level-j column around the block -- own rows at odd offsets from the block start, the partner's
// (one level-j row earlier each, received by shuffle) at even ones, so col[L-1 + 2r - k] is u[q - k] for the own row q of step r
// on either lane; v1[]: the lane's own V_j rows, which are all level j+1 needs (dilation 2 in level-j rows).  Taps ascending, as
// everywhere (ScalarOps.java:700-723).
template <int L> struct DirAnaCore {
    typedef DirTaps Params;
    static constexpr int R = VW_PAIR_R;
    static constexpr int LOOKBACK = L - 1 + L / 2;
#ifndef VW_DIR_CTAS
#define VW_DIR_CTAS 3
#endif
    static constexpr int CTAS = VW_DIR_CTAS;
    double col[L - 1 + 2 * R], v1[L - 1 + R], xprev;
    static __device__ __forceinline__ double gk(const Params &c, int k) { return (k & 1) ? -c.h[L - 1 - k] : c.h[L - 1 - k]; }
    __device__ __forceinline__ void init() {
#pragma unroll
        for (int j = 0; j < L - 1 + 2 * R; j++) col[j] = 0.0;
#pragma unroll
        for (int j = 0; j < L - 1 + R; j++) v1[j] = 0.0;
        xprev = 0.0;
    }
    __device__ __forceinline__ void row(const Params &c, int r, int rho, unsigned mask, double xv, double &w1, double &v2, double &w2) {
        const double un = shfl_partner(mask, rho ? xprev : xv);
        xprev = xv;
        col[L - 2 + 2 * r] = un;
        col[L - 1 + 2 * r] = xv;
        double ah = 0.0, ag = 0.0;
#pragma unroll
        for (int k = 0; k < L; k++) {
            ah = fma(c.h[k], col[L - 1 + 2 * r - k], ah);
            ag = fma(gk(c, k), col[L - 1 + 2 * r - k], ag);
        }
        w1 = ag;
        v1[L - 1 + r] = ah;
        double bh = 0.0, bg = 0.0;
#pragma unroll
        for (int k = 0; k < L; k++) {
            bh = fma(c.h[k], v1[L - 1 + r - k], bh);
            bg = fma(gk(c, k), v1[L - 1 + r - k], bg);
        }
        v2 = bh; w2 = bg;
    }
    __device__ __forceinline__ void end_block() {
#pragma unroll
        for (int j = 0; j < L - 1; j++) col[j] = col[j + 2 * R];
#pragma unroll
        for (int j = 0; j < L - 1; j++) v1[j] = v1[j + R];
    }
};

template <class Core>
__global__ void __launch_bounds__(kCThreads, Core::CTAS) k_column_analysis_pair(const __grid_constant__ ColPairT<typename Core::Params> a) {
    constexpr int R = kPR;
    constexpr int LEAD = ((Core::LOOKBACK + R - 1) / R) * R;     // warm-up own rows before the chunk: whole blocks
    static_assert(R % 2 == 0 && LEAD % 2 == 0, "delay slots must be compile-time registers");
    const long long gid = (long long)blockIdx.x * kCThreads + threadIdx.x;
    const long long d2 = 2 * a.d;
    const long long pid = gid >> 1;            // lane pair = one level-j column of one chunk
    const int rho = (int)(gid & 1);            // this lane's row parity inside the level-j column
    const long long chunk = pid / a.d;
    const long long c2 = (pid - chunk * a.d) + (rho ? a.d : 0);   // own level-(j+1) column
    const unsigned mask = __ballot_sync(0xffffffffu, chunk < a.chunks);
    if (chunk >= a.chunks) return;
    for (long long b = blockIdx.y; b < a.batch; b += gridDim.y) {
        const long long rows = a.n_out > c2 ? (a.n_out - c2 + d2 - 1) / d2 : 0;   // own rows inside the output range
        // chunk boundaries spread evenly over the longest column (multiples of 8 rows): a short last chunk would keep its warp
        // -- and with one wave per launch the whole kernel -- on the slow path long after the others have finished
        const long long rows_max = (a.n_out + d2 - 1) / d2;
        const long long i0 = ((chunk * rows_max) / a.chunks) & ~7ll;
        const long long i1 = chunk + 1 == a.chunks ? rows_max : (((chunk + 1) * rows_max) / a.chunks) & ~7ll;
        long long left64 = (i1 < rows ? i1 : rows) - i0;
        if (left64 < 0) left64 = 0;
        const int left = (int)left64;
        const int steps = __reduce_max_sync(mask, left) + LEAD;        // the lanes of a warp walk in step (shuffles)
        const long long p = a.t0 + c2 + i0 * d2;                       // position of the first own output row
        const long long p_lead = p - (long long)LEAD * d2;
        const double *x = a.x + b * a.ldx;
        const long long step = d2 * (8 * R);
        const long long back = d2 * (8 * LEAD);
        const char *xp = reinterpret_cast<const char *>(x + p) - back;               // own row 0 of the CURRENT block
        char *vp = reinterpret_cast<char *>(a.o0 + b * a.ldo0 + (p - a.t0)) - back;
        char *w1p = reinterpret_cast<char *>(a.o1 + b * a.ldo1 + (p - a.t0)) - back;
        char *w2p = reinterpret_cast<char *>(a.o2 + b * a.ldo2 + (p - a.t0)) - back;
        const int d2i = (int)d2;
        Core core;
        core.init();
        const int have = LEAD + left;          // own rows that exist from step 0 on (warm-up + outputs)
        constexpr int RING = kPD * R;          // rows in the ring (a power of two)
        static_assert((RING & (RING - 1)) == 0, "ring slots are taken modulo a power of two");
        const uint32_t ring = (uint32_t)__cvta_generic_to_shared(pair_ring) + threadIdx.x * 8u;
        auto slot = [&](int s) { return ring + (uint32_t)(s & (RING - 1)) * (kCThreads * 8u); };
        // request own row s (counted from the first warm-up row) into its ring slot
        auto fetch = [&](int s) {
            if (s >= have) { sts64(slot(s), 0.0); return; }
            const long long pos = p_lead + (long long)s * d2;
            if (pos >= 0 && pos < a.n_in) cp_async8(slot(s), x + pos);
            else sts64(slot(s), ext_load<true>(x, pos, a.n_in, a.mode));
        };
        // one commit group per block, so that "all but the newest kPD-1 groups" means "the current block" from the first iteration on
#pragma unroll
        for (int r = 0; r < (kPD - 1) * R; r++) {
            fetch(r);
            if ((r + 1) % R == 0) cp_async_commit();
        }
        for (int s0 = 0; s0 < steps; s0 += R) {
            // steady state for the whole warp: every lane stores this whole block, and the block requested now -- (kPD-1) blocks
            // ahead -- lies inside the row
            const bool fast = s0 >= LEAD && s0 + kPD * R <= have;
            const uint32_t cur = slot(s0), ahead = slot(s0 + (kPD - 1) * R);     // blocks never straddle the ring's end
            if (__all_sync(mask, fast)) {
#pragma unroll
                for (int r = 0; r < R; r++) cp_async8(ahead + r * (kCThreads * 8u), row_ptr(xp, d2i, (kPD - 1) * R + r));
                cp_async_commit();
                cp_async_wait<kPD - 1>();
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const double xv = lds64(cur + r * (kCThreads * 8u));
                    double w1, v2, w2;
                    core.row(a.c, r, rho, mask, xv, w1, v2, w2);
                    *row_ptr(w1p, d2i, r) = w1; *row_ptr(vp, d2i, r) = v2; *row_ptr(w2p, d2i, r) = w2;
                }
            } else {
#pragma unroll
                for (int r = 0; r < R; r++) fetch(s0 + (kPD - 1) * R + r);
                cp_async_commit();
                cp_async_wait<kPD - 1>();
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const double xv = lds64(cur + r * (kCThreads * 8u));
                    double w1, v2, w2;
                    core.row(a.c, r, rho, mask, xv, w1, v2, w2);
                    if (s0 + r >= LEAD && s0 + r < have) { *row_ptr(w1p, d2i, r) = w1; *row_ptr(vp, d2i, r) = v2; *row_ptr(w2p, d2i, r) = w2; }
                }
            }
            core.end_block();
            xp += step; vp += step; w1p += step; w2p += step;
        }
        cp_async_wait<0>();
    }
}

// Synthesis pair.  A lane consumes (V_{j+1}, W_{j+1}) at own row s, which completes V_j at own row s - (L-1); that value and
// W_j of the same row go into level j, whose outputs mix the parities (index rule t + k d, MultiLevelMODWTTransform.java:554-601):
// one value per row crosses the lane pair by shuffle.  The skeleton (lanes, chunks, prefetch, stores) is shared by two
// arithmetic cores: the lattice (long filters whose table fits one) and the direct transposed form (16-20-tap quadrature-mirror
// pairs, whose decimal tables fit no lattice).  The even lane's output lags its consumed row by LAG1 + LAG0 own rows, the odd
// lane's by one more.
template <int K> struct LatSynCore {
    typedef ColLat Params;
    static constexpr int LAG1 = 2 * K - 1;     // own rows between a consumed (V, W)_{j+1} row and the V_j row it completes
    static constexpr int LAG0 = K - 1;         // ... between that V_j row and the even lane's V_{j-1} row it completes
#ifndef VW_PAIR_DEPTH_SYN
#define VW_PAIR_DEPTH_SYN VW_PAIR_DEPTH
#endif
    static constexpr int CTAS = VW_PAIR_CTAS, DEPTH = VW_PAIR_DEPTH_SYN;
    double dl1[K - 1], dl2[K - 1][2], y0prev, z0prev;
    __device__ __forceinline__ void init() {
#pragma unroll
        for (int k = 0; k < K - 1; k++) { dl1[k] = 0.0; dl2[k][0] = dl2[k][1] = 0.0; }
        y0prev = z0prev = 0.0;
    }
    // V_{j-1}[q] = y0(q + L-2) + y1(q + L-1): one term from each lane of the pair
    __device__ __forceinline__ double row(const Params &c, int r, int rho, unsigned mask, double cv, double cw2, double cw1) {
        double aa = cv, bb = cw2;
#pragma unroll
        for (int k = K - 2; k >= 0; k--) {
            const double an = fma(-c.t[k], bb, aa);
            bb = fma(c.t[k], aa, bb);
            aa = dl2[k][r & 1];
            dl2[k][r & 1] = an;
        }
        const double y0 = fma(c.b[2], bb, c.b[0] * aa);
        const double y1 = fma(c.b[3], bb, c.b[1] * aa);
        aa = y0prev + y1;               // V_j at own row s - (L-1)
        y0prev = y0;
        bb = cw1;
#pragma unroll
        for (int k = K - 2; k >= 0; k--) {
            const double an = fma(-c.t[k], bb, aa);
            bb = fma(c.t[k], aa, bb);
            aa = dl1[k];
            dl1[k] = an;
        }
        const double z0 = fma(c.b[2], bb, c.b[0] * aa);
        const double z1 = fma(c.b[3], bb, c.b[1] * aa);
        const double z1n = shfl_partner(mask, z1);
        const double out = (rho ? z0prev : z0) + z1n;
        z0prev = z0;
        return out;
    }
    __device__ __forceinline__ void end_block() {}
};

// Direct (transposed) form.  acc2[j]: V_j at own row (block start - (L-1) + j), fed by every consumed row with all L taps;
// acc1[j]: V_{j-1} at the own output row that completes at in-block step j, fed per step by 8 even taps of the lane's own V_j
// row and 8 odd taps of the partner's.  The odd lane applies its own row one step late, which makes the accumulator indices
// the same compile-time constants on both lanes (its outputs then complete one step later than the even lane's: lag + 1).
template <int L> struct DirSynCore {
    typedef DirTaps Params;
    static constexpr int R = VW_PAIR_R, H = L / 2;
    static constexpr int LAG1 = L - 1, LAG0 = H - 1;
#ifndef VW_DIR_DEPTH
#define VW_DIR_DEPTH 2
#endif
    static constexpr int CTAS = VW_DIR_CTAS, DEPTH = VW_DIR_DEPTH;
    double acc2[L - 1 + R], acc1[H - 1 + R], v1prev, w1prev;
    static __device__ __forceinline__ double gk(const Params &c, int k) { return (k & 1) ? -c.h[L - 1 - k] : c.h[L - 1 - k]; }
    __device__ __forceinline__ void init() {
#pragma unroll
        for (int j = 0; j < L - 1 + R; j++) acc2[j] = 0.0;
#pragma unroll
        for (int j = 0; j < H - 1 + R; j++) acc1[j] = 0.0;
        v1prev = w1prev = 0.0;
    }
    __device__ __forceinline__ double row(const Params &c, int r, int rho, unsigned mask, double cv, double cw2, double cw1) {
#pragma unroll
        for (int k = 0; k < L; k++) {
            const int j = L - 1 + r - k;
            acc2[j] = fma(c.h[k], cv, acc2[j]);
            acc2[j] = fma(gk(c, k), cw2, acc2[j]);
        }
        const double v1 = acc2[r];                          // V_j at own row s - (L-1): complete
        const double pv = shfl_partner(mask, v1), pw = shfl_partner(mask, cw1);
        const double ov = rho ? v1prev : v1, ow = rho ? w1prev : cw1;
        v1prev = v1; w1prev = cw1;
#pragma unroll
        for (int kk = 0; kk < H; kk++) {
            const int j = H - 1 + r - kk;
            acc1[j] = fma(c.h[2 * kk], ov, acc1[j]);
            acc1[j] = fma(gk(c, 2 * kk), ow, acc1[j]);
            acc1[j] = fma(c.h[2 * kk + 1], pv, acc1[j]);
            acc1[j] = fma(gk(c, 2 * kk + 1), pw, acc1[j]);
        }
        return acc1[r];
    }
    __device__ __forceinline__ void end_block() {
#pragma unroll
        for (int j = 0; j < L - 1; j++) acc2[j] = acc2[j + R];
#pragma unroll
        for (int j = L - 1; j < L - 1 + R; j++) acc2[j] = 0.0;
#pragma unroll
        for (int j = 0; j < H - 1; j++) acc1[j] = acc1[j + R];
#pragma unroll
        for (int j = H - 1; j < H - 1 + R; j++) acc1[j] = 0.0;
    }
};

template <class Core, bool THR>
__global__ void __launch_bounds__(kCThreads, Core::CTAS) k_column_synthesis_pair(const __grid_constant__ ColPairT<typename Core::Params> a) {
    constexpr int R = kPR, LAG1 = Core::LAG1, PD = Core::DEPTH;
    static_assert(R % 2 == 0, "delay slots must be compile-time registers");
    const long long gid = (long long)blockIdx.x * kCThreads + threadIdx.x;
    const long long d2 = 2 * a.d;
    const int d2i = (int)d2;
    const long long pid = gid >> 1;
    const int rho = (int)(gid & 1);
    const long long chunk = pid / a.d;
    const long long c2 = (pid - chunk * a.d) + (rho ? a.d : 0);
    const unsigned mask = __ballot_sync(0xffffffffu, chunk < a.chunks);
    if (chunk >= a.chunks) return;
    const int lag = LAG1 + Core::LAG0 + rho;     // own rows between a consumed row and the output row it completes
    for (long long b = blockIdx.y; b < a.batch; b += gridDim.y) {
        const double *v2 = a.x + b * a.ldx;
        const double *w2 = a.wa + b * a.ldwa;
        const double *w1 = a.wb + b * a.ldwb;
        const long long rows = a.n_out > c2 ? (a.n_out - c2 + d2 - 1) / d2 : 0;
        const long long rows_max = (a.n_out + d2 - 1) / d2;           // evenly spread chunk boundaries: see the analysis kernel
        const long long i0 = ((chunk * rows_max) / a.chunks) & ~7ll;
        const long long i1 = chunk + 1 == a.chunks ? rows_max : (((chunk + 1) * rows_max) / a.chunks) & ~7ll;
        long long left64 = (i1 < rows ? i1 : rows) - i0;
        if (left64 < 0) left64 = 0;
        const int nout = (int)left64;
        const int steps = __reduce_max_sync(mask, nout + lag);     // consumed own rows: the warp walks in step
        const long long pin0 = a.t0 + c2 + i0 * d2;                // position of consumed own row 0
        // the pair consumes two detail levels, each with its own threshold: lam1 for W_j, lam2 for W_{j+1}
        const double lam1 = THR ? a.thr[a.thr_per_row ? b : 0] : 0.0;
        const double lam2 = THR ? a.thr[a.thr_lstride + (a.thr_per_row ? b : 0)] : 0.0;
        const bool thr_nonneg = !(lam1 < 0.0) && !(lam2 < 0.0);
        auto thr = [&](double v, double lam) { return THR ? (thr_nonneg ? vw_threshold_nonneg(v, lam, a.thr_soft) : vw_threshold_value(v, lam, a.thr_soft)) : v; };
        // rows this lane (or, one step later, its partner) still needs; a short last chunk must not keep loading -- wrapped
        // or not -- while the longer chunks of its warp finish
        const int need = nout + lag + 1;
        constexpr int RING = PD * R;
        static_assert((RING & (RING - 1)) == 0, "ring slots are taken modulo a power of two");
        const uint32_t ring = (uint32_t)__cvta_generic_to_shared(pair_ring) + threadIdx.x * 8u;
        constexpr uint32_t kRow = kCThreads * 8u, kStream = RING * kCThreads * 8u;     // bytes per ring row / per stream
        auto slot = [&](int s) { return ring + (uint32_t)(s & (RING - 1)) * kRow; };
        // request consumed row s of V_{j+1}, W_{j+1} and row s - LAG1 of W_j into their ring slots
        auto fetch2 = [&](const double *rowp, uint32_t dst, int s) {
            if (s < 0 || s >= need) { sts64(dst, 0.0); return; }
            const long long pos = pin0 + (long long)s * d2;
            if (pos < a.n_in) cp_async8(dst, rowp + pos);
            else sts64(dst, ext_load<true>(rowp, pos, a.n_in, a.mode));
        };
        auto fetch = [&](int s) {
            const uint32_t dst = slot(s);
            fetch2(v2, dst, s);
            fetch2(w2, dst + kStream, s);
            fetch2(w1, dst + 2 * kStream, s - LAG1);
        };
        const long long step = d2 * (8 * R);
        const char *v2p = reinterpret_cast<const char *>(v2 + pin0);                 // consumed own row 0 of the CURRENT block
        const char *w2p = reinterpret_cast<const char *>(w2 + pin0);
        const char *w1p = reinterpret_cast<const char *>(w1 + pin0) - d2 * (8 * LAG1);
        char *op = reinterpret_cast<char *>(a.o0 + b * a.ldo0 + c2 + i0 * d2) - d2 * (8 * (long long)lag);
        Core core;
        core.init();
        // one commit group per block, so that "all but the newest PD-1 groups" means "the current block" from the first iteration on
#pragma unroll
        for (int r = 0; r < (PD - 1) * R; r++) {
            fetch(r);
            if ((r + 1) % R == 0) cp_async_commit();
        }
        for (int s0 = 0; s0 < steps; s0 += R) {
            // steady state: every row of this block is stored; the block requested now -- (PD-1) blocks ahead -- exists in all
            // three streams and lies inside the row (only the last blocks of a row's last chunk reach past its end)
            const bool fast = s0 >= lag && s0 + R <= nout + lag && s0 + PD * R <= need && s0 + (PD - 1) * R >= LAG1 &&
                              pin0 + (long long)(s0 + PD * R) * d2 <= a.n_in;
            const uint32_t cur = slot(s0), ahead = slot(s0 + (PD - 1) * R);     // blocks never straddle the ring's end
            if (__all_sync(mask, fast)) {
#pragma unroll
                for (int r = 0; r < R; r++) {
                    cp_async8(ahead + r * kRow, row_ptr(v2p, d2i, (PD - 1) * R + r));
                    cp_async8(ahead + r * kRow + kStream, row_ptr(w2p, d2i, (PD - 1) * R + r));
                    cp_async8(ahead + r * kRow + 2 * kStream, row_ptr(w1p, d2i, (PD - 1) * R + r));
                }
                cp_async_commit();
                cp_async_wait<PD - 1>();
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const double cv = lds64(cur + r * kRow), cw2 = thr(lds64(cur + r * kRow + kStream), lam2), cw1 = thr(lds64(cur + r * kRow + 2 * kStream), lam1);
                    *row_ptr(op, d2i, r) = core.row(a.c, r, rho, mask, cv, cw2, cw1);
                }
            } else {
#pragma unroll
                for (int r = 0; r < R; r++) fetch(s0 + (PD - 1) * R + r);
                cp_async_commit();
                cp_async_wait<PD - 1>();
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const double cv = lds64(cur + r * kRow), cw2 = thr(lds64(cur + r * kRow + kStream), lam2), cw1 = thr(lds64(cur + r * kRow + 2 * kStream), lam1);
                    const double o = core.row(a.c, r, rho, mask, cv, cw2, cw1);
                    if (s0 + r >= lag && s0 + r < nout + lag) *row_ptr(op, d2i, r) = o;
                }
            }
            core.end_block();
            v2p += step; w2p += step; w1p += step; op += step;
        }
        cp_async_wait<0>();
    }
}

// the lattice builds exist for the lengths whose direct column kernels are FP64-bound
bool lattice_for(const vw_ctx *ctx, const VwFilt32 &f, int l, bool qmf, ColLat &c) {
    if (!(ctx->opt_lattice & 1) || !qmf || l != 30) return false;
    VwLattice lat;
    vw_lattice_fit(f.h, f.g, l, lat);
    if (!lat.ok) return false;
    for (int j = 0; j < 4; j++) c.b[j] = lat.b[j];
    for (int j = 0; j < VW_LATTICE_MAX_K - 1; j++) c.t[j] = j < lat.k - 1 ? lat.t[j] : 0.0;
    return true;
}

// short filters keep both tap arrays in uniform registers; from 12 taps on a quadrature-mirror pair takes the QMF build
#define VW_DISPATCH_CL(L, Q, CALL)                                  \
    switch (L) {                                                    \
        case 2: CALL(2, false); break;                              \
        case 4: CALL(4, false); break;                              \
        case 6: CALL(6, false); break;                              \
        case 8: CALL(8, false); break;                              \
        case 10: CALL(10, false); break;                            \
        case 12: if (Q) CALL(12, true); else CALL(12, false); break; \
        case 16: if (Q) CALL(16, true); else CALL(16, false); break; \
        case 18: if (Q) CALL(18, true); else CALL(18, false); break; \
        case 20: if (Q) CALL(20, true); else CALL(20, false); break; \
        case 30: if (Q) CALL(30, true); else CALL(30, false); break; \
        default: return VW_EUNSUPPORTED;                            \
    }

// per_sm = CTAs of this kernel build resident on one SM (occupancy query).  The grid is sized to a whole number of
// waves: with 2-3 resident CTAs per SM a naturally sized grid of ~1800 CTAs ran 4.1 or 6.15 waves, i.e. 12-18 % of the
// run with most SMs idle (and 2.05 waves -> 68 % at the 2^25-sample spans of an 8-GPU job).
int geometry(const vw_ctx *ctx, int64_t n_out, int64_t d, int64_t batch, int per_sm, dim3 &grid, int &rows_per_chunk,
             int &chunks_out, int64_t gran = kCR, int64_t want_mul = 6, int64_t min_rpc = 4 * kCR) {
    if (d < 1 || d > (1ll << 30)) return VW_EUNSUPPORTED;
    const int64_t rows = (n_out + d - 1) / d;
    // enough (chunk, column) threads to fill the machine several times over, but chunks long enough to amortise the
    // L-1 warm-up rows each chunk re-reads
    const int64_t want_threads = (int64_t)ctx->sm_count * 512 * want_mul;
    int64_t chunks = (want_threads + d * batch - 1) / (d * batch);
    if (chunks < 1) chunks = 1;
    int64_t rpc = (rows + chunks - 1) / chunks;
    {
        // chunks long enough to amortise the warm-up rows each of them re-reads -- but never fewer lanes than one full wave
        const int64_t one_wave = (n_out * batch) / ((int64_t)std::max(per_sm, 1) * ctx->sm_count * kCThreads);
        if (ctx->opt_colrpc > 0 && min_rpc != 4 * kCR) min_rpc = ctx->opt_colrpc;   // developer knob (lattice kernels only)
        const int64_t floor_rpc = std::max<int64_t>(4 * kCR, std::min(min_rpc, one_wave));
        if (rpc < floor_rpc) rpc = floor_rpc;
    }
    rpc = ((rpc + gran - 1) / gran) * gran;
    chunks = (rows + rpc - 1) / rpc;
    int64_t blocks = (chunks * d + kCThreads - 1) / kCThreads;
    const int64_t by = batch < 65535 ? batch : 65535;
    const int64_t resident = (int64_t)std::max(per_sm, 1) * ctx->sm_count;
    if (ctx->opt_wave != 0 && by == 1 && blocks > resident) {   // (batches already run thousands of short CTAs: quantisation is negligible)
        // shrink to a whole number of waves (never grow: longer chunks only amortise the warm-up better)
        const int64_t waves = (blocks * by) / resident;
        const int64_t target = std::max<int64_t>(1, waves * resident / by);            // blocks along x
        int64_t c2 = std::max<int64_t>(1, target * kCThreads / d);                      // chunks that fit the target
        int64_t r2 = (rows + c2 - 1) / c2;
        r2 = ((r2 + gran - 1) / gran) * gran;
        c2 = (rows + r2 - 1) / r2;
        const int64_t b2 = (c2 * d + kCThreads - 1) / kCThreads;
        if (b2 <= blocks && r2 < (1ll << 30)) { rpc = r2; chunks = c2; blocks = b2; }
    }
    if (blocks > 0x7fffffffll) return VW_EUNSUPPORTED;
    rows_per_chunk = (int)rpc;
    chunks_out = (int)chunks;
    grid = dim3((unsigned)blocks, (unsigned)by);
    return VW_OK;
}

}  // namespace

// The pair kernels spread their chunk boundaries evenly themselves (rows_per_chunk is not used), so the chunk count is free:
// in a batch (one grid row per signal) make the lanes of a signal fill whole CTAs -- 3 chunks x 32 lanes would leave a
// quarter of every CTA idle (config #3, levels 5-6: rows of 2048 own rows)
static void fill_ctas(int64_t n_out, int64_t d2, int64_t batch, int &chunks, dim3 &grid) {
    if (batch <= 1 || d2 >= kCThreads || (kCThreads % d2) != 0) return;
    const int64_t q = kCThreads / d2;                              // chunks per CTA
    const int64_t rows = (n_out + d2 - 1) / d2;
    int64_t c = ((chunks + q - 1) / q) * q;
    while (c > q && rows / c < 256) c -= q;                        // keep chunks long against their warm-up rows
    if (rows / c < 64) return;
    chunks = (int)c;
    grid.x = (unsigned)((c * d2 + kCThreads - 1) / kCThreads);
}
// dynamic shared memory of the pair kernels' input rings; above 48 KB a kernel needs the opt-in attribute once per device
constexpr size_t ring_bytes(int depth) { return (size_t)depth * kPR * kCThreads * 8; }
constexpr size_t kRingBytes = ring_bytes(kPD);
static int ring_optin(vw_ctx *ctx, const void *func, size_t bytes) {
    if (bytes <= 48 * 1024) return VW_OK;
    struct Entry { int device; const void *func; };
    static std::mutex mu;
    static std::vector<Entry> done;
    std::lock_guard<std::mutex> lk(mu);
    for (const auto &e : done)
        if (e.device == ctx->device && e.func == func) return VW_OK;
    int rc = vw_cuda_check(ctx, cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes),
                           "cudaFuncSetAttribute(max dynamic smem, pair kernel)");
    if (rc) return rc;
    done.push_back({ctx->device, func});
    return VW_OK;
}
// Levels j and j+1 (d = dilation of level j) in one pass; VW_EUNSUPPORTED when the pair form does not apply (the caller
// then runs the two levels one by one).
static bool pair_ok(const vw_ctx *ctx, const VwFilt &f, int l, int64_t d, int mode, ColLat &c) {
    if (!(ctx->opt_lattice & 2) || mode == VW_SYMMETRIC || d < 1 || d > (1ll << 28)) return false;
    VwFilt32 f32;
    if (l > VW_FUSED_MAX_L) return false;
    for (int k = 0; k < VW_FUSED_MAX_L; k++) { f32.h[k] = k < l ? f.h[k] : 0.0; f32.g[k] = k < l ? f.g[k] : 0.0; }
    return lattice_for(ctx, f32, l, vw_is_qmf(f32.h, f32.g, l), c);
}

template <class Core, class A>
static int launch_pair_analysis(vw_ctx *ctx, A &a, const double *x, int64_t ldx, double *w1, int64_t ldw1, double *w2, int64_t ldw2,
                                double *v2, int64_t ldv2, int64_t n_in, int64_t t0, int64_t n_out, int64_t batch, int64_t d, int mode) {
    a.x = x; a.ldx = ldx; a.wa = a.wb = nullptr; a.ldwa = a.ldwb = 0;
    a.o0 = v2; a.ldo0 = ldv2; a.o1 = w1; a.ldo1 = ldw1; a.o2 = w2; a.ldo2 = ldw2;
    a.n_in = n_in; a.t0 = t0; a.n_out = n_out; a.batch = batch; a.d = d; a.mode = mode;
    a.thr = nullptr; a.thr_per_row = 0; a.thr_soft = 0; a.thr_lstride = 0;
    int per_sm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_column_analysis_pair<Core>, kCThreads, kRingBytes);
    dim3 grid;
    // fewer, longer chunks than the single-level kernels: every chunk re-reads its warm-up rows
    if (int rc = geometry(ctx, n_out, 2 * d, batch, per_sm, grid, a.rows_per_chunk, a.chunks, 4 * kPR, 3, 768)) return rc;
    fill_ctas(n_out, 2 * d, batch, a.chunks, grid);
    k_column_analysis_pair<Core><<<grid, kCThreads, kRingBytes, ctx->stream>>>(a);
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "column analysis (pair) launch");
}

static bool dir_pair_ok(const vw_ctx *ctx, const VwFilt &f, int l, int64_t d, int mode, int bit) {
    return (ctx->opt_lattice & bit) && mode != VW_SYMMETRIC && d >= 1 && d <= (1ll << 28) && (l == 16 || l == 18 || l == 20) &&
           vw_is_qmf(f.h, f.g, l);
}

int vw_column_analysis2(vw_ctx *ctx, const double *x, int64_t ldx, double *w1, int64_t ldw1, double *w2, int64_t ldw2, double *v2,
                        int64_t ldv2, int64_t n_in, int64_t t0, int64_t n_out, int64_t batch, const VwFilt &f, int l, int64_t d,
                        int mode) {
    if (n_out < 1 || batch < 1) return VW_EUNSUPPORTED;
    if (l == 30) {
        ColPair a;
        if (!pair_ok(ctx, f, l, d, mode, a.c)) return VW_EUNSUPPORTED;
        return launch_pair_analysis<LatAnaCore<15>>(ctx, a, x, ldx, w1, ldw1, w2, ldw2, v2, ldv2, n_in, t0, n_out, batch, d, mode);
    }
    // 16-20-tap quadrature-mirror pairs: direct form (their decimal tables fit no lattice)
    if (!dir_pair_ok(ctx, f, l, d, mode, 8)) return VW_EUNSUPPORTED;
    ColPairT<DirTaps> a;
    for (int k = 0; k < VW_LEAN_MAX_L; k++) a.c.h[k] = k < l ? f.h[k] : 0.0;
    if (l == 16) return launch_pair_analysis<DirAnaCore<16>>(ctx, a, x, ldx, w1, ldw1, w2, ldw2, v2, ldv2, n_in, t0, n_out, batch, d, mode);
    if (l == 18) return launch_pair_analysis<DirAnaCore<18>>(ctx, a, x, ldx, w1, ldw1, w2, ldw2, v2, ldv2, n_in, t0, n_out, batch, d, mode);
    return launch_pair_analysis<DirAnaCore<20>>(ctx, a, x, ldx, w1, ldw1, w2, ldw2, v2, ldv2, n_in, t0, n_out, batch, d, mode);
}

template <class Core, class A>
static int launch_pair_synthesis(vw_ctx *ctx, A &a, int64_t n_out, int64_t d, int64_t batch, bool thr) {
    int per_sm = 0;
    dim3 grid;
    if (thr) {
        if (int rc = ring_optin(ctx, (const void *)k_column_synthesis_pair<Core, true>, 3 * ring_bytes(Core::DEPTH))) return rc;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_column_synthesis_pair<Core, true>, kCThreads, 3 * ring_bytes(Core::DEPTH));
        if (int rc = geometry(ctx, n_out, 2 * d, batch, per_sm, grid, a.rows_per_chunk, a.chunks, 4 * kPR, 3, 768)) return rc;
        fill_ctas(n_out, 2 * d, batch, a.chunks, grid);
        k_column_synthesis_pair<Core, true><<<grid, kCThreads, 3 * ring_bytes(Core::DEPTH), ctx->stream>>>(a);
    } else {
        if (int rc = ring_optin(ctx, (const void *)k_column_synthesis_pair<Core, false>, 3 * ring_bytes(Core::DEPTH))) return rc;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_column_synthesis_pair<Core, false>, kCThreads, 3 * ring_bytes(Core::DEPTH));
        if (int rc = geometry(ctx, n_out, 2 * d, batch, per_sm, grid, a.rows_per_chunk, a.chunks, 4 * kPR, 3, 768)) return rc;
        fill_ctas(n_out, 2 * d, batch, a.chunks, grid);
        k_column_synthesis_pair<Core, false><<<grid, kCThreads, 3 * ring_bytes(Core::DEPTH), ctx->stream>>>(a);
    }
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "column synthesis (pair) launch");
}

template <class A>
static void fill_pair_synthesis(A &a, const double *v2, int64_t ldv2, const double *w2, int64_t ldw2, const double *w1, int64_t ldw1,
                                double *out, int64_t ldo, int64_t n_in, int64_t t0, int64_t n_out, int64_t batch, int64_t d, int mode,
                                const double *thr_dev, int thr_per_row, int thr_soft, int64_t thr_lstride) {
    a.x = v2; a.ldx = ldv2; a.wa = w2; a.ldwa = ldw2; a.wb = w1; a.ldwb = ldw1;
    a.o0 = out; a.ldo0 = ldo; a.o1 = a.o2 = nullptr; a.ldo1 = a.ldo2 = 0;
    a.n_in = n_in; a.t0 = t0; a.n_out = n_out; a.batch = batch; a.d = d; a.mode = mode;
    a.thr = thr_dev; a.thr_per_row = thr_per_row; a.thr_soft = thr_soft; a.thr_lstride = thr_lstride;
}

int vw_column_synthesis2(vw_ctx *ctx, const double *v2, int64_t ldv2, const double *w2, int64_t ldw2, const double *w1,
                         int64_t ldw1, double *out, int64_t ldo, int64_t n_in, int64_t t0, int64_t n_out, int64_t batch,
                         const VwFilt &f, int l, int64_t d, int mode, const double *thr_dev, int thr_per_row, int thr_soft,
                         int64_t thr_lstride) {
    if (n_out < 1 || batch < 1 || !v2 || !w2 || !w1) return VW_EUNSUPPORTED;
    if (l == 30) {
        ColPair a;
        if (!pair_ok(ctx, f, l, d, mode, a.c)) return VW_EUNSUPPORTED;
        fill_pair_synthesis(a, v2, ldv2, w2, ldw2, w1, ldw1, out, ldo, n_in, t0, n_out, batch, d, mode, thr_dev, thr_per_row, thr_soft,
                            thr_lstride);
        return launch_pair_synthesis<LatSynCore<15>>(ctx, a, n_out, d, batch, thr_dev != nullptr);
    }
    // 16-20-tap quadrature-mirror pairs: direct form (their decimal tables fit no lattice)
    if (!dir_pair_ok(ctx, f, l, d, mode, 4)) return VW_EUNSUPPORTED;
    ColPairT<DirTaps> a;
    for (int k = 0; k < VW_LEAN_MAX_L; k++) a.c.h[k] = k < l ? f.h[k] : 0.0;
    fill_pair_synthesis(a, v2, ldv2, w2, ldw2, w1, ldw1, out, ldo, n_in, t0, n_out, batch, d, mode, thr_dev, thr_per_row, thr_soft,
                        thr_lstride);
    if (l == 16) return launch_pair_synthesis<DirSynCore<16>>(ctx, a, n_out, d, batch, thr_dev != nullptr);
    if (l == 18) return launch_pair_synthesis<DirSynCore<18>>(ctx, a, n_out, d, batch, thr_dev != nullptr);
    return launch_pair_synthesis<DirSynCore<20>>(ctx, a, n_out, d, batch, thr_dev != nullptr);
}

int vw_column_min_level(const vw_ctx *ctx, int l, bool forward) {
    if (ctx->opt_colmin > 0) return (int)ctx->opt_colmin;
    // measured on coif5 at 2^28 samples: analysis column 1.26 / 1.18 ms at dilation 4 / 8 vs 1.37 ms tile kernel; for the
    // synthesis the two are within noise of each other (the planner's small tile at those levels loses what the tile
    // kernel gains), so both directions switch at level 3
    (void)forward;
    if (l >= 24) return 3;
    return 6;
}

int vw_column_analysis(vw_ctx *ctx, const double *x, int64_t ldx, double *v, int64_t ldv, double *w, int64_t ldw,
                       int64_t n_in, int64_t t0, int64_t n_out, int64_t batch, const VwFilt &f, int l, int64_t d, int mode) {
    if (l < 2 || l > VW_FUSED_MAX_L || n_out < 1 || batch < 1) return VW_EUNSUPPORTED;
    ColArgs a;
    dim3 grid;
    a.x = x; a.ldx = ldx; a.w_in = nullptr; a.ldw_in = 0; a.v = v; a.ldv = ldv; a.w = w; a.ldw = ldw;
    a.thr = nullptr; a.thr_per_row = 0; a.thr_soft = 0;
    a.n_in = n_in; a.t0 = t0; a.n_out = n_out; a.batch = batch; a.d = d; a.off_h = a.off_g = 0;
    a.mode = mode;
    for (int k = 0; k < VW_FUSED_MAX_L; k++) { a.f.h[k] = k < l ? f.h[k] : 0.0; a.f.g[k] = k < l ? f.g[k] : 0.0; }
    const bool qmf = vw_is_qmf(a.f.h, a.f.g, l);
    int per_sm = 0;
    ColLat lat;
    if (lattice_for(ctx, a.f, l, qmf, lat)) {
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_column_analysis_lat<15>, kCThreads, 0);
        if (int rc = geometry(ctx, n_out, d, batch, per_sm, grid, a.rows_per_chunk, a.chunks, 4 * kLR, 6, 480)) return rc;
        k_column_analysis_lat<15><<<grid, kCThreads, 0, ctx->stream>>>(a, lat);
        ctx->launches++;
        return vw_cuda_check(ctx, cudaGetLastError(), "column analysis (lattice) launch");
    }
#define VW_CO(LL, QQ) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_column_analysis<LL, QQ>, kCThreads, 0)
    VW_DISPATCH_CL(l, qmf, VW_CO)
#undef VW_CO
    int rc = geometry(ctx, n_out, d, batch, per_sm, grid, a.rows_per_chunk, a.chunks);
    if (rc) return rc;
#define VW_CA(LL, QQ) k_column_analysis<LL, QQ><<<grid, kCThreads, 0, ctx->stream>>>(a)
    VW_DISPATCH_CL(l, qmf, VW_CA)
#undef VW_CA
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "column analysis launch");
}

int vw_column_synthesis(vw_ctx *ctx, const double *v, int64_t ldv, const double *w, int64_t ldw, double *out, int64_t ldo,
                        int64_t n_in, int64_t t0, int64_t n_out, int64_t batch, const VwFilt &f, int l, int64_t d, int mode,
                        vw_align al, const double *thr_dev, int thr_per_row, int thr_soft) {
    if (l < 2 || l > VW_FUSED_MAX_L || n_out < 1 || batch < 1) return VW_EUNSUPPORTED;
    ColArgs a;
    dim3 grid;
    a.x = v; a.ldx = ldv; a.w_in = w; a.ldw_in = ldw; a.v = out; a.ldv = ldo; a.w = nullptr; a.ldw = 0;
    a.thr = thr_dev; a.thr_per_row = thr_per_row; a.thr_soft = thr_soft;
    a.n_in = n_in; a.t0 = t0; a.n_out = n_out; a.batch = batch; a.d = d;
    a.mode = mode;
    // sigma=+1: sum_k f[k] S[p - tau + k d];  sigma=-1: sum_k f[k] S[p + tau - k d] = sum_k' f[L-1-k'] S[p + tau - (L-1)d + k' d]
    a.off_h = al.sigma_h > 0 ? -(int64_t)al.tau_h : (int64_t)al.tau_h - (int64_t)(l - 1) * d;
    a.off_g = al.sigma_g > 0 ? -(int64_t)al.tau_g : (int64_t)al.tau_g - (int64_t)(l - 1) * d;
    for (int k = 0; k < VW_FUSED_MAX_L; k++) {
        a.f.h[k] = k < l ? (al.sigma_h > 0 ? f.h[k] : f.h[l - 1 - k]) : 0.0;
        a.f.g[k] = k < l ? (al.sigma_g > 0 ? f.g[k] : f.g[l - 1 - k]) : 0.0;
    }
    const bool qmf = vw_is_qmf(a.f.h, a.f.g, l);   // on the arrays as the kernel sees them (sigma = -1 streams are reversed)
    int per_sm = 0;
    ColLat lat;
    if (lattice_for(ctx, a.f, l, qmf, lat)) {
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_column_synthesis_lat<15>, kCThreads, 0);
        if (int rc = geometry(ctx, n_out, d, batch, per_sm, grid, a.rows_per_chunk, a.chunks, 4 * kLR, 6, 480)) return rc;
        k_column_synthesis_lat<15><<<grid, kCThreads, 0, ctx->stream>>>(a, lat);
        ctx->launches++;
        return vw_cuda_check(ctx, cudaGetLastError(), "column synthesis (lattice) launch");
    }
#define VW_CO(LL, QQ) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_column_synthesis<LL, QQ>, kCThreads, 0)
    VW_DISPATCH_CL(l, qmf, VW_CO)
#undef VW_CO
    int rc = geometry(ctx, n_out, d, batch, per_sm, grid, a.rows_per_chunk, a.chunks);
    if (rc) return rc;
#define VW_CS(LL, QQ) k_column_synthesis<LL, QQ><<<grid, kCThreads, 0, ctx->stream>>>(a)
    VW_DISPATCH_CL(l, qmf, VW_CS)
#undef VW_CS
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "column synthesis launch");
}
