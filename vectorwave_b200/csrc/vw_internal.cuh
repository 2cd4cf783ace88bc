// vw_internal.cuh -- shared declarations of the MODWT engine's translation units.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <chrono>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "vw_modwt.h"

#define VW_MODE_LINEAR 4  // internal: span calls -- indices outside the provided buffer are skipped

// Pre-scaled base filters passed by value in kernel parameter space (constant bank).
struct VwFilt {
    double h[VW_MAX_FILTER_TAPS];
    double g[VW_MAX_FILTER_TAPS];
};

// Compact filter block of the fused kernels (L <= 32): fully unrolled tap loops read these
// straight from the constant bank as DFMA operands.
#define VW_FUSED_MAX_L 32
struct VwFilt32 {
    double h[VW_FUSED_MAX_L];
    double g[VW_FUSED_MAX_L];
};
#ifdef __CUDACC__
// high-pass tap k with compile-time k: f.g[k], or +-f.h[L-1-k] when the pair is a quadrature mirror
template <int L, bool QMF>
__device__ __forceinline__ double vw_tap_g(const VwFilt32 &f, int k) {
    return QMF ? ((k & 1) ? -f.h[L - 1 - k] : f.h[L - 1 - k]) : f.g[k];
}
#endif

// Orthogonal wavelets: g[k] = (-1)^k h[L-1-k] (quadrature mirror, CORE/api/Daubechies.java:323-330 and the Symlet /
// Coiflet twins); scaling by 1/sqrt(2) keeps the relation bit-exact.  When it holds, kernels for long filters read
// only the L low-pass taps -- 2L doubles no longer fit the 63 uniform registers of an SM sub-partition, L do -- and
// negate on the fly (free operand modifier).  Anything else (biorthogonal pairs, reversed streams) keeps both arrays.
inline bool vw_is_qmf(const double *h, const double *g, int l) {
    for (int k = 0; k < l; k++)
        if (g[k] != ((k & 1) ? -h[l - 1 - k] : h[l - 1 - k])) return false;
    return true;
}
struct VwPlanGroup { int first, nlev; int64_t tile; double cost; };

// Paraunitary lattice of a quadrature-mirror pair (vw_lattice.cu): E(z) = S_{k-1} Lam ... S_1 Lam B with
// S_j = [[1, t_j], [-t_j, 1]] and B = [[b0, b1], [b2, b3]] (carries the scale).  ok: the double-rounded parameters
// reproduce every tap of h and g to VW_LATTICE_TOL, so the lattice kernels may stand in for the direct form.
#define VW_LATTICE_MAX_K (VW_FUSED_MAX_L / 2)
#define VW_LATTICE_TOL 2.0e-16
struct VwLattice {
    int k = 0;
    bool ok = false;
    double tap_err = 0.0;
    double t[VW_LATTICE_MAX_K - 1] = {};
    double b[4] = {};
};
void vw_lattice_fit(const double *h, const double *g, int l, VwLattice &out);

struct vw_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    std::string err;
    int64_t launches = 0;
    int sm_count = 0;
    size_t smem_optin = 0;
    // grow-only device scratch (ping-pong V buffers, staged host I/O, selection workspaces)
    static const int kScratch = 6;         // per set; set 1 belongs to the second stream of the pipelined host path
    void *scratch[2 * kScratch] = {};
    size_t scratch_bytes[2 * kScratch] = {};
    int scratch_set = 0;
    cudaStream_t pipe_stream[2] = {nullptr, nullptr};   // created on first use by the pipelined host path
    int64_t opt_pipe_chunks = 8;
    int64_t opt_pipe_min = 64ll << 20;                  // staged bytes from which host calls are chunked and overlapped
    void *pinned = nullptr;  // small pinned mailbox for D2H scalars
    size_t pinned_bytes = 0;
    struct PlanEntry { bool forward, lean_ok; int l, levels; int64_t n; std::vector<VwPlanGroup> groups; };
    mutable std::vector<PlanEntry> plan_cache;   // launch plans by shape (the planner costs 2-35 us); cleared by vw_set_option
    // Scratch is per ctx, not per stream: a call that returned without synchronising (VW_FLAG_NO_SYNC) leaves an event
    // behind, and the next call that takes scratch on a DIFFERENT stream waits on it first (vw_scratch)
    bool capturing = false;   // between vw_graph_begin and vw_graph_end: calls are recorded, nothing may synchronise
    int call_depth = 0;       // public entry points nest (handle / *_all calls use the plain ones)
    int64_t opt_timing = 0;
    int64_t opt_zero_copy = 512 * 1024;   // bytes up to which PINNED host buffers are addressed in place by the kernels (vw_shim.cu: mapped_alias); measured on config #1: 28.4 -> 15.2 us per call, bit-identical results
    cudaEvent_t time_ev[2] = {nullptr, nullptr};
    int64_t time_launch0 = 0;
    std::chrono::steady_clock::time_point time_host0;
    float time_host_ms = 0.f;
    int32_t time_launches = 0;
    bool time_valid = false;
    cudaEvent_t scratch_event = nullptr;
    cudaStream_t scratch_stream = nullptr;
    bool scratch_pending = false;
    struct OccEntry { const void *func; int nthreads; size_t smem; int per_sm; };
    std::vector<OccEntry> occ_cache;   // occupancy queries of the tile kernels (vw_fused.cu: prefetch_distance)
    int64_t opt_lean = 3;    // issue-lean tile kernels (vw_lean.cu): bit 0 = filters up to 12 taps, bit 1 = 16..20-tap quadrature-mirror pairs
    // set by the cascade drivers for the duration of a call: can this call's tile launches take the lean kernels at all
    // (not SYMMETRIC, full detail mask; threshold-on-load is fine: the lean synthesis thresholds every W tile as it lands)?  The planner budgets shared memory / registers / threads for
    // the kernels that will really run.
    bool plan_lean_ok = true;
    int64_t opt_lean_small = 1;   // lean short filters: 128-thread CTAs on ~1024-sample tiles (vw_fused.cu: lean_small_tiles)
    int64_t opt_l2pf = 3;    // L2 prefetch mask of the tile kernels: 1 = the successor CTA's input tile (V + top W), 2 = a synthesis tile's own lower W levels (sym8 J = 8 inverse 2.08 -> 1.97 ms), 4 = the successor's lower W levels too (slower); 0 = off
    std::recursive_mutex mu;   // every public entry point holds it: calls on one ctx from several host threads serialise
    int64_t opt_tile = 0, opt_fuse = 0, opt_threads = 0, opt_poly = 1;
    int64_t opt_wave = 1;    // column kernels: size single-signal grids to whole waves
    int64_t opt_colmin = 0;  // first level the column kernels may take (0 = auto: see vw_column_min_level)
    int64_t opt_colrpc = 0;  // developer knob: minimum rows per chunk of the lattice column kernels (0 = built-in)
    int64_t opt_lattice = 15; // column kernels (vw_column.cu): bit 0 = lattice form for long quadrature-mirror pairs (>= 24 taps) whose taps fit one (vw_lattice.cu), bit 1 = two lattice levels per pass, bit 2 / bit 3 = two direct-form synthesis / analysis levels per pass for 16-20-tap pairs
};

// MutableMultiLevelMODWTResult.applyThresholdToArray (CORE/modwt/MutableMultiLevelMODWTResult.java:97-118):
// soft: |c| > t ? Math.signum(c) * (|c| - t) : 0;  hard: |c| <= t ? 0 : c.  One definition for every kernel that
// thresholds on the fly.
#ifdef __CUDACC__
__device__ __forceinline__ double vw_threshold_value(double c, double lam, int soft) {
    const double a = fabs(c), m = a - lam;
    if (soft) return a > lam ? (c > 0.0 ? m : (c < 0.0 ? -m : c * m)) : 0.0;
    return a <= lam ? 0.0 : c;
}
// same value for lam >= 0 (or NaN): |c| > lam then implies c != 0 and not NaN, so signum(c) * m == copysign(m, c) --
// two FP64-pipe instructions instead of five
__device__ __forceinline__ double vw_threshold_nonneg(double c, double lam, int soft) {
    const double a = fabs(c);
    if (soft) return a > lam ? copysign(a - lam, c) : 0.0;
    return a <= lam ? 0.0 : c;
}
#endif

int vw_fail(vw_ctx *ctx, int status, const char *fmt, ...);

// helpers of vw_shim.cu that the other host-side translation units (vw_multi.cu) use
namespace vwshim {
struct DeviceGuard {
    std::unique_lock<std::recursive_mutex> lk;
    vw_ctx *ctx = nullptr;
    int prev = -1;
    bool ranged = false, timed = false;
    explicit DeviceGuard(int dev);
    DeviceGuard(vw_ctx *ctx, const char *name);
    ~DeviceGuard();
    void enter(int dev);
};
int load_filters(vw_ctx *ctx, const double *hs, const double *gs, int l, VwFilt &f);
int check_mode(vw_ctx *ctx, int mode);
int check_levels(vw_ctx *ctx, int64_t n, int l, int levels);
int check_signal_args(vw_ctx *ctx, const void *x, int64_t batch, int64_t n, int64_t ld);
int check_finite(vw_ctx *ctx, const double *x_dev, int64_t batch, int64_t n, int64_t ld, const char *what);
int no_capture(vw_ctx *ctx, const char *what);
int pinned_mailbox(vw_ctx *ctx, size_t bytes, void **out);
int copy_rows(vw_ctx *ctx, void *dst, int64_t ld_dst, const void *src, int64_t ld_src, int64_t n, int64_t rows, cudaMemcpyKind kind);
int finish(vw_ctx *ctx, uint32_t flags, bool host_io);
int forward_device(vw_ctx *ctx, const double *x, int64_t batch, int64_t n, int64_t ldx, const VwFilt &f, int l, int levels,
                   int mode, double *w, int64_t ldw, int64_t lsw, double *vj, int64_t ldv, uint32_t flags);
int inverse_device(vw_ctx *ctx, const double *w, int64_t ldw, int64_t lsw, const double *vj, int64_t ldv, int64_t batch,
                   int64_t n, const VwFilt &f, int l, int levels, int mode, const vw_align *align, int order,
                   uint64_t detail_mask, int use_approx, double *xout, int64_t ldx, uint32_t flags, const double *thr_dev,
                   int thr_per_row, int thr_soft, int64_t thr_lstride);
int stream_level_device(vw_ctx *ctx, const double *vin, int64_t batch, int64_t ldin, int64_t hist, int64_t n, const VwFilt &f,
                        int l, int level, double *w, int64_t ldw, double *v, int64_t ldv, uint32_t flags);
int inverse_span_device(vw_ctx *ctx, const double *vin, const double *w, int64_t level_stride_w, int64_t halo, int64_t n_local,
                        const double *hs, const double *gs, int32_t l, int32_t first_level, int32_t nlevels, int32_t order,
                        double *vout, uint32_t flags, const double *thr_dev, int32_t thr_soft);
}  // namespace vwshim
int vw_cuda_check(vw_ctx *ctx, cudaError_t e, const char *what);
int vw_scratch(vw_ctx *ctx, int slot, size_t bytes, void **out);

// ---- generic per-level kernels (vw_generic.cu): any n, l, dilation, mode ------------------
int vw_launch_analysis_level(vw_ctx *ctx, const double *in, int64_t ld_in, double *v_out, int64_t ld_v,
                             double *w_out, int64_t ld_w, int64_t n_in, int64_t t0, int64_t n_out, int64_t batch,
                             const VwFilt &f, int l, int64_t d, int mode, bool exact);
int vw_launch_synthesis_level(vw_ctx *ctx, const double *v, int64_t ld_v, const double *w, int64_t ld_w, double *out,
                              int64_t ld_o, int64_t n_in, int64_t t0, int64_t n_out, int64_t batch, const VwFilt &f,
                              int l, int64_t d, int mode, vw_align al, bool pair, bool exact);
int vw_launch_conv_dense(vw_ctx *ctx, const double *x, int64_t n, const double *filter, int64_t lf, int mode,
                         double *out, bool exact);
int vw_launch_threshold(vw_ctx *ctx, double *c, int64_t batch, int64_t n, int64_t ld, const double *thr_dev,
                        int per_row, int soft);
int vw_launch_nonfinite_count(vw_ctx *ctx, const double *x, int64_t batch, int64_t n, int64_t ld,
                              unsigned long long *count_dev);
int vw_launch_energy(vw_ctx *ctx, const double *c, int64_t batch, int64_t n, int64_t ld, double *out_dev);

// ---- single level over packed rows of different lengths (vw_varlen.cu) ---------------------------------------
// off_dev: batch + 1 row offsets on the device (off_dev[b] - obase = start of row b in x / w / v, strictly increasing);
// total = off_dev[batch] - obase packed samples.  Synthesis: SYMMETRIC takes t - k, the other modes t + k.
int vw_launch_varlen_analysis(vw_ctx *ctx, const double *x, const int64_t *off_dev, int64_t batch, int64_t obase, int64_t total,
                              const VwFilt &f, int l, int mode, double *w, double *v, bool exact);
int vw_launch_varlen_synthesis(vw_ctx *ctx, const double *v, const double *w, const int64_t *off_dev, int64_t batch, int64_t obase,
                               int64_t total, const VwFilt &f, int l, int mode, double *out, bool exact);
// lowest index i < n with a[i] or b[i] (b may be null) NaN / Inf, atomically min-ed into *first_dev (preset to ~0)
int vw_launch_first_nonfinite(vw_ctx *ctx, const double *a, const double *b, int64_t n, unsigned long long *first_dev);

// ---- fused multi-level tile kernels (vw_fused.cu) ------------------------------------------
// Return VW_OK when the fused path ran, VW_EUNSUPPORTED when the shape is not eligible (caller
// falls back to the per-level kernels), anything else is an error.
struct VwFusedFwd {
    const double *x; int64_t ldx;            // V_{first-1}: [batch][n_in]
    double *w; int64_t ldw, lsw;             // W_j rows for j = first .. first+nlev-1
    double *v; int64_t ldv;                  // V_{first+nlev-1}
    int64_t batch, n_in, t0, n_out;          // outputs cover input positions [t0, t0+n_out)
    int l, first_level, nlevels, mode;
    int64_t tile;                            // 0 = choose here
};
int vw_fused_forward(vw_ctx *ctx, const VwFusedFwd &p, const VwFilt &f);
struct VwFusedInv {
    const double *v; int64_t ldv;            // V_top: [batch][n_in]  (nullptr => zeros)
    const double *w; int64_t ldw, lsw;       // W_j rows, j = first .. first+nlev-1
    uint64_t detail_mask;                    // bit (j-first) clear => zeros
    double *out; int64_t ldo;                // V_{first-1}
    int64_t batch, n_in, n_out;              // outputs cover positions [0, n_out) of the input buffers
    int l, first_level, nlevels, mode;
    const double *thr_dev; int thr_per_row; int thr_soft;  // optional fused thresholding of W on load
    int64_t tile;                            // 0 = choose here
    bool has_align = false;                  // single-level stage with a general (sigma, tau) alignment (any mode)
    vw_align align = {1, 0, 1, 0};
    int64_t thr_lstride = 0;                 // level first+i reads thr_dev[i * thr_lstride]; 0: one table for every level
};

// Level schedule: which consecutive levels share one fused launch and with which tile, from a small cost model
// (FP64-pipe cycles incl. halo recompute and ragged rounds vs HBM bytes incl. halo re-reads, overlapped across the
// CTAs that fit one SM).  tile < 0 marks a level that only the per-level kernels can take.
#include <vector>
int vw_plan_levels(const vw_ctx *ctx, bool forward, int l, int levels, int64_t n, std::vector<VwPlanGroup> &out);
int vw_fused_inverse(vw_ctx *ctx, const VwFusedInv &p, const VwFilt &f);

// ---- issue-lean tile kernels of the common case (vw_lean.cu); geometry chosen by vw_fused_forward / vw_fused_inverse ----
#define VW_LEAN_MAX_L 20
int vw_lean_forward(vw_ctx *ctx, const VwFusedFwd &p, const VwFilt32 &f, int64_t tile, int64_t htot, int64_t hexact,
                    bool use_stage, int nthreads);
int vw_lean_inverse(vw_ctx *ctx, const VwFusedInv &p, const VwFilt32 &f, int64_t tile, int64_t htot, int nthreads);

// first level (1-based) the column kernels take for filter length l: dilation >= 32 normally; FP64-bound filters
// (l >= 24) already from dilation 4 (analysis) / 16 (synthesis, whose two input streams suffer more from 32-byte row pieces)
int vw_column_min_level(const vw_ctx *ctx, int l, bool forward = true);
// ---- deep single levels, dilation >= 32 (vw_column.cu): register sliding window per dilation column ---------
int vw_column_analysis(vw_ctx *ctx, const double *x, int64_t ldx, double *v, int64_t ldv, double *w, int64_t ldw,
                       int64_t n_in, int64_t t0, int64_t n_out, int64_t batch, const VwFilt &f, int l, int64_t d, int mode);
int vw_column_synthesis(vw_ctx *ctx, const double *v, int64_t ldv, const double *w, int64_t ldw, double *out, int64_t ldo,
                        int64_t n_in, int64_t t0, int64_t n_out, int64_t batch, const VwFilt &f, int l, int64_t d, int mode,
                        vw_align al, const double *thr_dev = nullptr, int thr_per_row = 0, int thr_soft = 0);

// levels j and j+1 in one pass (lattice pair kernels; d = dilation of level j).  VW_EUNSUPPORTED: run them one by one.
int vw_column_analysis2(vw_ctx *ctx, const double *x, int64_t ldx, double *w1, int64_t ldw1, double *w2, int64_t ldw2, double *v2,
                        int64_t ldv2, int64_t n_in, int64_t t0, int64_t n_out, int64_t batch, const VwFilt &f, int l, int64_t d,
                        int mode);
int vw_column_synthesis2(vw_ctx *ctx, const double *v2, int64_t ldv2, const double *w2, int64_t ldw2, const double *w1,
                         int64_t ldw1, double *out, int64_t ldo, int64_t n_in, int64_t t0, int64_t n_out, int64_t batch,
                         const VwFilt &f, int l, int64_t d, int mode, const double *thr_dev, int thr_per_row, int thr_soft,
                         int64_t thr_lstride);

// ---- exact order statistics (vw_select.cu) ---------------------------------------------------
// median(|w1|) per row -> universal thresholds written to thr_dev[batch] (device).
int vw_launch_universal_threshold(vw_ctx *ctx, const double *w1, int64_t batch, int64_t n, int64_t ld,
                                  double *thr_dev);
// same selection, raw median(|c|) per row
int vw_launch_median_abs(vw_ctx *ctx, const double *c, int64_t batch, int64_t n, int64_t ld, double *med_dev);
// the span median's cross-rank reduction on the device (vw_swt_denoise_sharded): out = own + the other ranks' tables of
// gather[ranks][entries] (slot `self` is not read), and a fixed threshold stored without a host copy
int vw_launch_span_hist_sum(vw_ctx *ctx, const uint64_t *gather, const uint64_t *own, int ranks, int self, int entries,
                            uint64_t *out);
int vw_launch_span_fixed(vw_ctx *ctx, double *thr_dev, double value);
size_t vw_sure_workspace(int64_t batch, int64_t n);
int vw_launch_sure(vw_ctx *ctx, const double *c, int64_t batch, int64_t n, int64_t ld, const double *sigma_dev, void *ws,
                   double *thr_dev, double *risk_dev);
int vw_launch_mean_variance(vw_ctx *ctx, const double *c, int64_t batch, int64_t n, int64_t ld, double *mean_dev,
                            double *var_dev);
// WaveletDenoiser's threshold selectors (vw_select.cu: k_denoise_select) for `levels` x `batch` (level, row) pairs, in the
// reference's arithmetic.  The scalars that depend on n and j alone come from the host, computed as denoising.py does.
struct VwDenoiseSel {
    const double *med;       // [batch] median(|W_1|) per row
    const double *var;       // BAYES: [levels][batch] population variance of W_j per row
    const double *sure;      // SURE: [levels][batch] arg-min of the risk scan
    double *sig;             // non-null: write the per-(level, row) noise level s here instead of thresholds
    double *thr;             // [levels][batch] thresholds
    int64_t batch, n;
    int levels, method, multilevel;
    double root;             // sqrt(2 ln n)
    double log_n;            // ln n
    double minimax_c;        // 0.4745 + 0.1148 ln n
    double fixed;            // FIXED
    double level_scale[VW_MAX_LEVELS];   // sqrt(2^j), index j - 1
};
int vw_launch_denoise_select(vw_ctx *ctx, const VwDenoiseSel &a);
// the selectors' scalars that depend on n and j alone, as denoising.py computes them (math.log, math.sqrt: the same libm)
inline void vw_denoise_scalars(int64_t n, int levels, VwDenoiseSel &a) {
    a.n = n;
    a.log_n = log((double)n);
    a.root = sqrt(2.0 * log((double)n));
    a.minimax_c = 0.4745 + 0.1148 * a.log_n;
    for (int j = 1; j <= VW_MAX_LEVELS; j++) a.level_scale[j - 1] = j <= levels ? sqrt((double)((int64_t)1 << j)) : 0.0;
}
