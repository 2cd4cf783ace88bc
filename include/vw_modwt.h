/*
 * vw_modwt.h -- C ABI of the B200-native MODWT / SWT engine (libvwmodwt.so).
 *
 * This is the drop-in boundary for VectorWave's MODWT/SWT hot path.  The reference
 * (MorphIQ-Labs/VectorWave) is pure Java with no FFI; the entry points below are what a
 * Panama FFM (java.lang.foreign) binding of that path calls -- INTEGRATION.md shows the
 * downcall stubs.  Each function cites the reference interface it replaces
 * (CORE = vectorwave-core/src/main/java/com/morphiqlabs/wavelet,
 *  EXT  = vectorwave-extensions/src/main/java/com/morphiqlabs/wavelet).
 *
 * Conventions
 *  - Plain pointers and sizes only; no exceptions cross the ABI.  Every call returns a
 *    vw_status; vw_last_error(ctx) gives the message for the last failure on that ctx.
 *  - All data are IEEE fp64.  Signals are row-major [batch][n] with a row stride `ld`
 *    (in elements).  Multi-level details are [levels][batch][n]: level j (1-based,
 *    1 = finest, CORE/modwt/MultiLevelMODWTResult.java:32-99) starts at
 *    w + (j-1)*level_stride, signal b at + b*ld.
 *  - Filters cross the ABI ALREADY SCALED by 1/sqrt(2) (hs[k] = h[k]*(1.0/Math.sqrt(2.0)),
 *    one rounding, CORE/internal/ScalarOps.java:909-916, CORE/modwt/MODWTTransform.java:139-150)
 *    and NOT upsampled: the engine applies the a-trous spacing 2^(j-1) itself.  Wavelet
 *    tables, the level-cap policy and the SYMMETRIC alignment table stay on the host side
 *    so the reference's quirks stay the reference's (SURVEY.md 8b).
 *  - Data pointers are HOST pointers unless VW_FLAG_DEVICE_PTRS is set.  Host buffers are
 *    staged through ctx-owned device memory (pinned host memory from vw_alloc_pinned makes
 *    the copies asynchronous DMA).  There is no CPU compute path: without a CUDA device
 *    vw_init fails with VW_ECUDA and nothing else can be called.
 *  - A ctx is bound to one device and one stream.  Every call holds the ctx's mutex, so a ctx may be shared between host
 *    threads (the reference's transform objects are): concurrent calls on one ctx serialise; use one ctx per thread to
 *    overlap them.  vw_set_stream + the call that follows are two calls -- callers that rebind streams from several
 *    threads keep their own lock around the pair (the Python mirror does).
 */
#ifndef VW_MODWT_H
#define VW_MODWT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define VW_API __attribute__((visibility("default")))
#else
#define VW_API
#endif

#define VW_ABI_VERSION 2
#define VW_MAX_FILTER_TAPS 128 /* coif17 = 102 taps is the reference's longest table */
#define VW_MAX_LEVELS 32

/* Status codes; names follow CORE/exception/ErrorCode.java:24-118. */
typedef enum vw_status {
    VW_OK = 0,
    VW_ENULL = 1,        /* VAL_NULL_ARGUMENT   -> NullPointerException */
    VW_ENONFINITE = 3,   /* VAL_NON_FINITE_VALUES -> InvalidSignalException (ValidationUtils.validateFiniteValues) */
    VW_ETOOLARGE = 5,    /* VAL_TOO_LARGE: (L-1)*2^(j-1)+1 > n, CORE/modwt/MultiLevelMODWTTransform.java:717-729 */
    VW_EEMPTY = 6,       /* VAL_EMPTY           -> InvalidSignalException */
    VW_ELENGTH = 7,      /* VAL_LENGTH_MISMATCH -> IllegalArgumentException (shape errors, EXT/extensions/modwt/BatchMODWT.java:201-212) */
    VW_EBOUNDARY = 103,  /* CFG_UNSUPPORTED_BOUNDARY_MODE, CORE/modwt/MODWTTransform.java:96-110 */
    VW_ELEVEL = 104,     /* CFG_INVALID_DECOMPOSITION_LEVEL, CORE/modwt/MultiLevelMODWTTransform.java:226-239 */
    VW_ESTATE = 301,     /* STATE_CLOSED / STATE_INVALID */
    VW_EINVAL = 400,     /* other IllegalArgumentException */
    VW_ENOMEM = 500,     /* device or pinned allocation failed */
    VW_ECUDA = 501,      /* CUDA runtime error; message in vw_last_error */
    VW_EUNSUPPORTED = 502
} vw_status;

/* CORE/api/BoundaryMode.java:26-50.  CONSTANT is rejected exactly as the reference does. */
typedef enum vw_boundary {
    VW_PERIODIC = 0,
    VW_ZERO_PADDING = 1,
    VW_SYMMETRIC = 2,
    VW_CONSTANT = 3 /* always VW_EBOUNDARY */
} vw_boundary;

/* Summation order of one synthesis stage (SURVEY.md Appendix B / D5). */
typedef enum vw_synth_order {
    VW_ORDER_SPLIT = 0, /* all H taps, then all G taps: CORE/modwt/MultiLevelMODWTTransform.java:578-589,602-642 */
    VW_ORDER_PAIR = 1   /* sum += h*V + g*W per tap: CORE/modwt/MODWTTransform.java:246-295, MultiLevel ZERO :591-601 */
} vw_synth_order;

enum {
    VW_FLAG_DEVICE_PTRS = 1u << 0,  /* data pointers are device pointers on ctx's device */
    VW_FLAG_CHECK_FINITE = 1u << 1, /* reject NaN/Inf inputs (VW_ENONFINITE) like the Java API does */
    VW_FLAG_BITEXACT = 1u << 2,     /* separate multiply/add roundings in Java's tap order (no FMA);
                                       runs the per-level kernels; results are bit-identical to the JVM */
    VW_FLAG_NO_FUSE = 1u << 3,      /* force the per-level kernels (diagnostics) */
    VW_FLAG_NO_SYNC = 1u << 4       /* device-pointer calls only: return after enqueueing on the ctx stream */
};

/* Per-level alignment of one synthesis stage, generalising every inverse the reference has:
 *   out[t] = sum_k hs[k]*V[ext(t + sigma_h*(k*d - tau_h))] (+) gs[k]*W[ext(t + sigma_g*(k*d - tau_g))]
 * d = 2^(level-1).  PERIODIC / ZERO_PADDING and single-level batch SYMMETRIC: {+1,0,+1,0}
 * (t+l; CORE/modwt/MODWTTransform.java:246-272,672-684); single-level SYMMETRIC: {-1,0,-1,0}
 * (t-l; :277-295); multi-level SYMMETRIC: from SymmetricAlignmentStrategy.decide + computeTauJ
 * (CORE/modwt/SymmetricAlignmentStrategy.java:43-117, MultiLevelMODWTTransform.java:602-642,795-806). */
typedef struct vw_align {
    int32_t sigma_h; /* +1 "plus" orientation, -1 "minus" */
    int32_t tau_h;
    int32_t sigma_g;
    int32_t tau_g;
} vw_align;

typedef struct vw_ctx vw_ctx;

/* ---- lifecycle ------------------------------------------------------------------ */
/* device < 0 selects the current CUDA device.  Fails with VW_ECUDA when no device exists. */
VW_API int vw_init(int device, vw_ctx **out);
VW_API int vw_destroy(vw_ctx *ctx);
VW_API const char *vw_last_error(const vw_ctx *ctx);
VW_API const char *vw_status_name(int status);
VW_API int vw_abi_version(void);
/* Run on an existing cudaStream_t (e.g. the caller's framework stream).  The handle is used as is, so
 * NULL is CUDA's legacy default stream.  vw_reset_stream returns to the ctx-owned non-blocking stream. */
VW_API int vw_set_stream(vw_ctx *ctx, void *cuda_stream);
VW_API int vw_reset_stream(vw_ctx *ctx);
VW_API int vw_synchronize(vw_ctx *ctx);
VW_API int vw_device_index(const vw_ctx *ctx);
/* Tuning knobs: "tile" (samples per CTA tile), "fuse" (max levels per launch), "threads". 0 = auto. */
VW_API int vw_set_option(vw_ctx *ctx, const char *name, int64_t value);
/* Writes the level schedule the engine would use (which levels share one fused launch, tile sizes, modelled
 * cycles/sample) as text into out[0..cap).  Pure host logic: needs no device (assumes 227 KB shared memory per CTA).
 * forward != 0: analysis; else synthesis.  Returns the number of launch groups, or a negative vw_status. */
VW_API int vw_describe_plan(int forward, int32_t l, int32_t levels, int64_t n, int64_t tile, int32_t fuse, char *out,
                            size_t cap);
/* The same schedule as numbers: group g covers levels first[g] .. first[g]+nlev[g]-1.  Returns the group count
 * (<= cap) or a negative vw_status.  Used by the span-sharded host code to align halo exchanges with launches. */
VW_API int vw_plan_query(int forward, int32_t l, int32_t levels, int64_t n, int32_t *first, int32_t *nlev, int32_t cap);
/* Paraunitary lattice of the quadrature-mirror pair (hs, gs) as the column kernels of long filters use it (csrc/vw_lattice.cu):
 * writes t_1 .. t_{l/2-1} then the 2 x 2 base matrix row-major into coef[0..cap) and the largest deviation of the lattice's
 * taps from the given ones into *tap_err (either may be NULL).  Returns the number of coefficients (l/2 + 3) when the
 * lattice reproduces the taps to rounding and the engine will use it, 0 when the pair keeps the direct form, or a
 * negative vw_status.  Pure host logic: needs no device. */
VW_API int vw_lattice_query(const double *hs, const double *gs, int32_t l, double *coef, int32_t cap, double *tap_err);
/* Number of kernels this ctx has launched since creation (bench.py's gpu_launches). */
VW_API int64_t vw_launch_count(const vw_ctx *ctx);

/* ---- memory (Java: MemorySegment.reinterpret over these) ---------------------------- */
VW_API void *vw_alloc_pinned(size_t bytes);
VW_API void vw_free_pinned(void *p);
VW_API int vw_device_alloc(vw_ctx *ctx, size_t bytes, void **out);
VW_API int vw_device_free(vw_ctx *ctx, void *p);
VW_API int vw_copy_h2d(vw_ctx *ctx, void *dst_device, const void *src_host, size_t bytes);
VW_API int vw_copy_d2h(vw_ctx *ctx, void *dst_host, const void *src_device, size_t bytes);

/* ---- level admissibility ---------------------------------------------------------- */
/* CORE/modwt/MultiLevelMODWTTransform.java:455-501 calculateMaxLevels: 0 if n <= l, else the
 * largest j with (l-1)*2^(j-1)+1 <= n, found by `while (j < cap)` then `return j-1` -- so
 * cap = 10 (MAX_DECOMPOSITION_LEVELS) yields at most 9.  cap <= 0: no cap. */
VW_API int vw_max_levels(int64_t n, int32_t l, int32_t cap);

/* ---- primitives ------------------------------------------------------------------- */
/* WaveletOperations.{circular,zeroPadding,symmetric}ConvolveMODWT (CORE/WaveletOperations.java:29,48,59;
 * kernels CORE/internal/ScalarOps.java:700-723,790-808,818-835):
 *   out[t] = sum_{l<lf} x[ext(t-l)] * filter[l]   with an arbitrary dense (pre-scaled) filter. */
VW_API int vw_conv_modwt(vw_ctx *ctx, const double *x, int64_t n, const double *filter, int64_t lf, int32_t mode,
                  double *out, uint32_t flags);

/* ---- analysis --------------------------------------------------------------------- */
/* MODWTTransform.forward / forwardBatch (levels = 1; CORE/modwt/MODWTTransform.java:131,486),
 * MultiLevelMODWTTransform.decompose (CORE/modwt/MultiLevelMODWTTransform.java:209-255),
 * VectorWaveSwtAdapter.forward (CORE/swt/VectorWaveSwtAdapter.java:198-204),
 * BatchMODWT.singleLevelAoS / multiLevelAoS (EXT/extensions/modwt/BatchMODWT.java:62,90):
 *   V_0 = x;  W_j[t] = sum_k gs[k]*V_{j-1}[ext(t - k*2^(j-1))];  V_j likewise with hs.
 * Requires (l-1)*2^(levels-1)+1 <= n when levels > 1 (VW_ETOOLARGE); levels == 1 accepts any
 * n >= 1 (true multi-wrap, CORE/internal/ScalarOps.java:711-717).  The level CAP is host policy.
 * w: [levels][batch][n] with strides (level_stride_w, ldw); vj: [batch][n] stride ldv. */
VW_API int vw_modwt_forward(vw_ctx *ctx, const double *x, int64_t batch, int64_t n, int64_t ldx, const double *hs,
                     const double *gs, int32_t l, int32_t levels, int32_t mode, double *w, int64_t ldw,
                     int64_t level_stride_w, double *vj, int64_t ldv, uint32_t flags);

/* ---- synthesis -------------------------------------------------------------------- */
/* MODWTTransform.inverse / inverseBatch (CORE/modwt/MODWTTransform.java:203,531),
 * MultiLevelMODWTTransform.reconstruct / reconstructFromLevel / reconstructLevels (:339,361,398),
 * VectorWaveSwtAdapter.inverse (CORE/swt/VectorWaveSwtAdapter.java:435-474),
 * BatchMODWT.inverseSingleLevelAoS / inverseMultiLevelAoS (EXT/extensions/modwt/BatchMODWT.java:122,151).
 * align: levels entries (index j-1) or NULL for {+1,0,+1,0} at every level.
 * detail_mask bit (j-1) clear => W_j is treated as zeros (partial reconstruction);
 * use_approx == 0 => V_J is treated as zeros. */
VW_API int vw_modwt_inverse(vw_ctx *ctx, const double *w, int64_t ldw, int64_t level_stride_w, const double *vj,
                     int64_t ldv, int64_t batch, int64_t n, const double *hs, const double *gs, int32_t l,
                     int32_t levels, int32_t mode, const vw_align *align, int32_t order, uint64_t detail_mask,
                     int32_t use_approx, double *xout, int64_t ldx, uint32_t flags);

/* ---- single level over rows of different lengths -------------------------------------------------------------- */
/* MODWTTransform.forwardBatch over rows of different lengths (CORE/modwt/MODWTTransform.java:486-515), i.e. one
 * MODWTTransform.forward per row (:131-189): row b is x[offsets[b] .. offsets[b+1]), and its V and W are written at
 * the same packed positions of v and w.  Same per-row rules as vw_modwt_forward with levels = 1 (any n >= 1, true
 * multi-wrap when n < l).  offsets: a HOST array of batch + 1 values whatever the flags say, offsets[0] == 0, never
 * decreasing (else VW_ELENGTH).  Rows are validated in index order like the reference's per-row loop: the lowest row
 * that is empty (VW_EEMPTY) or, with VW_FLAG_CHECK_FINITE, holds a NaN / Inf (VW_ENONFINITE) fails the call, its index
 * in vw_last_error.  One kernel launch however many rows; not capturable into a graph (VW_ESTATE). */
VW_API int vw_modwt_forward_varlen(vw_ctx *ctx, const double *x, const int64_t *offsets, int64_t batch,
                                   const double *hs, const double *gs, int32_t l, int32_t mode,
                                   double *w, double *v, uint32_t flags);
/* MODWTTransform.inverse per row (:203-299): pair-added products; PERIODIC / ZERO_PADDING use t+l, SYMMETRIC uses
 * t-l (the rule inverseBatch applies when lengths differ).  Same packing as above; xout packed like w and v. */
VW_API int vw_modwt_inverse_varlen(vw_ctx *ctx, const double *w, const double *v, const int64_t *offsets,
                                   int64_t batch, const double *hs, const double *gs, int32_t l, int32_t mode,
                                   double *xout, uint32_t flags);

/* ---- thresholding / SWT denoise ------------------------------------------------------- */
/* MutableMultiLevelMODWTResult.applyThreshold (CORE/modwt/MutableMultiLevelMODWTResult.java:83-118):
 * in place over `batch` rows of n; soft: |c|>t ? sign(c)*(|c|-t) : 0; hard: |c|<=t ? 0 : c.
 * thresholds is a HOST array (1 value, or `batch` values when per_row != 0) regardless of flags. */
VW_API int vw_threshold(vw_ctx *ctx, double *coeffs, int64_t batch, int64_t n, int64_t ld, const double *thresholds,
                 int32_t per_row, int32_t soft, uint32_t flags);

/* VectorWaveSwtAdapter.applyUniversalThreshold's threshold (CORE/swt/VectorWaveSwtAdapter.java:505-520,627-645):
 * per row: median(|w1|)/0.6745*sqrt(2 ln n), median of an even count = mean of the two middle
 * order statistics (exact selection, no sort).  thresholds_out: `batch` doubles on the HOST. */
VW_API int vw_universal_threshold(vw_ctx *ctx, const double *w1, int64_t batch, int64_t n, int64_t ld,
                           double *thresholds_out, uint32_t flags);

/* VectorWaveSwtAdapter.denoise (CORE/swt/VectorWaveSwtAdapter.java:532-562): decompose, threshold every
 * detail level (threshold < 0 => universal, per signal), reconstruct.  thresholds_out may be NULL. */
VW_API int vw_swt_denoise(vw_ctx *ctx, const double *x, int64_t batch, int64_t n, int64_t ldx, const double *hs,
                   const double *gs, int32_t l, int32_t levels, int32_t mode, const vw_align *align, int32_t order,
                   double threshold, int32_t soft, double *out, int64_t ldo, double *thresholds_out, uint32_t flags);

/* WaveletDenoiser's threshold selection methods (CORE/denoising/WaveletDenoiser.java:602-632, same order as ThresholdMethod). */
typedef enum vw_threshold_method {
    VW_THR_UNIVERSAL = 0,
    VW_THR_SURE = 1,
    VW_THR_MINIMAX = 2,
    VW_THR_BAYES = 3,
    VW_THR_FIXED = 4
} vw_threshold_method;

/* WaveletDenoiser over a [batch][n] batch in one call, every row on its own noise level.
 * multilevel == 0: WaveletDenoiser.denoise / denoiseFixed (:111-145, :354-366): levels must be 1, any n >= 1 (multi-wrap
 *   as vw_modwt_forward at one level), sigma = median(|W_1|) / 0.6745 unscaled; FIXED uses fixed_threshold.
 * multilevel == 1: denoiseMultiLevel (:155-171, :183-231): sigma from each row's W_1, level j uses sigma / sqrt(2^j);
 *   levels > 31 (MAX_SAFE_LEVEL_FOR_SCALING) is VW_ETOOLARGE, FIXED is VW_EUNSUPPORTED.
 * UNIVERSAL s*sqrt(2 ln n); MINIMAX 0 (n <= 32), s*0.3936 + 0.1829*s*ln n (n <= 64), else s*(0.4745 + 0.1148 ln n);
 * BAYES s^2 / sqrt(max(0, var(W_j) - s^2) + 1e-10); SURE the risk arg-min of vw_sure_threshold (levels * batch * n^2 <= 2^44,
 * else VW_EUNSUPPORTED) capped at s*sqrt(2 ln n) -- each evaluated in the reference's operation order.  align / order are
 * those of the matching reconstruct (MODWTTransform.inverse or MultiLevelMODWTTransform.reconstruct), as in vw_swt_denoise.
 * The whole chain runs on the device with one synchronise at the end; the thresholds are applied as the synthesis loads W.
 * thresholds_out: NULL or levels * batch HOST doubles, [level][row].  Not capturable into a graph. */
VW_API int vw_wavelet_denoise(vw_ctx *ctx, const double *x, int64_t batch, int64_t n, int64_t ldx, const double *hs,
                              const double *gs, int32_t l, int32_t levels, int32_t mode, const vw_align *align, int32_t order,
                              int32_t multilevel, int32_t method, double fixed_threshold, int32_t soft, double *out, int64_t ldo,
                              double *thresholds_out, uint32_t flags);

/* WaveletDenoiser.estimateNoiseSigma's order statistic (CORE/denoising/WaveletDenoiser.java:376-387,587-597): the exact
 * median of |c| per row (even count: mean of the two middle values).  sigma = median / 0.6745 stays on the host.
 * out: `batch` doubles on the HOST. */
VW_API int vw_median_abs(vw_ctx *ctx, const double *c, int64_t batch, int64_t n, int64_t ld, double *out, uint32_t flags);

/* Mean and population variance about the mean per row -- the two loops of WaveletDenoiser.calculateBayesThreshold
 * (CORE/denoising/WaveletDenoiser.java:521-552).  mean_out, var_out: `batch` doubles each on the HOST. */
VW_API int vw_mean_variance(vw_ctx *ctx, const double *c, int64_t batch, int64_t n, int64_t ld, double *mean_out,
                     double *var_out, uint32_t flags);

/* BatchSIMDMODWT.batchMODWTSoA / batchMultiLevelMODWTSoA (EXT/extensions/modwt/BatchSIMDMODWT.java:64-81,343-424) on
 * the caller's SoA layout: soa_x[t*batch + b], PERIODIC; soa_w = `levels` pointers (a HOST array, like the reference's
 * double[][] soaDetailPerLevel) to n*batch doubles each, soa_v = n*batch doubles.  Runs on the flat array as one periodic signal of n*batch samples at dilation 2^(j-1)*batch --
 * no AoS<->SoA transposes anywhere.  hs/gs: the scaled taps (the reference's Haar special case passes literal +-0.5). */
VW_API int vw_modwt_forward_soa(vw_ctx *ctx, const double *soa_x, int64_t batch, int64_t n, const double *hs,
                         const double *gs, int32_t l, int32_t levels, double *const *soa_w, double *soa_v,
                         uint32_t flags);

/* WaveletDenoiser.calculateSUREThreshold (CORE/denoising/WaveletDenoiser.java:441-492) per row: the candidate t = |c_i|
 * of minimal Stein risk (first minimum in ascending t), every risk accumulated in the reference's coefficient order and
 * roundings (bit-identical to the JVM's O(n^2) double loop, which is what it costs here too: batch * n^2 <= 2^44), then
 * capped at sigma * sqrt(2 ln n).  sigma: `batch` doubles on the HOST (noise sigma per row); thr_out: `batch` doubles on
 * the HOST; risk_out (may be NULL): the minimal risk per row. */
VW_API int vw_sure_threshold(vw_ctx *ctx, const double *c, int64_t batch, int64_t n, int64_t ld, const double *sigma,
                      double *thr_out, double *risk_out, uint32_t flags);

/* sum of squares per row: MultiLevelMODWTResult.getDetailEnergyAtLevel / getApproximationEnergy
 * (CORE/modwt/MultiLevelMODWTResultImpl.java:91-139).  out: `batch` doubles on the HOST. */
VW_API int vw_energy(vw_ctx *ctx, const double *c, int64_t batch, int64_t n, int64_t ld, double *out, uint32_t flags);

/* ---- span-sharded long signals (one rank's part; halos already exchanged) ------------------ */
/* A rank owns samples [s, s+n_local) of one long signal.  For a group of `nlevels` levels starting
 * at `first_level`, analysis needs the halo = (l-1)*2^(first_level-1)*(2^nlevels-1) samples of
 * V_{first_level-1} that precede the span (from the left neighbour; the last rank for PERIODIC wrap).
 * vin points at the start of [halo | span] (halo+n_local contiguous samples, device memory).
 * Writes W_j[span] for the group's levels and V_{first_level+nlevels-1}[span].  No boundary rule is
 * applied: the halo IS the boundary (the host fills it per BoundaryMode).  Reference precedent for the
 * halo semantics: EXT/extensions/modwt/BatchSIMDMODWT.java:447-507 (left history of L_j-1 samples). */
VW_API int vw_modwt_forward_span(vw_ctx *ctx, const double *vin, int64_t halo, int64_t n_local, const double *hs,
                          const double *gs, int32_t l, int32_t first_level, int32_t nlevels, double *w,
                          int64_t level_stride_w, double *vout, uint32_t flags);
/* Synthesis of the same group: vin and each W_j are [span | halo] with the RIGHT halo
 * (first samples of the right neighbour), halo >= (l-1)*2^(first_level-1)*(2^nlevels-1); w rows are
 * level_stride_w apart, each halo+n_local long.  Writes V_{first_level-1}[span].  PERIODIC/ZERO index rule (t+k*d). */
VW_API int vw_modwt_inverse_span(vw_ctx *ctx, const double *vin, const double *w, int64_t level_stride_w, int64_t halo,
                          int64_t n_local, const double *hs, const double *gs, int32_t l, int32_t first_level,
                          int32_t nlevels, int32_t order, double *vout, uint32_t flags);
/* halo length the two calls above require */
VW_API int64_t vw_span_halo(int32_t l, int32_t first_level, int32_t nlevels);

/* ---- blockwise (streaming) batch analysis with carried left history ---------------------------------- */
/* One level of BatchStreamingMODWT.processSingleLevel / processMultiLevel / flush*
 * (EXT/extensions/modwt/BatchStreamingMODWT.java:55-163,183-276) on the history kernel's semantics
 * (EXT/extensions/modwt/BatchSIMDMODWT.java:447-507): every row of vin is [history | block], where history holds the
 * `hist` >= (l-1)*2^(level-1) samples of THIS level's input that precede the block (oldest first; the host fills it
 * with zeros, the symmetric reflection of the first block, or the tail of the previous block) and block has n samples:
 *   V[b][t] = sum_k hs[k] * ext[b][hist + t - k*2^(level-1)],  W likewise with gs,   t in [0, n).
 * vin: [batch] rows of hist + n samples, row stride ldin; w, v: [batch][n] with strides ldw, ldv.  v may point into
 * the next level's [history | block] buffer (the cascade then needs no copy).  Device pointers only. */
VW_API int vw_modwt_stream_level(vw_ctx *ctx, const double *vin, int64_t batch, int64_t ldin, int64_t hist, int64_t n,
                          const double *hs, const double *gs, int32_t l, int32_t level, double *w, int64_t ldw,
                          double *v, int64_t ldv, uint32_t flags);

/* ---- stream state on the device: the whole block cascade of BatchStreamingMODWT per call ------------------------- */
/* BatchStreamingMODWT.processSingleLevel / processMultiLevel / flushSingleLevel / flushMultiLevel
 * (EXT/extensions/modwt/BatchStreamingMODWT.java:55-276) with every level's left history kept in HBM by the handle:
 * level j keeps the last (l-1)*2^(j-1) samples of its own input.
 *  - create: mode ZERO_PADDING or SYMMETRIC (PERIODIC streaming is stateless: use vw_modwt_forward; anything else is
 *    VW_EBOUNDARY), levels 1..30 (else VW_ELEVEL).  The handle copies the taps and belongs to ctx's device.
 *  - process: x [batch][n] (row stride ldx) -> w [levels][batch][n] (strides level_stride_w, ldw), v = V_J [batch][n].
 *    Any n >= 1 (the history carries the left context).  The first block after create / reset, and a block whose batch
 *    differs from the previous one (:306-320), start the stream: level j's history is zeros, or for SYMMETRIC the
 *    half-sample mirror of level j's own first input (multi-wrap when n is shorter than the history, :326-334).  After
 *    every level the history becomes the last (l-1)*2^(j-1) samples of [history | input] (:336-350).
 *  - flush: the cascade over a tail of tail_length samples built from the level-1 history (zeros, or that history
 *    reversed for SYMMETRIC, :358-372); the histories are not advanced (:205-222,252-274).  VW_ESTATE before any block,
 *    VW_ELENGTH for tail_length > l - 1, VW_EEMPTY for tail_length < 1.  Outputs [levels][batch][tail_length].
 *  - reset: back to "no block seen" (no device work).
 * Pointers are host pointers (staged) unless VW_FLAG_DEVICE_PTRS; VW_FLAG_CHECK_FINITE checks x, VW_FLAG_BITEXACT gives
 * the reference's separate roundings, VW_FLAG_NO_FUSE forces the per-level kernels.  A failed call leaves the state as
 * it was.  Not capturable into a graph (VW_ESTATE): every call advances the state on the host side. */
typedef struct vw_stream_state vw_stream_state;
VW_API int vw_stream_create(vw_ctx *ctx, const double *hs, const double *gs, int32_t l, int32_t levels, int32_t mode,
                            vw_stream_state **out);
VW_API int vw_stream_destroy(vw_ctx *ctx, vw_stream_state *st);
VW_API int vw_stream_process(vw_ctx *ctx, vw_stream_state *st, const double *x, int64_t batch, int64_t n, int64_t ldx,
                             double *w, int64_t ldw, int64_t level_stride_w, double *v, int64_t ldv, uint32_t flags);
VW_API int vw_stream_flush(vw_ctx *ctx, vw_stream_state *st, int64_t tail_length, double *w, int64_t ldw,
                           int64_t level_stride_w, double *v, int64_t ldv, uint32_t flags);
VW_API int vw_stream_reset(vw_stream_state *st);

/* ---- span-sharded long signals, whole cascade per rank (up-front halo schedule) ---------------------------- */
/* The halo a rank needs is tiny next to its span ((l-1)*(2^levels-1) samples), so it is exchanged ONCE per direction:
 * before the analysis every rank receives the last `lead` samples of its left neighbour's x; before the synthesis the
 * first samples of its right neighbour's V_J and W_j rows (ring wrap for PERIODIC, zeros at the open ends for
 * ZERO_PADDING).  Every level then runs on a region that shrinks by its own halo -- no per-level synchronisation.
 * vw_span_plan_query gives the layout both directions share (pure host logic, no device needed):
 *   x work row   [lead | n_local]                 (the halo lands in front of the span)
 *   W rows       [lead_w | n_local | pad]          `levels` rows, row_stride >= lead_w + n_local + pad apart
 *   V_J row      [n_local | pad]
 * Halos are rounded up to 32 samples so every kernel sees sector-aligned rows.  Reference precedent for the halo
 * semantics: EXT/extensions/modwt/BatchSIMDMODWT.java:447-507; NOT StructuredParallelTransform.forwardChunked
 * (EXT/extensions/parallel/StructuredParallelTransform.java:313-341), which has no halo. */
#define VW_SPAN_MAX_GROUPS 16
typedef struct vw_span_plan {
    int32_t l, levels, world, reserved;
    int64_t n_local;
    int32_t ngroups_f, ngroups_i;                       /* launch groups of the analysis / synthesis cascade */
    int32_t first_f[VW_SPAN_MAX_GROUPS], nlev_f[VW_SPAN_MAX_GROUPS];
    int32_t first_i[VW_SPAN_MAX_GROUPS], nlev_i[VW_SPAN_MAX_GROUPS];
    int64_t halo_f[VW_SPAN_MAX_GROUPS], halo_i[VW_SPAN_MAX_GROUPS];   /* per group, rounded up to 32 samples */
    int64_t lead;          /* left halo of x: sum of halo_f */
    int64_t lead_w;        /* spare samples on the left of every W row: sum of halo_f[1..] */
    int64_t pad;           /* spare samples on the right of V_J and of every W row: sum of halo_i */
    int64_t inverse_msg;   /* doubles in one rank's synthesis halo message (vw_span_pack_inverse) */
} vw_span_plan;
/* VW_ELENGTH when the total halo exceeds n_local (use fewer ranks / levels, or the per-group calls above). */
VW_API int vw_span_plan_query(int32_t l, int32_t levels, int64_t n_local, int32_t world, vw_span_plan *out);
/* Analysis of one rank's span, all levels: xext = [lead | n_local] with the left neighbour's halo already in place.
 * Writes W_j[span] at w + (j-1)*row_stride + lead_w (the lead_w samples before it are engine work space) and V_J[span]
 * at v.  Device pointers only. */
VW_API int vw_modwt_forward_span_all(vw_ctx *ctx, const double *xext, const vw_span_plan *plan, const double *hs,
                              const double *gs, double *w, int64_t row_stride, double *v, uint32_t flags);
/* The synthesis halo message of this rank: the first samples of V_J and of every W_j row its LEFT neighbour needs,
 * gathered into `msg` (plan->inverse_msg doubles, device); unpack scatters a received message into the pad areas. */
VW_API int vw_span_pack_inverse(vw_ctx *ctx, const vw_span_plan *plan, const double *w, int64_t row_stride, const double *v,
                         double *msg, uint32_t flags);
VW_API int vw_span_unpack_inverse(vw_ctx *ctx, const vw_span_plan *plan, const double *msg, double *w, int64_t row_stride,
                           double *v, uint32_t flags);
/* Synthesis of one rank's span, all levels, halos already in the pad areas.  xout: n_local doubles. */
VW_API int vw_modwt_inverse_span_all(vw_ctx *ctx, const vw_span_plan *plan, const double *w, int64_t row_stride,
                              const double *v, const double *hs, const double *gs, int32_t order, double *xout,
                              uint32_t flags);
/* The same synthesis of the soft (soft != 0) or hard thresholded W: thr_dev is ONE device double, applied to every W
 * sample the kernels load -- the halo included, which holds the neighbour's raw coefficients that the neighbour thresholds
 * on load too, so the ranks together give the whole-signal synthesis of the thresholded coefficients.  V_J is not
 * thresholded; W and V are read only (the per-level kernels of VW_FLAG_BITEXACT / VW_FLAG_NO_FUSE threshold a scratch copy). */
VW_API int vw_modwt_inverse_span_all_thr(vw_ctx *ctx, const vw_span_plan *plan, const double *w, int64_t row_stride,
                                         const double *v, const double *hs, const double *gs, int32_t order,
                                         const double *thr_dev, int32_t soft, double *xout, uint32_t flags);

/* ---- exact median of |c| over a signal split into spans (the universal threshold of a span-sharded signal) ---------- */
/* The seven digit rounds of vw_universal_threshold's selection with the histogram reduction left to the caller, so ranks
 * in separate processes (NCCL, one GPU each) can drive it.  Per rank: allocate vw_span_median_state_bytes(n_local) bytes of
 * device memory, vw_span_median_init once, then for round = 0 .. VW_SPAN_MEDIAN_ROUNDS-1:
 *   vw_span_median_hist(own span -> hist, vw_span_median_bins(round) uint64 entries);
 *   the caller sums hist over the ranks (e.g. ncclAllReduce with ncclUint64 / ncclSum) into hist_sum;
 *   vw_span_median_pick(hist_sum)  -- every rank picks from the identical sum, so every rank's state stays identical;
 * finally vw_span_median_value writes median(|c|) / 0.6745 * factor, or the raw median for factor < 0 (even n_total: the mean
 * of the two middle order statistics), to one device double.  The universal threshold uses factor = sqrt(2 ln n_total).
 * Candidate buffers stay rank-local: a rank whose round-2 bucket overflows them (a constant span) histograms its full span
 * in the later rounds, the sum is still exact.  All pointers are device pointers on ctx's device; every call only
 * enqueues on ctx's stream and nothing synchronises. */
#define VW_SPAN_MEDIAN_ROUNDS 7
VW_API int32_t vw_span_median_bins(int32_t round);   /* 2 * 4096 (rounds 0, 1), 2 * 256 (rounds 2..6), 0 outside */
VW_API size_t vw_span_median_state_bytes(int64_t n_local);
VW_API int vw_span_median_init(vw_ctx *ctx, void *state, int64_t n_total);
VW_API int vw_span_median_hist(vw_ctx *ctx, void *state, const double *c, int64_t n_local, int32_t round, uint64_t *hist);
VW_API int vw_span_median_pick(vw_ctx *ctx, void *state, int32_t round, const uint64_t *hist_sum);
VW_API int vw_span_median_value(vw_ctx *ctx, const void *state, double factor, double *out_dev);

/* ---- several GPUs driven by ONE host thread (the JVM case) ------------------------------------------------------ */
/* vw_init_multi opens one ctx per listed device and enables peer access between ring neighbours.  The sharded calls
 * take one DEVICE pointer per device (allocated with vw_device_alloc on vw_multi_ctx(m, r)), enqueue the halo
 * exchange as peer copies over NVLink (cudaMemcpyPeerAsync; ring wrap for PERIODIC) and the per-device cascades on
 * each device's own stream, and return when every device has finished (or right after enqueueing with
 * VW_FLAG_NO_SYNC; vw_multi_synchronize then waits).  Batches need no such call: signals are independent, use one ctx
 * per device.  SURVEY.md 8(b)/(e). */
typedef struct vw_multi vw_multi;
VW_API int vw_init_multi(const int *devices, int32_t ndev, vw_multi **out);
VW_API int vw_destroy_multi(vw_multi *m);
VW_API int32_t vw_multi_size(const vw_multi *m);
VW_API vw_ctx *vw_multi_ctx(vw_multi *m, int32_t rank);
VW_API const char *vw_multi_last_error(const vw_multi *m);
VW_API int vw_multi_synchronize(vw_multi *m);
/* xext[r]: [lead | n_local] on device r with the span filled (the engine fills the lead); w[r]: `levels` rows of
 * row_stride; v[r]: [n_local | pad].  mode: VW_PERIODIC or VW_ZERO_PADDING.  exchange_ms (may be NULL): device time of
 * the slowest halo copy, measured with events (forces a synchronise). */
VW_API int vw_modwt_forward_sharded(vw_multi *m, const vw_span_plan *plan, double *const *xext, const double *hs,
                             const double *gs, int32_t mode, double *const *w, int64_t row_stride, double *const *v,
                             float *exchange_ms, uint32_t flags);
VW_API int vw_modwt_inverse_sharded(vw_multi *m, const vw_span_plan *plan, double *const *w, int64_t row_stride,
                             double *const *v, const double *hs, const double *gs, int32_t mode, int32_t order,
                             double *const *xout, float *exchange_ms, uint32_t flags);
/* VectorWaveSwtAdapter.denoise (CORE/swt/VectorWaveSwtAdapter.java:532-562) of ONE signal of world * n_local samples spread
 * over the devices, i.e. vw_swt_denoise with batch = 1 on the whole signal: vw_modwt_forward_sharded, then (threshold < 0)
 * the universal threshold median(|W_1|)/0.6745 * sqrt(2 ln N) with the exact median over all ranks (the vw_span_median_*
 * rounds, histograms summed on the devices: every device pulls the others' tables with cudaMemcpyPeerAsync, ordered by
 * events, no host round trip between rounds) or the fixed `threshold`, then the synthesis exchange and
 * vw_modwt_inverse_span_all_thr on every device.  The same threshold applies to every detail level; V_J is untouched.
 * Buffers as vw_modwt_forward_sharded / vw_modwt_inverse_sharded (w and v receive the raw coefficients).
 * VW_FLAG_CHECK_FINITE checks every span first: VW_ENONFINITE names the rank and nothing is written to xout.
 * threshold_out (may be NULL): the threshold on the HOST (for the universal threshold this waits for rank 0's stream).
 * One synchronise at the end, none with VW_FLAG_NO_SYNC (vw_multi_synchronize then waits). */
VW_API int vw_swt_denoise_sharded(vw_multi *m, const vw_span_plan *plan, double *const *xext, const double *hs,
                                  const double *gs, int32_t mode, int32_t order, double threshold, int32_t soft,
                                  double *const *w, int64_t row_stride, double *const *v, double *const *xout,
                                  double *threshold_out, uint32_t flags);

/* ---- device-resident results (MultiLevelMODWTResult kept on the GPU between calls) ------------------------------ */
/* CORE/modwt/MultiLevelMODWTResultImpl.java:51-139 and MutableMultiLevelMODWTResultImpl are opaque enough to be backed
 * by device memory: decompose once, threshold / measure / reconstruct without the coefficients ever crossing PCIe; a
 * level is copied to the host only when the caller asks for it (getDetailCoeffsAtLevel -> vw_result_get_level).
 * A decompose -> threshold -> reconstruct pipeline then moves 16 B/sample over PCIe instead of 16*(levels+2). */
typedef struct vw_result vw_result;
/* x: host (staged) or device pointer per flags.  *res == NULL: a new result is allocated; otherwise *res is reused when
 * its shape matches (no allocation on the steady state) and replaced when it does not. */
VW_API int vw_modwt_decompose_h(vw_ctx *ctx, const double *x, int64_t batch, int64_t n, int64_t ldx, const double *hs,
                         const double *gs, int32_t l, int32_t levels, int32_t mode, vw_result **res, uint32_t flags);
VW_API int vw_result_shape(const vw_result *res, int64_t *batch, int64_t *n, int32_t *levels);
/* level 1..levels: W_level; level 0: V_J.  dst: [batch][n] rows of stride ld; host unless VW_FLAG_DEVICE_PTRS. */
VW_API int vw_result_get_level(vw_ctx *ctx, const vw_result *res, int32_t level, double *dst, int64_t ld, uint32_t flags);
/* MutableMultiLevelMODWTResult.setDetailCoeffs / setApproximationCoeffs: overwrite one level from src. */
VW_API int vw_result_set_level(vw_ctx *ctx, vw_result *res, int32_t level, const double *src, int64_t ld, uint32_t flags);
/* zero-copy device view of one level (row stride n): for callers that keep working on the device */
VW_API double *vw_result_device_ptr(const vw_result *res, int32_t level);
/* MutableMultiLevelMODWTResult.applyThreshold on level `level` (1..levels), or on every detail level when level == 0;
 * thresholds: 1 or (per_row) batch HOST values. */
VW_API int vw_result_threshold(vw_ctx *ctx, vw_result *res, int32_t level, const double *thresholds, int32_t per_row,
                        int32_t soft);
/* VectorWaveSwtAdapter.applyUniversalThreshold: per-row universal threshold from W_1, applied to every detail level;
 * thresholds_out (may be NULL): batch HOST doubles. */
VW_API int vw_result_universal_threshold(vw_ctx *ctx, vw_result *res, int32_t soft, double *thresholds_out);
/* getDetailEnergyAtLevel (level >= 1) / getApproximationEnergy (level 0): batch HOST doubles. */
VW_API int vw_result_energy(vw_ctx *ctx, const vw_result *res, int32_t level, double *out);
/* MultiLevelMODWTTransform.reconstruct / reconstructFromLevel / reconstructLevels from the resident coefficients. */
VW_API int vw_modwt_reconstruct_h(vw_ctx *ctx, const vw_result *res, const double *hs, const double *gs, int32_t l,
                           int32_t mode, const vw_align *align, int32_t order, uint64_t detail_mask, int32_t use_approx,
                           double *xout, int64_t ldx, uint32_t flags);
VW_API int vw_result_free(vw_ctx *ctx, vw_result *res);

/* ---- replaying a fixed call sequence as one CUDA graph (small, latency-bound shapes) --------------------------- */
/* Between vw_graph_begin and vw_graph_end every engine call on this ctx is captured instead of executed (calls must
 * not need a device->host answer: no VW_FLAG_CHECK_FINITE, no threshold selectors; host buffers must be pinned and
 * stay valid; run the same calls once un-captured first so the scratch buffers exist).  vw_graph_launch replays the
 * whole sequence -- copies included -- with one launch.  Reference shape: config #1/#2's small transforms, which the
 * JVM runs in 117-358 us (docs/BENCHMARK-RESULTS.md:26). */
typedef struct vw_graph vw_graph;
VW_API int vw_graph_begin(vw_ctx *ctx);
VW_API int vw_graph_end(vw_ctx *ctx, vw_graph **out);
VW_API int vw_graph_launch(vw_ctx *ctx, vw_graph *g, uint32_t flags);
VW_API int vw_graph_destroy(vw_ctx *ctx, vw_graph *g);

/* ---- timing of the last call (SURVEY.md section 5) ----------------------------------------------------------------- */
/* With vw_set_option(ctx, "timing", 1) every public call brackets its device work with CUDA events; vw_last_timing
 * reports the last call: device milliseconds (first enqueue to last), host milliseconds inside the call, kernels
 * launched.  Also wraps each call in an NVTX range ("vw_modwt_forward", ...) visible to Nsight tools. */
typedef struct vw_timing { float device_ms; float host_ms; int32_t launches; int32_t reserved; } vw_timing;
VW_API int vw_last_timing(vw_ctx *ctx, vw_timing *out);
/* The FP64 roofline denominator measured on this device: sustained TFLOP/s of the DFMA stream the tile kernels are made
 * of (one uniform-register operand, 8 independent chains, 64 warps per SM, a few milliseconds).  MEASURED_PEAKS.json has
 * no FP64 figure; bench.py calls this once per run.  sm_mhz_out (may be NULL): the device's maximum SM clock. */
VW_API int vw_probe_fp64(vw_ctx *ctx, double *tflops_out, double *sm_mhz_out);

#ifdef __cplusplus
}
#endif
#endif /* VW_MODWT_H */
