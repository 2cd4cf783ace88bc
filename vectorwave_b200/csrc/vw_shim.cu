// vw_shim.cu -- the C ABI of include/vw_modwt.h: argument validation with the reference's error
// vocabulary, host<->device staging, and the level schedule (which levels fuse into which launch).
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include <chrono>

#include "vw_internal.cuh"

// ------------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------------
int vw_fail(vw_ctx *ctx, int status, const char *fmt, ...) {
    if (ctx) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        ctx->err = buf;
    }
    return status;
}

int vw_cuda_check(vw_ctx *ctx, cudaError_t e, const char *what) {
    if (e == cudaSuccess) return VW_OK;
    return vw_fail(ctx, e == cudaErrorMemoryAllocation ? VW_ENOMEM : VW_ECUDA, "CUDA error in %s: %s (%s)", what,
                   cudaGetErrorName(e), cudaGetErrorString(e));
}

int vw_scratch(vw_ctx *ctx, int slot, size_t bytes, void **out) {
    if (bytes == 0) bytes = 16;
    slot += ctx->scratch_set * vw_ctx::kScratch;
    if (ctx->capturing && ctx->scratch_bytes[slot] < bytes)
        return vw_fail(ctx, VW_ESTATE, "scratch buffer %d would have to grow during graph capture: run the same calls once "
                                       "before vw_graph_begin", slot);
    if (ctx->scratch_pending && ctx->scratch_stream != ctx->stream && !ctx->capturing) {
        // the previous un-synchronised call may still be using the scratch on its own stream: order this stream after it
        int rc = vw_cuda_check(ctx, cudaStreamWaitEvent(ctx->stream, ctx->scratch_event, 0), "scratch hand-over between streams");
        if (rc) return rc;
        ctx->scratch_stream = ctx->stream;   // this stream now runs after it; later calls on it need no second wait
    }
    if (ctx->scratch_bytes[slot] < bytes) {
        if (ctx->scratch[slot]) {
            cudaStreamSynchronize(ctx->stream);
            cudaFree(ctx->scratch[slot]);
            ctx->scratch[slot] = nullptr;
            ctx->scratch_bytes[slot] = 0;
        }
        size_t want = (bytes + ((size_t)1 << 20) - 1) & ~(((size_t)1 << 20) - 1);
        int rc = vw_cuda_check(ctx, cudaMalloc(&ctx->scratch[slot], want), "scratch cudaMalloc");
        if (rc) return rc;
        ctx->scratch_bytes[slot] = want;
    }
    *out = ctx->scratch[slot];
    return VW_OK;
}

namespace vwshim {

// DeviceGuard (vw_internal.cuh) is held for the duration of a public call: the ctx's mutex (scratch buffers, stream
// binding, error string and launch counter are per ctx, so concurrent callers of one ctx serialise -- the reference's
// transforms are shared across threads), the ctx's device as the current one, an NVTX range named after the entry
// point, and -- with vw_set_option("timing", 1) -- a CUDA event pair around the call's device work.
void DeviceGuard::enter(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
}
DeviceGuard::DeviceGuard(int dev) { enter(dev); }
DeviceGuard::DeviceGuard(vw_ctx *c, const char *name) : lk(c->mu), ctx(c) {
    enter(c->device);
    if (++c->call_depth > 1) return;          // nested public calls (the *_all and handle entry points) report as one
    if (name) { nvtxRangePushA(name); ranged = true; }
    if (c->opt_timing && !c->capturing) {
        if (!c->time_ev[0]) {
            cudaEventCreate(&c->time_ev[0]);
            cudaEventCreate(&c->time_ev[1]);
        }
        cudaEventRecord(c->time_ev[0], c->stream);
        c->time_launch0 = c->launches;
        c->time_host0 = std::chrono::steady_clock::now();
        timed = true;
    }
}
DeviceGuard::~DeviceGuard() {
    if (ctx && --ctx->call_depth == 0) {
        if (timed) {
            cudaEventRecord(ctx->time_ev[1], ctx->stream);
            ctx->time_host_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - ctx->time_host0).count();
            ctx->time_launches = (int32_t)(ctx->launches - ctx->time_launch0);
            ctx->time_valid = true;
        }
        if (ranged) nvtxRangePop();
    }
    if (prev >= 0) cudaSetDevice(prev);
}

int pinned_mailbox(vw_ctx *ctx, size_t bytes, void **out) {
    if (ctx->pinned_bytes < bytes) {
        if (ctx->pinned) cudaFreeHost(ctx->pinned);
        ctx->pinned = nullptr;
        ctx->pinned_bytes = 0;
        size_t want = std::max(bytes, (size_t)4096);
        int rc = vw_cuda_check(ctx, cudaMallocHost(&ctx->pinned, want), "pinned mailbox");
        if (rc) return rc;
        ctx->pinned_bytes = want;
    }
    *out = ctx->pinned;
    return VW_OK;
}

int load_filters(vw_ctx *ctx, const double *hs, const double *gs, int l, VwFilt &f) {
    if (!hs || !gs) return vw_fail(ctx, VW_ENULL, "filter pointer is null");
    if (l < 1 || l > VW_MAX_FILTER_TAPS)
        return vw_fail(ctx, VW_EINVAL, "filter length %d outside [1, %d]", l, VW_MAX_FILTER_TAPS);
    memset(&f, 0, sizeof f);
    memcpy(f.h, hs, sizeof(double) * l);
    memcpy(f.g, gs, sizeof(double) * l);
    return VW_OK;
}

int check_mode(vw_ctx *ctx, int mode) {
    if (mode == VW_PERIODIC || mode == VW_ZERO_PADDING || mode == VW_SYMMETRIC) return VW_OK;
    return vw_fail(ctx, VW_EBOUNDARY, "MODWT only supports PERIODIC, ZERO_PADDING, and SYMMETRIC boundary modes (got %d)",
                   mode);
}

// (l-1)*2^(levels-1)+1 <= n  (CORE/modwt/MultiLevelMODWTTransform.java:717-729); single level takes any n >= 1
int check_levels(vw_ctx *ctx, int64_t n, int l, int levels) {
    if (levels < 1 || levels > VW_MAX_LEVELS)
        return vw_fail(ctx, VW_ELEVEL, "Invalid number of decomposition levels: %d", levels);
    if (levels > 1) {
        long double lj = (long double)(l - 1) * (long double)((int64_t)1 << (levels - 1)) + 1;
        if (lj > (long double)n)
            return vw_fail(ctx, VW_ETOOLARGE,
                           "Upsampled filter length %.0Lf at level %d exceeds signal length %lld", lj, levels,
                           (long long)n);
    }
    return VW_OK;
}

// entry points that need an answer from the device (or a host-side wait) cannot be captured into a graph
int no_capture(vw_ctx *ctx, const char *what) {
    if (ctx->capturing) return vw_fail(ctx, VW_ESTATE, "%s needs a device-to-host answer and cannot be captured into a graph", what);
    return VW_OK;
}

int check_finite(vw_ctx *ctx, const double *x_dev, int64_t batch, int64_t n, int64_t ld, const char *what) {
    if (int rc0 = no_capture(ctx, "VW_FLAG_CHECK_FINITE")) return rc0;
    void *cnt = nullptr, *mb = nullptr;
    int rc = vw_scratch(ctx, 5, 64, &cnt);
    if (rc) return rc;
    if ((rc = pinned_mailbox(ctx, 64, &mb))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaMemsetAsync(cnt, 0, 8, ctx->stream), "small copy"))) return rc;
    if ((rc = vw_launch_nonfinite_count(ctx, x_dev, batch, n, ld, (unsigned long long *)cnt))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(mb, cnt, 8, cudaMemcpyDeviceToHost, ctx->stream), "small copy"))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaStreamSynchronize(ctx->stream), "finite check"))) return rc;
    unsigned long long bad = *(unsigned long long *)mb;
    if (bad) return vw_fail(ctx, VW_ENONFINITE, "%s contains %llu non-finite value(s) (NaN or Infinity)", what, bad);
    return VW_OK;
}

// 2-D strided copies between host rows and packed device rows
int copy_rows(vw_ctx *ctx, void *dst, int64_t ld_dst, const void *src, int64_t ld_src, int64_t n, int64_t rows,
              cudaMemcpyKind kind) {
    if (n <= 0 || rows <= 0) return VW_OK;
    return vw_cuda_check(ctx,
                         cudaMemcpy2DAsync(dst, (size_t)ld_dst * 8, src, (size_t)ld_src * 8, (size_t)n * 8,
                                           (size_t)rows, kind, ctx->stream),
                         "strided copy");
}

int finish(vw_ctx *ctx, uint32_t flags, bool host_io) {
    if (ctx->capturing) return VW_OK;   // nothing runs now; the graph launch decides about synchronising
    if (host_io || !(flags & VW_FLAG_NO_SYNC)) {
        int rc = vw_cuda_check(ctx, cudaStreamSynchronize(ctx->stream), "synchronize");
        if (ctx->scratch_stream == ctx->stream) ctx->scratch_pending = false;   // the stream the scratch was last used on has drained
        return rc;
    }
    // returning with work in flight: mark where the scratch buffers become free again (the outermost call does it once)
    if (ctx->call_depth > 1) return VW_OK;
    if (!ctx->scratch_event) {
        int rc = vw_cuda_check(ctx, cudaEventCreateWithFlags(&ctx->scratch_event, cudaEventDisableTiming), "scratch event");
        if (rc) return rc;
    }
    int rc = vw_cuda_check(ctx, cudaEventRecord(ctx->scratch_event, ctx->stream), "scratch event record");
    if (rc) return rc;
    ctx->scratch_pending = true;
    ctx->scratch_stream = ctx->stream;
    return VW_OK;
}

// ------------------------------------------------------------------------------------------------
// device-resident cores.  All pointers are device pointers here.
// ------------------------------------------------------------------------------------------------

vw_align default_align() { return vw_align{1, 0, 1, 0}; }

// One level of a streaming block over [history | block] rows (vw_modwt_stream_level and the per-level path of the
// stream state): the row is a linear span, so the tile kernel (any dilation whose halo fits) or, for deep levels, the
// column kernel -- the same kernels as the whole-signal path -- and the generic kernel for the rest and for BITEXACT.
int stream_level_device(vw_ctx *ctx, const double *vin, int64_t batch, int64_t ldin, int64_t hist, int64_t n, const VwFilt &f,
                        int l, int level, double *w, int64_t ldw, double *v, int64_t ldv, uint32_t flags) {
    const int64_t d = (int64_t)1 << (level - 1), n_in = hist + n;
    const bool exact = flags & VW_FLAG_BITEXACT;
    ctx->plan_lean_ok = true;
    int rc = VW_EUNSUPPORTED;
    if (!exact && !(flags & VW_FLAG_NO_FUSE)) {
        VwFusedFwd p{vin, ldin, w, ldw, 0, v, ldv, batch, n_in, hist, n, l, level, 1, VW_MODE_LINEAR, 0};
        rc = vw_fused_forward(ctx, p, f);
        if (rc != VW_OK && rc != VW_EUNSUPPORTED) return rc;
        if (rc == VW_EUNSUPPORTED && d >= 4 && ctx->opt_poly != 0) {
            rc = vw_column_analysis(ctx, vin, ldin, v, ldv, w, ldw, n_in, hist, n, batch, f, l, d, VW_MODE_LINEAR);
            if (rc != VW_OK && rc != VW_EUNSUPPORTED) return rc;
        }
    }
    if (rc == VW_EUNSUPPORTED)
        rc = vw_launch_analysis_level(ctx, vin, ldin, v, ldv, w, ldw, n_in, hist, n, batch, f, l, d, VW_MODE_LINEAR, exact);
    return rc;
}

// Analysis cascade over device buffers.  Groups of levels come from the planner; a group the fused kernel declines
// (unaligned rows, exotic filter length, ...) runs level by level on the generic kernels.
int forward_device(vw_ctx *ctx, const double *x, int64_t batch, int64_t n, int64_t ldx, const VwFilt &f, int l,
                   int levels, int mode, double *w, int64_t ldw, int64_t lsw, double *vj, int64_t ldv, uint32_t flags) {
    const bool exact = flags & VW_FLAG_BITEXACT;
    const bool allow_fused = !exact && !(flags & VW_FLAG_NO_FUSE);
    std::vector<VwPlanGroup> plan;
    ctx->plan_lean_ok = true;   // the lean analysis takes every boundary mode
    if (allow_fused) vw_plan_levels(ctx, true, l, levels, n, plan);
    else for (int j = 1; j <= levels; j++) plan.push_back(VwPlanGroup{j, 1, -1, 0.0});
    double *buf[2] = {nullptr, nullptr};
    const double *cur = x;
    int64_t ld_cur = ldx;
    int pp = 0;
    // destination of the approximation leaving level `end`: the caller's V_J for the last level, else ping-pong scratch
    auto pick_out = [&](int end, double *&vout, int64_t &ld_vout) -> int {
        if (end == levels) { vout = vj; ld_vout = ldv; return VW_OK; }
        if (!buf[pp]) {
            void *p;
            int r = vw_scratch(ctx, pp, (size_t)batch * (size_t)n * 8, &p);
            if (r) return r;
            buf[pp] = (double *)p;
        }
        vout = buf[pp];
        ld_vout = n;
        return VW_OK;
    };
    for (const VwPlanGroup &g : plan) {
        int rc = VW_EUNSUPPORTED;
        double *vout = nullptr;
        int64_t ld_vout = 0;
        if (allow_fused && g.tile > 0) {
            if ((rc = pick_out(g.first + g.nlev - 1, vout, ld_vout))) return rc;
            VwFusedFwd p{cur, ld_cur, w + (int64_t)(g.first - 1) * lsw, ldw, lsw, vout, ld_vout, batch, n, 0, n,
                         l, g.first, g.nlev, mode, g.tile};
            rc = vw_fused_forward(ctx, p, f);
            if (rc != VW_OK && rc != VW_EUNSUPPORTED) return rc;
            if (rc == VW_OK) { cur = vout; ld_cur = ld_vout; pp ^= 1; }
        } else if (allow_fused && g.tile == -2 && g.nlev == 2) {
            // two column levels in one pass (lattice pair kernels): V of the first level never exists in memory
            if ((rc = pick_out(g.first + 1, vout, ld_vout))) return rc;
            rc = vw_column_analysis2(ctx, cur, ld_cur, w + (int64_t)(g.first - 1) * lsw, ldw, w + (int64_t)g.first * lsw, ldw, vout,
                                     ld_vout, n, 0, n, batch, f, l, (int64_t)1 << (g.first - 1), mode);
            if (rc != VW_OK && rc != VW_EUNSUPPORTED) return rc;
            if (rc == VW_OK) { cur = vout; ld_cur = ld_vout; pp ^= 1; }
        }
        if (rc == VW_EUNSUPPORTED) {
            for (int level = g.first; level < g.first + g.nlev; level++) {
                if ((rc = pick_out(level, vout, ld_vout))) return rc;
                rc = VW_EUNSUPPORTED;
                if (allow_fused && level >= vw_column_min_level(ctx, l) && ctx->opt_poly != 0) {
                    rc = vw_column_analysis(ctx, cur, ld_cur, vout, ld_vout, w + (int64_t)(level - 1) * lsw, ldw, n, 0, n,
                                            batch, f, l, (int64_t)1 << (level - 1), mode);
                    if (rc != VW_OK && rc != VW_EUNSUPPORTED) return rc;
                }
                if (rc == VW_EUNSUPPORTED)
                    rc = vw_launch_analysis_level(ctx, cur, ld_cur, vout, ld_vout, w + (int64_t)(level - 1) * lsw, ldw, n,
                                                  0, n, batch, f, l, (int64_t)1 << (level - 1), mode, exact);
                if (rc) return rc;
                cur = vout; ld_cur = ld_vout; pp ^= 1;
            }
        }
    }
    return VW_OK;
}

int inverse_device(vw_ctx *ctx, const double *w, int64_t ldw, int64_t lsw, const double *vj, int64_t ldv,
                   int64_t batch, int64_t n, const VwFilt &f, int l, int levels, int mode, const vw_align *align,
                   int order, uint64_t detail_mask, int use_approx, double *xout, int64_t ldx, uint32_t flags,
                   const double *thr_dev, int thr_per_row, int thr_soft, int64_t thr_lstride) {
    const bool exact = flags & VW_FLAG_BITEXACT;
    // thresholds of level j start at thr_dev + (j-1) * thr_lstride (stride 0: one table for every level); a stage gets
    // the table of its first level, and a multi-level stage the stride to reach the others
    auto thr_at = [&](int level) { return thr_dev ? thr_dev + (int64_t)(level - 1) * thr_lstride : nullptr; };
    // the fused synthesis kernels implement the {+1,0,+1,0} index rule (t + k*d) -- PERIODIC and ZERO_PADDING
    bool plain = true;
    if (align)
        for (int j = 0; j < levels; j++)
            plain = plain && align[j].sigma_h == 1 && align[j].sigma_g == 1 && align[j].tau_h == 0 && align[j].tau_g == 0;
    const bool allow_fused = !exact && !(flags & VW_FLAG_NO_FUSE) && plain && mode != VW_SYMMETRIC;
    std::vector<VwPlanGroup> plan;
    {
        const uint64_t full = levels >= 64 ? ~0ull : ((1ull << levels) - 1);
        ctx->plan_lean_ok = mode != VW_SYMMETRIC && use_approx && (detail_mask & full) == full;
    }
    if (allow_fused) vw_plan_levels(ctx, false, l, levels, n, plan);
    else for (int j = 1; j <= levels; j++) plan.push_back(VwPlanGroup{j, 1, -1, 0.0});
    double *buf[2] = {nullptr, nullptr};
    const double *cur = use_approx ? vj : nullptr;
    int64_t ld_cur = ldv;
    int pp = 0;
    auto pick_out = [&](int first, double *&out, int64_t &ld_out) -> int {
        if (first == 1) { out = xout; ld_out = ldx; return VW_OK; }
        if (!buf[pp]) {
            void *p;
            int r = vw_scratch(ctx, pp, (size_t)batch * (size_t)n * 8, &p);
            if (r) return r;
            buf[pp] = (double *)p;
        }
        out = buf[pp];
        ld_out = n;
        return VW_OK;
    };
    for (int gi = (int)plan.size() - 1; gi >= 0; gi--) {
        const VwPlanGroup &g = plan[gi];
        int rc = VW_EUNSUPPORTED;
        double *out = nullptr;
        int64_t ld_out = 0;
        if (allow_fused && g.tile > 0) {
            if ((rc = pick_out(g.first, out, ld_out))) return rc;
            VwFusedInv p{cur, ld_cur, w + (int64_t)(g.first - 1) * lsw, ldw, lsw,
                         (detail_mask >> (g.first - 1)) & ((g.nlev >= 64 ? ~0ull : ((1ull << g.nlev) - 1))),
                         out, ld_out, batch, n, n, l, g.first, g.nlev, mode, thr_at(g.first), thr_per_row, thr_soft, g.tile};
            p.thr_lstride = thr_lstride;
            rc = vw_fused_inverse(ctx, p, f);
            if (rc != VW_OK && rc != VW_EUNSUPPORTED) return rc;
            if (rc == VW_OK) { cur = out; ld_cur = ld_out; pp ^= 1; }
        } else if (allow_fused && g.tile == -2 && g.nlev == 2 && cur && ((detail_mask >> (g.first - 1)) & 3ull) == 3ull) {
            if ((rc = pick_out(g.first, out, ld_out))) return rc;
            rc = vw_column_synthesis2(ctx, cur, ld_cur, w + (int64_t)g.first * lsw, ldw, w + (int64_t)(g.first - 1) * lsw, ldw, out,
                                      ld_out, n, 0, n, batch, f, l, (int64_t)1 << (g.first - 1), mode, thr_at(g.first), thr_per_row,
                                      thr_soft, thr_lstride);
            if (rc != VW_OK && rc != VW_EUNSUPPORTED) return rc;
            if (rc == VW_OK) { cur = out; ld_cur = ld_out; pp ^= 1; }
        }
        if (rc == VW_EUNSUPPORTED) {
            for (int level = g.first + g.nlev - 1; level >= g.first; level--) {
                if ((rc = pick_out(level, out, ld_out))) return rc;
                vw_align al = align ? align[level - 1] : default_align();
                const double *wj = ((detail_mask >> (level - 1)) & 1ull) ? w + (int64_t)(level - 1) * lsw : nullptr;
                rc = VW_EUNSUPPORTED;
                const bool fast = !exact && !(flags & VW_FLAG_NO_FUSE);
                // aligned (sigma, tau) stages have no multi-level fused form: column kernels from dilation 4, and the
                // single-level tile kernel (stream offsets + reversed taps) below that
                const int col_min = allow_fused ? vw_column_min_level(ctx, l, false) : std::min(3, vw_column_min_level(ctx, l, false));
                if (fast && level >= col_min && ctx->opt_poly != 0) {
                    rc = vw_column_synthesis(ctx, cur, ld_cur, wj, ldw, out, ld_out, n, 0, n, batch, f, l,
                                             (int64_t)1 << (level - 1), mode, al, thr_at(level), thr_per_row, thr_soft);
                    if (rc != VW_OK && rc != VW_EUNSUPPORTED) return rc;
                }
                if (rc == VW_EUNSUPPORTED && fast && !allow_fused) {
                    VwFusedInv p{cur, ld_cur, w + (int64_t)(level - 1) * lsw, ldw, lsw, wj ? 1ull : 0ull, out, ld_out, batch, n, n,
                                 l, level, 1, mode, thr_at(level), thr_per_row, thr_soft, 0};
                    p.has_align = true;
                    p.align = al;
                    rc = vw_fused_inverse(ctx, p, f);
                    if (rc != VW_OK && rc != VW_EUNSUPPORTED) return rc;
                }
                if (rc == VW_EUNSUPPORTED) {
                    // the per-level kernels have no threshold-on-load: threshold this level in place first (only the
                    // denoisers pass thr_dev, and their W is engine scratch)
                    if (thr_dev && wj &&
                        (rc = vw_launch_threshold(ctx, const_cast<double *>(wj), batch, n, ldw, thr_at(level), thr_per_row, thr_soft)))
                        return rc;
                    rc = vw_launch_synthesis_level(ctx, cur, ld_cur, wj, ldw, out, ld_out, n, 0, n, batch, f, l,
                                                   (int64_t)1 << (level - 1), mode, al, order == VW_ORDER_PAIR, exact);
                }
                if (rc) return rc;
                cur = out; ld_cur = ld_out; pp ^= 1;
            }
        }
    }
    return VW_OK;
}

// ------------------------------------------------------------------------------------------------
// host-buffer calls on large batches: chunk the batch and alternate two streams, so the H2D copy of chunk c+1, the
// kernels of chunk c and the D2H copy of chunk c-1 overlap (PCIe is full duplex and the copy engines are separate;
// the double[] API moves (levels + 2) * 8 bytes per sample each way, which is what bounds e2e throughput).
// Every stream owns its own scratch set.  Signals are independent, so chunking by rows changes no result.
// ------------------------------------------------------------------------------------------------
struct PipeGuard {
    vw_ctx *ctx;
    cudaStream_t saved;
    explicit PipeGuard(vw_ctx *c) : ctx(c), saved(c->stream) {}
    // every exit path, errors included: chunks already enqueued may still be copying into the caller's buffers and
    // using both scratch sets, so nothing is handed back before both pipeline streams have drained
    ~PipeGuard() {
        for (int i = 0; i < 2; i++) if (ctx->pipe_stream[i]) cudaStreamSynchronize(ctx->pipe_stream[i]);
        ctx->stream = saved; ctx->scratch_set = 0;
    }
};

int pipe_streams(vw_ctx *ctx) {
    for (int i = 0; i < 2; i++)
        if (!ctx->pipe_stream[i]) {
            int rc = vw_cuda_check(ctx, cudaStreamCreateWithFlags(&ctx->pipe_stream[i], cudaStreamNonBlocking), "pipeline stream");
            if (rc) return rc;
        }
    return VW_OK;
}

// rows per chunk: chunks of >= 16 MB staged bytes, at most `pipe_chunks` of them (the first chunk's H2D and the last
// chunk's D2H overlap nothing: more chunks = a shorter fill and drain), at least 2
int64_t pipe_rows(const vw_ctx *ctx, int64_t batch, int64_t n, int levels) {
    const double total = (double)batch * (double)n * 8.0 * (levels + 2);
    if (ctx->opt_pipe_min <= 0 || batch < 2 || total < (double)ctx->opt_pipe_min || ctx->capturing) return 0;
    int64_t chunks = (int64_t)(total / (16.0 * 1048576.0));
    chunks = std::max<int64_t>(2, std::min<int64_t>(std::min<int64_t>(chunks, std::max<int64_t>(ctx->opt_pipe_chunks, 2)), batch));
    return (batch + chunks - 1) / chunks;
}

// runs chunk(c) for c = 0 .. nchunks-1, chunk c enqueued on pipeline stream c & 1 with scratch set c & 1; returns when
// both streams have drained
template <class Chunk>
int run_pipelined(vw_ctx *ctx, int64_t nchunks, Chunk &&chunk) {
    int rc;
    if ((rc = pipe_streams(ctx))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaStreamSynchronize(ctx->stream), "synchronize"))) return rc;
    PipeGuard guard(ctx);
    for (int64_t c = 0; c < nchunks; c++) {
        ctx->scratch_set = (int)(c & 1);
        ctx->stream = ctx->pipe_stream[c & 1];
        if ((rc = chunk(c))) return rc;
    }
    for (int i = 0; i < 2; i++)
        if ((rc = vw_cuda_check(ctx, cudaStreamSynchronize(ctx->pipe_stream[i]), "pipeline synchronize"))) return rc;
    return VW_OK;
}

int forward_host_pipelined(vw_ctx *ctx, const double *x, int64_t batch, int64_t n, int64_t ldx, const VwFilt &f, int l,
                           int levels, int mode, double *w, int64_t ldw, int64_t lsw, double *vj, int64_t ldv, uint32_t flags,
                           int64_t rows) {
    return run_pipelined(ctx, (batch + rows - 1) / rows, [&](int64_t c) -> int {
        int rc;
        const int64_t b0 = c * rows, rb = std::min(rows, batch - b0);
        void *px, *pw;
        const size_t bn = (size_t)rb * (size_t)n;
        if ((rc = vw_scratch(ctx, 2, (size_t)rows * (size_t)n * 8, &px))) return rc;
        if ((rc = vw_scratch(ctx, 3, (size_t)rows * (size_t)n * 8 * (size_t)(levels + 1), &pw))) return rc;
        double *xd = (double *)px, *wd = (double *)pw, *vd = wd + bn * (size_t)levels;
        if ((rc = copy_rows(ctx, xd, n, x + b0 * ldx, ldx, n, rb, cudaMemcpyHostToDevice))) return rc;
        if (flags & VW_FLAG_CHECK_FINITE) if ((rc = check_finite(ctx, xd, rb, n, n, "signal"))) return rc;
        if ((rc = forward_device(ctx, xd, rb, n, n, f, l, levels, mode, wd, n, (int64_t)bn, vd, n, flags))) return rc;
        for (int j = 0; j < levels; j++)
            if ((rc = copy_rows(ctx, w + (int64_t)j * lsw + b0 * ldw, ldw, wd + (size_t)j * bn, n, n, rb, cudaMemcpyDeviceToHost))) return rc;
        return copy_rows(ctx, vj + b0 * ldv, ldv, vd, n, n, rb, cudaMemcpyDeviceToHost);
    });
}

int inverse_host_pipelined(vw_ctx *ctx, const double *w, int64_t ldw, int64_t lsw, const double *vj, int64_t ldv,
                           int64_t batch, int64_t n, const VwFilt &f, int l, int levels, int mode, const vw_align *align,
                           int order, uint64_t detail_mask, int use_approx, double *xout, int64_t ldx, uint32_t flags,
                           int64_t rows) {
    return run_pipelined(ctx, (batch + rows - 1) / rows, [&](int64_t c) -> int {
        int rc;
        const int64_t b0 = c * rows, rb = std::min(rows, batch - b0);
        void *px, *pw;
        const size_t bn = (size_t)rb * (size_t)n;
        if ((rc = vw_scratch(ctx, 2, (size_t)rows * (size_t)n * 8, &px))) return rc;
        if ((rc = vw_scratch(ctx, 3, (size_t)rows * (size_t)n * 8 * (size_t)(levels + 1), &pw))) return rc;
        double *xd = (double *)px, *wd = (double *)pw, *vd = wd + bn * (size_t)levels;
        for (int j = 0; j < levels; j++)
            if ((rc = copy_rows(ctx, wd + (size_t)j * bn, n, w + (int64_t)j * lsw + b0 * ldw, ldw, n, rb, cudaMemcpyHostToDevice))) return rc;
        if ((rc = copy_rows(ctx, vd, n, vj + b0 * ldv, ldv, n, rb, cudaMemcpyHostToDevice))) return rc;
        if (flags & VW_FLAG_CHECK_FINITE)
            if ((rc = check_finite(ctx, wd, (int64_t)(levels + 1) * rb, n, n, "coefficients"))) return rc;
        if ((rc = inverse_device(ctx, wd, n, (int64_t)bn, vd, n, rb, n, f, l, levels, mode, align, order, detail_mask,
                                 use_approx, xd, n, flags, nullptr, 0, 0, 0))) return rc;
        return copy_rows(ctx, xout + b0 * ldx, ldx, xd, n, n, rb, cudaMemcpyDeviceToHost);
    });
}

// Small host-buffer calls on PINNED memory skip the staging copies altogether: page-locked allocations are mapped into the
// device's address space (unified addressing), so the kernels read the signal and write the coefficients over PCIe
// themselves -- one launch + one synchronise instead of H2D + launch + 2 D2H + synchronise, each with its own DMA set-up
// (config #1, 1 x 4096 db4 J = 1: 28.4 -> 15.2 us per call, bit-identical results).  Capturable: it is one kernel launch.  Returns the device alias of a mapped host pointer, or nullptr
// (pageable memory, or a device that cannot map host memory).
const void *mapped_alias(const void *host) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    if (at.type != cudaMemoryTypeHost || !at.devicePointer) return nullptr;
    return at.devicePointer;
}

int check_signal_args(vw_ctx *ctx, const void *x, int64_t batch, int64_t n, int64_t ld) {
    if (!x) return vw_fail(ctx, VW_ENULL, "signal cannot be null");
    if (batch < 1) return vw_fail(ctx, VW_ELENGTH, "signals must be non-null and non-empty (batch=%lld)", (long long)batch);
    if (n < 1) return vw_fail(ctx, VW_EEMPTY, "Signal cannot be empty");
    if (ld < n) return vw_fail(ctx, VW_ELENGTH, "row stride %lld shorter than signal length %lld", (long long)ld, (long long)n);
    return VW_OK;
}

// ---- packed rows of different lengths (vw_modwt_forward_varlen / vw_modwt_inverse_varlen) ---------------------------
// offsets: HOST array of batch + 1 values, offsets[0] == 0, never decreasing.  *first_empty: the lowest empty row, or batch.
int check_offsets(vw_ctx *ctx, const int64_t *off, int64_t batch, int64_t *first_empty) {
    if (!off) return vw_fail(ctx, VW_ENULL, "offsets cannot be null");
    if (batch < 1) return vw_fail(ctx, VW_ELENGTH, "signals must be non-null and non-empty (batch=%lld)", (long long)batch);
    if (off[0] != 0) return vw_fail(ctx, VW_ELENGTH, "offsets[0] must be 0 (got %lld)", (long long)off[0]);
    *first_empty = batch;
    for (int64_t b = 0; b < batch; b++) {
        if (off[b + 1] < off[b])
            return vw_fail(ctx, VW_ELENGTH, "offsets decrease at row %lld (%lld -> %lld)", (long long)b, (long long)off[b],
                           (long long)off[b + 1]);
        if (off[b + 1] == off[b] && *first_empty == batch) *first_empty = b;
    }
    return VW_OK;
}

// row holding packed position p (empty rows hold none)
int64_t row_of(const int64_t *off, int64_t batch, int64_t p) {
    return (int64_t)(std::upper_bound(off, off + batch + 1, p) - off) - 1;
}

// lowest packed index i < n with a[i] or b[i] (b may be null) NaN / Inf, or -1.  Device pointers.
int first_nonfinite(vw_ctx *ctx, const double *a, const double *b, int64_t n, int64_t *idx) {
    *idx = -1;
    if (n <= 0) return VW_OK;
    void *slot = nullptr, *mb = nullptr;
    int rc;
    if ((rc = vw_scratch(ctx, 5, 64, &slot))) return rc;
    if ((rc = pinned_mailbox(ctx, 64, &mb))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaMemsetAsync(slot, 0xff, 8, ctx->stream), "small copy"))) return rc;
    if ((rc = vw_launch_first_nonfinite(ctx, a, b, n, (unsigned long long *)slot))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(mb, slot, 8, cudaMemcpyDeviceToHost, ctx->stream), "small copy"))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaStreamSynchronize(ctx->stream), "finite check"))) return rc;
    const unsigned long long first = *(unsigned long long *)mb;
    if (first != ~0ull) *idx = (int64_t)first;
    return VW_OK;
}

// VW_ENONFINITE naming the row of the first bad packed index (chunk-local index q of a chunk starting at s0), if any
int varlen_finite(vw_ctx *ctx, const double *a, const double *b, int64_t n, const int64_t *off, int64_t batch, int64_t s0,
                  const char *what) {
    int64_t q;
    if (int rc = first_nonfinite(ctx, a, b, n, &q)) return rc;
    if (q < 0) return VW_OK;
    return vw_fail(ctx, VW_ENONFINITE, "row %lld: %s contain(s) non-finite values (NaN or Infinity)",
                   (long long)row_of(off, batch, s0 + q), what);
}

// The reference's loop over rows (forwardBatch / inverseBatch with mixed lengths, one forward / inverse per row)
// validates rows in index order and throws at the first bad one.  An empty row therefore fails the call, but only after
// the rows before it were scanned for NaN / Inf.  a, b: the packed inputs (b may be null), host unless dev.
int varlen_empty_row(vw_ctx *ctx, const double *a, const double *b, const int64_t *off, int64_t batch, int64_t empty, bool dev,
                     bool check, const char *what) {
    const int64_t lim = off[empty];
    if (check && lim > 0) {
        int rc;
        if (!dev) {
            void *p;
            if ((rc = vw_scratch(ctx, 2, (size_t)lim * 8 * (b ? 2 : 1), &p))) return rc;
            double *ad = (double *)p, *bd = b ? ad + lim : nullptr;
            if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(ad, a, (size_t)lim * 8, cudaMemcpyHostToDevice, ctx->stream), "h2d"))) return rc;
            if (b && (rc = vw_cuda_check(ctx, cudaMemcpyAsync(bd, b, (size_t)lim * 8, cudaMemcpyHostToDevice, ctx->stream), "h2d"))) return rc;
            a = ad; b = bd;
        }
        if ((rc = varlen_finite(ctx, a, b, lim, off, batch, 0, what))) return rc;
    }
    return vw_fail(ctx, VW_EEMPTY, "row %lld: Signal cannot be empty", (long long)empty);
}

// row boundaries of the pipelined host path: about equal packed samples per chunk, cut between rows; a single cut
// (one row holding nearly everything) means nothing to overlap
std::vector<int64_t> varlen_chunks(const vw_ctx *ctx, const int64_t *off, int64_t batch) {
    const int64_t total = off[batch];
    const double bytes = (double)total * 8.0 * 3.0;
    std::vector<int64_t> cut{0};
    if (ctx->opt_pipe_min <= 0 || batch < 2 || bytes < (double)ctx->opt_pipe_min) return cut;
    int64_t chunks = (int64_t)(bytes / (16.0 * 1048576.0));
    chunks = std::max<int64_t>(2, std::min<int64_t>(std::min<int64_t>(chunks, std::max<int64_t>(ctx->opt_pipe_chunks, 2)), batch));
    for (int64_t c = 1; c < chunks; c++) {
        const int64_t b = (int64_t)(std::lower_bound(off, off + batch + 1, (int64_t)((double)total * c / chunks)) - off);
        if (b > cut.back() && b < batch) cut.push_back(b);
    }
    cut.push_back(batch);
    if (cut.size() < 3) cut.resize(1);
    return cut;
}

// The denoisers' chain over one batch: stage x, decompose into scratch, let `select` put the thresholds on the device
// (select(W, thr, per_row, level_stride); W is [levels][batch][n] scratch), reconstruct with them applied as the
// synthesis loads W (MutableMultiLevelMODWTResult.applyThreshold :97-118 fused into the load; stages without a fused form
// threshold their level in place just before consuming it), stage the result back.  The caller synchronises.
template <class Select>
int denoise_chain(vw_ctx *ctx, const double *x, int64_t batch, int64_t n, int64_t ldx, const VwFilt &f, int l, int levels,
                  int mode, const vw_align *align, int order, int soft, double *out, int64_t ldo, uint32_t flags, Select &&select) {
    int rc;
    const bool dev = flags & VW_FLAG_DEVICE_PTRS;
    size_t bn = (size_t)batch * (size_t)n;
    void *pw;
    if ((rc = vw_scratch(ctx, 3, bn * 8 * (size_t)(levels + 1), &pw))) return rc;
    double *wd = (double *)pw, *vd = wd + bn * (size_t)levels;
    const double *xd = x;
    double *od = out;
    int64_t ldxd = ldx, ldod = ldo;
    if (!dev) {
        void *p;
        if ((rc = vw_scratch(ctx, 2, bn * 8, &p))) return rc;
        if ((rc = copy_rows(ctx, p, n, x, ldx, n, batch, cudaMemcpyHostToDevice))) return rc;
        xd = (const double *)p; od = (double *)p; ldxd = n; ldod = n;
    }
    if (flags & VW_FLAG_CHECK_FINITE) if ((rc = check_finite(ctx, xd, batch, n, ldxd, "signal"))) return rc;
    if ((rc = forward_device(ctx, xd, batch, n, ldxd, f, l, levels, mode, wd, n, (int64_t)bn, vd, n, flags))) return rc;
    const double *thr = nullptr;
    int per_row = 0;
    int64_t lstride = 0;
    if ((rc = select((const double *)wd, thr, per_row, lstride))) return rc;
    uint64_t mask = levels >= 64 ? ~0ull : ((1ull << levels) - 1);
    if ((rc = inverse_device(ctx, wd, n, (int64_t)bn, vd, n, batch, n, f, l, levels, mode, align, order, mask, 1, od,
                             ldod, flags, thr, per_row, soft, lstride))) return rc;
    if (!dev) if ((rc = copy_rows(ctx, out, ldo, od, n, n, batch, cudaMemcpyDeviceToHost))) return rc;
    return VW_OK;
}

}  // namespace vwshim
using namespace vwshim;

// ------------------------------------------------------------------------------------------------
// extern "C"
// ------------------------------------------------------------------------------------------------
extern "C" {

int vw_abi_version(void) { return VW_ABI_VERSION; }

const char *vw_status_name(int s) {
    switch (s) {
        case VW_OK: return "OK";
        case VW_ENULL: return "VAL_NULL_ARGUMENT";
        case VW_ENONFINITE: return "VAL_NON_FINITE_VALUES";
        case VW_ETOOLARGE: return "VAL_TOO_LARGE";
        case VW_EEMPTY: return "VAL_EMPTY";
        case VW_ELENGTH: return "VAL_LENGTH_MISMATCH";
        case VW_EBOUNDARY: return "CFG_UNSUPPORTED_BOUNDARY_MODE";
        case VW_ELEVEL: return "CFG_INVALID_DECOMPOSITION_LEVEL";
        case VW_ESTATE: return "STATE_INVALID";
        case VW_EINVAL: return "ILLEGAL_ARGUMENT";
        case VW_ENOMEM: return "OUT_OF_MEMORY";
        case VW_ECUDA: return "CUDA_ERROR";
        case VW_EUNSUPPORTED: return "UNSUPPORTED";
        default: return "UNKNOWN";
    }
}

int vw_init(int device, vw_ctx **out) {
    if (!out) return VW_ENULL;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) return VW_ECUDA;  // no CPU path exists: fail loudly
    if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) return VW_ECUDA; }
    if (device >= count) return VW_EINVAL;
    DeviceGuard g(device);
    vw_ctx *ctx = new vw_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete ctx; return VW_ECUDA; }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return VW_ECUDA; }
    ctx->stream = ctx->own_stream;
    *out = ctx;
    return VW_OK;
}

int vw_destroy(vw_ctx *ctx) {
    if (!ctx) return VW_ENULL;
    {
        DeviceGuard g(ctx, "vw_destroy");   // released before the ctx (and its mutex) goes away
        cudaStreamSynchronize(ctx->stream);
        for (int i = 0; i < 2 * vw_ctx::kScratch; i++) if (ctx->scratch[i]) cudaFree(ctx->scratch[i]);
        for (int i = 0; i < 2; i++) if (ctx->pipe_stream[i]) cudaStreamDestroy(ctx->pipe_stream[i]);
        if (ctx->pinned) cudaFreeHost(ctx->pinned);
        if (ctx->scratch_event) cudaEventDestroy(ctx->scratch_event);
        for (int i = 0; i < 2; i++) if (ctx->time_ev[i]) cudaEventDestroy(ctx->time_ev[i]);
        if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    }
    delete ctx;
    return VW_OK;
}

const char *vw_last_error(const vw_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int vw_set_stream(vw_ctx *ctx, void *s) {
    if (!ctx) return VW_ENULL;
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    ctx->stream = (cudaStream_t)s;
    return VW_OK;
}

int vw_reset_stream(vw_ctx *ctx) {
    if (!ctx) return VW_ENULL;
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    ctx->stream = ctx->own_stream;
    return VW_OK;
}

int vw_synchronize(vw_ctx *ctx) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_synchronize");
    if (int rc0 = no_capture(ctx, "vw_synchronize")) return rc0;
    return vw_cuda_check(ctx, cudaStreamSynchronize(ctx->stream), "synchronize");
}

int vw_device_index(const vw_ctx *ctx) { return ctx ? ctx->device : -1; }

int vw_set_option(vw_ctx *ctx, const char *name, int64_t value) {
    if (!ctx || !name) return VW_ENULL;
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    if (!strcmp(name, "tile")) ctx->opt_tile = value;
    else if (!strcmp(name, "fuse")) ctx->opt_fuse = value;
    else if (!strcmp(name, "threads")) ctx->opt_threads = value;
    else if (!strcmp(name, "poly")) ctx->opt_poly = value;
    else if (!strcmp(name, "colmin")) ctx->opt_colmin = value;
    else if (!strcmp(name, "lattice")) ctx->opt_lattice = value;
    else if (!strcmp(name, "colrpc")) ctx->opt_colrpc = value;
    else if (!strcmp(name, "wave")) ctx->opt_wave = value;
    else if (!strcmp(name, "l2pf")) ctx->opt_l2pf = value;
    else if (!strcmp(name, "lean")) ctx->opt_lean = value;
    else if (!strcmp(name, "lean_small")) ctx->opt_lean_small = value;
    else if (!strcmp(name, "pipe_chunks")) ctx->opt_pipe_chunks = value;   // most chunks a pipelined host call is cut into
    else if (!strcmp(name, "pipe_min")) ctx->opt_pipe_min = value;   // bytes; <= 0 disables the pipelined host path
    else if (!strcmp(name, "timing")) ctx->opt_timing = value;
    else if (!strcmp(name, "zero_copy")) ctx->opt_zero_copy = value;   // bytes up to which pinned host buffers are addressed in place; 0 = always stage       // event pair around every public call (vw_last_timing)
    else return vw_fail(ctx, VW_EINVAL, "unknown option '%s'", name);
    ctx->plan_cache.clear();   // plans depend on the knobs
    return VW_OK;
}

int64_t vw_launch_count(const vw_ctx *ctx) { return ctx ? ctx->launches : -1; }

int vw_plan_query(int forward, int32_t l, int32_t levels, int64_t n, int32_t *first, int32_t *nlev, int32_t cap) {
    if (!first || !nlev) return -VW_ENULL;
    if (l < 1 || levels < 1 || levels > VW_MAX_LEVELS || n < 1) return -VW_EINVAL;
    vw_ctx fake;
    fake.smem_optin = 227 * 1024;
    fake.sm_count = 148;
    std::vector<VwPlanGroup> plan;
    vw_plan_levels(&fake, forward != 0, l, levels, n, plan);
    if ((int)plan.size() > cap) return -VW_ELENGTH;
    for (size_t i = 0; i < plan.size(); i++) { first[i] = plan[i].first; nlev[i] = plan[i].nlev; }
    return (int)plan.size();
}

int vw_describe_plan(int forward, int32_t l, int32_t levels, int64_t n, int64_t tile, int32_t fuse, char *out, size_t cap) {
    if (!out || cap == 0) return -VW_ENULL;
    if (l < 1 || levels < 1 || levels > VW_MAX_LEVELS || n < 1) return -VW_EINVAL;
    vw_ctx fake;
    fake.smem_optin = 227 * 1024;
    fake.sm_count = 148;
    fake.opt_tile = tile;
    fake.opt_fuse = fuse;
    std::vector<VwPlanGroup> plan;
    vw_plan_levels(&fake, forward != 0, l, levels, n, plan);
    size_t used = 0;
    out[0] = 0;
    for (const VwPlanGroup &g : plan) {
        int k = snprintf(out + used, cap - used, "levels %d-%d: %s tile=%lld halo=%lld cost=%.2f cyc/sample/SM\n", g.first,
                         g.first + g.nlev - 1, g.tile > 0 ? "fused" : (g.tile == -2 ? "column" : "per-level"), (long long)g.tile,
                         (long long)((int64_t)(l - 1) * ((int64_t)1 << (g.first - 1)) * (((int64_t)1 << g.nlev) - 1)), g.cost);
        if (k < 0 || (size_t)k >= cap - used) break;
        used += (size_t)k;
    }
    return (int)plan.size();
}

void *vw_alloc_pinned(size_t bytes) {
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 16) != cudaSuccess) return nullptr;
    return p;
}
void vw_free_pinned(void *p) { if (p) cudaFreeHost(p); }

int vw_device_alloc(vw_ctx *ctx, size_t bytes, void **out) {
    if (!ctx || !out) return VW_ENULL;
    DeviceGuard g(ctx, "vw_device_alloc");
    return vw_cuda_check(ctx, cudaMalloc(out, bytes ? bytes : 16), "vw_device_alloc");
}
int vw_device_free(vw_ctx *ctx, void *p) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_device_free");
    if (int rc0 = no_capture(ctx, "vw_device_free")) return rc0;
    cudaStreamSynchronize(ctx->stream);
    return vw_cuda_check(ctx, cudaFree(p), "vw_device_free");
}
int vw_copy_h2d(vw_ctx *ctx, void *dst, const void *src, size_t bytes) {
    if (!ctx || !dst || !src) return VW_ENULL;
    DeviceGuard g(ctx, "vw_copy_h2d");
    if (int rc0 = no_capture(ctx, "vw_copy_h2d")) return rc0;
    int rc = vw_cuda_check(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream), "h2d");
    return rc ? rc : vw_cuda_check(ctx, cudaStreamSynchronize(ctx->stream), "h2d sync");
}
int vw_copy_d2h(vw_ctx *ctx, void *dst, const void *src, size_t bytes) {
    if (!ctx || !dst || !src) return VW_ENULL;
    DeviceGuard g(ctx, "vw_copy_d2h");
    if (int rc0 = no_capture(ctx, "vw_copy_d2h")) return rc0;
    int rc = vw_cuda_check(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream), "d2h");
    return rc ? rc : vw_cuda_check(ctx, cudaStreamSynchronize(ctx->stream), "d2h sync");
}

int vw_max_levels(int64_t n, int32_t l, int32_t cap) {
    if (n <= l) return 0;
    int limit = cap > 0 ? cap : 62;
    int max_level = 1;
    while (max_level < limit) {
        long double lj = (long double)(l - 1) * (long double)((int64_t)1 << (max_level - 1)) + 1;
        if (lj > (long double)n) break;
        max_level++;
    }
    return max_level - 1;
}

int64_t vw_span_halo(int32_t l, int32_t first_level, int32_t nlevels) {
    if (l < 1 || first_level < 1 || nlevels < 1 || first_level + nlevels > 62) return -1;
    return (int64_t)(l - 1) * ((int64_t)1 << (first_level - 1)) * (((int64_t)1 << nlevels) - 1);
}

int vw_conv_modwt(vw_ctx *ctx, const double *x, int64_t n, const double *filter, int64_t lf, int32_t mode, double *out,
                  uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_conv_modwt");
    if (!x || !filter || !out) return vw_fail(ctx, VW_ENULL, "signal, filter and output cannot be null");
    int rc;
    if ((rc = check_mode(ctx, mode))) return rc;
    if (n < 1) return vw_fail(ctx, VW_EEMPTY, "Signal cannot be empty");
    if (lf < 1) return vw_fail(ctx, VW_EEMPTY, "Filter cannot be empty");
    const bool dev = flags & VW_FLAG_DEVICE_PTRS;
    const double *xd = x, *fd = filter;
    double *od = out;
    if (!dev) {
        void *p;
        if ((rc = vw_scratch(ctx, 2, (size_t)(2 * n + lf) * 8, &p))) return rc;
        double *base = (double *)p;
        if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(base, x, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream), "small copy"))) return rc;
        if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(base + 2 * n, filter, (size_t)lf * 8, cudaMemcpyHostToDevice, ctx->stream), "small copy"))) return rc;
        xd = base; od = base + n; fd = base + 2 * n;
    }
    if (flags & VW_FLAG_CHECK_FINITE) if ((rc = check_finite(ctx, xd, 1, n, n, "signal"))) return rc;
    if ((rc = vw_launch_conv_dense(ctx, xd, n, fd, lf, mode, od, flags & VW_FLAG_BITEXACT))) return rc;
    if (!dev && (rc = vw_cuda_check(ctx, cudaMemcpyAsync(out, od, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream), "small copy"))) return rc;
    return finish(ctx, flags, !dev);
}

int vw_modwt_forward(vw_ctx *ctx, const double *x, int64_t batch, int64_t n, int64_t ldx, const double *hs,
                     const double *gs, int32_t l, int32_t levels, int32_t mode, double *w, int64_t ldw,
                     int64_t level_stride_w, double *vj, int64_t ldv, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_modwt_forward");
    int rc;
    if ((rc = check_mode(ctx, mode))) return rc;
    if ((rc = check_signal_args(ctx, x, batch, n, ldx))) return rc;
    if (!w || !vj) return vw_fail(ctx, VW_ENULL, "output buffers cannot be null");
    VwFilt f;
    if ((rc = load_filters(ctx, hs, gs, l, f))) return rc;
    if ((rc = check_levels(ctx, n, l, levels))) return rc;
    if (ldw < n || ldv < n || (levels > 1 && level_stride_w < (batch - 1) * ldw + n))
        return vw_fail(ctx, VW_ELENGTH, "output strides too small for [levels][batch][n]");
    const bool dev = flags & VW_FLAG_DEVICE_PTRS;
    if (dev) {
        if (flags & VW_FLAG_CHECK_FINITE) if ((rc = check_finite(ctx, x, batch, n, ldx, "signal"))) return rc;
        if ((rc = forward_device(ctx, x, batch, n, ldx, f, l, levels, mode, w, ldw, level_stride_w, vj, ldv, flags))) return rc;
        return finish(ctx, flags, false);
    }
    // small pinned host buffers: zero-copy (the kernels address the mapped host memory directly)
    if (ctx->opt_zero_copy > 0 && (double)batch * (double)n * 8.0 * (levels + 2) <= (double)ctx->opt_zero_copy) {
        const double *xa = (const double *)mapped_alias(x);
        double *wa = xa ? (double *)mapped_alias(w) : nullptr, *va = wa ? (double *)mapped_alias(vj) : nullptr;
        if (xa && wa && va) {
            if (flags & VW_FLAG_CHECK_FINITE) if ((rc = check_finite(ctx, xa, batch, n, ldx, "signal"))) return rc;
            if ((rc = forward_device(ctx, xa, batch, n, ldx, f, l, levels, mode, wa, ldw, level_stride_w, va, ldv, flags))) return rc;
            return finish(ctx, flags, true);
        }
    }
    // host buffers: stage x -> device (packed rows), run, stage W and V_J back
    if (const int64_t rows = pipe_rows(ctx, batch, n, levels))
        return forward_host_pipelined(ctx, x, batch, n, ldx, f, l, levels, mode, w, ldw, level_stride_w, vj, ldv, flags, rows);
    void *px, *pw;
    size_t bn = (size_t)batch * (size_t)n;
    if ((rc = vw_scratch(ctx, 2, bn * 8, &px))) return rc;
    if ((rc = vw_scratch(ctx, 3, bn * 8 * (size_t)(levels + 1), &pw))) return rc;
    double *xd = (double *)px, *wd = (double *)pw, *vd = wd + bn * (size_t)levels;
    if ((rc = copy_rows(ctx, xd, n, x, ldx, n, batch, cudaMemcpyHostToDevice))) return rc;
    if (flags & VW_FLAG_CHECK_FINITE) if ((rc = check_finite(ctx, xd, batch, n, n, "signal"))) return rc;
    if ((rc = forward_device(ctx, xd, batch, n, n, f, l, levels, mode, wd, n, (int64_t)bn, vd, n, flags))) return rc;
    for (int j = 0; j < levels; j++)
        if ((rc = copy_rows(ctx, w + (int64_t)j * level_stride_w, ldw, wd + (size_t)j * bn, n, n, batch, cudaMemcpyDeviceToHost))) return rc;
    if ((rc = copy_rows(ctx, vj, ldv, vd, n, n, batch, cudaMemcpyDeviceToHost))) return rc;
    return finish(ctx, flags, true);
}

// SoA batches are one flat periodic signal of n*batch samples whose level-j dilation is 2^(j-1) * batch:
// x[t*B+b] and x[((t-k d) mod n)*B+b] are d*B apart, and the wrap of the flat index mod n*B is the wrap of t mod n.
// The column kernels take any integer dilation, so the cascade runs in place on the caller's layout -- no transposes.
int vw_modwt_forward_soa(vw_ctx *ctx, const double *soa_x, int64_t batch, int64_t n, const double *hs, const double *gs,
                         int32_t l, int32_t levels, double *const *soa_w, double *soa_v, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_modwt_forward_soa");
    int rc;
    if ((rc = check_signal_args(ctx, soa_x, batch, n, n))) return rc;
    if (!soa_w || !soa_v) return vw_fail(ctx, VW_ENULL, "output buffers cannot be null");
    VwFilt f;
    if ((rc = load_filters(ctx, hs, gs, l, f))) return rc;
    if ((rc = check_levels(ctx, n, l, levels))) return rc;
    const int64_t tot = batch * n;
    for (int j = 0; j < levels; j++)
        if (!soa_w[j]) return vw_fail(ctx, VW_ENULL, "detail buffer of level %d cannot be null", j + 1);
    const bool dev = flags & VW_FLAG_DEVICE_PTRS;
    const bool exact = flags & VW_FLAG_BITEXACT;
    const double *xd = soa_x;
    double *wd = nullptr, *vd = soa_v;
    if (!dev) {
        void *px, *pw;
        if ((rc = vw_scratch(ctx, 2, (size_t)tot * 8, &px))) return rc;
        if ((rc = vw_scratch(ctx, 3, (size_t)tot * 8 * (size_t)(levels + 1), &pw))) return rc;
        if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(px, soa_x, (size_t)tot * 8, cudaMemcpyHostToDevice, ctx->stream), "h2d"))) return rc;
        xd = (const double *)px; wd = (double *)pw; vd = wd + (size_t)tot * (size_t)levels;
    }
    if (flags & VW_FLAG_CHECK_FINITE) if ((rc = check_finite(ctx, xd, 1, tot, tot, "signal"))) return rc;
    const double *cur = xd;
    double *buf[2] = {nullptr, nullptr};
    int pp = 0;
    for (int level = 1; level <= levels; level++) {
        double *vout = vd;
        if (level != levels) {
            if (!buf[pp]) {
                void *p;
                if ((rc = vw_scratch(ctx, pp, (size_t)tot * 8, &p))) return rc;
                buf[pp] = (double *)p;
            }
            vout = buf[pp];
        }
        const int64_t d = ((int64_t)1 << (level - 1)) * batch;
        double *wj = dev ? soa_w[level - 1] : wd + (size_t)(level - 1) * (size_t)tot;
        rc = VW_EUNSUPPORTED;
        if (!exact && !(flags & VW_FLAG_NO_FUSE) && d >= 32 && ctx->opt_poly != 0) {
            rc = vw_column_analysis(ctx, cur, 0, vout, 0, wj, 0, tot, 0, tot, 1, f, l, d, VW_PERIODIC);
            if (rc != VW_OK && rc != VW_EUNSUPPORTED) return rc;
        }
        if (rc == VW_EUNSUPPORTED)   // narrow batches at the first levels, exotic filter lengths, bit-exact order
            rc = vw_launch_analysis_level(ctx, cur, 0, vout, 0, wj, 0, tot, 0, tot, 1, f, l, d, VW_PERIODIC, exact);
        if (rc) return rc;
        cur = vout; pp ^= 1;
    }
    if (!dev) {
        for (int j = 0; j < levels; j++)
            if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(soa_w[j], wd + (size_t)j * (size_t)tot, (size_t)tot * 8,
                                                         cudaMemcpyDeviceToHost, ctx->stream), "d2h"))) return rc;
        if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(soa_v, vd, (size_t)tot * 8, cudaMemcpyDeviceToHost, ctx->stream), "d2h"))) return rc;
    }
    return finish(ctx, flags, !dev);
}

int vw_modwt_inverse(vw_ctx *ctx, const double *w, int64_t ldw, int64_t level_stride_w, const double *vj, int64_t ldv,
                     int64_t batch, int64_t n, const double *hs, const double *gs, int32_t l, int32_t levels,
                     int32_t mode, const vw_align *align, int32_t order, uint64_t detail_mask, int32_t use_approx,
                     double *xout, int64_t ldx, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_modwt_inverse");
    int rc;
    if ((rc = check_mode(ctx, mode))) return rc;
    if (!w || !vj) return vw_fail(ctx, VW_ENULL, "coefficient buffers cannot be null");
    if ((rc = check_signal_args(ctx, xout, batch, n, ldx))) return rc;
    VwFilt f;
    if ((rc = load_filters(ctx, hs, gs, l, f))) return rc;
    if ((rc = check_levels(ctx, n, l, levels))) return rc;
    if (order != VW_ORDER_SPLIT && order != VW_ORDER_PAIR) return vw_fail(ctx, VW_EINVAL, "unknown synthesis order %d", order);
    if (align)
        for (int j = 0; j < levels; j++) {
            const vw_align &a = align[j];
            if ((a.sigma_h != 1 && a.sigma_h != -1) || (a.sigma_g != 1 && a.sigma_g != -1))
                return vw_fail(ctx, VW_EINVAL, "alignment sigma must be +1 or -1 (level %d)", j + 1);
            if (order == VW_ORDER_PAIR && (a.sigma_h != a.sigma_g || a.tau_h != a.tau_g))
                return vw_fail(ctx, VW_EINVAL, "pair-added synthesis needs identical H and G alignment (level %d)", j + 1);
        }
    if (ldw < n || ldv < n) return vw_fail(ctx, VW_ELENGTH, "coefficient strides shorter than the signal length");
    const bool dev = flags & VW_FLAG_DEVICE_PTRS;
    if (dev) {
        if (flags & VW_FLAG_CHECK_FINITE) {
            if ((rc = check_finite(ctx, vj, batch, n, ldv, "approximation coefficients"))) return rc;
            for (int j = 0; j < levels; j++)
                if ((rc = check_finite(ctx, w + (int64_t)j * level_stride_w, batch, n, ldw, "detail coefficients"))) return rc;
        }
        if ((rc = inverse_device(ctx, w, ldw, level_stride_w, vj, ldv, batch, n, f, l, levels, mode, align, order,
                                 detail_mask, use_approx, xout, ldx, flags, nullptr, 0, 0, 0))) return rc;
        return finish(ctx, flags, false);
    }
    if (ctx->opt_zero_copy > 0 && (double)batch * (double)n * 8.0 * (levels + 2) <= (double)ctx->opt_zero_copy &&
        (levels == 1 || level_stride_w >= (batch - 1) * ldw + n)) {
        const double *wa = (const double *)mapped_alias(w);
        const double *va = wa ? (const double *)mapped_alias(vj) : nullptr;
        double *xa = va ? (double *)mapped_alias(xout) : nullptr;
        if (wa && va && xa) {
            if (flags & VW_FLAG_CHECK_FINITE) {
                if ((rc = check_finite(ctx, va, batch, n, ldv, "approximation coefficients"))) return rc;
                for (int j = 0; j < levels; j++)
                    if ((rc = check_finite(ctx, wa + (int64_t)j * level_stride_w, batch, n, ldw, "detail coefficients"))) return rc;
            }
            if ((rc = inverse_device(ctx, wa, ldw, level_stride_w, va, ldv, batch, n, f, l, levels, mode, align, order, detail_mask,
                                     use_approx, xa, ldx, flags, nullptr, 0, 0, 0))) return rc;
            return finish(ctx, flags, true);
        }
    }
    if (const int64_t rows = pipe_rows(ctx, batch, n, levels))
        return inverse_host_pipelined(ctx, w, ldw, level_stride_w, vj, ldv, batch, n, f, l, levels, mode, align, order,
                                      detail_mask, use_approx, xout, ldx, flags, rows);
    void *px, *pw;
    size_t bn = (size_t)batch * (size_t)n;
    if ((rc = vw_scratch(ctx, 2, bn * 8, &px))) return rc;
    if ((rc = vw_scratch(ctx, 3, bn * 8 * (size_t)(levels + 1), &pw))) return rc;
    double *xd = (double *)px, *wd = (double *)pw, *vd = wd + bn * (size_t)levels;
    for (int j = 0; j < levels; j++)
        if ((rc = copy_rows(ctx, wd + (size_t)j * bn, n, w + (int64_t)j * level_stride_w, ldw, n, batch, cudaMemcpyHostToDevice))) return rc;
    if ((rc = copy_rows(ctx, vd, n, vj, ldv, n, batch, cudaMemcpyHostToDevice))) return rc;
    if (flags & VW_FLAG_CHECK_FINITE)
        if ((rc = check_finite(ctx, wd, (int64_t)(levels + 1) * batch, n, n, "coefficients"))) return rc;
    if ((rc = inverse_device(ctx, wd, n, (int64_t)bn, vd, n, batch, n, f, l, levels, mode, align, order, detail_mask,
                             use_approx, xd, n, flags, nullptr, 0, 0, 0))) return rc;
    if ((rc = copy_rows(ctx, xout, ldx, xd, n, n, batch, cudaMemcpyDeviceToHost))) return rc;
    return finish(ctx, flags, true);
}

// MODWTTransform.forwardBatch / inverseBatch over rows of different lengths: one launch per direction (vw_varlen.cu)
int vw_modwt_forward_varlen(vw_ctx *ctx, const double *x, const int64_t *offsets, int64_t batch, const double *hs,
                            const double *gs, int32_t l, int32_t mode, double *w, double *v, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_modwt_forward_varlen");
    if (int rc0 = no_capture(ctx, "vw_modwt_forward_varlen (host offsets)")) return rc0;
    int rc;
    if ((rc = check_mode(ctx, mode))) return rc;
    if (!x) return vw_fail(ctx, VW_ENULL, "signal cannot be null");
    if (!w || !v) return vw_fail(ctx, VW_ENULL, "output buffers cannot be null");
    int64_t empty;
    if ((rc = check_offsets(ctx, offsets, batch, &empty))) return rc;
    VwFilt f;
    if ((rc = load_filters(ctx, hs, gs, l, f))) return rc;
    const bool dev = flags & VW_FLAG_DEVICE_PTRS, check = flags & VW_FLAG_CHECK_FINITE, exact = flags & VW_FLAG_BITEXACT;
    if (empty < batch) return varlen_empty_row(ctx, x, nullptr, offsets, batch, empty, dev, check, "signal");
    const int64_t total = offsets[batch];
    void *po;
    if ((rc = vw_scratch(ctx, 4, (size_t)(batch + 1) * 8, &po))) return rc;
    int64_t *off_dev = (int64_t *)po;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(off_dev, offsets, (size_t)(batch + 1) * 8, cudaMemcpyHostToDevice, ctx->stream),
                            "offsets copy"))) return rc;
    // rows [b0, b1) of the call, packed at xd / wd / vd
    auto run = [&](const double *xd, double *wd, double *vd, int64_t b0, int64_t b1) -> int {
        const int64_t s0 = offsets[b0], m = offsets[b1] - s0;
        int r;
        if (check && (r = varlen_finite(ctx, xd, nullptr, m, offsets, batch, s0, "signal"))) return r;
        return vw_launch_varlen_analysis(ctx, xd, off_dev + b0, b1 - b0, s0, m, f, l, mode, wd, vd, exact);
    };
    if (dev) {
        if ((rc = run(x, w, v, 0, batch))) return rc;
        return finish(ctx, flags, false);
    }
    if (ctx->opt_zero_copy > 0 && (double)total * 24.0 <= (double)ctx->opt_zero_copy) {
        const double *xa = (const double *)mapped_alias(x);
        double *wa = xa ? (double *)mapped_alias(w) : nullptr, *va = wa ? (double *)mapped_alias(v) : nullptr;
        if (xa && wa && va) {
            if ((rc = run(xa, wa, va, 0, batch))) return rc;
            return finish(ctx, flags, true);
        }
    }
    const std::vector<int64_t> cut = varlen_chunks(ctx, offsets, batch);
    if (cut.size() > 2) {
        int64_t most = 0;
        for (size_t c = 0; c + 1 < cut.size(); c++) most = std::max(most, offsets[cut[c + 1]] - offsets[cut[c]]);
        return run_pipelined(ctx, (int64_t)cut.size() - 1, [&](int64_t c) -> int {
            const int64_t b0 = cut[c], b1 = cut[c + 1], s0 = offsets[b0], m = offsets[b1] - s0;
            void *px, *pw;
            int r;
            if ((r = vw_scratch(ctx, 2, (size_t)most * 8, &px))) return r;
            if ((r = vw_scratch(ctx, 3, (size_t)most * 16, &pw))) return r;
            double *xd = (double *)px, *wd = (double *)pw, *vd = wd + m;
            if ((r = vw_cuda_check(ctx, cudaMemcpyAsync(xd, x + s0, (size_t)m * 8, cudaMemcpyHostToDevice, ctx->stream), "h2d"))) return r;
            if ((r = run(xd, wd, vd, b0, b1))) return r;
            if ((r = vw_cuda_check(ctx, cudaMemcpyAsync(w + s0, wd, (size_t)m * 8, cudaMemcpyDeviceToHost, ctx->stream), "d2h"))) return r;
            return vw_cuda_check(ctx, cudaMemcpyAsync(v + s0, vd, (size_t)m * 8, cudaMemcpyDeviceToHost, ctx->stream), "d2h");
        });
    }
    void *px, *pw;
    if ((rc = vw_scratch(ctx, 2, (size_t)total * 8, &px))) return rc;
    if ((rc = vw_scratch(ctx, 3, (size_t)total * 16, &pw))) return rc;
    double *xd = (double *)px, *wd = (double *)pw, *vd = wd + total;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(xd, x, (size_t)total * 8, cudaMemcpyHostToDevice, ctx->stream), "h2d"))) return rc;
    if ((rc = run(xd, wd, vd, 0, batch))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(w, wd, (size_t)total * 8, cudaMemcpyDeviceToHost, ctx->stream), "d2h"))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(v, vd, (size_t)total * 8, cudaMemcpyDeviceToHost, ctx->stream), "d2h"))) return rc;
    return finish(ctx, flags, true);
}

int vw_modwt_inverse_varlen(vw_ctx *ctx, const double *w, const double *v, const int64_t *offsets, int64_t batch,
                            const double *hs, const double *gs, int32_t l, int32_t mode, double *xout, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_modwt_inverse_varlen");
    if (int rc0 = no_capture(ctx, "vw_modwt_inverse_varlen (host offsets)")) return rc0;
    int rc;
    if ((rc = check_mode(ctx, mode))) return rc;
    if (!w || !v) return vw_fail(ctx, VW_ENULL, "coefficient buffers cannot be null");
    if (!xout) return vw_fail(ctx, VW_ENULL, "output buffer cannot be null");
    int64_t empty;
    if ((rc = check_offsets(ctx, offsets, batch, &empty))) return rc;
    VwFilt f;
    if ((rc = load_filters(ctx, hs, gs, l, f))) return rc;
    const bool dev = flags & VW_FLAG_DEVICE_PTRS, check = flags & VW_FLAG_CHECK_FINITE, exact = flags & VW_FLAG_BITEXACT;
    if (empty < batch) return varlen_empty_row(ctx, w, v, offsets, batch, empty, dev, check, "coefficients");
    const int64_t total = offsets[batch];
    void *po;
    if ((rc = vw_scratch(ctx, 4, (size_t)(batch + 1) * 8, &po))) return rc;
    int64_t *off_dev = (int64_t *)po;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(off_dev, offsets, (size_t)(batch + 1) * 8, cudaMemcpyHostToDevice, ctx->stream),
                            "offsets copy"))) return rc;
    auto run = [&](const double *wd, const double *vd, double *xd, int64_t b0, int64_t b1) -> int {
        const int64_t s0 = offsets[b0], m = offsets[b1] - s0;
        int r;
        if (check && (r = varlen_finite(ctx, wd, vd, m, offsets, batch, s0, "coefficients"))) return r;
        return vw_launch_varlen_synthesis(ctx, vd, wd, off_dev + b0, b1 - b0, s0, m, f, l, mode, xd, exact);
    };
    if (dev) {
        if ((rc = run(w, v, xout, 0, batch))) return rc;
        return finish(ctx, flags, false);
    }
    if (ctx->opt_zero_copy > 0 && (double)total * 24.0 <= (double)ctx->opt_zero_copy) {
        const double *wa = (const double *)mapped_alias(w);
        const double *va = wa ? (const double *)mapped_alias(v) : nullptr;
        double *xa = va ? (double *)mapped_alias(xout) : nullptr;
        if (wa && va && xa) {
            if ((rc = run(wa, va, xa, 0, batch))) return rc;
            return finish(ctx, flags, true);
        }
    }
    const std::vector<int64_t> cut = varlen_chunks(ctx, offsets, batch);
    if (cut.size() > 2) {
        int64_t most = 0;
        for (size_t c = 0; c + 1 < cut.size(); c++) most = std::max(most, offsets[cut[c + 1]] - offsets[cut[c]]);
        return run_pipelined(ctx, (int64_t)cut.size() - 1, [&](int64_t c) -> int {
            const int64_t b0 = cut[c], b1 = cut[c + 1], s0 = offsets[b0], m = offsets[b1] - s0;
            void *px, *pw;
            int r;
            if ((r = vw_scratch(ctx, 2, (size_t)most * 8, &px))) return r;
            if ((r = vw_scratch(ctx, 3, (size_t)most * 16, &pw))) return r;
            double *xd = (double *)px, *wd = (double *)pw, *vd = wd + m;
            if ((r = vw_cuda_check(ctx, cudaMemcpyAsync(wd, w + s0, (size_t)m * 8, cudaMemcpyHostToDevice, ctx->stream), "h2d"))) return r;
            if ((r = vw_cuda_check(ctx, cudaMemcpyAsync(vd, v + s0, (size_t)m * 8, cudaMemcpyHostToDevice, ctx->stream), "h2d"))) return r;
            if ((r = run(wd, vd, xd, b0, b1))) return r;
            return vw_cuda_check(ctx, cudaMemcpyAsync(xout + s0, xd, (size_t)m * 8, cudaMemcpyDeviceToHost, ctx->stream), "d2h");
        });
    }
    void *px, *pw;
    if ((rc = vw_scratch(ctx, 2, (size_t)total * 8, &px))) return rc;
    if ((rc = vw_scratch(ctx, 3, (size_t)total * 16, &pw))) return rc;
    double *xd = (double *)px, *wd = (double *)pw, *vd = wd + total;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(wd, w, (size_t)total * 8, cudaMemcpyHostToDevice, ctx->stream), "h2d"))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(vd, v, (size_t)total * 8, cudaMemcpyHostToDevice, ctx->stream), "h2d"))) return rc;
    if ((rc = run(wd, vd, xd, 0, batch))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(xout, xd, (size_t)total * 8, cudaMemcpyDeviceToHost, ctx->stream), "d2h"))) return rc;
    return finish(ctx, flags, true);
}

int vw_threshold(vw_ctx *ctx, double *coeffs, int64_t batch, int64_t n, int64_t ld, const double *thresholds,
                 int32_t per_row, int32_t soft, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_threshold");
    if (int rc0 = no_capture(ctx, "vw_threshold (host thresholds)")) return rc0;
    int rc;
    if ((rc = check_signal_args(ctx, coeffs, batch, n, ld))) return rc;
    if (!thresholds) return vw_fail(ctx, VW_ENULL, "thresholds cannot be null");
    const bool dev = flags & VW_FLAG_DEVICE_PTRS;
    int64_t nthr = per_row ? batch : 1;
    void *pt;
    if ((rc = vw_scratch(ctx, 5, (size_t)nthr * 8 + 64, &pt))) return rc;
    double *thr_dev = (double *)((char *)pt + 64);
    // thresholds are always read from the host (they come from vw_universal_threshold or the caller)
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(thr_dev, thresholds, (size_t)nthr * 8, cudaMemcpyHostToDevice, ctx->stream), "small copy"))) return rc;
    double *cd = coeffs;
    if (!dev) {
        void *p;
        if ((rc = vw_scratch(ctx, 2, (size_t)batch * (size_t)n * 8, &p))) return rc;
        cd = (double *)p;
        if ((rc = copy_rows(ctx, cd, n, coeffs, ld, n, batch, cudaMemcpyHostToDevice))) return rc;
    }
    if ((rc = vw_launch_threshold(ctx, cd, batch, n, dev ? ld : n, thr_dev, per_row, soft))) return rc;
    if (!dev) if ((rc = copy_rows(ctx, coeffs, ld, cd, n, n, batch, cudaMemcpyDeviceToHost))) return rc;
    return finish(ctx, flags & ~VW_FLAG_NO_SYNC, !dev);  // thresholds buffer is host memory: always complete
}

int vw_universal_threshold(vw_ctx *ctx, const double *w1, int64_t batch, int64_t n, int64_t ld, double *thresholds_out,
                           uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_universal_threshold");
    if (int rc0 = no_capture(ctx, "vw_universal_threshold")) return rc0;
    int rc;
    if ((rc = check_signal_args(ctx, w1, batch, n, ld))) return rc;
    if (!thresholds_out) return vw_fail(ctx, VW_ENULL, "thresholds_out cannot be null");
    const bool dev = flags & VW_FLAG_DEVICE_PTRS;
    const double *wd = w1;
    int64_t ldd = ld;
    if (!dev) {
        void *p;
        if ((rc = vw_scratch(ctx, 2, (size_t)batch * (size_t)n * 8, &p))) return rc;
        if ((rc = copy_rows(ctx, p, n, w1, ld, n, batch, cudaMemcpyHostToDevice))) return rc;
        wd = (const double *)p;
        ldd = n;
    }
    void *pt;
    if ((rc = vw_scratch(ctx, 5, (size_t)batch * 8 + 64, &pt))) return rc;
    double *thr_dev = (double *)((char *)pt + 64);
    if ((rc = vw_launch_universal_threshold(ctx, wd, batch, n, ldd, thr_dev))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(thresholds_out, thr_dev, (size_t)batch * 8, cudaMemcpyDeviceToHost, ctx->stream), "small copy"))) return rc;
    return vw_cuda_check(ctx, cudaStreamSynchronize(ctx->stream), "universal threshold");
}

int vw_swt_denoise(vw_ctx *ctx, const double *x, int64_t batch, int64_t n, int64_t ldx, const double *hs,
                   const double *gs, int32_t l, int32_t levels, int32_t mode, const vw_align *align, int32_t order,
                   double threshold, int32_t soft, double *out, int64_t ldo, double *thresholds_out, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_swt_denoise");
    if (int rc0 = no_capture(ctx, "vw_swt_denoise")) return rc0;
    int rc;
    if ((rc = check_mode(ctx, mode))) return rc;
    if ((rc = check_signal_args(ctx, x, batch, n, ldx))) return rc;
    if ((rc = check_signal_args(ctx, out, batch, n, ldo))) return rc;
    VwFilt f;
    if ((rc = load_filters(ctx, hs, gs, l, f))) return rc;
    if ((rc = check_levels(ctx, n, l, levels))) return rc;
    if (order != VW_ORDER_SPLIT && order != VW_ORDER_PAIR) return vw_fail(ctx, VW_EINVAL, "unknown synthesis order %d", order);
    void *pt;
    if ((rc = vw_scratch(ctx, 5, (size_t)batch * 8 + 64, &pt))) return rc;
    double *thr_dev = (double *)((char *)pt + 64);
    int per_row = 0;
    rc = denoise_chain(ctx, x, batch, n, ldx, f, l, levels, mode, align, order, soft, out, ldo, flags,
                       [&](const double *wd, const double *&thr, int &thr_per_row, int64_t &lstride) -> int {
        if (threshold < 0) {
            per_row = 1;
            if (int r = vw_launch_universal_threshold(ctx, wd, batch, n, n, thr_dev)) return r;
        } else {
            if (int r = vw_cuda_check(ctx, cudaMemcpyAsync(thr_dev, &threshold, 8, cudaMemcpyHostToDevice, ctx->stream), "small copy")) return r;
            cudaStreamSynchronize(ctx->stream);  // &threshold is a stack address
        }
        thr = thr_dev; thr_per_row = per_row; lstride = 0;   // one table for every level
        return VW_OK;
    });
    if (rc) return rc;
    if (thresholds_out) {
        if (per_row) {
            if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(thresholds_out, thr_dev, (size_t)batch * 8, cudaMemcpyDeviceToHost, ctx->stream), "small copy"))) return rc;
        } else {
            for (int64_t b = 0; b < batch; b++) thresholds_out[b] = threshold;
        }
    }
    return vw_cuda_check(ctx, cudaStreamSynchronize(ctx->stream), "denoise");
}

int vw_wavelet_denoise(vw_ctx *ctx, const double *x, int64_t batch, int64_t n, int64_t ldx, const double *hs,
                       const double *gs, int32_t l, int32_t levels, int32_t mode, const vw_align *align, int32_t order,
                       int32_t multilevel, int32_t method, double fixed_threshold, int32_t soft, double *out, int64_t ldo,
                       double *thresholds_out, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_wavelet_denoise");
    if (int rc0 = no_capture(ctx, "vw_wavelet_denoise")) return rc0;
    int rc;
    if ((rc = check_mode(ctx, mode))) return rc;
    if ((rc = check_signal_args(ctx, x, batch, n, ldx))) return rc;
    if ((rc = check_signal_args(ctx, out, batch, n, ldo))) return rc;
    VwFilt f;
    if ((rc = load_filters(ctx, hs, gs, l, f))) return rc;
    if (multilevel != 0 && multilevel != 1) return vw_fail(ctx, VW_EINVAL, "multilevel must be 0 or 1 (got %d)", multilevel);
    if (method < VW_THR_UNIVERSAL || method > VW_THR_FIXED) return vw_fail(ctx, VW_EINVAL, "Unknown threshold selection method %d", method);
    if (!multilevel && levels != 1) return vw_fail(ctx, VW_EINVAL, "single-level denoise takes levels = 1 (got %d)", levels);
    if (multilevel && levels > 31)   // WaveletDenoiser.MAX_SAFE_LEVEL_FOR_SCALING (:57)
        return vw_fail(ctx, VW_ETOOLARGE, "Decomposition level %d exceeds safe limit for scale-dependent thresholds", levels);
    if ((rc = check_levels(ctx, n, l, levels))) return rc;
    if (order != VW_ORDER_SPLIT && order != VW_ORDER_PAIR) return vw_fail(ctx, VW_EINVAL, "unknown synthesis order %d", order);
    if (multilevel && method == VW_THR_FIXED)
        return vw_fail(ctx, VW_EUNSUPPORTED, "Fixed threshold method requires explicit threshold value");
    if (method == VW_THR_SURE && (double)levels * (double)batch * (double)n * (double)n > 17592186044416.0)
        return vw_fail(ctx, VW_EUNSUPPORTED, "SURE scores n candidates against n coefficients (as the reference does): "
                                             "levels * batch * n^2 = %.3g exceeds 2^44",
                       (double)levels * (double)batch * (double)n * (double)n);
    const int64_t jb = (int64_t)levels * batch;
    // slot 5 past the finite check's 64 bytes: med [batch] | thr, sig, mean, var, sure, risk [levels][batch]
    void *pt;
    if ((rc = vw_scratch(ctx, 5, (size_t)(batch + 6 * jb) * 8 + 64, &pt))) return rc;
    double *med = (double *)((char *)pt + 64), *thr_dev = med + batch, *sig = thr_dev + jb, *mean = sig + jb, *var = mean + jb,
           *sure = var + jb, *risk = sure + jb;
    VwDenoiseSel sel;
    vw_denoise_scalars(n, levels, sel);
    sel.med = med; sel.var = var; sel.sure = sure; sel.sig = nullptr; sel.thr = thr_dev;
    sel.batch = batch; sel.levels = levels; sel.method = method; sel.multilevel = multilevel; sel.fixed = fixed_threshold;
    rc = denoise_chain(ctx, x, batch, n, ldx, f, l, levels, mode, align, order, soft, out, ldo, flags,
                       [&](const double *wd, const double *&thr, int &thr_per_row, int64_t &lstride) -> int {
        // W is [levels][batch][n] contiguous: the per-(level, row) statistics are one launch over levels * batch rows
        if (int r = vw_launch_median_abs(ctx, wd, batch, n, n, med)) return r;
        if (method == VW_THR_BAYES)
            if (int r = vw_launch_mean_variance(ctx, wd, jb, n, n, mean, var)) return r;
        if (method == VW_THR_SURE) {
            VwDenoiseSel s = sel;
            s.sig = sig;   // the noise level each row's risk scan scores against
            if (int r = vw_launch_denoise_select(ctx, s)) return r;
            void *ws;
            if (int r = vw_scratch(ctx, 4, vw_sure_workspace(jb, n), &ws)) return r;
            if (int r = vw_launch_sure(ctx, wd, jb, n, n, sig, ws, sure, risk)) return r;
        }
        if (int r = vw_launch_denoise_select(ctx, sel)) return r;
        thr = thr_dev; thr_per_row = 1; lstride = batch;
        return VW_OK;
    });
    if (rc) return rc;
    if (thresholds_out &&
        (rc = vw_cuda_check(ctx, cudaMemcpyAsync(thresholds_out, thr_dev, (size_t)jb * 8, cudaMemcpyDeviceToHost, ctx->stream), "small copy")))
        return rc;
    return vw_cuda_check(ctx, cudaStreamSynchronize(ctx->stream), "denoise");
}

int vw_median_abs(vw_ctx *ctx, const double *c, int64_t batch, int64_t n, int64_t ld, double *out, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_median_abs");
    if (int rc0 = no_capture(ctx, "vw_median_abs")) return rc0;
    int rc;
    if ((rc = check_signal_args(ctx, c, batch, n, ld))) return rc;
    if (!out) return vw_fail(ctx, VW_ENULL, "out cannot be null");
    const double *cd = c;
    int64_t ldd = ld;
    if (!(flags & VW_FLAG_DEVICE_PTRS)) {
        void *p;
        if ((rc = vw_scratch(ctx, 2, (size_t)batch * (size_t)n * 8, &p))) return rc;
        if ((rc = copy_rows(ctx, p, n, c, ld, n, batch, cudaMemcpyHostToDevice))) return rc;
        cd = (const double *)p; ldd = n;
    }
    void *pt;
    if ((rc = vw_scratch(ctx, 5, (size_t)batch * 8 + 64, &pt))) return rc;
    double *med = (double *)((char *)pt + 64);
    if ((rc = vw_launch_median_abs(ctx, cd, batch, n, ldd, med))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(out, med, (size_t)batch * 8, cudaMemcpyDeviceToHost, ctx->stream), "small copy"))) return rc;
    return vw_cuda_check(ctx, cudaStreamSynchronize(ctx->stream), "median");
}

int vw_mean_variance(vw_ctx *ctx, const double *c, int64_t batch, int64_t n, int64_t ld, double *mean_out, double *var_out,
                     uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_mean_variance");
    if (int rc0 = no_capture(ctx, "vw_mean_variance")) return rc0;
    int rc;
    if ((rc = check_signal_args(ctx, c, batch, n, ld))) return rc;
    if (!mean_out || !var_out) return vw_fail(ctx, VW_ENULL, "out cannot be null");
    const double *cd = c;
    int64_t ldd = ld;
    if (!(flags & VW_FLAG_DEVICE_PTRS)) {
        void *p;
        if ((rc = vw_scratch(ctx, 2, (size_t)batch * (size_t)n * 8, &p))) return rc;
        if ((rc = copy_rows(ctx, p, n, c, ld, n, batch, cudaMemcpyHostToDevice))) return rc;
        cd = (const double *)p; ldd = n;
    }
    void *pt;
    if ((rc = vw_scratch(ctx, 5, (size_t)batch * 16 + 64, &pt))) return rc;
    double *md = (double *)((char *)pt + 64), *vd = md + batch;
    if ((rc = vw_launch_mean_variance(ctx, cd, batch, n, ldd, md, vd))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(mean_out, md, (size_t)batch * 8, cudaMemcpyDeviceToHost, ctx->stream), "small copy"))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(var_out, vd, (size_t)batch * 8, cudaMemcpyDeviceToHost, ctx->stream), "small copy"))) return rc;
    return vw_cuda_check(ctx, cudaStreamSynchronize(ctx->stream), "mean/variance");
}

int vw_sure_threshold(vw_ctx *ctx, const double *c, int64_t batch, int64_t n, int64_t ld, const double *sigma,
                      double *thr_out, double *risk_out, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_sure_threshold");
    if (int rc0 = no_capture(ctx, "vw_sure_threshold")) return rc0;
    int rc;
    if ((rc = check_signal_args(ctx, c, batch, n, ld))) return rc;
    if (!sigma || !thr_out) return vw_fail(ctx, VW_ENULL, "sigma and thr_out cannot be null");
    if ((double)batch * (double)n * (double)n > 17592186044416.0)   // 2^44 candidate x coefficient pairs, a few seconds
        return vw_fail(ctx, VW_EUNSUPPORTED, "SURE scores n candidates against n coefficients (as the reference does): "
                                             "batch * n^2 = %.3g exceeds 2^44", (double)batch * (double)n * (double)n);
    const double *cd = c;
    int64_t ldd = ld;
    if (!(flags & VW_FLAG_DEVICE_PTRS)) {
        void *p;
        if ((rc = vw_scratch(ctx, 2, (size_t)batch * (size_t)n * 8, &p))) return rc;
        if ((rc = copy_rows(ctx, p, n, c, ld, n, batch, cudaMemcpyHostToDevice))) return rc;
        cd = (const double *)p; ldd = n;
    }
    void *pt, *ws;
    if ((rc = vw_scratch(ctx, 5, (size_t)batch * 24 + 64, &pt))) return rc;
    if ((rc = vw_scratch(ctx, 4, vw_sure_workspace(batch, n), &ws))) return rc;
    double *sd = (double *)((char *)pt + 64), *td = sd + batch, *rd = td + batch;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(sd, sigma, (size_t)batch * 8, cudaMemcpyHostToDevice, ctx->stream), "sigma copy")))
        return rc;
    if ((rc = vw_launch_sure(ctx, cd, batch, n, ldd, sd, ws, td, rd))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(thr_out, td, (size_t)batch * 8, cudaMemcpyDeviceToHost, ctx->stream), "small copy"))) return rc;
    if (risk_out && (rc = vw_cuda_check(ctx, cudaMemcpyAsync(risk_out, rd, (size_t)batch * 8, cudaMemcpyDeviceToHost, ctx->stream), "small copy"))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaStreamSynchronize(ctx->stream), "sure"))) return rc;
    const double root = sqrt(2.0 * log((double)n));
    for (int64_t b = 0; b < batch; b++) {                           // :465-469 compare with the universal threshold
        const double universal = sigma[b] * root;
        if (thr_out[b] > universal) thr_out[b] = universal;
    }
    return VW_OK;
}

int vw_energy(vw_ctx *ctx, const double *c, int64_t batch, int64_t n, int64_t ld, double *out, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_energy");
    if (int rc0 = no_capture(ctx, "vw_energy")) return rc0;
    int rc;
    if ((rc = check_signal_args(ctx, c, batch, n, ld))) return rc;
    if (!out) return vw_fail(ctx, VW_ENULL, "out cannot be null");
    const bool dev = flags & VW_FLAG_DEVICE_PTRS;
    const double *cd = c;
    int64_t ldd = ld;
    if (!dev) {
        void *p;
        if ((rc = vw_scratch(ctx, 2, (size_t)batch * (size_t)n * 8, &p))) return rc;
        if ((rc = copy_rows(ctx, p, n, c, ld, n, batch, cudaMemcpyHostToDevice))) return rc;
        cd = (const double *)p; ldd = n;
    }
    void *pe;
    if ((rc = vw_scratch(ctx, 5, (size_t)batch * 8 + 64, &pe))) return rc;
    double *ed = (double *)((char *)pe + 64);
    if ((rc = vw_launch_energy(ctx, cd, batch, n, ldd, ed))) return rc;
    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(out, ed, (size_t)batch * 8, cudaMemcpyDeviceToHost, ctx->stream), "small copy"))) return rc;
    return vw_cuda_check(ctx, cudaStreamSynchronize(ctx->stream), "energy");
}

int vw_modwt_forward_span(vw_ctx *ctx, const double *vin, int64_t halo, int64_t n_local, const double *hs,
                          const double *gs, int32_t l, int32_t first_level, int32_t nlevels, double *w,
                          int64_t level_stride_w, double *vout, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_modwt_forward_span");
    ctx->plan_lean_ok = true;
    int rc;
    if (!(flags & VW_FLAG_DEVICE_PTRS)) return vw_fail(ctx, VW_EUNSUPPORTED, "span calls take device pointers only");
    if (!vin || !w || !vout) return vw_fail(ctx, VW_ENULL, "span buffers cannot be null");
    if (n_local < 1) return vw_fail(ctx, VW_EEMPTY, "span cannot be empty");
    VwFilt f;
    if ((rc = load_filters(ctx, hs, gs, l, f))) return rc;
    int64_t need = vw_span_halo(l, first_level, nlevels);
    if (need < 0) return vw_fail(ctx, VW_ELEVEL, "invalid level group [%d, %d)", first_level, first_level + nlevels);
    if (halo < need) return vw_fail(ctx, VW_ELENGTH, "halo %lld shorter than the %lld samples levels %d..%d need",
                                    (long long)halo, (long long)need, first_level, first_level + nlevels - 1);
    const bool exact = flags & VW_FLAG_BITEXACT;
    const int64_t n_in = halo + n_local;
    rc = VW_EUNSUPPORTED;
    // same kernel choice as the unsharded path: a single level at or above the column threshold runs on the column kernel
    const bool column_first = nlevels == 1 && first_level >= vw_column_min_level(ctx, l) && ctx->opt_poly != 0;
    if (!exact && !(flags & VW_FLAG_NO_FUSE) && nlevels == 2 && first_level >= vw_column_min_level(ctx, l) && ctx->opt_poly != 0) {
        rc = vw_column_analysis2(ctx, vin, 0, w, 0, w + level_stride_w, 0, vout, 0, n_in, halo, n_local, 1, f, l,
                                 (int64_t)1 << (first_level - 1), VW_MODE_LINEAR);
        if (rc != VW_OK && rc != VW_EUNSUPPORTED) return rc;
    }
    if (rc == VW_EUNSUPPORTED && !exact && !(flags & VW_FLAG_NO_FUSE) && !column_first) {
        VwFusedFwd p{vin, n_in, w, n_local, level_stride_w, vout, n_local, 1, n_in, halo, n_local,
                     l, first_level, nlevels, VW_MODE_LINEAR, 0};
        rc = vw_fused_forward(ctx, p, f);
        if (rc != VW_OK && rc != VW_EUNSUPPORTED) return rc;
    }
    if (rc == VW_EUNSUPPORTED) {
        // per-level: level i of the group must be produced on [halo - rem_i, n_in) where rem_i is the halo
        // the later levels of the group still need
        double *buf[2] = {nullptr, nullptr};
        const double *cur = vin;
        int64_t cur_off = 0;  // cur[0] is input position cur_off
        for (int i = 0; i < nlevels; i++) {
            int level = first_level + i;
            int64_t d = (int64_t)1 << (level - 1);
            int64_t rem = (i + 1 < nlevels) ? vw_span_halo(l, level + 1, nlevels - i - 1) : 0;
            int64_t start = halo - rem;  // first position produced at this level
            bool last = i + 1 == nlevels;
            double *vdst;
            if (last) vdst = vout;
            else {
                void *p;
                if ((rc = vw_scratch(ctx, i & 1, (size_t)n_in * 8, &p))) return rc;
                buf[i & 1] = (double *)p;
                vdst = buf[i & 1];
            }
            // analysis over input coords: in = cur (position cur_off at index 0), outputs [start, n_in)
            // W rows only exist for the span: write them via a second launch restricted to [halo, n_in)
            rc = VW_EUNSUPPORTED;
            if (last && nlevels == 1 && !exact && !(flags & VW_FLAG_NO_FUSE) && d >= ((int64_t)1 << (vw_column_min_level(ctx, l) - 1)) && ctx->opt_poly != 0) {
                rc = vw_column_analysis(ctx, cur, 0, vout, 0, w, 0, n_in, halo, n_local, 1, f, l, d, VW_MODE_LINEAR);
                if (rc != VW_OK && rc != VW_EUNSUPPORTED) return rc;
            }
            if (rc == VW_EUNSUPPORTED)
                rc = vw_launch_analysis_level(ctx, cur, 0, last ? vout : vdst, 0, last ? w + (int64_t)i * level_stride_w : nullptr,
                                              0, n_in - cur_off, (last ? halo : start) - cur_off, last ? n_local : n_in - start,
                                              1, f, l, d, VW_MODE_LINEAR, exact);
            if (rc) return rc;
            if (!last) {
                rc = vw_launch_analysis_level(ctx, cur, 0, nullptr, 0, w + (int64_t)i * level_stride_w, 0, n_in - cur_off,
                                              halo - cur_off, n_local, 1, f, l, d, VW_MODE_LINEAR, exact);
                if (rc) return rc;
                cur = vdst;
                cur_off = start;
            }
        }
    }
    return finish(ctx, flags, false);
}

int vw_modwt_stream_level(vw_ctx *ctx, const double *vin, int64_t batch, int64_t ldin, int64_t hist, int64_t n,
                          const double *hs, const double *gs, int32_t l, int32_t level, double *w, int64_t ldw,
                          double *v, int64_t ldv, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_modwt_stream_level");
    ctx->plan_lean_ok = true;
    int rc;
    if (!(flags & VW_FLAG_DEVICE_PTRS)) return vw_fail(ctx, VW_EUNSUPPORTED, "streaming calls take device pointers only");
    if (!vin || !w || !v) return vw_fail(ctx, VW_ENULL, "stream buffers cannot be null");
    if (batch < 1) return vw_fail(ctx, VW_ELENGTH, "block must be non-null (batch=%lld)", (long long)batch);
    if (n < 1) return vw_fail(ctx, VW_EEMPTY, "block length must be > 0");
    if (level < 1 || level > 30) return vw_fail(ctx, VW_ELEVEL, "Invalid level: %d", level);
    VwFilt f;
    if ((rc = load_filters(ctx, hs, gs, l, f))) return rc;
    const int64_t d = (int64_t)1 << (level - 1);
    const int64_t need = (int64_t)(l - 1) * d;
    if (hist < need) return vw_fail(ctx, VW_ELENGTH, "history %lld shorter than the %lld samples level %d needs",
                                    (long long)hist, (long long)need, level);
    if (ldin < hist + n || ldw < n || ldv < n) return vw_fail(ctx, VW_ELENGTH, "row stride shorter than the row");
    if ((rc = stream_level_device(ctx, vin, batch, ldin, hist, n, f, l, level, w, ldw, v, ldv, flags))) return rc;
    return finish(ctx, flags, false);
}

int vw_modwt_inverse_span(vw_ctx *ctx, const double *vin, const double *w, int64_t level_stride_w, int64_t halo,
                          int64_t n_local, const double *hs, const double *gs, int32_t l, int32_t first_level,
                          int32_t nlevels, int32_t order, double *vout, uint32_t flags) {
    return vwshim::inverse_span_device(ctx, vin, w, level_stride_w, halo, n_local, hs, gs, l, first_level, nlevels, order, vout,
                                       flags, nullptr, 0);
}

}  // extern "C"

namespace vwshim {
// vw_modwt_inverse_span, optionally with one threshold (device scalar) applied to every W sample the group reads, halo
// included: the tile, column and column-pair kernels threshold on load; the per-level kernels have no such form, so each
// level's W row is thresholded into a scratch copy first (the caller's W stays as it is)
int inverse_span_device(vw_ctx *ctx, const double *vin, const double *w, int64_t level_stride_w, int64_t halo, int64_t n_local,
                        const double *hs, const double *gs, int32_t l, int32_t first_level, int32_t nlevels, int32_t order,
                        double *vout, uint32_t flags, const double *thr_dev, int32_t thr_soft) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_modwt_inverse_span");
    ctx->plan_lean_ok = true;
    int rc;
    if (!(flags & VW_FLAG_DEVICE_PTRS)) return vw_fail(ctx, VW_EUNSUPPORTED, "span calls take device pointers only");
    if (!vin || !w || !vout) return vw_fail(ctx, VW_ENULL, "span buffers cannot be null");
    if (n_local < 1) return vw_fail(ctx, VW_EEMPTY, "span cannot be empty");
    VwFilt f;
    if ((rc = load_filters(ctx, hs, gs, l, f))) return rc;
    int64_t need = vw_span_halo(l, first_level, nlevels);
    if (need < 0) return vw_fail(ctx, VW_ELEVEL, "invalid level group [%d, %d)", first_level, first_level + nlevels);
    if (halo < need) return vw_fail(ctx, VW_ELENGTH, "halo %lld shorter than the %lld samples levels %d..%d need",
                                    (long long)halo, (long long)need, first_level, first_level + nlevels - 1);
    const bool exact = flags & VW_FLAG_BITEXACT;
    const int64_t n_in = halo + n_local;
    rc = VW_EUNSUPPORTED;
    const bool column_first = nlevels == 1 && first_level >= vw_column_min_level(ctx, l, false) && ctx->opt_poly != 0;
    if (!exact && !(flags & VW_FLAG_NO_FUSE) && nlevels == 2 && first_level >= vw_column_min_level(ctx, l, false) && ctx->opt_poly != 0) {
        rc = vw_column_synthesis2(ctx, vin, 0, w + level_stride_w, 0, w, 0, vout, 0, n_in, 0, n_local, 1, f, l,
                                  (int64_t)1 << (first_level - 1), VW_MODE_LINEAR, thr_dev, 0, thr_soft, 0);
        if (rc != VW_OK && rc != VW_EUNSUPPORTED) return rc;
    }
    if (rc == VW_EUNSUPPORTED && !exact && !(flags & VW_FLAG_NO_FUSE) && !column_first) {
        VwFusedInv p{vin, n_in, w, n_in, level_stride_w, nlevels >= 64 ? ~0ull : ((1ull << nlevels) - 1), vout, n_local,
                     1, n_in, n_local, l, first_level, nlevels, VW_MODE_LINEAR, thr_dev, 0, thr_soft, 0};
        rc = vw_fused_inverse(ctx, p, f);
        if (rc != VW_OK && rc != VW_EUNSUPPORTED) return rc;
    }
    if (rc == VW_EUNSUPPORTED) {
        // per-level, top of the group first; level j output must cover [0, n_local + halo of the levels below)
        const double *cur = vin;
        for (int i = nlevels - 1; i >= 0; i--) {
            int level = first_level + i;
            int64_t d = (int64_t)1 << (level - 1);
            int64_t below = i > 0 ? vw_span_halo(l, first_level, i) : 0;
            int64_t n_out = n_local + below;
            double *dst = vout;
            if (i > 0) {
                void *p;
                if ((rc = vw_scratch(ctx, i & 1, (size_t)n_in * 8, &p))) return rc;
                dst = (double *)p;
            }
            rc = VW_EUNSUPPORTED;
            if (nlevels == 1 && !exact && !(flags & VW_FLAG_NO_FUSE) && d >= ((int64_t)1 << (vw_column_min_level(ctx, l, false) - 1)) && ctx->opt_poly != 0) {
                rc = vw_column_synthesis(ctx, cur, 0, w, 0, dst, 0, n_in, 0, n_out, 1, f, l, d, VW_MODE_LINEAR, default_align(), thr_dev,
                                         0, thr_soft);
                if (rc != VW_OK && rc != VW_EUNSUPPORTED) return rc;
            }
            if (rc == VW_EUNSUPPORTED) {
                const double *wj = w + (int64_t)i * level_stride_w;
                if (thr_dev) {
                    void *p;
                    if ((rc = vw_scratch(ctx, 4, (size_t)n_in * 8, &p))) return rc;
                    if ((rc = vw_cuda_check(ctx, cudaMemcpyAsync(p, wj, (size_t)n_in * 8, cudaMemcpyDeviceToDevice, ctx->stream), "d2d")))
                        return rc;
                    if ((rc = vw_launch_threshold(ctx, (double *)p, 1, n_in, n_in, thr_dev, 0, thr_soft))) return rc;
                    wj = (const double *)p;
                }
                rc = vw_launch_synthesis_level(ctx, cur, 0, wj, 0, dst, 0, n_in, 0, n_out, 1, f, l, d, VW_MODE_LINEAR, default_align(),
                                               order == VW_ORDER_PAIR, exact);
            }
            if (rc) return rc;
            cur = dst;
        }
    }
    return finish(ctx, flags, false);
}
}  // namespace vwshim
