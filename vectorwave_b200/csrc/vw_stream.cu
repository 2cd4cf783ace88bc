// vw_stream.cu -- BatchStreamingMODWT below the C ABI (EXT/extensions/modwt/BatchStreamingMODWT.java:55-276): a handle
// keeps every level's left history in HBM, and one call runs a block's whole cascade.
//
// Histories: level j keeps H_j = (l-1)*2^(j-1) samples per row, [batch][H_j] at hist + batch*(l-1)*(2^(j-1)-1).
//
// Fused path (k_stream): one CTA per row runs all J levels in shared memory.  Two buffers of H_J + n doubles take turns:
// level j holds [history_j | input_j] in one, reads its history from HBM (or builds it from the block on the first
// block, or builds the flush tail from the level-1 history), computes exactly n outputs, writes W_j to HBM and V_j into
// the block part of the other buffer (level j+1's input), and writes its new history -- the last H_j samples of
// [history_j | input_j] -- back in place: a row's histories belong to one CTA, so nothing races.  HBM traffic: the block
// in, W_1..W_J and V_J out, and the histories in and out: 8*(J+2) bytes per sample plus 16*sum(H_j) per row.  Taps run
// ascending with V and W in separate accumulators; EXACT rounds every product and sum separately in the reference's
// order, bit for bit with the JVM.
//
// Per-level path: rows whose two buffers do not fit one CTA's shared memory, filter lengths without a compiled kernel,
// pairs that are not quadrature mirrors and VW_FLAG_NO_FUSE run level by level on the kernels of vw_modwt_stream_level
// over handle-owned [history | block] rows; the history copies are 2-D async copies and the first-block / tail fills
// one small kernel.
#include <string.h>

#include <algorithm>

#include "vw_internal.cuh"

using namespace vwshim;

struct vw_stream_state {
    int device = 0;
    int l = 0, levels = 0, mode = 0;
    bool qmf = false;
    VwFilt f;
    int64_t batch = -1;                          // rows of the running stream; -1: no block since create / reset
    double *hist = nullptr;                      // every level's history (layout above)
    size_t hist_bytes = 0;
    double *ext = nullptr;                       // per-level path: two [batch][ld] work buffers
    size_t ext_bytes = 0;
};

namespace {

constexpr int kMaxThreads = 512;

__device__ __forceinline__ int mirror(int i, int n) {   // CORE/util/MathUtils.java:30-51, i < 0 here
    const int p = 2 * n;
    i %= p;
    if (i < 0) i += p;
    return i < n ? i : p - 1 - i;
}

template <bool EXACT>
__device__ __forceinline__ double mac(double acc, double a, double b) {
    if (EXACT) return __dadd_rn(acc, __dmul_rn(a, b));
    return fma(a, b, acc);
}

struct VwStreamArgs {
    const double *x; int64_t ldx;        // level-1 block [batch][n]; nullptr: flush, the tail comes from the level-1 history
    double *hist;
    double *w; int64_t ldw, lsw;
    double *v; int64_t ldv;
    int64_t batch;
    int n, levels, mode;
    int init;                            // first block: every history is built from the level's own input
    int update;                          // advance the histories (0: flush)
};

template <int L, bool EXACT>
__global__ void __launch_bounds__(kMaxThreads)
k_stream(const VwStreamArgs a, const __grid_constant__ VwFilt32 f) {
    extern __shared__ double smem[];
    const int64_t b = blockIdx.x;
    const int n = a.n, nt = blockDim.x, tid = threadIdx.x;
    double *cur = smem, *nxt = smem + ((L - 1) << (a.levels - 1)) + n;
    double *hist = a.hist;
    for (int j = 1; j <= a.levels; j++) {
        const int d = 1 << (j - 1), H = (L - 1) * d;
        double *hrow = hist + b * H;
        if (j == 1 && a.x) {
            const double *xrow = a.x + b * a.ldx;
            for (int t = tid; t < n; t += nt) cur[H + t] = xrow[t];
        }
        if (!a.init)
            for (int i = tid; i < H; i += nt) cur[i] = hrow[i];
        __syncthreads();
        if (a.init) {          // zeros, or the input reflected about its left edge (:326-334)
            for (int i = tid; i < H; i += nt) cur[i] = a.mode == VW_ZERO_PADDING ? 0.0 : cur[H + mirror(i - H, n)];
            __syncthreads();
        } else if (j == 1 && !a.x) {   // flush tail: zeros, or the level-1 history reversed (:358-372)
            for (int t = tid; t < n; t += nt) cur[H + t] = a.mode == VW_ZERO_PADDING ? 0.0 : cur[H - 1 - t];
            __syncthreads();
        }
        double *wrow = a.w + (int64_t)(j - 1) * a.lsw + b * a.ldw;
        double *vrow = j < a.levels ? nxt + 2 * H : a.v + b * a.ldv;   // next level's block part, or V_J
#pragma unroll 1
        for (int t = tid; t < n; t += nt) {
            const double *s = cur + H + t;
            double av = 0.0, aw = 0.0;
#pragma unroll
            for (int k = 0; k < L; k++) {
                const double xv = s[-k * d];
                av = mac<EXACT>(av, xv, f.h[k]);
                aw = mac<EXACT>(aw, xv, vw_tap_g<L, true>(f, k));
            }
            wrow[t] = aw;
            vrow[t] = av;
        }
        if (a.update)          // the last H samples of [history | input] (:336-350)
            for (int i = tid; i < H; i += nt) hrow[i] = cur[n + i];
        __syncthreads();
        hist += a.batch * H;
        double *tmp = cur; cur = nxt; nxt = tmp;
    }
}

// per-level path: rows e[b] = [history (H) | block (n)] of stride ld.  init: history from the block (zeros / mirror);
// else the flush tail: block from the history (zeros / reversed)
__global__ void __launch_bounds__(256)
k_stream_fill(double *e, int64_t ld, int64_t batch, int64_t H, int64_t n, int mode, int init) {
    const int64_t cnt = init ? H : n, tot = batch * cnt;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < tot; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = q / cnt, i = q - b * cnt;
        double *r = e + b * ld;
        if (init) {
            int64_t m = (i - H) % (2 * n);
            if (m < 0) m += 2 * n;
            r[i] = mode == VW_ZERO_PADDING ? 0.0 : r[H + (m < n ? m : 2 * n - 1 - m)];
        } else {
            r[H + i] = mode == VW_ZERO_PADDING ? 0.0 : r[H - 1 - i];
        }
    }
}

int launch_fill(vw_ctx *ctx, double *e, int64_t ld, int64_t batch, int64_t H, int64_t n, int mode, bool init) {
    const int64_t tot = batch * (init ? H : n);
    if (tot <= 0) return VW_OK;
    const int64_t blocks = std::min<int64_t>((tot + 255) / 256, (int64_t)ctx->sm_count * 8);
    k_stream_fill<<<(unsigned)blocks, 256, 0, ctx->stream>>>(e, ld, batch, H, n, mode, init);
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "stream fill launch");
}

int64_t hist_len(const vw_stream_state *st, int j) { return (int64_t)(st->l - 1) << (j - 1); }
int64_t hist_offset(const vw_stream_state *st, int j) { return st->batch * (int64_t)(st->l - 1) * (((int64_t)1 << (j - 1)) - 1); }

size_t fused_smem(int l, int levels, int64_t n) { return (size_t)(2 * (((int64_t)(l - 1) << (levels - 1)) + n)) * 8; }

bool compiled_length(int l) {
    switch (l) {
        case 2: case 4: case 6: case 8: case 10: case 12: case 16: case 18: case 20: case 30: return true;
        default: return false;
    }
}

// the compile-time filter lengths of vw_varlen.cu
#define VW_STREAM_DISPATCH(CALL)      \
    switch (st->l) {                  \
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
        default: return VW_EUNSUPPORTED; \
    }

int launch_fused(vw_ctx *ctx, const vw_stream_state *st, const VwStreamArgs &a, bool exact) {
    VwFilt32 f32;
    memset(&f32, 0, sizeof f32);
    memcpy(f32.h, st->f.h, sizeof(double) * st->l);
    const size_t smem = fused_smem(st->l, st->levels, a.n);
    const int nt = (int)std::min<int64_t>(kMaxThreads, std::max<int64_t>(128, (a.n + 127) / 128 * 128));
    int rc = VW_OK;
#define VW_SK(LC)                                                                                                      \
    {                                                                                                                  \
        auto kern = exact ? k_stream<LC, true> : k_stream<LC, false>;                                                 \
        if (smem > 48 * 1024 &&                                                                                        \
            (rc = vw_cuda_check(ctx, cudaFuncSetAttribute((const void *)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                                          (int)smem), "cudaFuncSetAttribute(stream smem)")))            \
            return rc;                                                                                                 \
        kern<<<(unsigned)a.batch, nt, smem, ctx->stream>>>(a, f32);                                                    \
    }
    VW_STREAM_DISPATCH(VW_SK)
#undef VW_SK
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "stream cascade launch");
}

// The fused kernel takes a row when its two level buffers fit one CTA's shared memory, the filter length is compiled and
// the pair is a quadrature mirror (every orthogonal wavelet of the reference): it reads only the low-pass taps.
bool use_fused(const vw_ctx *ctx, const vw_stream_state *st, int64_t n, uint32_t flags) {
    if ((flags & VW_FLAG_NO_FUSE) || !st->qmf || !compiled_length(st->l) || st->batch >= ((int64_t)1 << 31)) return false;
    return fused_smem(st->l, st->levels, n) <= ctx->smem_optin;
}

int grow(vw_ctx *ctx, double *&p, size_t &cap, size_t bytes, const char *what) {
    if (cap >= bytes) return VW_OK;
    if (p) {
        cudaStreamSynchronize(ctx->stream);
        cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    int rc = vw_cuda_check(ctx, cudaMalloc((void **)&p, bytes), what);
    if (rc) return rc;
    cap = bytes;
    return VW_OK;
}

// One block (x != nullptr) or the flush tail (x == nullptr) through every level.  Device pointers; st->batch is set.
int cascade(vw_ctx *ctx, vw_stream_state *st, const double *x, int64_t ldx, int64_t n, double *w, int64_t ldw, int64_t lsw,
            double *v, int64_t ldv, bool init, uint32_t flags) {
    const bool exact = flags & VW_FLAG_BITEXACT, update = x != nullptr;
    const int64_t batch = st->batch;
    if (use_fused(ctx, st, n, flags)) {
        VwStreamArgs a{x, ldx, st->hist, w, ldw, lsw, v, ldv, batch, (int)n, st->levels, st->mode, init, update};
        int rc = launch_fused(ctx, st, a, exact);
        if (rc != VW_EUNSUPPORTED) return rc;
    }
    // per-level: ping-pong [history | block] rows, even stride (16-byte aligned rows for the tile kernels' bulk copies)
    auto ld_of = [&](int j) { const int64_t r = hist_len(st, j) + n; return r + (r & 1); };
    const int64_t ldmax = ld_of(st->levels);
    int rc = grow(ctx, st->ext, st->ext_bytes, (size_t)batch * (size_t)ldmax * 16, "stream work buffers");
    if (rc) return rc;
    double *buf[2] = {st->ext, st->ext + (size_t)batch * (size_t)ldmax};
    for (int j = 1; j <= st->levels; j++) {
        const int64_t H = hist_len(st, j), ld = ld_of(j);
        double *e = buf[(j - 1) & 1], *hrow = st->hist + hist_offset(st, j);
        if (j == 1 && x)
            if ((rc = copy_rows(ctx, e + H, ld, x, ldx, n, batch, cudaMemcpyDeviceToDevice))) return rc;
        if (init) rc = launch_fill(ctx, e, ld, batch, H, n, st->mode, true);
        else rc = copy_rows(ctx, e, ld, hrow, H, H, batch, cudaMemcpyDeviceToDevice);
        if (rc) return rc;
        if (j == 1 && !x && (rc = launch_fill(ctx, e, ld, batch, H, n, st->mode, false))) return rc;
        double *vout = v;
        int64_t ldvout = ldv;
        if (j < st->levels) { vout = buf[j & 1] + hist_len(st, j + 1); ldvout = ld_of(j + 1); }
        if ((rc = stream_level_device(ctx, e, batch, ld, H, n, st->f, st->l, j, w + (int64_t)(j - 1) * lsw, ldw, vout, ldvout,
                                      flags)))
            return rc;
        if (update && (rc = copy_rows(ctx, hrow, H, e + n, ld, H, batch, cudaMemcpyDeviceToDevice))) return rc;
    }
    return VW_OK;
}

int check_handle(vw_ctx *ctx, const vw_stream_state *st) {
    if (!st) return vw_fail(ctx, VW_ENULL, "stream state cannot be null");
    if (st->device != ctx->device)
        return vw_fail(ctx, VW_EINVAL, "stream state belongs to device %d, the context to device %d", st->device, ctx->device);
    return VW_OK;
}

int check_outputs(vw_ctx *ctx, const vw_stream_state *st, const double *w, int64_t ldw, int64_t lsw, const double *v,
                  int64_t ldv, int64_t batch, int64_t n) {
    if (!w || !v) return vw_fail(ctx, VW_ENULL, "output buffers cannot be null");
    if (ldw < n || ldv < n || (st->levels > 1 && lsw < (batch - 1) * ldw + n))
        return vw_fail(ctx, VW_ELENGTH, "output strides too small for [levels][batch][n]");
    return VW_OK;
}

// device outputs, or host outputs staged through scratch slot 3 and copied back after the cascade
template <class Run>
int with_outputs(vw_ctx *ctx, const vw_stream_state *st, int64_t batch, int64_t n, double *w, int64_t ldw, int64_t lsw,
                 double *v, int64_t ldv, uint32_t flags, Run run) {
    const bool dev = flags & VW_FLAG_DEVICE_PTRS;
    int rc;
    if (dev) {
        if ((rc = run(w, ldw, lsw, v, ldv))) return rc;
        return finish(ctx, flags, false);
    }
    const size_t bn = (size_t)batch * (size_t)n;
    void *pw;
    if ((rc = vw_scratch(ctx, 3, bn * 8 * (size_t)(st->levels + 1), &pw))) return rc;
    double *wd = (double *)pw, *vd = wd + bn * (size_t)st->levels;
    if ((rc = run(wd, n, (int64_t)bn, vd, n))) return rc;
    for (int j = 0; j < st->levels; j++)
        if ((rc = copy_rows(ctx, w + (int64_t)j * lsw, ldw, wd + (size_t)j * bn, n, n, batch, cudaMemcpyDeviceToHost))) return rc;
    if ((rc = copy_rows(ctx, v, ldv, vd, n, n, batch, cudaMemcpyDeviceToHost))) return rc;
    return finish(ctx, flags, true);
}

}  // namespace

extern "C" {

int vw_stream_create(vw_ctx *ctx, const double *hs, const double *gs, int32_t l, int32_t levels, int32_t mode,
                     vw_stream_state **out) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_stream_create");
    if (!out) return vw_fail(ctx, VW_ENULL, "output handle pointer cannot be null");
    if (mode != VW_ZERO_PADDING && mode != VW_SYMMETRIC)
        return vw_fail(ctx, VW_EBOUNDARY, "stream state supports ZERO_PADDING and SYMMETRIC (PERIODIC streaming is stateless), got %d",
                       mode);
    if (levels < 1 || levels > 30) return vw_fail(ctx, VW_ELEVEL, "Invalid number of decomposition levels: %d", levels);
    VwFilt f;
    if (int rc = load_filters(ctx, hs, gs, l, f)) return rc;
    if (l < 2) return vw_fail(ctx, VW_EINVAL, "filter length %d: streaming needs at least 2 taps", l);
    vw_stream_state *st = new vw_stream_state;
    st->device = ctx->device;
    st->l = l;
    st->levels = levels;
    st->mode = mode;
    st->qmf = vw_is_qmf(hs, gs, l);
    st->f = f;
    *out = st;
    return VW_OK;
}

int vw_stream_destroy(vw_ctx *ctx, vw_stream_state *st) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_stream_destroy");
    if (!st) return VW_OK;
    if (int rc = check_handle(ctx, st)) return rc;
    cudaStreamSynchronize(ctx->stream);
    cudaError_t e = cudaSuccess;
    if (st->hist) e = cudaFree(st->hist);
    if (st->ext && e == cudaSuccess) e = cudaFree(st->ext);
    delete st;
    return vw_cuda_check(ctx, e, "vw_stream_destroy");
}

int vw_stream_reset(vw_stream_state *st) {
    if (!st) return VW_ENULL;
    st->batch = -1;
    return VW_OK;
}

int vw_stream_process(vw_ctx *ctx, vw_stream_state *st, const double *x, int64_t batch, int64_t n, int64_t ldx, double *w,
                      int64_t ldw, int64_t level_stride_w, double *v, int64_t ldv, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_stream_process");
    int rc;
    if ((rc = no_capture(ctx, "vw_stream_process"))) return rc;
    if ((rc = check_handle(ctx, st))) return rc;
    if ((rc = check_signal_args(ctx, x, batch, n, ldx))) return rc;
    if ((rc = check_outputs(ctx, st, w, ldw, level_stride_w, v, ldv, batch, n))) return rc;
    const bool dev = flags & VW_FLAG_DEVICE_PTRS;
    const double *xd = x;
    int64_t ldxd = ldx;
    if (!dev) {
        void *px;
        if ((rc = vw_scratch(ctx, 2, (size_t)batch * (size_t)n * 8, &px))) return rc;
        if ((rc = copy_rows(ctx, px, n, x, ldx, n, batch, cudaMemcpyHostToDevice))) return rc;
        xd = (const double *)px;
        ldxd = n;
    }
    if (flags & VW_FLAG_CHECK_FINITE) if ((rc = check_finite(ctx, xd, batch, n, ldxd, "signal"))) return rc;
    // a new batch size restarts the stream (BatchStreamingMODWT.java:306-320); the state changes only once the call runs
    const bool init = st->batch != batch;
    const int64_t hist_total = batch * (int64_t)(st->l - 1) * (((int64_t)1 << st->levels) - 1);
    if ((rc = grow(ctx, st->hist, st->hist_bytes, (size_t)hist_total * 8, "stream histories"))) return rc;
    st->batch = batch;
    rc = with_outputs(ctx, st, batch, n, w, ldw, level_stride_w, v, ldv, flags,
                      [&](double *wd, int64_t lw, int64_t ls, double *vd, int64_t lv) {
                          return cascade(ctx, st, xd, ldxd, n, wd, lw, ls, vd, lv, init, flags);
                      });
    if (rc && init) st->batch = -1;   // a stream that failed to start has not started
    return rc;
}

int vw_stream_flush(vw_ctx *ctx, vw_stream_state *st, int64_t tail_length, double *w, int64_t ldw, int64_t level_stride_w,
                    double *v, int64_t ldv, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_stream_flush");
    int rc;
    if ((rc = no_capture(ctx, "vw_stream_flush"))) return rc;
    if ((rc = check_handle(ctx, st))) return rc;
    if (st->batch < 0) return vw_fail(ctx, VW_ESTATE, "No prior blocks processed; cannot flush");
    if (tail_length < 1) return vw_fail(ctx, VW_EEMPTY, "tail length must be > 0");
    if (tail_length > st->l - 1)
        return vw_fail(ctx, VW_ELENGTH, "tailLength (%lld) exceeds maximum allowed across levels (%d)", (long long)tail_length,
                       st->l - 1);
    if ((rc = check_outputs(ctx, st, w, ldw, level_stride_w, v, ldv, st->batch, tail_length))) return rc;
    return with_outputs(ctx, st, st->batch, tail_length, w, ldw, level_stride_w, v, ldv, flags,
                        [&](double *wd, int64_t lw, int64_t ls, double *vd, int64_t lv) {
                            return cascade(ctx, st, nullptr, 0, tail_length, wd, lw, ls, vd, lv, false, flags);
                        });
}

}  // extern "C"
