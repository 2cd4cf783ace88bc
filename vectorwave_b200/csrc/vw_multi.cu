// vw_multi.cu -- the host-side pieces of the C ABI that sit above the single-call engine:
//   * span-sharded cascades with the up-front halo schedule (one rank's part: vw_modwt_*_span_all, message packing),
//   * several GPUs driven by one host thread (vw_init_multi, vw_modwt_*_sharded: peer copies over NVLink),
//   * device-resident results (vw_result: MultiLevelMODWTResult kept in HBM between decompose and reconstruct),
//   * CUDA-graph replay of a fixed call sequence, and the timing record of the last call.
// No kernels here: everything runs on the tile / column / per-level kernels through the same entry points.
//
// Reference semantics: the sharded transform equals the UNSHARDED MultiLevelMODWTTransform.decompose / reconstruct
// (CORE/modwt/MultiLevelMODWTTransform.java:209-255,339-349,554-601); halo precedent
// EXT/extensions/modwt/BatchSIMDMODWT.java:447-507.  Result objects: CORE/modwt/MultiLevelMODWTResultImpl.java:51-139,
// CORE/modwt/MutableMultiLevelMODWTResult.java:83-118.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <condition_variable>
#include <functional>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "vw_internal.cuh"

using namespace vwshim;

namespace {

int64_t halo_up(int64_t v) { return (v + 31) & ~(int64_t)31; }   // whole 256-byte rows: every offset stays sector aligned

struct SpanSchedule {
    // rf[g]: left halo still needed AFTER forward group g; si_out / si_in: right halo on the outputs / inputs of inverse group g
    int64_t rf[VW_SPAN_MAX_GROUPS], si_out[VW_SPAN_MAX_GROUPS], si_in[VW_SPAN_MAX_GROUPS];
};

SpanSchedule schedule_of(const vw_span_plan &p) {
    SpanSchedule s;
    for (int g = 0; g < p.ngroups_f; g++) {
        s.rf[g] = 0;
        for (int k = g + 1; k < p.ngroups_f; k++) s.rf[g] += p.halo_f[k];
    }
    int64_t acc = 0;
    for (int g = 0; g < p.ngroups_i; g++) {
        s.si_out[g] = acc;
        acc += p.halo_i[g];
        s.si_in[g] = acc;
    }
    return s;
}

// One launch gathers (pack) or scatters (unpack) every piece of a synthesis halo message: piece i is `count[i]` doubles of
// row i (row 0 = V_J, rows 1.. = the W_j rows in message order) starting at element `off[i]` of that row's base pointer.
// Eleven cudaMemcpyAsync calls per rank and direction made the one-host-thread driver launch-bound at 8 GPUs.
constexpr int kMaxPieces = VW_MAX_LEVELS + 1;
struct HaloPieces {
    double *row[kMaxPieces];        // base pointer of every row (V_J row, W_j rows)
    long long off[kMaxPieces];      // first element of the piece inside its row
    int count[kMaxPieces];
    int start[kMaxPieces + 1];      // prefix sums: position of the piece inside the message
    int n;
    double *msg;                    // nullptr on unpack: fill with zeros (open end of a ZERO_PADDING signal)
    int pack;
};
__global__ void __launch_bounds__(256) k_span_halo_pieces(const __grid_constant__ HaloPieces a) {
    const int total = a.start[a.n];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        int p = 0;
        while (i >= a.start[p + 1]) p++;
        double *cell = a.row[p] + a.off[p] + (i - a.start[p]);
        if (a.pack) a.msg[i] = *cell;
        else *cell = a.msg ? a.msg[i] : 0.0;
    }
}

int check_plan(vw_ctx *ctx, const vw_span_plan *p) {
    if (!p) return vw_fail(ctx, VW_ENULL, "span plan cannot be null");
    if (p->ngroups_f < 1 || p->ngroups_f > VW_SPAN_MAX_GROUPS || p->ngroups_i < 1 || p->ngroups_i > VW_SPAN_MAX_GROUPS ||
        p->n_local < 1 || p->levels < 1 || p->l < 1)
        return vw_fail(ctx, VW_EINVAL, "span plan is not initialised (vw_span_plan_query)");
    return VW_OK;
}

}  // namespace

// message layout: V_J[0 .. si_in[top]), then for every inverse group g (ascending) its rows W_j[0 .. si_in[g]).
// pack reads the FIRST samples of every row (what the left neighbour needs), unpack writes behind the span (the pad areas).
static int halo_pieces(vw_ctx *ctx, const vw_span_plan &p, double *w, int64_t row_stride, double *v, double *msg, bool pack) {
    const SpanSchedule s = schedule_of(p);
    HaloPieces a;
    a.n = 0; a.msg = msg; a.pack = pack ? 1 : 0; a.start[0] = 0;
    const int64_t behind = pack ? 0 : p.n_local;
    auto add = [&](double *row, int64_t off, int64_t count) {
        a.row[a.n] = row; a.off[a.n] = off; a.count[a.n] = (int)count;
        a.start[a.n + 1] = a.start[a.n] + (int)count;
        a.n++;
    };
    add(v, behind, s.si_in[p.ngroups_i - 1]);
    for (int gi = 0; gi < p.ngroups_i; gi++)
        for (int i = 0; i < p.nlev_i[gi]; i++)
            add(w + (int64_t)(p.first_i[gi] - 1 + i) * row_stride, p.lead_w + behind, s.si_in[gi]);
    const int total = a.start[a.n];
    if (total <= 0) return VW_OK;
    k_span_halo_pieces<<<std::min(ctx->sm_count, (total + 255) / 256), 256, 0, ctx->stream>>>(a);
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "halo pack / unpack launch");
}

// One enqueueing thread per device.  The caller drives everything from ONE thread, but a cascade is ~20 launches per
// device and direction: enqueued one device after the other, eight devices cost the host more time than the kernels take
// (measured at 8 GPUs: 5.2 ms per step against 3.6 ms of device time).  Every ctx has its own mutex and stream, so the
// per-device cascades are enqueued in parallel; the halo copies and their cross-device events stay on the calling thread.
struct DeviceWorker {
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    std::function<int()> task;
    bool has = false, done = false, stop = false;
    int rc = 0;
    void loop() {
        std::unique_lock<std::mutex> lk(mu);
        for (;;) {
            cv.wait(lk, [&] { return has || stop; });
            if (stop) return;
            has = false;
            lk.unlock();
            const int r = task();
            lk.lock();
            rc = r;
            done = true;
            cv.notify_all();
        }
    }
};

struct vw_multi {
    std::vector<std::unique_ptr<DeviceWorker>> workers;   // empty for a single device
    std::vector<vw_ctx *> ctx;
    std::vector<cudaEvent_t> ev_ready;   // per device: "my outgoing halo source is complete / my stream reached the exchange"
    std::vector<cudaEvent_t> ev_t0, ev_t1;   // per device: around the halo copy this device RECEIVES
    std::vector<double *> msg_send, msg_recv;   // synthesis halo messages (device memory, grow-only)
    std::vector<size_t> msg_cap;
    std::vector<char *> den_buf;   // vw_swt_denoise_sharded per device: threshold, median state and histograms (grow-only)
    std::vector<size_t> den_cap;
    std::string err;
};

struct vw_result {
    int device = 0;
    int64_t batch = 0, n = 0;
    int32_t levels = 0;
    double *base = nullptr;   // [levels + 1][batch][n]: W_1 .. W_J, then V_J
    double *level_ptr(int32_t level) const {   // level 0 = approximation
        const size_t bn = (size_t)batch * (size_t)n;
        return base + (level == 0 ? (size_t)levels * bn : (size_t)(level - 1) * bn);
    }
};

struct vw_graph {
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
};

// runs fn(r) for every device -- in parallel on the device workers when there are several -- and returns the first failure
static int run_on_all_devices(vw_multi *m, const std::function<int(int)> &fn, std::vector<int> &rcs) {
    const int P = (int)m->ctx.size();
    rcs.assign(P, VW_OK);
    if (m->workers.empty()) {
        for (int r = 0; r < P; r++) rcs[r] = fn(r);
    } else {
        for (int r = 0; r < P; r++) {
            DeviceWorker &w = *m->workers[r];
            std::lock_guard<std::mutex> lk(w.mu);
            w.task = [&fn, r] { return fn(r); };
            w.done = false;
            w.has = true;
            w.cv.notify_all();
        }
        for (int r = 0; r < P; r++) {
            DeviceWorker &w = *m->workers[r];
            std::unique_lock<std::mutex> lk(w.mu);
            w.cv.wait(lk, [&] { return w.done; });
            rcs[r] = w.rc;
        }
    }
    for (int r = 0; r < P; r++) if (rcs[r] != VW_OK) return rcs[r];
    return VW_OK;
}

extern "C" {

// ------------------------------------------------------------------------------------------------
// span plan (host logic only)
// ------------------------------------------------------------------------------------------------
int vw_span_plan_query(int32_t l, int32_t levels, int64_t n_local, int32_t world, vw_span_plan *out) {
    if (!out) return VW_ENULL;
    memset(out, 0, sizeof *out);
    if (l < 1 || levels < 1 || levels > VW_MAX_LEVELS || n_local < 1 || world < 1) return VW_EINVAL;
    const int64_t n_total = n_local * (int64_t)world;
    if ((long double)(l - 1) * (long double)((int64_t)1 << (levels - 1)) + 1 > (long double)n_total) return VW_ETOOLARGE;
    int32_t first[64], nlev[64];
    for (int dir = 0; dir < 2; dir++) {
        const int ng = vw_plan_query(dir == 0, l, levels, n_total, first, nlev, 64);
        if (ng < 0) return -ng;
        if (ng > VW_SPAN_MAX_GROUPS) return VW_EUNSUPPORTED;
        for (int g = 0; g < ng; g++) {
            const int64_t h = halo_up(vw_span_halo(l, first[g], nlev[g]));
            if (dir == 0) { out->first_f[g] = first[g]; out->nlev_f[g] = nlev[g]; out->halo_f[g] = h; }
            else { out->first_i[g] = first[g]; out->nlev_i[g] = nlev[g]; out->halo_i[g] = h; }
        }
        if (dir == 0) out->ngroups_f = ng; else out->ngroups_i = ng;
    }
    out->l = l; out->levels = levels; out->world = world; out->n_local = n_local;
    for (int g = 0; g < out->ngroups_f; g++) { out->lead += out->halo_f[g]; if (g > 0) out->lead_w += out->halo_f[g]; }
    for (int g = 0; g < out->ngroups_i; g++) out->pad += out->halo_i[g];
    const SpanSchedule s = schedule_of(*out);
    out->inverse_msg = s.si_in[out->ngroups_i - 1];
    for (int g = 0; g < out->ngroups_i; g++) out->inverse_msg += (int64_t)out->nlev_i[g] * s.si_in[g];
    if (std::max(out->lead, out->pad) > n_local) return VW_ELENGTH;   // a neighbour cannot supply more than its own span
    return VW_OK;
}

// ------------------------------------------------------------------------------------------------
// one rank's cascades (halos already exchanged)
// ------------------------------------------------------------------------------------------------
int vw_modwt_forward_span_all(vw_ctx *ctx, const double *xext, const vw_span_plan *plan, const double *hs, const double *gs,
                              double *w, int64_t row_stride, double *v, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_modwt_forward_span_all");
    int rc;
    if ((rc = check_plan(ctx, plan))) return rc;
    if (!(flags & VW_FLAG_DEVICE_PTRS)) return vw_fail(ctx, VW_EUNSUPPORTED, "span calls take device pointers only");
    if (!xext || !w || !v) return vw_fail(ctx, VW_ENULL, "span buffers cannot be null");
    const vw_span_plan &p = *plan;
    if (row_stride < p.lead_w + p.n_local + p.pad)
        return vw_fail(ctx, VW_ELENGTH, "W row stride %lld shorter than lead_w + n_local + pad = %lld", (long long)row_stride,
                       (long long)(p.lead_w + p.n_local + p.pad));
    const SpanSchedule s = schedule_of(p);
    const int64_t n = p.n_local, lead = p.lead;
    // position 0 of the span sits at index `lead` in every work buffer; group g reads [-(have), n) and writes [-(keep), n)
    double *buf[2] = {nullptr, nullptr};
    const double *cur = xext;
    int64_t have = lead;
    int pp = 0;
    const uint32_t fl = (flags & (VW_FLAG_BITEXACT | VW_FLAG_NO_FUSE)) | VW_FLAG_DEVICE_PTRS | VW_FLAG_NO_SYNC;
    for (int gi = 0; gi < p.ngroups_f; gi++) {
        const int64_t keep = s.rf[gi];
        const bool last = gi + 1 == p.ngroups_f;
        double *vout = v;
        if (!last) {
            if (!buf[pp]) {
                void *q;
                // slots 2 / 3: the per-group call below ping-pongs its own levels through slots 0 / 1
                if ((rc = vw_scratch(ctx, 2 + pp, (size_t)(lead + n) * 8, &q))) return rc;
                buf[pp] = (double *)q;
            }
            vout = buf[pp] + (lead - keep);
        }
        rc = vw_modwt_forward_span(ctx, cur + (lead - have), have - keep, keep + n, hs, gs, p.l, p.first_f[gi], p.nlev_f[gi],
                                   w + (int64_t)(p.first_f[gi] - 1) * row_stride + (p.lead_w - keep), row_stride, vout, fl);
        if (rc) return rc;
        if (!last) { cur = buf[pp]; pp ^= 1; }
        have = keep;
    }
    return finish(ctx, flags, false);
}

// message layout: V_J[0 .. si_in[top]), then for every inverse group g (ascending) its rows W_j[0 .. si_in[g])
int vw_span_pack_inverse(vw_ctx *ctx, const vw_span_plan *plan, const double *w, int64_t row_stride, const double *v,
                         double *msg, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_span_pack_inverse");
    int rc;
    if ((rc = check_plan(ctx, plan))) return rc;
    if (!w || !v || !msg) return vw_fail(ctx, VW_ENULL, "span buffers cannot be null");
    if ((rc = halo_pieces(ctx, *plan, const_cast<double *>(w), row_stride, const_cast<double *>(v), msg, true))) return rc;
    return finish(ctx, flags | VW_FLAG_NO_SYNC, false);
}

int vw_span_unpack_inverse(vw_ctx *ctx, const vw_span_plan *plan, const double *msg, double *w, int64_t row_stride, double *v,
                           uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_span_unpack_inverse");
    int rc;
    if ((rc = check_plan(ctx, plan))) return rc;
    if (!w || !v) return vw_fail(ctx, VW_ENULL, "span buffers cannot be null");
    // msg == NULL: the open end of a ZERO_PADDING signal -- the halo is zeros
    if ((rc = halo_pieces(ctx, *plan, w, row_stride, v, const_cast<double *>(msg), false))) return rc;
    return finish(ctx, flags | VW_FLAG_NO_SYNC, false);
}

}  // extern "C"

// thr_dev == nullptr: the plain synthesis; otherwise one threshold applied to every W sample as the kernels load it
static int inverse_span_all(vw_ctx *ctx, const vw_span_plan *plan, const double *w, int64_t row_stride, const double *v,
                            const double *hs, const double *gs, int32_t order, const double *thr_dev, int32_t soft, double *xout,
                            uint32_t flags, const char *name) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, name);
    int rc;
    if ((rc = check_plan(ctx, plan))) return rc;
    if (!(flags & VW_FLAG_DEVICE_PTRS)) return vw_fail(ctx, VW_EUNSUPPORTED, "span calls take device pointers only");
    if (!w || !v || !xout) return vw_fail(ctx, VW_ENULL, "span buffers cannot be null");
    const vw_span_plan &p = *plan;
    if (row_stride < p.lead_w + p.n_local + p.pad) return vw_fail(ctx, VW_ELENGTH, "W row stride shorter than lead_w + n_local + pad");
    const SpanSchedule s = schedule_of(p);
    const int64_t n = p.n_local;
    double *work[2] = {nullptr, nullptr};
    const double *vext = v;
    int cur = 0;
    const uint32_t fl = (flags & (VW_FLAG_BITEXACT | VW_FLAG_NO_FUSE)) | VW_FLAG_DEVICE_PTRS | VW_FLAG_NO_SYNC;
    for (int gi = p.ngroups_i - 1; gi >= 0; gi--) {
        const int64_t s_in = s.si_in[gi], s_out = s.si_out[gi];
        double *dst = xout;
        if (gi > 0) {
            if (!work[cur]) {
                void *q;
                if ((rc = vw_scratch(ctx, 2 + cur, (size_t)(n + p.pad) * 8, &q))) return rc;
                work[cur] = (double *)q;
            }
            dst = work[cur];
        }
        rc = inverse_span_device(ctx, vext, w + (int64_t)(p.first_i[gi] - 1) * row_stride + p.lead_w, row_stride, s_in - s_out,
                                 n + s_out, hs, gs, p.l, p.first_i[gi], p.nlev_i[gi], order, dst, fl, thr_dev, soft);
        if (rc) return rc;
        if (gi > 0) { vext = work[cur]; cur ^= 1; }
    }
    return finish(ctx, flags, false);
}

extern "C" {

int vw_modwt_inverse_span_all(vw_ctx *ctx, const vw_span_plan *plan, const double *w, int64_t row_stride, const double *v,
                              const double *hs, const double *gs, int32_t order, double *xout, uint32_t flags) {
    return inverse_span_all(ctx, plan, w, row_stride, v, hs, gs, order, nullptr, 0, xout, flags, "vw_modwt_inverse_span_all");
}

int vw_modwt_inverse_span_all_thr(vw_ctx *ctx, const vw_span_plan *plan, const double *w, int64_t row_stride, const double *v,
                                  const double *hs, const double *gs, int32_t order, const double *thr_dev, int32_t soft,
                                  double *xout, uint32_t flags) {
    if (ctx && !thr_dev) {
        DeviceGuard g(ctx, "vw_modwt_inverse_span_all_thr");
        return vw_fail(ctx, VW_ENULL, "threshold pointer cannot be null");
    }
    return inverse_span_all(ctx, plan, w, row_stride, v, hs, gs, order, thr_dev, soft, xout, flags, "vw_modwt_inverse_span_all_thr");
}

// ------------------------------------------------------------------------------------------------
// several GPUs, one host thread
// ------------------------------------------------------------------------------------------------
static int multi_fail(vw_multi *m, int status, const std::string &msg) {
    if (m) m->err = msg;
    return status;
}
static int multi_from_ctx(vw_multi *m, int r, int rc) {
    if (rc != VW_OK) m->err = "device " + std::to_string(m->ctx[r]->device) + ": " + vw_last_error(m->ctx[r]);
    return rc;
}

int vw_init_multi(const int *devices, int32_t ndev, vw_multi **out) {
    if (!out) return VW_ENULL;
    *out = nullptr;
    if (ndev < 1 || ndev > 64) return VW_EINVAL;
    vw_multi *m = new vw_multi();
    for (int r = 0; r < ndev; r++) {
        vw_ctx *c = nullptr;
        int rc = vw_init(devices ? devices[r] : r, &c);
        if (rc) { vw_destroy_multi(m); return rc; }
        m->ctx.push_back(c);
    }
    for (int r = 0; r < ndev; r++) {
        DeviceGuard g(m->ctx[r]->device);
        cudaEvent_t e0, e1, e2;
        if (cudaEventCreateWithFlags(&e0, cudaEventDisableTiming) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess ||
            cudaEventCreate(&e2) != cudaSuccess) { vw_destroy_multi(m); return VW_ECUDA; }
        m->ev_ready.push_back(e0); m->ev_t0.push_back(e1); m->ev_t1.push_back(e2);
        m->msg_send.push_back(nullptr); m->msg_recv.push_back(nullptr); m->msg_cap.push_back(0);
        m->den_buf.push_back(nullptr); m->den_cap.push_back(0);
        // peer access to both ring neighbours (NVLink through NVSwitch on the box; cudaMemcpyPeerAsync falls back to a
        // staged copy where access cannot be enabled, so a refusal is not fatal)
        for (int nb : {(r + 1) % ndev, (r + ndev - 1) % ndev}) {
            if (nb == r || m->ctx[nb]->device == m->ctx[r]->device) continue;
            int can = 0;
            cudaDeviceCanAccessPeer(&can, m->ctx[r]->device, m->ctx[nb]->device);
            if (can) {
                cudaError_t e = cudaDeviceEnablePeerAccess(m->ctx[nb]->device, 0);
                if (e != cudaSuccess) cudaGetLastError();   // cudaErrorPeerAccessAlreadyEnabled included
            }
        }
    }
    if (ndev > 1)
        for (int r = 0; r < ndev; r++) {
            m->workers.emplace_back(new DeviceWorker());
            DeviceWorker *w = m->workers.back().get();
            w->th = std::thread([w] { w->loop(); });
        }
    *out = m;
    return VW_OK;
}

int vw_destroy_multi(vw_multi *m) {
    if (!m) return VW_ENULL;
    for (auto &w : m->workers) {
        { std::lock_guard<std::mutex> lk(w->mu); w->stop = true; w->cv.notify_all(); }
        if (w->th.joinable()) w->th.join();
    }
    for (size_t r = 0; r < m->ctx.size(); r++) {
        {
            DeviceGuard g(m->ctx[r]->device);
            cudaStreamSynchronize(m->ctx[r]->stream);
            if (r < m->ev_ready.size()) { cudaEventDestroy(m->ev_ready[r]); cudaEventDestroy(m->ev_t0[r]); cudaEventDestroy(m->ev_t1[r]); }
            if (r < m->msg_send.size()) { if (m->msg_send[r]) cudaFree(m->msg_send[r]); if (m->msg_recv[r]) cudaFree(m->msg_recv[r]); }
            if (r < m->den_buf.size() && m->den_buf[r]) cudaFree(m->den_buf[r]);
        }
        vw_destroy(m->ctx[r]);
    }
    delete m;
    return VW_OK;
}

int32_t vw_multi_size(const vw_multi *m) { return m ? (int32_t)m->ctx.size() : 0; }
vw_ctx *vw_multi_ctx(vw_multi *m, int32_t rank) { return (m && rank >= 0 && rank < (int32_t)m->ctx.size()) ? m->ctx[rank] : nullptr; }
const char *vw_multi_last_error(const vw_multi *m) { return m ? m->err.c_str() : "null multi-device context"; }

int vw_multi_synchronize(vw_multi *m) {
    if (!m) return VW_ENULL;
    for (size_t r = 0; r < m->ctx.size(); r++)
        if (int rc = multi_from_ctx(m, (int)r, vw_synchronize(m->ctx[r]))) return rc;
    return VW_OK;
}

static int multi_check(vw_multi *m, const vw_span_plan *plan, int32_t mode) {
    if (!m) return VW_ENULL;
    if (!plan) return multi_fail(m, VW_ENULL, "span plan cannot be null");
    if (plan->world != (int32_t)m->ctx.size())
        return multi_fail(m, VW_EINVAL, "the span plan was made for " + std::to_string(plan->world) + " ranks, this context has " +
                                            std::to_string(m->ctx.size()) + " devices");
    if (mode != VW_PERIODIC && mode != VW_ZERO_PADDING)
        return multi_fail(m, VW_EBOUNDARY, "span sharding supports PERIODIC and ZERO_PADDING (SYMMETRIC synthesis is two-sided per "
                                           "level; shard those by signal instead)");
    return VW_OK;
}

// elapsed time of the slowest receiving halo copy (all devices idle afterwards)
static int exchange_time(vw_multi *m, float *exchange_ms) {
    if (int rc = vw_multi_synchronize(m)) return rc;
    float worst = 0.f;
    for (size_t r = 0; r < m->ctx.size(); r++) {
        DeviceGuard g(m->ctx[r]->device);
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, m->ev_t0[r], m->ev_t1[r]) == cudaSuccess) worst = std::max(worst, ms);
        else cudaGetLastError();
    }
    *exchange_ms = worst;
    return VW_OK;
}

int vw_modwt_forward_sharded(vw_multi *m, const vw_span_plan *plan, double *const *xext, const double *hs, const double *gs,
                             int32_t mode, double *const *w, int64_t row_stride, double *const *v, float *exchange_ms,
                             uint32_t flags) {
    int rc;
    if ((rc = multi_check(m, plan, mode))) return rc;
    if (!xext || !w || !v) return multi_fail(m, VW_ENULL, "per-device pointer arrays cannot be null");
    const int P = (int)m->ctx.size();
    const vw_span_plan &p = *plan;
    const int64_t n = p.n_local, lead = p.lead;
    for (int r = 0; r < P; r++) if (!xext[r] || !w[r] || !v[r]) return multi_fail(m, VW_ENULL, "a per-device buffer is null");
    // 1. every device marks the point where its span (the source of its right neighbour's halo) is ready
    for (int r = 0; r < P; r++) {
        DeviceGuard g(m->ctx[r], "vw_modwt_forward_sharded");
        if ((rc = multi_from_ctx(m, r, vw_cuda_check(m->ctx[r], cudaEventRecord(m->ev_ready[r], m->ctx[r]->stream), "event record")))) return rc;
    }
    // 2. the halo of rank r = the last `lead` samples of rank r-1's span, pulled on r's stream (ring wrap for PERIODIC,
    //    zeros in front of rank 0 for ZERO_PADDING)
    for (int r = 0; r < P && lead > 0; r++) {
        vw_ctx *c = m->ctx[r];
        DeviceGuard g(c, "vw_modwt_forward_sharded");
        const int left = (r + P - 1) % P;
        // the timing events bracket the copy alone: the wait for the neighbour's data is in front of them
        cudaError_t e = cudaSuccess;
        const bool open_end = r == 0 && mode == VW_ZERO_PADDING;
        if (!open_end && left != r) e = cudaStreamWaitEvent(c->stream, m->ev_ready[left], 0);
        if (e == cudaSuccess) e = cudaEventRecord(m->ev_t0[r], c->stream);
        if (e == cudaSuccess)
            e = open_end ? cudaMemsetAsync(xext[r], 0, (size_t)lead * 8, c->stream)
                         : cudaMemcpyPeerAsync(xext[r], c->device, xext[left] + n, m->ctx[left]->device, (size_t)lead * 8, c->stream);
        if (e == cudaSuccess) e = cudaEventRecord(m->ev_t1[r], c->stream);
        if ((rc = multi_from_ctx(m, r, vw_cuda_check(c, e, "halo exchange (analysis)")))) return rc;
    }
    // 3. the cascades, one per device, all enqueued (in parallel, one worker per device) before anything is waited for
    {
        std::vector<int> rcs;
        const uint32_t fl = (flags & ~VW_FLAG_CHECK_FINITE) | VW_FLAG_DEVICE_PTRS | VW_FLAG_NO_SYNC;
        run_on_all_devices(m, [&](int r) { return vw_modwt_forward_span_all(m->ctx[r], xext[r], plan, hs, gs, w[r], row_stride, v[r], fl); }, rcs);
        for (int r = 0; r < P; r++) if ((rc = multi_from_ctx(m, r, rcs[r]))) return rc;
    }
    if (exchange_ms) return exchange_time(m, exchange_ms);
    if (!(flags & VW_FLAG_NO_SYNC)) return vw_multi_synchronize(m);
    return VW_OK;
}

}  // extern "C"

// thr == nullptr: the plain synthesis; else thr[r] is device r's threshold, applied to W on load (vw_modwt_inverse_span_all_thr)
static int inverse_sharded(vw_multi *m, const vw_span_plan *plan, double *const *w, int64_t row_stride, double *const *v,
                           const double *hs, const double *gs, int32_t mode, int32_t order, double *const *xout,
                           float *exchange_ms, uint32_t flags, const double *const *thr, int32_t soft) {
    int rc;
    if ((rc = multi_check(m, plan, mode))) return rc;
    if (!xout || !w || !v) return multi_fail(m, VW_ENULL, "per-device pointer arrays cannot be null");
    const int P = (int)m->ctx.size();
    const vw_span_plan &p = *plan;
    for (int r = 0; r < P; r++) if (!xout[r] || !w[r] || !v[r]) return multi_fail(m, VW_ENULL, "a per-device buffer is null");
    const size_t msg_bytes = (size_t)p.inverse_msg * 8;
    // 1. every device gathers the message its LEFT neighbour needs (first samples of V_J and of every W_j row)
    for (int r = 0; r < P; r++) {
        vw_ctx *c = m->ctx[r];
        DeviceGuard g(c, "vw_modwt_inverse_sharded");
        if (m->msg_cap[r] < msg_bytes) {
            cudaStreamSynchronize(c->stream);
            if (m->msg_send[r]) cudaFree(m->msg_send[r]);
            if (m->msg_recv[r]) cudaFree(m->msg_recv[r]);
            m->msg_send[r] = m->msg_recv[r] = nullptr; m->msg_cap[r] = 0;
            if ((rc = multi_from_ctx(m, r, vw_cuda_check(c, cudaMalloc(&m->msg_send[r], msg_bytes), "halo message buffer")))) return rc;
            if ((rc = multi_from_ctx(m, r, vw_cuda_check(c, cudaMalloc(&m->msg_recv[r], msg_bytes), "halo message buffer")))) return rc;
            m->msg_cap[r] = msg_bytes;
        }
        if ((rc = multi_from_ctx(m, r, vw_span_pack_inverse(c, plan, w[r], row_stride, v[r], m->msg_send[r], VW_FLAG_DEVICE_PTRS)))) return rc;
        if ((rc = multi_from_ctx(m, r, vw_cuda_check(c, cudaEventRecord(m->ev_ready[r], c->stream), "event record")))) return rc;
    }
    // 2. rank r pulls its right neighbour's message and scatters it into its pad areas (ring wrap / zeros at the open end)
    for (int r = 0; r < P; r++) {
        vw_ctx *c = m->ctx[r];
        DeviceGuard g(c, "vw_modwt_inverse_sharded");
        const int right = (r + 1) % P;
        const bool open_end = r == P - 1 && mode == VW_ZERO_PADDING;
        cudaError_t e = cudaSuccess;
        if (!open_end && right != r) e = cudaStreamWaitEvent(c->stream, m->ev_ready[right], 0);
        if (e == cudaSuccess) e = cudaEventRecord(m->ev_t0[r], c->stream);
        if (e == cudaSuccess && !open_end)
            e = cudaMemcpyPeerAsync(m->msg_recv[r], c->device, m->msg_send[right], m->ctx[right]->device, msg_bytes, c->stream);
        if (e == cudaSuccess) e = cudaEventRecord(m->ev_t1[r], c->stream);
        if ((rc = multi_from_ctx(m, r, vw_cuda_check(c, e, "halo exchange (synthesis)")))) return rc;
        if ((rc = multi_from_ctx(m, r, vw_span_unpack_inverse(c, plan, open_end ? nullptr : m->msg_recv[r], w[r], row_stride, v[r],
                                                               VW_FLAG_DEVICE_PTRS)))) return rc;
    }
    // 3. the cascades
    {
        std::vector<int> rcs;
        const uint32_t fl = (flags & ~VW_FLAG_CHECK_FINITE) | VW_FLAG_DEVICE_PTRS | VW_FLAG_NO_SYNC;
        run_on_all_devices(m, [&](int r) {
            return thr ? vw_modwt_inverse_span_all_thr(m->ctx[r], plan, w[r], row_stride, v[r], hs, gs, order, thr[r], soft, xout[r], fl)
                       : vw_modwt_inverse_span_all(m->ctx[r], plan, w[r], row_stride, v[r], hs, gs, order, xout[r], fl);
        }, rcs);
        for (int r = 0; r < P; r++) if ((rc = multi_from_ctx(m, r, rcs[r]))) return rc;
    }
    // msg_send of rank r is read by rank r-1's stream: the next pack on r must not overwrite it early.  Both streams are
    // drained below unless the caller asked for an asynchronous return, in which case the next call's event wait orders it.
    if (exchange_ms) return exchange_time(m, exchange_ms);
    if (!(flags & VW_FLAG_NO_SYNC)) return vw_multi_synchronize(m);
    // asynchronous return: make every sender wait until its message has been consumed before it may run later work
    for (int r = 0; r < P; r++) {
        vw_ctx *c = m->ctx[r];
        DeviceGuard g(c->device);
        cudaEventRecord(m->ev_ready[r], c->stream);   // after r's unpack: r has consumed right's message
    }
    for (int r = 0; r < P; r++) {
        const int left = (r + P - 1) % P;
        if (left == r) continue;
        DeviceGuard g(m->ctx[r]->device);
        cudaStreamWaitEvent(m->ctx[r]->stream, m->ev_ready[left], 0);
    }
    return VW_OK;
}

extern "C" {

int vw_modwt_inverse_sharded(vw_multi *m, const vw_span_plan *plan, double *const *w, int64_t row_stride, double *const *v,
                             const double *hs, const double *gs, int32_t mode, int32_t order, double *const *xout,
                             float *exchange_ms, uint32_t flags) {
    return inverse_sharded(m, plan, w, row_stride, v, hs, gs, mode, order, xout, exchange_ms, flags, nullptr, 0);
}

// One long signal denoised across the devices: analysis, the exact median of |W_1| over the whole signal, synthesis with
// the threshold applied on load.  The median runs select_median's seven rounds with the histograms reduced ON the
// devices: after each rank's histogram every device pulls the others' tables (cudaMemcpyPeerAsync, ordered by the
// ranks' events) and sums them itself, so all devices pick from the same sum with no host round trip between rounds.
// Each round's own table has its own slot, so a table is never rewritten while a peer may still be reading it.
int vw_swt_denoise_sharded(vw_multi *m, const vw_span_plan *plan, double *const *xext, const double *hs, const double *gs,
                           int32_t mode, int32_t order, double threshold, int32_t soft, double *const *w, int64_t row_stride,
                           double *const *v, double *const *xout, double *threshold_out, uint32_t flags) {
    int rc;
    if ((rc = multi_check(m, plan, mode))) return rc;
    if (!xext || !w || !v || !xout) return multi_fail(m, VW_ENULL, "per-device pointer arrays cannot be null");
    const int P = (int)m->ctx.size();
    const vw_span_plan &p = *plan;
    for (int r = 0; r < P; r++)
        if (!xext[r] || !w[r] || !v[r] || !xout[r]) return multi_fail(m, VW_ENULL, "a per-device buffer is null");
    if (order != VW_ORDER_SPLIT && order != VW_ORDER_PAIR) return multi_fail(m, VW_EINVAL, "unknown synthesis order " + std::to_string(order));
    if (p.ngroups_f < 1 || p.ngroups_i < 1 || p.n_local < 1) return multi_fail(m, VW_EINVAL, "span plan is not initialised (vw_span_plan_query)");
    const int64_t n = p.n_local, n_total = n * (int64_t)P;
    // 0. every span is checked before anything is computed (nothing is written to xout on failure)
    if (flags & VW_FLAG_CHECK_FINITE)
        for (int r = 0; r < P; r++) {
            vw_ctx *c = m->ctx[r];
            DeviceGuard g(c, "vw_swt_denoise_sharded");
            if ((rc = check_finite(c, xext[r] + p.lead, 1, n, n, "signal")))
                return multi_fail(m, rc, "rank " + std::to_string(r) + " (device " + std::to_string(c->device) + "): " + vw_last_error(c));
        }
    const uint32_t fl = (flags & ~VW_FLAG_CHECK_FINITE) | VW_FLAG_NO_SYNC;
    // 1. analysis
    if ((rc = vw_modwt_forward_sharded(m, plan, xext, hs, gs, mode, w, row_stride, v, nullptr, fl))) return rc;
    // 2. per-device work space: [threshold | summed table | one own table per round | the ranks' tables | median state]
    constexpr int kEntries = 2 << 12;   // the largest round's table (vw_span_median_bins)
    const size_t tab = (size_t)kEntries * 8;
    const size_t off_sum = 256, off_own = off_sum + tab, off_gather = off_own + VW_SPAN_MEDIAN_ROUNDS * tab,
                 off_state = off_gather + (size_t)P * tab;
    const size_t need = off_state + vw_span_median_state_bytes(n);
    bool grow = false;
    for (int r = 0; r < P; r++) grow = grow || m->den_cap[r] < need;
    // a peer may still be reading an earlier call's tables from its own stream: every device drains before any regrowth
    if (grow && (rc = vw_multi_synchronize(m))) return rc;
    for (int r = 0; r < P; r++) {
        vw_ctx *c = m->ctx[r];
        if (m->den_cap[r] >= need) continue;
        DeviceGuard g(c, "vw_swt_denoise_sharded");
        if (m->den_buf[r]) cudaFree(m->den_buf[r]);
        m->den_buf[r] = nullptr; m->den_cap[r] = 0;
        if ((rc = multi_from_ctx(m, r, vw_cuda_check(c, cudaMalloc((void **)&m->den_buf[r], need), "denoise work space")))) return rc;
        m->den_cap[r] = need;
    }
    std::vector<double *> thr(P);
    for (int r = 0; r < P; r++) thr[r] = (double *)m->den_buf[r];
    // 3. the threshold: the same value on every device
    if (threshold < 0) {
        auto at = [&](int r, size_t off) { return m->den_buf[r] + off; };
        for (int r = 0; r < P; r++)
            if ((rc = multi_from_ctx(m, r, vw_span_median_init(m->ctx[r], at(r, off_state), n_total)))) return rc;
        for (int round = 0; round < VW_SPAN_MEDIAN_ROUNDS; round++) {
            const int entries = vw_span_median_bins(round);
            for (int r = 0; r < P; r++) {
                vw_ctx *c = m->ctx[r];
                uint64_t *own = (uint64_t *)(at(r, off_own) + (size_t)round * tab);
                if ((rc = multi_from_ctx(m, r, vw_span_median_hist(c, at(r, off_state), w[r] + p.lead_w, n, round, own)))) return rc;
                DeviceGuard g(c->device);
                if ((rc = multi_from_ctx(m, r, vw_cuda_check(c, cudaEventRecord(m->ev_ready[r], c->stream), "event record")))) return rc;
            }
            for (int r = 0; r < P; r++) {
                vw_ctx *c = m->ctx[r];
                uint64_t *gather = (uint64_t *)at(r, off_gather);
                {
                    DeviceGuard g(c->device);
                    for (int q = 0; q < P; q++) {
                        if (q == r) continue;
                        cudaError_t e = cudaStreamWaitEvent(c->stream, m->ev_ready[q], 0);
                        if (e == cudaSuccess)
                            e = cudaMemcpyPeerAsync(gather + (size_t)q * entries, c->device, at(q, off_own) + (size_t)round * tab,
                                                    m->ctx[q]->device, (size_t)entries * 8, c->stream);
                        if ((rc = multi_from_ctx(m, r, vw_cuda_check(c, e, "median histogram exchange")))) return rc;
                    }
                }
                uint64_t *sum = (uint64_t *)at(r, off_sum);
                {
                    DeviceGuard g(c, "vw_swt_denoise_sharded");
                    rc = vw_launch_span_hist_sum(c, gather, (const uint64_t *)(at(r, off_own) + (size_t)round * tab), P, r, entries, sum);
                }
                if ((rc = multi_from_ctx(m, r, rc))) return rc;
                if ((rc = multi_from_ctx(m, r, vw_span_median_pick(c, at(r, off_state), round, sum)))) return rc;
            }
        }
        const double factor = sqrt(2.0 * log((double)n_total));   // k_select_finish's factor, from the total length
        for (int r = 0; r < P; r++)
            if ((rc = multi_from_ctx(m, r, vw_span_median_value(m->ctx[r], at(r, off_state), factor, thr[r])))) return rc;
    } else {
        for (int r = 0; r < P; r++) {
            DeviceGuard g(m->ctx[r], "vw_swt_denoise_sharded");
            if ((rc = multi_from_ctx(m, r, vw_launch_span_fixed(m->ctx[r], thr[r], threshold)))) return rc;
        }
    }
    // 4. the synthesis exchange and the thresholded cascades
    if ((rc = inverse_sharded(m, plan, w, row_stride, v, hs, gs, mode, order, xout, nullptr, fl, thr.data(), soft))) return rc;
    if (threshold_out) {
        if (threshold < 0) {
            vw_ctx *c = m->ctx[0];
            DeviceGuard g(c->device);
            if ((rc = multi_from_ctx(m, 0, vw_cuda_check(c, cudaMemcpyAsync(threshold_out, thr[0], 8, cudaMemcpyDeviceToHost, c->stream), "small copy"))))
                return rc;
            if ((rc = multi_from_ctx(m, 0, vw_cuda_check(c, cudaStreamSynchronize(c->stream), "threshold copy")))) return rc;
        } else {
            *threshold_out = threshold;
        }
    }
    if (!(flags & VW_FLAG_NO_SYNC)) return vw_multi_synchronize(m);
    return VW_OK;
}

// ------------------------------------------------------------------------------------------------
// device-resident results
// ------------------------------------------------------------------------------------------------
int vw_modwt_decompose_h(vw_ctx *ctx, const double *x, int64_t batch, int64_t n, int64_t ldx, const double *hs, const double *gs,
                         int32_t l, int32_t levels, int32_t mode, vw_result **res, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_modwt_decompose_h");
    int rc;
    if (!res) return vw_fail(ctx, VW_ENULL, "result handle pointer cannot be null");
    if ((rc = check_mode(ctx, mode))) return rc;
    if ((rc = check_signal_args(ctx, x, batch, n, ldx))) return rc;
    VwFilt f;
    if ((rc = load_filters(ctx, hs, gs, l, f))) return rc;
    if ((rc = check_levels(ctx, n, l, levels))) return rc;
    vw_result *r = *res;
    if (r && (r->device != ctx->device || r->batch != batch || r->n != n || r->levels != levels)) {
        if ((rc = vw_result_free(ctx, r))) return rc;
        r = *res = nullptr;
    }
    if (!r) {
        if ((rc = no_capture(ctx, "allocating a result"))) return rc;
        r = new vw_result();
        r->device = ctx->device; r->batch = batch; r->n = n; r->levels = levels;
        rc = vw_cuda_check(ctx, cudaMalloc(&r->base, (size_t)(levels + 1) * (size_t)batch * (size_t)n * 8), "result cudaMalloc");
        if (rc) { delete r; return rc; }
        *res = r;
    }
    const bool dev = flags & VW_FLAG_DEVICE_PTRS;
    const size_t bn = (size_t)batch * (size_t)n;
    const double *xd = x;
    int64_t ldxd = ldx;
    if (!dev) {
        void *px;
        if ((rc = vw_scratch(ctx, 2, bn * 8, &px))) return rc;
        if ((rc = copy_rows(ctx, px, n, x, ldx, n, batch, cudaMemcpyHostToDevice))) return rc;
        xd = (const double *)px; ldxd = n;
    }
    if (flags & VW_FLAG_CHECK_FINITE) if ((rc = check_finite(ctx, xd, batch, n, ldxd, "signal"))) return rc;
    if ((rc = forward_device(ctx, xd, batch, n, ldxd, f, l, levels, mode, r->base, n, (int64_t)bn, r->level_ptr(0), n, flags))) return rc;
    // host input: the staged copy must have been read before the caller may reuse x -- the kernels are ordered after it on
    // the stream, so an asynchronous return is fine for pinned memory; pageable memory was copied synchronously by the driver
    return finish(ctx, flags, false);
}

int vw_result_shape(const vw_result *res, int64_t *batch, int64_t *n, int32_t *levels) {
    if (!res) return VW_ENULL;
    if (batch) *batch = res->batch;
    if (n) *n = res->n;
    if (levels) *levels = res->levels;
    return VW_OK;
}

double *vw_result_device_ptr(const vw_result *res, int32_t level) {
    if (!res || level < 0 || level > res->levels) return nullptr;
    return res->level_ptr(level);
}

static int result_level_ok(vw_ctx *ctx, const vw_result *res, int32_t level, int32_t lo) {
    if (!res) return vw_fail(ctx, VW_ENULL, "result handle cannot be null");
    if (res->device != ctx->device) return vw_fail(ctx, VW_EINVAL, "result lives on device %d, ctx on device %d", res->device, ctx->device);
    if (level < lo || level > res->levels)
        return vw_fail(ctx, VW_ELEVEL, "Level must be between %d and %d, got: %d", lo, res->levels, level);   // MultiLevelMODWTResultImpl.java:74-80
    return VW_OK;
}

int vw_result_get_level(vw_ctx *ctx, const vw_result *res, int32_t level, double *dst, int64_t ld, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_result_get_level");
    int rc;
    if ((rc = result_level_ok(ctx, res, level, 0))) return rc;
    if (!dst) return vw_fail(ctx, VW_ENULL, "destination cannot be null");
    if (ld < res->n) return vw_fail(ctx, VW_ELENGTH, "row stride %lld shorter than signal length %lld", (long long)ld, (long long)res->n);
    const bool dev = flags & VW_FLAG_DEVICE_PTRS;
    if ((rc = copy_rows(ctx, dst, ld, res->level_ptr(level), res->n, res->n, res->batch, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost)))
        return rc;
    return finish(ctx, flags, !dev);
}

int vw_result_set_level(vw_ctx *ctx, vw_result *res, int32_t level, const double *src, int64_t ld, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_result_set_level");
    int rc;
    if ((rc = result_level_ok(ctx, res, level, 0))) return rc;
    if (!src) return vw_fail(ctx, VW_ENULL, "source cannot be null");
    if (ld < res->n) return vw_fail(ctx, VW_ELENGTH, "row stride %lld shorter than signal length %lld", (long long)ld, (long long)res->n);
    const bool dev = flags & VW_FLAG_DEVICE_PTRS;
    if ((rc = copy_rows(ctx, res->level_ptr(level), res->n, src, ld, res->n, res->batch, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice)))
        return rc;
    return finish(ctx, flags, !dev);
}

int vw_result_threshold(vw_ctx *ctx, vw_result *res, int32_t level, const double *thresholds, int32_t per_row, int32_t soft) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_result_threshold");
    int rc;
    if ((rc = result_level_ok(ctx, res, level, 0))) return rc;
    if (!thresholds) return vw_fail(ctx, VW_ENULL, "thresholds cannot be null");
    // level 0 = every detail level: they are contiguous rows [levels * batch][n]; per-row thresholds then repeat per level
    if (level == 0 && !per_row)
        return vw_threshold(ctx, res->base, (int64_t)res->levels * res->batch, res->n, res->n, thresholds, 0, soft, VW_FLAG_DEVICE_PTRS);
    const int lo = level == 0 ? 1 : level, hi = level == 0 ? res->levels : level;
    for (int j = lo; j <= hi; j++)
        if ((rc = vw_threshold(ctx, res->level_ptr(j), res->batch, res->n, res->n, thresholds, per_row, soft, VW_FLAG_DEVICE_PTRS))) return rc;
    return VW_OK;
}

int vw_result_universal_threshold(vw_ctx *ctx, vw_result *res, int32_t soft, double *thresholds_out) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_result_universal_threshold");
    int rc;
    if ((rc = result_level_ok(ctx, res, 1, 1))) return rc;
    if ((rc = no_capture(ctx, "vw_result_universal_threshold"))) return rc;
    // thresholds stay on the device: select per row from W_1, then one in-place pass per detail level
    void *pt;
    if ((rc = vw_scratch(ctx, 5, (size_t)res->batch * 8 + 64, &pt))) return rc;
    double *thr_dev = (double *)((char *)pt + 64);
    if ((rc = vw_launch_universal_threshold(ctx, res->level_ptr(1), res->batch, res->n, res->n, thr_dev))) return rc;
    for (int j = 1; j <= res->levels; j++)
        if ((rc = vw_launch_threshold(ctx, res->level_ptr(j), res->batch, res->n, res->n, thr_dev, 1, soft))) return rc;
    if (thresholds_out &&
        (rc = vw_cuda_check(ctx, cudaMemcpyAsync(thresholds_out, thr_dev, (size_t)res->batch * 8, cudaMemcpyDeviceToHost, ctx->stream), "small copy")))
        return rc;
    return finish(ctx, 0, true);
}

int vw_result_energy(vw_ctx *ctx, const vw_result *res, int32_t level, double *out) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_result_energy");
    if (int rc = result_level_ok(ctx, res, level, 0)) return rc;
    return vw_energy(ctx, res->level_ptr(level), res->batch, res->n, res->n, out, VW_FLAG_DEVICE_PTRS);
}

int vw_modwt_reconstruct_h(vw_ctx *ctx, const vw_result *res, const double *hs, const double *gs, int32_t l, int32_t mode,
                           const vw_align *align, int32_t order, uint64_t detail_mask, int32_t use_approx, double *xout, int64_t ldx,
                           uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_modwt_reconstruct_h");
    int rc;
    if ((rc = result_level_ok(ctx, res, 0, 0))) return rc;
    const bool dev = flags & VW_FLAG_DEVICE_PTRS;
    const int64_t batch = res->batch, n = res->n;
    const size_t bn = (size_t)batch * (size_t)n;
    if (dev)
        return vw_modwt_inverse(ctx, res->base, n, (int64_t)bn, res->level_ptr(0), n, batch, n, hs, gs, l, res->levels, mode, align,
                                order, detail_mask, use_approx, xout, ldx, flags);
    // host output: reconstruct into scratch, then one D2H copy of the signal (8 B/sample instead of 8 * (levels + 2))
    if ((rc = check_signal_args(ctx, xout, batch, n, ldx))) return rc;
    void *px;
    if ((rc = vw_scratch(ctx, 2, bn * 8, &px))) return rc;
    rc = vw_modwt_inverse(ctx, res->base, n, (int64_t)bn, res->level_ptr(0), n, batch, n, hs, gs, l, res->levels, mode, align, order,
                          detail_mask, use_approx, (double *)px, n, (flags & ~VW_FLAG_CHECK_FINITE) | VW_FLAG_DEVICE_PTRS | VW_FLAG_NO_SYNC);
    if (rc) return rc;
    if ((rc = copy_rows(ctx, xout, ldx, px, n, n, batch, cudaMemcpyDeviceToHost))) return rc;
    return finish(ctx, flags, true);
}

int vw_result_free(vw_ctx *ctx, vw_result *res) {
    if (!ctx) return VW_ENULL;
    if (!res) return VW_OK;
    DeviceGuard g(ctx, "vw_result_free");
    if (int rc = no_capture(ctx, "vw_result_free")) return rc;
    cudaStreamSynchronize(ctx->stream);
    cudaError_t e = res->base ? cudaFree(res->base) : cudaSuccess;
    delete res;
    return vw_cuda_check(ctx, e, "vw_result_free");
}

// ------------------------------------------------------------------------------------------------
// CUDA-graph replay
// ------------------------------------------------------------------------------------------------
int vw_graph_begin(vw_ctx *ctx) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_graph_begin");
    if (ctx->capturing) return vw_fail(ctx, VW_ESTATE, "a graph capture is already open on this ctx");
    // relaxed: the host side of the captured calls may still query occupancy / function attributes
    int rc = vw_cuda_check(ctx, cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeRelaxed), "cudaStreamBeginCapture");
    if (rc) return rc;
    ctx->capturing = true;
    return VW_OK;
}

int vw_graph_end(vw_ctx *ctx, vw_graph **out) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_graph_end");
    if (!out) return vw_fail(ctx, VW_ENULL, "graph handle pointer cannot be null");
    if (!ctx->capturing) return vw_fail(ctx, VW_ESTATE, "no graph capture is open on this ctx");
    ctx->capturing = false;
    vw_graph *gr = new vw_graph();
    int rc = vw_cuda_check(ctx, cudaStreamEndCapture(ctx->stream, &gr->graph), "cudaStreamEndCapture");
    if (!rc) rc = vw_cuda_check(ctx, cudaGraphInstantiate(&gr->exec, gr->graph, 0), "cudaGraphInstantiate");
    if (rc) {
        if (gr->graph) cudaGraphDestroy(gr->graph);
        delete gr;
        return rc;
    }
    *out = gr;
    return VW_OK;
}

int vw_graph_launch(vw_ctx *ctx, vw_graph *gr, uint32_t flags) {
    if (!ctx) return VW_ENULL;
    DeviceGuard g(ctx, "vw_graph_launch");
    if (!gr || !gr->exec) return vw_fail(ctx, VW_ENULL, "graph handle cannot be null");
    if (ctx->capturing) return vw_fail(ctx, VW_ESTATE, "cannot launch a graph while capturing");
    int rc = vw_cuda_check(ctx, cudaGraphLaunch(gr->exec, ctx->stream), "cudaGraphLaunch");
    if (rc) return rc;
    ctx->launches++;
    return finish(ctx, flags, false);
}

int vw_graph_destroy(vw_ctx *ctx, vw_graph *gr) {
    if (!ctx) return VW_ENULL;
    if (!gr) return VW_OK;
    DeviceGuard g(ctx, "vw_graph_destroy");
    cudaStreamSynchronize(ctx->stream);
    if (gr->exec) cudaGraphExecDestroy(gr->exec);
    if (gr->graph) cudaGraphDestroy(gr->graph);
    delete gr;
    return VW_OK;
}

// ------------------------------------------------------------------------------------------------
// timing record
// ------------------------------------------------------------------------------------------------
int vw_last_timing(vw_ctx *ctx, vw_timing *out) {
    if (!ctx || !out) return VW_ENULL;
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    DeviceGuard g(ctx->device);
    if (!ctx->time_valid) return vw_fail(ctx, VW_ESTATE, "no timed call yet: vw_set_option(ctx, \"timing\", 1) first");
    int rc = vw_cuda_check(ctx, cudaEventSynchronize(ctx->time_ev[1]), "timing event");
    if (rc) return rc;
    float ms = 0.f;
    if ((rc = vw_cuda_check(ctx, cudaEventElapsedTime(&ms, ctx->time_ev[0], ctx->time_ev[1]), "timing event"))) return rc;
    out->device_ms = ms;
    out->host_ms = ctx->time_host_ms;
    out->launches = ctx->time_launches;
    out->reserved = 0;
    return VW_OK;
}

}  // extern "C"
