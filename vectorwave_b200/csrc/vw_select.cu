// vw_select.cu -- exact per-signal median of |W_1| for the universal threshold.
//
// Replaces VectorWaveSwtAdapter.estimateNoiseSigma's full Arrays.sort
// (CORE/swt/VectorWaveSwtAdapter.java:627-645) with an MSB-first radix select on the IEEE bit
// pattern of |x| (order-isomorphic to the value for finite non-negative doubles).  Both middle order
// statistics of an even-length row are tracked in the same passes.  Result per row:
//   thr = (median / 0.6745) * sqrt(2 ln n)        (CORE/swt/VectorWaveSwtAdapter.java:505-520)
#include "vw_internal.cuh"

namespace {

// Passes over the data: two 12-bit digits (exponent, then the top 12 mantissa bits) on the full row, then one pass
// that compacts the keys sharing the 24 decided bits (a few dozen per million N(0,1) samples) into a candidate
// buffer; the remaining 40 bits are resolved by five 8-bit passes over the candidates only.  24 B/sample instead of
// the 64 B/sample of eight full passes.  A row whose bucket overflows the buffer (heavy ties, e.g. a constant
// signal) keeps running the 8-bit passes over the full row -- still exact, just slower.
struct SelState {           // per row
    unsigned long long prefix[2];  // key bits decided so far (high bits), for rank lo / hi
    unsigned long long rank[2];    // remaining 0-based rank inside the current prefix bucket
    unsigned int count[2];         // candidates collected for lo / hi
    unsigned int pad[2];
};

constexpr int kBig = 12;                 // bits per digit of the two full-row passes
constexpr int kBigBins = 1 << kBig;

__global__ void k_select_init(SelState *st, int64_t batch, int64_t n) {
    int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= batch) return;
    st[b].prefix[0] = st[b].prefix[1] = 0ull;
    st[b].rank[1] = (unsigned long long)(n / 2);
    st[b].rank[0] = (n % 2 == 0) ? (unsigned long long)(n / 2 - 1) : (unsigned long long)(n / 2);
    st[b].count[0] = st[b].count[1] = 0u;
}

__device__ __forceinline__ unsigned long long key_of(double v) { return (unsigned long long)__double_as_longlong(fabs(v)); }

// histogram of the next BITS-bit digit among keys that match each tracked prefix.
// cand != nullptr: rows whose candidate buffers did not overflow read their candidates instead of the full row.
template <int BITS>
__global__ void __launch_bounds__(256)
k_select_hist(const double *__restrict__ w, int64_t batch, int64_t n, int64_t ld, const SelState *__restrict__ st, int shift,
              unsigned int *__restrict__ hist /*[batch][2][1 << BITS]*/, const double *__restrict__ cand, unsigned int cap) {
    constexpr int BINS = 1 << BITS;
    __shared__ unsigned int sh[2][BINS];
    const int64_t b = blockIdx.y + (int64_t)blockIdx.z * gridDim.y;   // batches beyond 32768 rows spill into grid.z
    if (b >= batch) return;
    for (int i = threadIdx.x; i < 2 * BINS; i += blockDim.x) (&sh[0][0])[i] = 0;
    __syncthreads();
    const unsigned long long p0 = st[b].prefix[0], p1 = st[b].prefix[1];
    const bool same = p0 == p1;
    const int hs = shift + BITS;  // bits above the current digit
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool use_cand = cand != nullptr && st[b].count[0] <= cap && st[b].count[1] <= cap;
    if (!use_cand) {
        const double *row = w + b * ld;
        for (int64_t t = t0; t < n; t += stride) {
            const unsigned long long key = key_of(row[t]);
            const unsigned long long hi = hs >= 64 ? 0ull : (key >> hs);
            const unsigned int dg = (unsigned int)(key >> shift) & (BINS - 1);
            if (hi == p0) atomicAdd(&sh[0][dg], 1u);
            if (!same && hi == p1) atomicAdd(&sh[1][dg], 1u);
        }
    } else {
        // candidates of rank lo and of rank hi sit in separate buffers (identical content when the prefixes agree)
        for (int which = 0; which < (same ? 1 : 2); which++) {
            const double *src = cand + ((size_t)b * 2 + which) * cap;
            const unsigned long long pw = which ? p1 : p0;
            const int64_t len = st[b].count[which];
            for (int64_t t = t0; t < len; t += stride) {
                const unsigned long long key = key_of(src[t]);
                const unsigned long long hi = hs >= 64 ? 0ull : (key >> hs);
                if (hi == pw) atomicAdd(&sh[which][(unsigned int)(key >> shift) & (BINS - 1)], 1u);
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < BINS; i += blockDim.x) {
        const unsigned int c0 = sh[0][i], c1 = same ? c0 : sh[1][i];
        if (c0) atomicAdd(&hist[((size_t)b * 2 + 0) * BINS + i], c0);
        if (c1) atomicAdd(&hist[((size_t)b * 2 + 1) * BINS + i], c1);
    }
}

// one block per (row, which): find the bin holding the rank (parallel prefix over the bins), clear the bins
template <int BITS>
__global__ void __launch_bounds__(256) k_select_pick(SelState *st, unsigned int *hist) {
    constexpr int BINS = 1 << BITS, PER = BINS / 256 > 0 ? BINS / 256 : 1;
    __shared__ unsigned long long part[256];
    const int64_t i = blockIdx.x;
    const int64_t b = i >> 1; const int which = (int)(i & 1);
    unsigned int *h = hist + (size_t)i * BINS;
    const int tid = threadIdx.x;
    unsigned long long mine = 0;
    unsigned int loc[PER];
#pragma unroll
    for (int q = 0; q < PER; q++) { const int bin = tid * PER + q; loc[q] = bin < BINS ? h[bin] : 0u; mine += loc[q]; }
    part[tid] = mine;
    __syncthreads();
    if (tid == 0) {   // 256-entry exclusive scan: tiny
        unsigned long long run = 0;
        for (int q = 0; q < 256; q++) { const unsigned long long c = part[q]; part[q] = run; run += c; }
    }
    __syncthreads();
    const unsigned long long r = st[b].rank[which];
    unsigned long long cum = part[tid];
    __syncthreads();
    if (r >= cum && r < cum + mine) {
#pragma unroll
        for (int q = 0; q < PER; q++) {
            if (r < cum + loc[q]) {
                st[b].rank[which] = r - cum;
                st[b].prefix[which] = (st[b].prefix[which] << BITS) | (unsigned long long)(tid * PER + q);
                break;
            }
            cum += loc[q];
        }
    }
#pragma unroll
    for (int q = 0; q < PER; q++) { const int bin = tid * PER + q; if (bin < BINS) h[bin] = 0; }
}

// compact the keys that share the decided high bits into the per-(row, which) candidate buffers
__global__ void __launch_bounds__(256)
k_select_collect(const double *__restrict__ w, int64_t batch, int64_t n, int64_t ld, SelState *st, int decided_bits,
                 double *cand, unsigned int cap) {
    const int64_t b = blockIdx.y + (int64_t)blockIdx.z * gridDim.y;
    if (b >= batch) return;
    const unsigned long long p0 = st[b].prefix[0], p1 = st[b].prefix[1];
    const bool same = p0 == p1;
    const int hs = 64 - decided_bits;
    const double *row = w + b * ld;
    double *c0 = cand + ((size_t)b * 2 + 0) * cap, *c1 = cand + ((size_t)b * 2 + 1) * cap;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        const double v = fabs(row[t]);
        const unsigned long long hi = key_of(v) >> hs;
        if (hi == p0) {   // one bucket for both ranks: fill both buffers, the prefixes may part ways in a later digit
            const unsigned int k = atomicAdd(&st[b].count[0], 1u);
            if (k < cap) { c0[k] = v; if (same) c1[k] = v; }
        }
        if (!same && hi == p1) { const unsigned int k = atomicAdd(&st[b].count[1], 1u); if (k < cap) c1[k] = v; }
    }
}
__global__ void k_select_mirror_count(SelState *st, int64_t batch) {   // same prefix: hi shares lo's candidates
    int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= batch) return;
    if (st[b].prefix[0] == st[b].prefix[1]) st[b].count[1] = st[b].count[0];
}

// factor >= 0: universal threshold (median / 0.6745) * factor (0 for n = 1); factor < 0: the raw median
__global__ void k_select_finish(const SelState *st, int64_t batch, int64_t n, double factor, double *thr) {
    int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= batch) return;
    double lo = __longlong_as_double((long long)st[b].prefix[0]);
    double hi = __longlong_as_double((long long)st[b].prefix[1]);
    double med = (n % 2 == 0) ? __ddiv_rn(__dadd_rn(lo, hi), 2.0) : hi;
    thr[b] = factor >= 0.0 ? __dmul_rn(__ddiv_rn(med, 0.6745), factor) : med;
}

}  // namespace

static int select_median(vw_ctx *ctx, const double *w1, int64_t batch, int64_t n, int64_t ld, double *thr_dev, double factor);

int vw_launch_universal_threshold(vw_ctx *ctx, const double *w1, int64_t batch, int64_t n, int64_t ld,
                                  double *thr_dev) {
    // Math.sqrt(2 * Math.log(n)), CORE/swt/VectorWaveSwtAdapter.java:512
    return select_median(ctx, w1, batch, n, ld, thr_dev, sqrt(2.0 * log((double)n)));
}

int vw_launch_median_abs(vw_ctx *ctx, const double *c, int64_t batch, int64_t n, int64_t ld, double *med_dev) {
    return select_median(ctx, c, batch, n, ld, med_dev, -1.0);
}

static int select_median(vw_ctx *ctx, const double *w1, int64_t batch, int64_t n, int64_t ld, double *thr_dev, double factor) {
    if (batch <= 0 || n <= 0) return VW_OK;
    void *ws = nullptr;
    int64_t cap64 = n / 64;
    if (cap64 < 1024) cap64 = 1024;
    if (cap64 > (1 << 20)) cap64 = 1 << 20;
    const unsigned int cap = (unsigned int)cap64;
    const size_t st_bytes = ((size_t)batch * sizeof(SelState) + 255) & ~(size_t)255;
    const size_t hist_bytes = (size_t)batch * 2 * kBigBins * sizeof(unsigned int);
    const size_t cand_bytes = (size_t)batch * 2 * cap * sizeof(double);
    int rc = vw_scratch(ctx, 4, st_bytes + hist_bytes + cand_bytes, &ws);
    if (rc) return rc;
    SelState *st = (SelState *)ws;
    unsigned int *hist = (unsigned int *)((char *)ws + st_bytes);
    double *cand = (double *)((char *)ws + st_bytes + hist_bytes);
    rc = vw_cuda_check(ctx, cudaMemsetAsync(hist, 0, hist_bytes, ctx->stream), "select memset");
    if (rc) return rc;
    const unsigned nb = (unsigned)((batch + 127) / 128);
    k_select_init<<<nb, 128, 0, ctx->stream>>>(st, batch, n);
    ctx->launches++;
    int64_t chunks = (n + 256 * 16 - 1) / (256 * 16);
    const int64_t capc = ((int64_t)ctx->sm_count * 16 + batch - 1) / batch;
    if (chunks > capc) chunks = capc;
    if (chunks < 1) chunks = 1;
    // one row per grid.y slot; gridDim.y stops at 65535, so rows beyond 32768 go to grid.z
    const unsigned gy = (unsigned)(batch < 32768 ? batch : 32768);
    const dim3 grid((unsigned)chunks, gy, (unsigned)((batch + gy - 1) / gy));
    // two 12-bit digits over the full rows: bits 63..52 (sign 0 + exponent), bits 51..40
    for (int shift = 64 - kBig; shift >= 64 - 2 * kBig; shift -= kBig) {
        k_select_hist<kBig><<<grid, 256, 0, ctx->stream>>>(w1, batch, n, ld, st, shift, hist, nullptr, 0u);
        k_select_pick<kBig><<<(unsigned)(batch * 2), 256, 0, ctx->stream>>>(st, hist);
        ctx->launches += 2;
    }
    k_select_collect<<<grid, 256, 0, ctx->stream>>>(w1, batch, n, ld, st, 2 * kBig, cand, cap);
    k_select_mirror_count<<<nb, 128, 0, ctx->stream>>>(st, batch);
    ctx->launches += 2;
    // remaining 40 bits, 8 at a time, over the candidates (or the full row where they overflowed)
    for (int shift = 64 - 2 * kBig - 8; shift >= 0; shift -= 8) {
        k_select_hist<8><<<grid, 256, 0, ctx->stream>>>(w1, batch, n, ld, st, shift, hist, cand, cap);
        k_select_pick<8><<<(unsigned)(batch * 2), 256, 0, ctx->stream>>>(st, hist);
        ctx->launches += 2;
    }
    k_select_finish<<<nb, 128, 0, ctx->stream>>>(st, batch, n, factor, thr_dev);
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "universal threshold launch");
}

// ---- the same selection over a signal split into spans on several ranks -------------------------------------------
// select_median's seven digit rounds with the histogram handed out between "histogram" and "pick": every rank counts
// its own span into a u64 table, the caller sums the tables over the ranks, and every rank picks from the identical sum,
// so the decided prefixes and remaining ranks stay identical everywhere.  The candidate buffer of round 2 is rank-local:
// a rank whose bucket overflows it (a constant span) keeps histogramming its full span, the others their candidates,
// and the sum is the same exact count either way.
namespace {
struct SpanSel {             // device state blob: SelState first (the per-row kernels above run on it with batch 1)
    SelState s;
    long long n_total;
    long long pad[3];
};
static_assert(sizeof(SpanSel) <= 256, "span selection state fits its 256-byte header");

constexpr int kSpanRounds = VW_SPAN_MEDIAN_ROUNDS;
int span_bits(int round) { return round < 2 ? kBig : 8; }
int span_shift(int round) { return round < 2 ? 64 - kBig * (round + 1) : 64 - 2 * kBig - 8 * (round - 1); }
unsigned int span_cap(int64_t n_local) {
    int64_t cap64 = n_local / 64;
    if (cap64 < 1024) cap64 = 1024;
    if (cap64 > (1 << 20)) cap64 = 1 << 20;
    return (unsigned int)cap64;
}

__global__ void k_span_init(SpanSel *st, long long n_total) {
    st->s.prefix[0] = st->s.prefix[1] = 0ull;
    st->s.rank[1] = (unsigned long long)(n_total / 2);
    st->s.rank[0] = (n_total % 2 == 0) ? (unsigned long long)(n_total / 2 - 1) : (unsigned long long)(n_total / 2);
    st->s.count[0] = st->s.count[1] = 0u;
    st->n_total = n_total;
}

// k_select_hist on one span, accumulated into a u64 table [2][1 << BITS] (the sum over ranks may exceed 2^32)
template <int BITS>
__global__ void __launch_bounds__(256)
k_span_hist(const double *__restrict__ w, int64_t n, const SpanSel *__restrict__ st, int shift,
            unsigned long long *__restrict__ hist, const double *__restrict__ cand, unsigned int cap) {
    constexpr int BINS = 1 << BITS;
    __shared__ unsigned int sh[2][BINS];
    for (int i = threadIdx.x; i < 2 * BINS; i += blockDim.x) (&sh[0][0])[i] = 0;
    __syncthreads();
    const unsigned long long p0 = st->s.prefix[0], p1 = st->s.prefix[1];
    const bool same = p0 == p1;
    const int hs = shift + BITS;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool use_cand = cand != nullptr && st->s.count[0] <= cap && st->s.count[1] <= cap;
    if (!use_cand) {
        for (int64_t t = t0; t < n; t += stride) {
            const unsigned long long key = key_of(w[t]);
            const unsigned long long hi = hs >= 64 ? 0ull : (key >> hs);
            const unsigned int dg = (unsigned int)(key >> shift) & (BINS - 1);
            if (hi == p0) atomicAdd(&sh[0][dg], 1u);
            if (!same && hi == p1) atomicAdd(&sh[1][dg], 1u);
        }
    } else {
        for (int which = 0; which < (same ? 1 : 2); which++) {
            const double *src = cand + (size_t)which * cap;
            const unsigned long long pw = which ? p1 : p0;
            const int64_t len = st->s.count[which];
            for (int64_t t = t0; t < len; t += stride) {
                const unsigned long long key = key_of(src[t]);
                const unsigned long long hi = hs >= 64 ? 0ull : (key >> hs);
                if (hi == pw) atomicAdd(&sh[which][(unsigned int)(key >> shift) & (BINS - 1)], 1u);
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < BINS; i += blockDim.x) {
        const unsigned int c0 = sh[0][i], c1 = same ? c0 : sh[1][i];
        if (c0) atomicAdd(&hist[i], (unsigned long long)c0);
        if (c1) atomicAdd(&hist[BINS + i], (unsigned long long)c1);
    }
}

// k_select_pick on a summed u64 table (left as it is: it belongs to the caller); one block per tracked rank
template <int BITS>
__global__ void __launch_bounds__(256) k_span_pick(SpanSel *st, const unsigned long long *__restrict__ hist) {
    constexpr int BINS = 1 << BITS, PER = BINS / 256 > 0 ? BINS / 256 : 1;
    __shared__ unsigned long long part[256];
    const int which = (int)blockIdx.x;
    const unsigned long long *h = hist + (size_t)which * BINS;
    const int tid = threadIdx.x;
    unsigned long long mine = 0;
    unsigned long long loc[PER];
#pragma unroll
    for (int q = 0; q < PER; q++) { const int bin = tid * PER + q; loc[q] = bin < BINS ? h[bin] : 0ull; mine += loc[q]; }
    part[tid] = mine;
    __syncthreads();
    if (tid == 0) {
        unsigned long long run = 0;
        for (int q = 0; q < 256; q++) { const unsigned long long c = part[q]; part[q] = run; run += c; }
    }
    __syncthreads();
    const unsigned long long r = st->s.rank[which];
    unsigned long long cum = part[tid];
    __syncthreads();
    if (r >= cum && r < cum + mine) {
#pragma unroll
        for (int q = 0; q < PER; q++) {
            if (r < cum + loc[q]) {
                st->s.rank[which] = r - cum;
                st->s.prefix[which] = (st->s.prefix[which] << BITS) | (unsigned long long)(tid * PER + q);
                break;
            }
            cum += loc[q];
        }
    }
}

// k_select_finish with the total length from the state
__global__ void k_span_finish(const SpanSel *st, double factor, double *thr) {
    const double lo = __longlong_as_double((long long)st->s.prefix[0]);
    const double hi = __longlong_as_double((long long)st->s.prefix[1]);
    const double med = (st->n_total % 2 == 0) ? __ddiv_rn(__dadd_rn(lo, hi), 2.0) : hi;
    *thr = factor >= 0.0 ? __dmul_rn(__ddiv_rn(med, 0.6745), factor) : med;
}

// out[i] = own[i] + sum over the other ranks' tables (gather[q], q != self), in rank order
__global__ void __launch_bounds__(256) k_span_hist_sum(const unsigned long long *__restrict__ gather,
                                                       const unsigned long long *__restrict__ own, int ranks, int self,
                                                       int entries, unsigned long long *__restrict__ out) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < entries; i += gridDim.x * blockDim.x) {
        unsigned long long s = 0;
        for (int q = 0; q < ranks; q++) s += q == self ? own[i] : gather[(size_t)q * entries + i];
        out[i] = s;
    }
}

__global__ void k_span_fixed(double *thr, double value) { *thr = value; }
}  // namespace

static int vw_span_rounds_check(vw_ctx *ctx, int32_t round) {
    if (round < 0 || round >= kSpanRounds) return vw_fail(ctx, VW_EINVAL, "median round %d outside 0..%d", round, kSpanRounds - 1);
    return VW_OK;
}

int vw_launch_span_hist_sum(vw_ctx *ctx, const uint64_t *gather, const uint64_t *own, int ranks, int self, int entries,
                            uint64_t *out) {
    k_span_hist_sum<<<(entries + 255) / 256, 256, 0, ctx->stream>>>((const unsigned long long *)gather, (const unsigned long long *)own,
                                                                     ranks, self, entries, (unsigned long long *)out);
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "median histogram sum launch");
}

int vw_launch_span_fixed(vw_ctx *ctx, double *thr_dev, double value) {
    k_span_fixed<<<1, 1, 0, ctx->stream>>>(thr_dev, value);
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "threshold store launch");
}

extern "C" {

int32_t vw_span_median_bins(int32_t round) {
    if (round < 0 || round >= kSpanRounds) return 0;
    return 2 << span_bits(round);
}

size_t vw_span_median_state_bytes(int64_t n_local) {
    if (n_local < 1) return 0;
    return 256 + (size_t)2 * span_cap(n_local) * sizeof(double);
}

int vw_span_median_init(vw_ctx *ctx, void *state, int64_t n_total) {
    if (!ctx) return VW_ENULL;
    vwshim::DeviceGuard g(ctx, "vw_span_median_init");
    if (!state) return vw_fail(ctx, VW_ENULL, "median state cannot be null");
    if (n_total < 1) return vw_fail(ctx, VW_EEMPTY, "signal cannot be empty");
    k_span_init<<<1, 1, 0, ctx->stream>>>((SpanSel *)state, (long long)n_total);
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "median init launch");
}

int vw_span_median_hist(vw_ctx *ctx, void *state, const double *c, int64_t n_local, int32_t round, uint64_t *hist) {
    if (!ctx) return VW_ENULL;
    vwshim::DeviceGuard g(ctx, "vw_span_median_hist");
    int rc;
    if ((rc = vw_span_rounds_check(ctx, round))) return rc;
    if (!state || !c || !hist) return vw_fail(ctx, VW_ENULL, "median buffers cannot be null");
    if (n_local < 1) return vw_fail(ctx, VW_EEMPTY, "span cannot be empty");
    SpanSel *st = (SpanSel *)state;
    const unsigned int cap = span_cap(n_local);
    double *cand = (double *)((char *)state + 256);
    const int bits = span_bits(round), shift = span_shift(round);
    if ((rc = vw_cuda_check(ctx, cudaMemsetAsync(hist, 0, (size_t)(2 << bits) * sizeof(uint64_t), ctx->stream), "median memset")))
        return rc;
    int64_t chunks = (n_local + 256 * 16 - 1) / (256 * 16);
    if (chunks > (int64_t)ctx->sm_count * 16) chunks = (int64_t)ctx->sm_count * 16;
    if (chunks < 1) chunks = 1;
    if (round == 2) {
        // the 24 decided bits are the same on every rank: compact this span's keys that share them
        const dim3 grid((unsigned)chunks, 1, 1);
        k_select_collect<<<grid, 256, 0, ctx->stream>>>(c, 1, n_local, n_local, &st->s, 2 * kBig, cand, cap);
        k_select_mirror_count<<<1, 128, 0, ctx->stream>>>(&st->s, 1);
        ctx->launches += 2;
    }
    unsigned long long *h = (unsigned long long *)hist;
    if (bits == kBig) k_span_hist<kBig><<<(unsigned)chunks, 256, 0, ctx->stream>>>(c, n_local, st, shift, h, nullptr, 0u);
    else k_span_hist<8><<<(unsigned)chunks, 256, 0, ctx->stream>>>(c, n_local, st, shift, h, cand, cap);
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "median histogram launch");
}

int vw_span_median_pick(vw_ctx *ctx, void *state, int32_t round, const uint64_t *hist_sum) {
    if (!ctx) return VW_ENULL;
    vwshim::DeviceGuard g(ctx, "vw_span_median_pick");
    int rc;
    if ((rc = vw_span_rounds_check(ctx, round))) return rc;
    if (!state || !hist_sum) return vw_fail(ctx, VW_ENULL, "median buffers cannot be null");
    const unsigned long long *h = (const unsigned long long *)hist_sum;
    if (span_bits(round) == kBig) k_span_pick<kBig><<<2, 256, 0, ctx->stream>>>((SpanSel *)state, h);
    else k_span_pick<8><<<2, 256, 0, ctx->stream>>>((SpanSel *)state, h);
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "median pick launch");
}

int vw_span_median_value(vw_ctx *ctx, const void *state, double factor, double *out_dev) {
    if (!ctx) return VW_ENULL;
    vwshim::DeviceGuard g(ctx, "vw_span_median_value");
    if (!state || !out_dev) return vw_fail(ctx, VW_ENULL, "median buffers cannot be null");
    k_span_finish<<<1, 1, 0, ctx->stream>>>((const SpanSel *)state, factor, out_dev);
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "median value launch");
}

}  // extern "C"

// ---- SURE threshold (CORE/denoising/WaveletDenoiser.java:441-492) -------------------------------------------------
// The reference scores every candidate threshold t = |c_i| with a full pass over the coefficients (an O(n^2) double
// loop) and keeps the first minimum in ascending order of t.  Here one thread owns kSureCand candidates and walks the
// coefficients in the reference's order with the reference's roundings (separate multiplies and adds, no contraction),
// so every risk is bit-identical to the JVM's; (|c|, c*c) pairs are staged through shared memory and broadcast.  The
// sort disappears: "first minimum in ascending t" = the smallest t among the candidates of minimal risk.
namespace {
constexpr int kSureThreads = 256, kSureCand = 4, kSureChunk = 2048;

struct SureBest { double risk, t; };

__device__ __forceinline__ SureBest sure_better(SureBest a, SureBest b) {
    if (a.risk < b.risk) return a;
    if (b.risk < a.risk) return b;
    a.t = a.t < b.t ? a.t : b.t;
    return a;
}

__global__ void __launch_bounds__(kSureThreads) k_sure_scan(const double *__restrict__ c, int64_t batch, int64_t n, int64_t ld,
                                                            const double *__restrict__ sigma, SureBest *partial) {
    __shared__ double2 sm[kSureChunk];
    __shared__ SureBest red[kSureThreads / 32];
    for (int64_t row = blockIdx.y; row < batch; row += gridDim.y) {
        const double *r = c + row * ld;
        const double sigma2 = __dmul_rn(sigma[row], sigma[row]);             // :479
        double t[kSureCand], risk[kSureCand];
        const int64_t i0 = ((int64_t)blockIdx.x * kSureThreads + threadIdx.x) * kSureCand;
#pragma unroll
        for (int q = 0; q < kSureCand; q++) {
            t[q] = i0 + q < n ? fabs(r[i0 + q]) : 0.0;
            risk[q] = __dmul_rn((double)(-(long long)n), sigma2);            // :480  -n * sigma2
        }
        for (int64_t j0 = 0; j0 < n; j0 += kSureChunk) {
            const int m = (int)(n - j0 < kSureChunk ? n - j0 : kSureChunk);
            __syncthreads();
            for (int j = threadIdx.x; j < m; j += kSureThreads) {
                const double x = r[j0 + j];
                sm[j] = make_double2(fabs(x), __dmul_rn(x, x));
            }
            __syncthreads();
#pragma unroll 4
            for (int j = 0; j < m; j++) {
                const double2 p = sm[j];
#pragma unroll
                for (int q = 0; q < kSureCand; q++) {
                    const double d = __dsub_rn(p.x, t[q]);
                    const double over = __dadd_rn(sigma2, __dmul_rn(d, d));  // :487
                    risk[q] = __dadd_rn(risk[q], p.x <= t[q] ? p.y : over);  // :484-488 (NaN compares false: else branch)
                }
            }
        }
        SureBest best{INFINITY, 0.0};                                        // :452-453 minRisk = +inf, bestThreshold = 0
#pragma unroll
        for (int q = 0; q < kSureCand; q++) {
            const double rk = __ddiv_rn(risk[q], (double)n);                 // :491
            if (i0 + q < n && rk < INFINITY) best = sure_better(best, SureBest{rk, t[q]});   // `risk < minRisk` never takes NaN / +inf
        }
        for (int o = 16; o > 0; o >>= 1) {
            SureBest other{__shfl_down_sync(0xffffffffu, best.risk, o), __shfl_down_sync(0xffffffffu, best.t, o)};
            best = sure_better(best, other);
        }
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = best;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < kSureThreads / 32; w++) best = sure_better(best, red[w]);
            partial[row * gridDim.x + blockIdx.x] = best;
        }
    }
}

__global__ void __launch_bounds__(256) k_sure_finish(const SureBest *partial, int per_row, double *thr_out, double *risk_out) {
    __shared__ SureBest red[8];
    SureBest best{INFINITY, 0.0};
    for (int i = threadIdx.x; i < per_row; i += 256) best = sure_better(best, partial[(int64_t)blockIdx.x * per_row + i]);
    for (int o = 16; o > 0; o >>= 1) {
        SureBest other{__shfl_down_sync(0xffffffffu, best.risk, o), __shfl_down_sync(0xffffffffu, best.t, o)};
        best = sure_better(best, other);
    }
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; w++) best = sure_better(best, red[w]);
        thr_out[blockIdx.x] = best.t;
        risk_out[blockIdx.x] = best.risk;
    }
}
}  // namespace

size_t vw_sure_workspace(int64_t batch, int64_t n) {
    const int64_t per_row = (n + kSureThreads * kSureCand - 1) / (kSureThreads * kSureCand);
    return (size_t)batch * (size_t)per_row * sizeof(SureBest);
}

int vw_launch_sure(vw_ctx *ctx, const double *c, int64_t batch, int64_t n, int64_t ld, const double *sigma_dev, void *ws,
                   double *thr_dev, double *risk_dev) {
    if (batch <= 0 || n <= 0) return VW_OK;
    const int64_t per_row = (n + kSureThreads * kSureCand - 1) / (kSureThreads * kSureCand);
    const dim3 grid((unsigned)per_row, (unsigned)(batch < 65535 ? batch : 65535));
    k_sure_scan<<<grid, kSureThreads, 0, ctx->stream>>>(c, batch, n, ld, sigma_dev, (SureBest *)ws);
    k_sure_finish<<<(unsigned)batch, 256, 0, ctx->stream>>>((const SureBest *)ws, (int)per_row, thr_dev, risk_dev);
    ctx->launches += 2;
    return vw_cuda_check(ctx, cudaGetLastError(), "sure launch");
}

// ---- WaveletDenoiser's threshold selectors (CORE/denoising/WaveletDenoiser.java:391-552) ---------------------------------
// One thread per (level, row).  The device does only correctly rounded operations in denoising.py's left-to-right order
// (no contraction), so every threshold is the one the single-signal path computes on the host from the same medians,
// variances and SURE arg-mins.
namespace {
__global__ void k_denoise_select(const VwDenoiseSel a) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)a.levels * a.batch) return;
    const int j = (int)(i / a.batch);                          // level j + 1
    const int64_t b = i - (int64_t)j * a.batch;
    const double sigma = __ddiv_rn(a.med[b], 0.6745);          // estimateNoiseSigma (:376-387)
    const double s = a.multilevel ? __ddiv_rn(sigma, a.level_scale[j]) : sigma;   // sigma / sqrt(2^j) (:221)
    if (a.sig) { a.sig[i] = s; return; }
    double t;
    switch (a.method) {
        case VW_THR_UNIVERSAL: t = __dmul_rn(s, a.root); break;
        case VW_THR_MINIMAX:                                   // :497-509
            if (a.n <= 32) t = 0.0;
            else if (a.n <= 64) t = __dadd_rn(__dmul_rn(s, 0.3936), __dmul_rn(__dmul_rn(0.1829, s), a.log_n));
            else t = __dmul_rn(s, a.minimax_c);
            break;
        case VW_THR_BAYES: {                                   // :521-552; Python's max(0.0, d) keeps 0.0 unless d > 0
            const double s2 = __dmul_rn(s, s);
            const double d = __dsub_rn(a.var[i], s2);
            const double sx = __dsqrt_rn(__dadd_rn(d > 0.0 ? d : 0.0, 1e-10));
            t = __ddiv_rn(s2, sx);
            break;
        }
        case VW_THR_SURE: {                                    // :465-469 capped at the universal threshold
            const double u = __dmul_rn(s, a.root);
            t = a.sure[i] > u ? u : a.sure[i];
            break;
        }
        default: t = a.fixed; break;                           // VW_THR_FIXED
    }
    a.thr[i] = t;
}
}  // namespace

int vw_launch_denoise_select(vw_ctx *ctx, const VwDenoiseSel &a) {
    const int64_t count = (int64_t)a.levels * a.batch;
    if (count <= 0) return VW_OK;
    k_denoise_select<<<(unsigned)((count + 127) / 128), 128, 0, ctx->stream>>>(a);
    ctx->launches++;
    return vw_cuda_check(ctx, cudaGetLastError(), "denoise select launch");
}
