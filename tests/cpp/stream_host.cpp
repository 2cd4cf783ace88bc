// BatchStreamingMODWT of the C++ host mirror (include/vw_modwt.hpp) -- the engine's stream state -- against the CPU
// oracle: a ZERO_PADDING stream's concatenated blocks equal the whole-signal ZERO_PADDING decomposition, and a SYMMETRIC
// first block equals the SYMMETRIC decomposition of that block.  Prints "ok" on success.
#include <cmath>
#include <cstdio>
#include <random>
#include <vector>

#include "vw_modwt.hpp"

extern "C" int vwo_decompose(const double *x, int64_t n, const double *h, const double *g, int64_t l, int levels, int mode,
                             int dense, double *w, double *v);

using namespace vectorwave;

int main() {
    std::mt19937_64 rng(11);
    std::normal_distribution<double> nd(0.0, 1.0);
    const int batch = 3, total = 3000;
    std::vector<std::vector<double>> x(batch, std::vector<double>(total));
    double amax = 0.0;
    for (auto &r : x) for (double &v : r) { v = nd(rng); amax = std::fmax(amax, std::fabs(v)); }
    const double tol = 1e-12 * amax;
    int bad = 0;
    struct Case { Wavelet w; int levels; };
    for (const Case &c : {Case{wavelets::haar(), 5}, Case{wavelets::db4(), 4}, Case{wavelets::sym8(), 3}, Case{wavelets::coif5(), 2}}) {
        const std::vector<double> h = c.w.lowPassDecomposition(), g = c.w.highPassDecomposition();
        const int J = c.levels;
        // ZERO_PADDING: blocks of odd sizes, one shorter than every history
        BatchStreamingMODWT zp(c.w, BoundaryMode::ZERO_PADDING, J);
        std::vector<double> w((size_t)J * batch * total), v((size_t)batch * total);
        int at = 0;
        for (int len : {700, 3, 997, 1300}) {
            std::vector<std::vector<double>> blk(batch);
            for (int b = 0; b < batch; b++) blk[b].assign(x[b].begin() + at, x[b].begin() + at + len);
            const BatchMODWT::MultiLevelResult r = zp.processMultiLevel(blk);
            for (int j = 0; j < J; j++)
                for (int b = 0; b < batch; b++)
                    for (int t = 0; t < len; t++)
                        w[((size_t)j * batch + b) * total + at + t] = r.detailPerLevel[((size_t)j * batch + b) * len + t];
            for (int b = 0; b < batch; b++)
                for (int t = 0; t < len; t++) v[(size_t)b * total + at + t] = r.finalApprox[(size_t)b * len + t];
            at += len;
        }
        for (int b = 0; b < batch; b++) {
            std::vector<double> wo((size_t)J * total), vo(total);
            vwo_decompose(x[b].data(), total, h.data(), g.data(), (int64_t)h.size(), J, VW_ZERO_PADDING, 0, wo.data(), vo.data());
            double err = 0.0;
            for (int t = 0; t < total; t++) {
                err = std::fmax(err, std::fabs(v[(size_t)b * total + t] - vo[t]));
                for (int j = 0; j < J; j++) err = std::fmax(err, std::fabs(w[((size_t)j * batch + b) * total + t] - wo[(size_t)j * total + t]));
            }
            if (!(err <= tol)) { std::printf("%s ZERO_PADDING row %d: max error %.3e\n", c.w.name().c_str(), b, err); bad++; }
        }
        // SYMMETRIC: the first block equals the SYMMETRIC decomposition of that block
        const int n = 512;
        BatchStreamingMODWT sy(c.w, BoundaryMode::SYMMETRIC, J);
        std::vector<std::vector<double>> blk(batch);
        for (int b = 0; b < batch; b++) blk[b].assign(x[b].begin(), x[b].begin() + n);
        const BatchMODWT::MultiLevelResult r = sy.processMultiLevel(blk);
        for (int b = 0; b < batch; b++) {
            std::vector<double> wo((size_t)J * n), vo(n);
            vwo_decompose(blk[b].data(), n, h.data(), g.data(), (int64_t)h.size(), J, VW_SYMMETRIC, 0, wo.data(), vo.data());
            double err = 0.0;
            for (int t = 0; t < n; t++) {
                err = std::fmax(err, std::fabs(r.finalApprox[(size_t)b * n + t] - vo[t]));
                for (int j = 0; j < J; j++) err = std::fmax(err, std::fabs(r.detailPerLevel[((size_t)j * batch + b) * n + t] - wo[(size_t)j * n + t]));
            }
            if (!(err <= tol)) { std::printf("%s SYMMETRIC row %d: max error %.3e\n", c.w.name().c_str(), b, err); bad++; }
        }
        // flush: one call, the tail of every row
        const BatchMODWT::MultiLevelResult f = sy.flushMultiLevel(sy.getMinFlushTailLength());
        if (f.batch != batch || f.n != (int)h.size() - 1) { std::printf("%s flush shape %d x %d\n", c.w.name().c_str(), f.batch, f.n); bad++; }
    }
    try {
        BatchStreamingMODWT(wavelets::db4(), BoundaryMode::SYMMETRIC, 2).flushMultiLevel(3);
        std::printf("flush before any block accepted\n");
        bad++;
    } catch (const IllegalStateException &) {
    }
    if (bad) return 1;
    std::printf("ok\n");
    return 0;
}
