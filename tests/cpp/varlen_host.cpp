// Mixed-length MODWTTransform::forwardBatch of the C++ host mirror (include/vw_modwt.hpp) -- one
// vw_modwt_forward_varlen call -- against the CPU oracle, row by row, in every boundary mode.  Prints "ok" on success.
#include <cmath>
#include <cstdio>
#include <random>
#include <vector>

#include "vw_modwt.hpp"

extern "C" void vwo_forward_single(const double *x, int64_t n, const double *h, const double *g, int64_t l, int mode,
                                   double *v, double *w);

using namespace vectorwave;

int main() {
    std::mt19937_64 rng(7);
    std::normal_distribution<double> nd(0.0, 1.0);
    const std::vector<int> lengths = {1, 2, 3, 5, 7, 16, 31, 64, 97, 1000, 4099, 1 << 16, 1, 3};
    std::vector<std::vector<double>> rows;
    double amax = 0.0;
    for (int n : lengths) {
        std::vector<double> r(n);
        for (double &x : r) { x = nd(rng); amax = std::fmax(amax, std::fabs(x)); }
        rows.push_back(r);
    }
    const double tol = 1e-12 * std::fmax(1.0, amax);
    int bad = 0;
    for (const Wavelet &wv : {wavelets::db4(), wavelets::sym8(), wavelets::coif5()}) {
        const std::vector<double> h = wv.lowPassDecomposition(), g = wv.highPassDecomposition();
        for (BoundaryMode m : {BoundaryMode::PERIODIC, BoundaryMode::ZERO_PADDING, BoundaryMode::SYMMETRIC}) {
            const std::vector<MODWTResult> out = MODWTTransform(wv, m).forwardBatch(rows);
            if (out.size() != rows.size()) { std::printf("%s: %zu results\n", wv.name().c_str(), out.size()); return 1; }
            for (size_t b = 0; b < rows.size(); b++) {
                const int64_t n = (int64_t)rows[b].size();
                std::vector<double> v(n), w(n);
                vwo_forward_single(rows[b].data(), n, h.data(), g.data(), (int64_t)h.size(), (int)m, v.data(), w.data());
                const std::vector<double> gv = out[b].approximationCoeffs(), gw = out[b].detailCoeffs();
                double err = 0.0;
                for (int64_t t = 0; t < n; t++) err = std::fmax(err, std::fmax(std::fabs(gv[t] - v[t]), std::fabs(gw[t] - w[t])));
                if (!(err <= tol)) {
                    std::printf("%s mode %d row %zu (n = %lld): max error %.3e\n", wv.name().c_str(), (int)m, b, (long long)n, err);
                    bad++;
                }
            }
        }
    }
    // an empty row fails the whole batch with the reference's VAL_EMPTY
    try {
        MODWTTransform(wavelets::db4(), BoundaryMode::PERIODIC).forwardBatch({{1.0, 2.0, 3.0}, {}, {4.0}});
        std::printf("empty row accepted\n");
        bad++;
    } catch (const InvalidSignalException &e) {
        if (e.code != "VAL_006") { std::printf("empty row: code %s\n", e.code.c_str()); bad++; }
    }
    if (bad) return 1;
    std::printf("ok\n");
    return 0;
}
