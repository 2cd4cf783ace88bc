// vw_modwt.hpp -- C++17 host-side mirror of VectorWave's MODWT / SWT classes over the C ABI of vw_modwt.h.
//
// The reference (MorphIQ-Labs/VectorWave) is Java and the build image has no JDK, so next to the Java FFM binding
// (java/, source only) and the Python mirror (vectorwave_b200/*.py, used by the test-suite) this header gives a
// compiled-language host: the same class and method names, argument meaning and error behaviour as the reference
// for the path, header-only, linking nothing but libvwmodwt.so.  CORE = vectorwave-core/src/main/java/com/
// morphiqlabs/wavelet, EXT = vectorwave-extensions/src/main/java/com/morphiqlabs/wavelet.
//
//   vectorwave::MODWTTransform            CORE/modwt/MODWTTransform.java:91-299,486-559
//   vectorwave::MultiLevelMODWTTransform  CORE/modwt/MultiLevelMODWTTransform.java:181-446
//   vectorwave::VectorWaveSwtAdapter      CORE/swt/VectorWaveSwtAdapter.java:184-562
//   vectorwave::BatchMODWT                EXT/extensions/modwt/BatchMODWT.java:62-178
//   vectorwave::SymmetricAlignmentStrategy / computeTauJ   CORE/modwt/SymmetricAlignmentStrategy.java:43-117,
//                                                          MultiLevelMODWTTransform.java:795-806
// What stays on this side of the ABI is exactly what INTEGRATION.md lists: tables, the 1/sqrt(2) scaling, the level cap
// of 9, the alignment table, result types and exceptions.  There is no CPU compute path: Engine() throws when no CUDA
// device exists.
#pragma once
#include <cmath>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "vw_modwt.h"

namespace vectorwave {

// ---- exceptions (CORE/exception/*.java; codes CORE/exception/ErrorCode.java:24-118) -------------------------------
struct WaveletTransformException : std::runtime_error {
    std::string code;
    WaveletTransformException(const std::string &m, std::string c = "") : std::runtime_error(m), code(std::move(c)) {}
};
struct InvalidSignalException : WaveletTransformException { using WaveletTransformException::WaveletTransformException; };
struct InvalidArgumentException : WaveletTransformException { using WaveletTransformException::WaveletTransformException; };
struct IllegalArgumentException : std::invalid_argument { using std::invalid_argument::invalid_argument; };
struct NativeEngineError : std::runtime_error { using std::runtime_error::runtime_error; };

// ---- BoundaryMode (CORE/api/BoundaryMode.java:26-50); values are vw_boundary ----------------------------------------
enum class BoundaryMode : int { PERIODIC = VW_PERIODIC, ZERO_PADDING = VW_ZERO_PADDING, SYMMETRIC = VW_SYMMETRIC, CONSTANT = VW_CONSTANT };

// ---- wavelets: orthogonal tables as data (Haar.java:39-43, Daubechies.java:61-160, Symlet.java:91-161,
//      Coiflet.java:63-178); g[i] = (-1)^i h[L-1-i] (Daubechies.java:323-330); reconstruction == decomposition ----------
class Wavelet {
public:
    enum class Id { OTHER, HAAR, DB6, DB8, SYM4, SYM8, COIF2, COIF3 };   // the identities SymmetricAlignmentStrategy tests
    Wavelet(std::string name, std::vector<double> h, Id id = Id::OTHER) : name_(std::move(name)), h_(std::move(h)), id_(id) {}
    const std::string &name() const { return name_; }
    Id id() const { return id_; }
    std::vector<double> lowPassDecomposition() const { return h_; }
    std::vector<double> highPassDecomposition() const {
        const size_t l = h_.size();
        std::vector<double> g(l);
        for (size_t i = 0; i < l; i++) g[i] = (i % 2 == 0 ? 1.0 : -1.0) * h_[l - 1 - i];
        return g;
    }
    std::vector<double> lowPassReconstruction() const { return lowPassDecomposition(); }
    std::vector<double> highPassReconstruction() const { return highPassDecomposition(); }

private:
    std::string name_;
    std::vector<double> h_;
    Id id_;
};

namespace wavelets {
inline Wavelet haar() { const double s = 1.0 / std::sqrt(2.0); return Wavelet("Haar", {s, s}, Wavelet::Id::HAAR); }
inline Wavelet db2() { return Wavelet("db2", {0.4829629131445341, 0.8365163037378079, 0.2241438680420134, -0.1294095225512603}); }
inline Wavelet db4() {
    return Wavelet("db4", {0.2303778133088964, 0.7148465705529154, 0.6308807679298587, -0.0279837693982488,
                           -0.1870348117190931, 0.0308413818355607, 0.0328830116668852, -0.0105974017850690});
}
inline Wavelet db8() {
    return Wavelet("db8", {0.0544158422431049, 0.3128715909143031, 0.6756307362972904, 0.5853546836541907,
                           -0.0158291052563816, -0.2840155429615702, 0.0004724845739124, 0.1287474266204837,
                           -0.0173693010018083, -0.0440882539307952, 0.0139810279173995, 0.0087460940474061,
                           -0.0048703529934518, -0.0003917403733770, 0.0006754494064506, -0.0001174767841248}, Wavelet::Id::DB8);
}
inline Wavelet sym4() {
    return Wavelet("sym4", {0.03222310060407815, -0.01260396726226383, -0.09921954357695636, 0.29785779560553225,
                            0.80373875180591614, 0.49761866763256292, -0.02963552764596039, -0.07576571478935668}, Wavelet::Id::SYM4);
}
inline Wavelet sym8() {
    return Wavelet("sym8", {-0.003382415951359, -0.000542132331635, 0.031695087810979, 0.007607487324918,
                            -0.143294238350810, -0.061273359067938, 0.481359651258372, 0.777185751700574,
                            0.364441894835509, -0.051945838107658, -0.027219029168752, 0.049137179673713,
                            0.003808752013903, -0.014952258336792, -0.000302920514551, 0.001889950332768}, Wavelet::Id::SYM8);
}
inline Wavelet coif5() {
    return Wavelet("coif5", {-0.0000000960401011, -0.0000001623799517, 0.0000020612203986, 0.0000037007277113,
                             -0.0000212702216725, -0.0000412198619243, 0.0001403563281237, 0.0003018579416682,
                             -0.0006375589261259, -0.0016616273039299, 0.0024315754425383, 0.0067615202206204,
                             -0.0091595073386762, -0.0197583916009655, 0.0326747994670574, 0.0412875304721178,
                             -0.1055631513073372, -0.0620377515749820, 0.4379823066591634, 0.7742936228603274,
                             0.4215712667307543, -0.0520466702535548, -0.0919215880600861, 0.0281697442705324,
                             0.0234083221189278, -0.0101315848469003, -0.0041593126275786, 0.0021782943778457,
                             0.0003585777411618, -0.0002120818620675});
}
}  // namespace wavelets

// ---- engine handle ----------------------------------------------------------------------------------------------
class Engine {
public:
    explicit Engine(int device = -1) {
        const int rc = vw_init(device, &ctx_);
        if (rc != VW_OK) throw NativeEngineError(std::string("vw_init failed: ") + vw_status_name(rc) + " (the MODWT engine has no CPU path)");
    }
    ~Engine() { if (ctx_) vw_destroy(ctx_); }
    Engine(const Engine &) = delete;
    Engine &operator=(const Engine &) = delete;
    vw_ctx *ctx() const { return ctx_; }
    static Engine &get() { static thread_local Engine e; return e; }   // one ctx per host thread (vw_modwt.h)

    // status -> the reference's exception vocabulary (same table as vectorwave_b200/_native.py:_STATUS)
    void check(int rc) const {
        if (rc == VW_OK) return;
        const std::string msg = vw_last_error(ctx_);
        switch (rc) {
            case VW_ENONFINITE: throw InvalidSignalException(msg, "VAL_003");
            case VW_EEMPTY: throw InvalidSignalException(msg, "VAL_006");
            case VW_ETOOLARGE: throw InvalidArgumentException(msg, "VAL_005");
            case VW_EBOUNDARY: throw InvalidArgumentException(msg, "CFG_003");
            case VW_ELEVEL: throw InvalidArgumentException(msg, "CFG_004");
            case VW_ENULL: case VW_ELENGTH: case VW_EINVAL: throw IllegalArgumentException(msg);
            default: throw NativeEngineError(msg);
        }
    }

private:
    vw_ctx *ctx_ = nullptr;
};

namespace detail {
inline const double kScale = 1.0 / std::sqrt(2.0);   // 1.0 / Math.sqrt(2.0)
inline std::vector<double> scaled(const std::vector<double> &f) {
    std::vector<double> s(f.size());
    for (size_t i = 0; i < f.size(); i++) s[i] = f[i] * kScale;   // one rounding per tap, ScalarOps.java:909-916
    return s;
}
inline void require_mode(BoundaryMode m) {
    if (m != BoundaryMode::PERIODIC && m != BoundaryMode::ZERO_PADDING && m != BoundaryMode::SYMMETRIC)
        throw InvalidArgumentException("MODWT only supports PERIODIC, ZERO_PADDING, and SYMMETRIC boundary modes", "CFG_003");
}
}  // namespace detail

// ---- SymmetricAlignmentStrategy.decide (:43-117) and computeTauJ (:795-806) ------------------------------------------
struct SymmetricAlignmentStrategy {
    struct Decision { bool approxPlus; int deltaH; bool detailPlus; int deltaG; };
    static Decision decide(const Wavelet &w, int level) {
        const int l0 = (int)w.lowPassReconstruction().size();
        if (l0 <= 2) return {true, level <= 1 ? 0 : -1, true, 0};
        bool ap = false, dp = true;
        int dh = 0, dg = 0;
        switch (w.id()) {
            case Wavelet::Id::DB6: dh = level <= 1 ? 0 : -1; dg = level >= 3 ? 1 : 0; break;
            case Wavelet::Id::DB8: dh = level <= 1 ? 0 : 1; dg = level >= 2 ? 1 : 0; break;
            case Wavelet::Id::SYM4: ap = true; dp = false; break;
            case Wavelet::Id::SYM8: if (level == 2) dh = 1; else if (level > 2) { dh = 1; dg = 1; } break;
            case Wavelet::Id::COIF2: ap = true; dp = false; dh = level <= 1 ? 0 : 1; break;
            case Wavelet::Id::COIF3: dp = false; if (level > 1) { dh = -1; dg = 1; } break;
            default:
                if (l0 >= 12) dh = dg = (level <= 1 || level % 2 == 0) ? 0 : -1;
                else if (level > 1) dh = -1;
        }
        return {ap, dh, dp, dg};
    }
    static int computeTauJ(int baseFilterLength, int level) {
        const int lm1 = baseFilterLength - 1;
        if (level <= 1) return lm1 / 2 > 0 ? lm1 / 2 : 0;
        return (int)(((int64_t)lm1 * ((int64_t)1 << (level - 1))) / 2);
    }
};

// ---- results ----------------------------------------------------------------------------------------------------
class MODWTResult {   // CORE/modwt/MODWTResult.java:25-110: two same-length arrays, copies out
public:
    MODWTResult(std::vector<double> approx, std::vector<double> detail) : a_(std::move(approx)), d_(std::move(detail)) {
        if (a_.size() != d_.size()) throw IllegalArgumentException("Approximation and detail coefficients must have the same length");
        if (a_.empty()) throw IllegalArgumentException("Coefficient arrays cannot be empty");
    }
    static MODWTResult create(std::vector<double> a, std::vector<double> d) { return MODWTResult(std::move(a), std::move(d)); }
    std::vector<double> approximationCoeffs() const { return a_; }
    std::vector<double> detailCoeffs() const { return d_; }
    int getSignalLength() const { return (int)a_.size(); }

private:
    std::vector<double> a_, d_;
};

class MultiLevelMODWTResult {   // CORE/modwt/MultiLevelMODWTResult.java:32-99: level 1 = finest, every array length N
public:
    MultiLevelMODWTResult(int levels, int n) : levels_(levels), n_(n), w_((size_t)levels * n), v_(n) {}
    int getLevels() const { return levels_; }
    int getSignalLength() const { return n_; }
    std::vector<double> getDetailCoeffsAtLevel(int level) const {
        if (level < 1 || level > levels_) throw InvalidArgumentException("Invalid level: " + std::to_string(level), "CFG_004");
        return std::vector<double>(w_.begin() + (size_t)(level - 1) * n_, w_.begin() + (size_t)level * n_);
    }
    std::vector<double> getApproximationCoeffs() const { return v_; }
    double getDetailEnergyAtLevel(int level) const { double e = 0; for (double c : getDetailCoeffsAtLevel(level)) e += c * c; return e; }
    double getApproximationEnergy() const { double e = 0; for (double c : v_) e += c * c; return e; }
    // live storage ([J][N] block + V_J), as MutableMultiLevelMODWTResult exposes it
    double *detailData() { return w_.data(); }
    const double *detailData() const { return w_.data(); }
    double *approxData() { return v_.data(); }
    const double *approxData() const { return v_.data(); }

private:
    int levels_, n_;
    std::vector<double> w_, v_;
};

// ---- MODWTTransform -------------------------------------------------------------------------------------------------
class MODWTTransform {
public:
    MODWTTransform(Wavelet w, BoundaryMode m) : wavelet_(std::move(w)), mode_(m) {
        detail::require_mode(m);
        hs_ = detail::scaled(wavelet_.lowPassDecomposition());
        gs_ = detail::scaled(wavelet_.highPassDecomposition());
    }
    const Wavelet &getWavelet() const { return wavelet_; }
    BoundaryMode getBoundaryMode() const { return mode_; }

    MODWTResult forward(const std::vector<double> &signal) const {   // :131-189
        if (signal.empty()) throw InvalidSignalException("Signal cannot be empty", "VAL_006");
        const int64_t n = (int64_t)signal.size();
        std::vector<double> v(n), w(n);
        Engine &e = Engine::get();
        e.check(vw_modwt_forward(e.ctx(), signal.data(), 1, n, n, hs_.data(), gs_.data(), (int)hs_.size(), 1, (int)mode_, w.data(), n,
                                 n, v.data(), n, VW_FLAG_CHECK_FINITE));
        return MODWTResult(std::move(v), std::move(w));
    }
    std::vector<double> inverse(const MODWTResult &r) const {   // :203-299: pair-added; SYMMETRIC uses t - l
        const int64_t n = r.getSignalLength();
        const std::vector<double> v = r.approximationCoeffs(), w = r.detailCoeffs();
        std::vector<double> x(n);
        const vw_align sym{-1, 0, -1, 0};
        Engine &e = Engine::get();
        e.check(vw_modwt_inverse(e.ctx(), w.data(), n, n, v.data(), n, 1, n, hs_.data(), gs_.data(), (int)hs_.size(), 1, (int)mode_,
                                 mode_ == BoundaryMode::SYMMETRIC ? &sym : nullptr, VW_ORDER_PAIR, 1ull, 1, x.data(), n, 0));
        return x;
    }
    std::vector<MODWTResult> forwardBatch(const std::vector<std::vector<double>> &signals) const {   // :486-515
        std::vector<MODWTResult> out;
        if (signals.empty()) return out;
        const int64_t b = (int64_t)signals.size(), n = (int64_t)signals[0].size();
        bool same = true;
        for (const auto &s : signals) same = same && (int64_t)s.size() == n;
        if (!same) return forwardMixed(signals);
        if (n == 0) throw InvalidSignalException("Signal cannot be empty", "VAL_006");
        std::vector<double> x((size_t)b * n), w((size_t)b * n), v((size_t)b * n);
        for (int64_t i = 0; i < b; i++) std::copy(signals[i].begin(), signals[i].end(), x.begin() + i * n);
        Engine &e = Engine::get();
        e.check(vw_modwt_forward(e.ctx(), x.data(), b, n, n, hs_.data(), gs_.data(), (int)hs_.size(), 1, (int)mode_, w.data(), n,
                                 b * n, v.data(), n, VW_FLAG_CHECK_FINITE));
        for (int64_t i = 0; i < b; i++)
            out.emplace_back(std::vector<double>(v.begin() + i * n, v.begin() + (i + 1) * n),
                             std::vector<double>(w.begin() + i * n, w.begin() + (i + 1) * n));
        return out;
    }

private:
    // rows of different lengths: one packed vw_modwt_forward_varlen call; rows are validated in index order (the first
    // empty or non-finite row throws, as forward() per row would)
    std::vector<MODWTResult> forwardMixed(const std::vector<std::vector<double>> &signals) const {
        const int64_t b = (int64_t)signals.size();
        std::vector<int64_t> off((size_t)b + 1, 0);
        for (int64_t i = 0; i < b; i++) off[i + 1] = off[i] + (int64_t)signals[i].size();
        std::vector<double> x((size_t)off[b]), w((size_t)off[b]), v((size_t)off[b]);
        for (int64_t i = 0; i < b; i++) std::copy(signals[i].begin(), signals[i].end(), x.begin() + off[i]);
        Engine &e = Engine::get();
        e.check(vw_modwt_forward_varlen(e.ctx(), x.data(), off.data(), b, hs_.data(), gs_.data(), (int)hs_.size(), (int)mode_,
                                        w.data(), v.data(), VW_FLAG_CHECK_FINITE));
        std::vector<MODWTResult> out;
        out.reserve((size_t)b);
        for (int64_t i = 0; i < b; i++)
            out.emplace_back(std::vector<double>(v.begin() + off[i], v.begin() + off[i + 1]),
                             std::vector<double>(w.begin() + off[i], w.begin() + off[i + 1]));
        return out;
    }

    Wavelet wavelet_;
    BoundaryMode mode_;
    std::vector<double> hs_, gs_;
};

// ---- MultiLevelMODWTTransform -----------------------------------------------------------------------------------------
class MultiLevelMODWTTransform {
public:
    static constexpr int MAX_DECOMPOSITION_LEVELS = 10;   // :117 (the loop below caps at 9, pinned by the reference's tests)
    MultiLevelMODWTTransform(Wavelet w, BoundaryMode m) : wavelet_(std::move(w)), mode_(m) {
        detail::require_mode(m);
        hs_ = detail::scaled(wavelet_.lowPassDecomposition());
        gs_ = detail::scaled(wavelet_.highPassDecomposition());
    }
    int getMaximumLevels(int signalLength) const { return vw_max_levels(signalLength, (int)hs_.size(), MAX_DECOMPOSITION_LEVELS); }   // :455-501

    MultiLevelMODWTResult decompose(const std::vector<double> &signal, int levels = 0) const {   // :195-255
        const int n = (int)signal.size();
        if (n == 0) throw InvalidSignalException("Signal cannot be empty for multi-level MODWT", "VAL_006");
        const int maxLevels = getMaximumLevels(n);
        if (levels == 0) levels = maxLevels;
        if (levels < 1 || levels > maxLevels)
            throw InvalidArgumentException("Invalid number of decomposition levels: " + std::to_string(levels), "CFG_004");
        MultiLevelMODWTResult r(levels, n);
        Engine &e = Engine::get();
        e.check(vw_modwt_forward(e.ctx(), signal.data(), 1, n, n, hs_.data(), gs_.data(), (int)hs_.size(), levels, (int)mode_,
                                 r.detailData(), n, n, r.approxData(), n, VW_FLAG_CHECK_FINITE));
        return r;
    }
    std::vector<double> reconstruct(const MultiLevelMODWTResult &r) const { return run(r, mask(1, r.getLevels()), true); }   // :339-349
    std::vector<double> reconstructFromLevel(const MultiLevelMODWTResult &r, int startLevel) const {   // :361-386
        if (startLevel < 1 || startLevel > r.getLevels()) throw InvalidArgumentException("Invalid start level", "CFG_004");
        return run(r, mask(startLevel, r.getLevels()), true);
    }
    std::vector<double> reconstructLevels(const MultiLevelMODWTResult &r, int minLevel, int maxLevel) const {   // :398-446
        if (minLevel < 1 || maxLevel > r.getLevels() || minLevel > maxLevel)
            throw InvalidArgumentException("Invalid level range for partial reconstruction", "CFG_004");
        return run(r, mask(minLevel, maxLevel), r.getLevels() <= maxLevel);
    }
    // per-level (sigma, tau) of the SYMMETRIC inverse (:602-642) and the summation order of each mode (:578-601)
    std::vector<vw_align> alignment(int levels, int &order) const {
        std::vector<vw_align> al;
        order = mode_ == BoundaryMode::ZERO_PADDING ? VW_ORDER_PAIR : VW_ORDER_SPLIT;
        if (mode_ != BoundaryMode::SYMMETRIC) return al;
        const int l = (int)hs_.size();
        for (int level = 1; level <= levels; level++) {
            const auto d = SymmetricAlignmentStrategy::decide(wavelet_, level);
            al.push_back(vw_align{d.approxPlus ? 1 : -1, SymmetricAlignmentStrategy::computeTauJ(l, level) + d.deltaH,
                                  d.detailPlus ? 1 : -1, SymmetricAlignmentStrategy::computeTauJ(l, level) + d.deltaG});
        }
        return al;
    }
    const std::vector<double> &scaledLow() const { return hs_; }
    const std::vector<double> &scaledHigh() const { return gs_; }
    BoundaryMode getBoundaryMode() const { return mode_; }

private:
    static uint64_t mask(int lo, int hi) { uint64_t m = 0; for (int j = lo; j <= hi; j++) m |= 1ull << (j - 1); return m; }
    std::vector<double> run(const MultiLevelMODWTResult &r, uint64_t detailMask, bool useApprox) const {
        const int64_t n = r.getSignalLength();
        int order;
        const std::vector<vw_align> al = alignment(r.getLevels(), order);
        std::vector<double> x(n);
        Engine &e = Engine::get();
        e.check(vw_modwt_inverse(e.ctx(), r.detailData(), n, n, r.approxData(), n, 1, n, hs_.data(), gs_.data(), (int)hs_.size(),
                                 r.getLevels(), (int)mode_, al.empty() ? nullptr : al.data(), order, detailMask, useApprox ? 1 : 0,
                                 x.data(), n, 0));
        return x;
    }
    Wavelet wavelet_;
    BoundaryMode mode_;
    std::vector<double> hs_, gs_;
};

// ---- device-resident result (GpuResidentResult.java): MutableMultiLevelMODWTResult whose coefficients stay in HBM --------
class ResidentResult {
public:
    // MultiLevelMODWTTransform.decomposeMutable (:284-330) with the result kept on the device
    ResidentResult(const MultiLevelMODWTTransform &t, const std::vector<double> &signal, int levels) : t_(t), n_((int64_t)signal.size()), levels_(levels) {
        if (signal.empty()) throw InvalidSignalException("Signal cannot be empty for multi-level MODWT", "VAL_006");
        if (levels < 1 || levels > t.getMaximumLevels((int)signal.size()))
            throw InvalidArgumentException("Invalid number of decomposition levels: " + std::to_string(levels), "CFG_004");
        Engine &e = Engine::get();
        e.check(vw_modwt_decompose_h(e.ctx(), signal.data(), 1, n_, n_, t.scaledLow().data(), t.scaledHigh().data(), (int)t.scaledLow().size(),
                                     levels, (int)t.getBoundaryMode(), &res_, VW_FLAG_CHECK_FINITE));
    }
    ~ResidentResult() { if (res_) vw_result_free(Engine::get().ctx(), res_); }
    ResidentResult(const ResidentResult &) = delete;
    ResidentResult &operator=(const ResidentResult &) = delete;
    int getLevels() const { return levels_; }
    std::vector<double> getDetailCoeffsAtLevel(int level) const { return fetch(level, 1); }
    std::vector<double> getApproximationCoeffs() const { return fetch(0, 0); }
    void applyThreshold(int level, double threshold, bool soft) {   // MutableMultiLevelMODWTResult.applyThreshold (:83-118)
        Engine &e = Engine::get();
        e.check(vw_result_threshold(e.ctx(), res_, level, &threshold, 0, soft ? 1 : 0));
    }
    double applyUniversalThreshold(bool soft) {                     // VectorWaveSwtAdapter.applyUniversalThreshold (:505-520)
        double thr = 0.0;
        Engine &e = Engine::get();
        e.check(vw_result_universal_threshold(e.ctx(), res_, soft ? 1 : 0, &thr));
        return thr;
    }
    double getDetailEnergyAtLevel(int level) const { double v = 0; Engine &e = Engine::get(); e.check(vw_result_energy(e.ctx(), res_, level, &v)); return v; }
    std::vector<double> reconstruct() const {                       // MultiLevelMODWTTransform.reconstruct (:339-349)
        int order;
        const std::vector<vw_align> al = t_.alignment(levels_, order);
        std::vector<double> x((size_t)n_);
        Engine &e = Engine::get();
        e.check(vw_modwt_reconstruct_h(e.ctx(), res_, t_.scaledLow().data(), t_.scaledHigh().data(), (int)t_.scaledLow().size(),
                                       (int)t_.getBoundaryMode(), al.empty() ? nullptr : al.data(), order, (1ull << levels_) - 1, 1,
                                       x.data(), n_, 0));
        return x;
    }

private:
    std::vector<double> fetch(int level, int lo) const {
        if (level < lo || level > levels_) throw IllegalArgumentException("Level must be between 1 and " + std::to_string(levels_));
        std::vector<double> out((size_t)n_);
        Engine &e = Engine::get();
        e.check(vw_result_get_level(e.ctx(), res_, level, out.data(), n_, 0));
        return out;
    }
    const MultiLevelMODWTTransform &t_;
    int64_t n_;
    int levels_;
    vw_result *res_ = nullptr;
};

// ---- one long signal over several GPUs, driven by one host thread (vw_init_multi; INTEGRATION.md section 3) ---------------
class ShardedMODWT {
public:
    // devices: one entry per span (a device may be listed more than once); PERIODIC or ZERO_PADDING
    ShardedMODWT(const Wavelet &w, BoundaryMode m, int levels, int64_t n_local, const std::vector<int> &devices)
        : mode_(m), levels_(levels), n_(n_local), hs_(detail::scaled(w.lowPassDecomposition())), gs_(detail::scaled(w.highPassDecomposition())) {
        int rc = vw_span_plan_query((int)hs_.size(), levels, n_local, (int)devices.size(), &plan_);
        if (rc != VW_OK) throw IllegalArgumentException(std::string("vw_span_plan_query: ") + vw_status_name(rc));
        rc = vw_init_multi(devices.data(), (int)devices.size(), &m_);
        if (rc != VW_OK) throw NativeEngineError(std::string("vw_init_multi failed: ") + vw_status_name(rc));
        row_ = plan_.lead_w + n_ + plan_.pad;
        for (size_t r = 0; r < devices.size(); r++) {
            void *x, *wv, *v, *o;
            vw_ctx *c = vw_multi_ctx(m_, (int)r);
            if (vw_device_alloc(c, (size_t)(plan_.lead + n_) * 8, &x) || vw_device_alloc(c, (size_t)levels * row_ * 8, &wv) ||
                vw_device_alloc(c, (size_t)(n_ + plan_.pad) * 8, &v) || vw_device_alloc(c, (size_t)n_ * 8, &o))
                throw NativeEngineError("device allocation failed");
            xext_.push_back((double *)x); w_.push_back((double *)wv); v_.push_back((double *)v); out_.push_back((double *)o);
        }
    }
    ~ShardedMODWT() {
        for (size_t r = 0; r < xext_.size(); r++) {
            vw_ctx *c = vw_multi_ctx(m_, (int)r);
            vw_device_free(c, xext_[r]); vw_device_free(c, w_[r]); vw_device_free(c, v_[r]); vw_device_free(c, out_[r]);
        }
        if (m_) vw_destroy_multi(m_);
    }
    ShardedMODWT(const ShardedMODWT &) = delete;
    ShardedMODWT &operator=(const ShardedMODWT &) = delete;
    // signal: world * n_local samples on the host; details come back as [levels][world * n_local], approximation [world * n_local]
    void decompose(const std::vector<double> &signal, std::vector<double> &details, std::vector<double> &approx) {
        const size_t world = xext_.size(), total = world * (size_t)n_;
        if (signal.size() != total) throw IllegalArgumentException("signal length must be world * n_local");
        for (size_t r = 0; r < world; r++)
            chk(r, vw_copy_h2d(vw_multi_ctx(m_, (int)r), xext_[r] + plan_.lead, signal.data() + r * n_, (size_t)n_ * 8));
        mchk(vw_modwt_forward_sharded(m_, &plan_, xext_.data(), hs_.data(), gs_.data(), (int)mode_, w_.data(), row_, v_.data(), nullptr, 0));
        details.resize((size_t)levels_ * total); approx.resize(total);
        for (size_t r = 0; r < world; r++) {
            vw_ctx *c = vw_multi_ctx(m_, (int)r);
            for (int j = 0; j < levels_; j++)
                chk(r, vw_copy_d2h(c, details.data() + (size_t)j * total + r * n_, w_[r] + (size_t)j * row_ + plan_.lead_w, (size_t)n_ * 8));
            chk(r, vw_copy_d2h(c, approx.data() + r * n_, v_[r], (size_t)n_ * 8));
        }
    }
    // reconstruct from the coefficients the last decompose left on the devices
    std::vector<double> reconstruct() {
        const size_t world = xext_.size();
        mchk(vw_modwt_inverse_sharded(m_, &plan_, w_.data(), row_, v_.data(), hs_.data(), gs_.data(), (int)mode_,
                                      mode_ == BoundaryMode::ZERO_PADDING ? VW_ORDER_PAIR : VW_ORDER_SPLIT, out_.data(), nullptr, 0));
        std::vector<double> x(world * (size_t)n_);
        for (size_t r = 0; r < world; r++) chk(r, vw_copy_d2h(vw_multi_ctx(m_, (int)r), x.data() + r * n_, out_[r], (size_t)n_ * 8));
        return x;
    }
    // VectorWaveSwtAdapter.denoise of the whole signal (vw_swt_denoise_sharded): threshold < 0 selects the universal
    // threshold from the exact median of |W_1| over every span; *threshold_out (may be null) receives the value used.
    // The coefficients stay on the devices unthresholded, so reconstruct() afterwards gives the plain reconstruction.
    std::vector<double> denoise(const std::vector<double> &signal, double threshold = -1.0, bool soft = true,
                                double *threshold_out = nullptr) {
        const size_t world = xext_.size(), total = world * (size_t)n_;
        if (signal.size() != total) throw IllegalArgumentException("signal length must be world * n_local");
        for (size_t r = 0; r < world; r++)
            chk(r, vw_copy_h2d(vw_multi_ctx(m_, (int)r), xext_[r] + plan_.lead, signal.data() + r * n_, (size_t)n_ * 8));
        double thr = 0.0;
        const int rc = vw_swt_denoise_sharded(m_, &plan_, xext_.data(), hs_.data(), gs_.data(), (int)mode_,
                                              mode_ == BoundaryMode::ZERO_PADDING ? VW_ORDER_PAIR : VW_ORDER_SPLIT, threshold,
                                              soft ? 1 : 0, w_.data(), row_, v_.data(), out_.data(), &thr, VW_FLAG_CHECK_FINITE);
        if (rc == VW_ENONFINITE) throw InvalidSignalException(vw_multi_last_error(m_), "VAL_003");
        mchk(rc);
        if (threshold_out) *threshold_out = thr;
        std::vector<double> x(total);
        for (size_t r = 0; r < world; r++) chk(r, vw_copy_d2h(vw_multi_ctx(m_, (int)r), x.data() + r * n_, out_[r], (size_t)n_ * 8));
        return x;
    }

private:
    void mchk(int rc) const { if (rc != VW_OK) throw NativeEngineError(vw_multi_last_error(m_)); }
    void chk(size_t r, int rc) const { if (rc != VW_OK) throw NativeEngineError(vw_last_error(vw_multi_ctx(m_, (int)r))); }
    BoundaryMode mode_;
    int levels_;
    int64_t n_, row_ = 0;
    std::vector<double> hs_, gs_;
    vw_span_plan plan_{};
    vw_multi *m_ = nullptr;
    std::vector<double *> xext_, w_, v_, out_;
};

// ---- VectorWaveSwtAdapter ---------------------------------------------------------------------------------------------
class VectorWaveSwtAdapter {
public:
    VectorWaveSwtAdapter(Wavelet w, BoundaryMode m = BoundaryMode::PERIODIC) : t_(std::move(w), m) {}
    MultiLevelMODWTResult forward(const std::vector<double> &signal, int levels) const { return t_.decompose(signal, levels); }   // :184-204
    std::vector<double> inverse(const MultiLevelMODWTResult &r) const { return t_.reconstruct(r); }                                 // :435-474
    // :489-493 -- level 0 addresses the approximation, like MutableMultiLevelMODWTResult.applyThreshold
    void applyThreshold(MultiLevelMODWTResult &r, int level, double threshold, bool soft) const {
        if (level < 0 || level > r.getLevels()) throw InvalidArgumentException("Invalid level: " + std::to_string(level), "CFG_004");
        double *c = level == 0 ? r.approxData() : r.detailData() + (size_t)(level - 1) * r.getSignalLength();
        Engine &e = Engine::get();
        e.check(vw_threshold(e.ctx(), c, 1, r.getSignalLength(), r.getSignalLength(), &threshold, 0, soft ? 1 : 0, 0));
    }
    // :505-520 -- sigma = median|W_1| / 0.6745, thr = sigma * sqrt(2 ln N), every detail level; returns the threshold
    double applyUniversalThreshold(MultiLevelMODWTResult &r, bool soft) const {
        const int64_t n = r.getSignalLength();
        double thr = 0.0;
        Engine &e = Engine::get();
        e.check(vw_universal_threshold(e.ctx(), r.detailData(), 1, n, n, &thr, 0));
        e.check(vw_threshold(e.ctx(), r.detailData(), r.getLevels(), n, n, &thr, 0, soft ? 1 : 0, 0));
        return thr;
    }
    // :532-562 as ONE native call; threshold < 0 selects the universal threshold
    std::vector<double> denoise(const std::vector<double> &signal, int levels, double threshold = -1.0, bool soft = true) const {
        const int64_t n = (int64_t)signal.size();
        if (n == 0) throw InvalidSignalException("Signal cannot be empty for SWT", "VAL_006");
        const int maxLevels = t_.getMaximumLevels((int)n);
        if (levels < 1 || levels > maxLevels) throw InvalidArgumentException("Invalid SWT decomposition levels: " + std::to_string(levels), "CFG_004");
        int order;
        const std::vector<vw_align> al = t_.alignment(levels, order);
        std::vector<double> out(n);
        Engine &e = Engine::get();
        e.check(vw_swt_denoise(e.ctx(), signal.data(), 1, n, n, t_.scaledLow().data(), t_.scaledHigh().data(), (int)t_.scaledLow().size(),
                               levels, (int)t_.getBoundaryMode(), al.empty() ? nullptr : al.data(), order, threshold, soft ? 1 : 0,
                               out.data(), n, nullptr, VW_FLAG_CHECK_FINITE));
        return out;
    }

private:
    MultiLevelMODWTTransform t_;
};

// ---- BatchMODWT (PERIODIC, AoS rows) ------------------------------------------------------------------------------------
struct BatchMODWT {
    struct MultiLevelResult { std::vector<double> detailPerLevel /*[J][B][N]*/, finalApprox /*[B][N]*/; int levels, batch, n; };
    static MultiLevelResult multiLevelAoS(const Wavelet &w, const std::vector<std::vector<double>> &signals, int levels) {   // :90-111
        if (levels < 1) throw IllegalArgumentException("levels must be >= 1");
        if (signals.empty()) throw IllegalArgumentException("signals must be non-null and non-empty");
        const int64_t b = (int64_t)signals.size(), n = (int64_t)signals[0].size();
        if (n == 0) throw IllegalArgumentException("signal length must be > 0");
        for (const auto &s : signals) if ((int64_t)s.size() != n) throw IllegalArgumentException("all signals must be non-null and same length");
        const std::vector<double> hs = detail::scaled(w.lowPassDecomposition()), gs = detail::scaled(w.highPassDecomposition());
        std::vector<double> x((size_t)b * n);
        for (int64_t i = 0; i < b; i++) std::copy(signals[i].begin(), signals[i].end(), x.begin() + i * n);
        MultiLevelResult r{std::vector<double>((size_t)levels * b * n), std::vector<double>((size_t)b * n), levels, (int)b, (int)n};
        Engine &e = Engine::get();
        e.check(vw_modwt_forward(e.ctx(), x.data(), b, n, n, hs.data(), gs.data(), (int)hs.size(), levels, VW_PERIODIC,
                                 r.detailPerLevel.data(), n, b * n, r.finalApprox.data(), n, 0));
        return r;
    }
    static std::vector<double> inverseMultiLevelAoS(const Wavelet &w, const MultiLevelResult &r) {   // :151-178 (split order)
        const std::vector<double> hs = detail::scaled(w.lowPassReconstruction()), gs = detail::scaled(w.highPassReconstruction());
        std::vector<double> x((size_t)r.batch * r.n);
        Engine &e = Engine::get();
        e.check(vw_modwt_inverse(e.ctx(), r.detailPerLevel.data(), r.n, (int64_t)r.batch * r.n, r.finalApprox.data(), r.n, r.batch, r.n,
                                 hs.data(), gs.data(), (int)hs.size(), r.levels, VW_PERIODIC, nullptr, VW_ORDER_SPLIT,
                                 (r.levels >= 64 ? ~0ull : ((1ull << r.levels) - 1)), 1, x.data(), r.n, 0));
        return x;
    }
};

// ---- BatchStreamingMODWT (EXT/extensions/modwt/BatchStreamingMODWT.java:55-276) ----------------------------------------
// ZERO_PADDING / SYMMETRIC blocks continue each other through histories the engine keeps in HBM (vw_stream_state, owned
// here: RAII); PERIODIC has no state and transforms each block on its own (:62-64,113-115).
struct IllegalStateException : std::logic_error { using std::logic_error::logic_error; };
struct UnsupportedOperationException : std::logic_error { using std::logic_error::logic_error; };

class BatchStreamingMODWT {
public:
    struct SingleLevelResult { std::vector<double> approx /*[B][N]*/, detail /*[B][N]*/; int batch, n; };
    using MultiLevelResult = BatchMODWT::MultiLevelResult;

    BatchStreamingMODWT(const Wavelet &w, BoundaryMode mode, int levels = 1)
        : mode_(mode), levels_(levels), hs_(detail::scaled(w.lowPassDecomposition())), gs_(detail::scaled(w.highPassDecomposition())) {
        if (levels < 1) throw IllegalArgumentException("levels must be >= 1");
        detail::require_mode(mode);
    }
    ~BatchStreamingMODWT() { if (st_) vw_stream_destroy(Engine::get().ctx(), st_); }
    BatchStreamingMODWT(const BatchStreamingMODWT &) = delete;
    BatchStreamingMODWT &operator=(const BatchStreamingMODWT &) = delete;

    SingleLevelResult processSingleLevel(const std::vector<std::vector<double>> &signals) {   // :55-103
        if (levels_ != 1) throw IllegalStateException("This instance is configured for levels=" + std::to_string(levels_) + ", expected=1");
        MultiLevelResult r = processMultiLevel(signals);
        return {std::move(r.finalApprox), std::move(r.detailPerLevel), r.batch, r.n};
    }
    MultiLevelResult processMultiLevel(const std::vector<std::vector<double>> &signals) {    // :111-163
        if (signals.empty()) throw IllegalArgumentException("signals must be non-null and non-empty");
        const int64_t b = (int64_t)signals.size(), n = (int64_t)signals[0].size();
        if (n == 0) throw IllegalArgumentException("signal length must be > 0");
        for (const auto &s : signals) if ((int64_t)s.size() != n) throw IllegalArgumentException("all signals must be non-null and same length");
        std::vector<double> x((size_t)b * n);
        for (int64_t i = 0; i < b; i++) std::copy(signals[i].begin(), signals[i].end(), x.begin() + i * n);
        MultiLevelResult r{std::vector<double>((size_t)levels_ * b * n), std::vector<double>((size_t)b * n), levels_, (int)b, (int)n};
        Engine &e = Engine::get();
        if (mode_ == BoundaryMode::PERIODIC) {
            e.check(vw_modwt_forward(e.ctx(), x.data(), b, n, n, hs_.data(), gs_.data(), (int)hs_.size(), levels_, VW_PERIODIC,
                                     r.detailPerLevel.data(), n, b * n, r.finalApprox.data(), n, 0));
            return r;
        }
        if (!st_) e.check(vw_stream_create(e.ctx(), hs_.data(), gs_.data(), (int)hs_.size(), levels_, (int)mode_, &st_));
        e.check(vw_stream_process(e.ctx(), st_, x.data(), b, n, n, r.detailPerLevel.data(), n, b * n, r.finalApprox.data(), n, 0));
        batch_ = (int)b;
        return r;
    }
    SingleLevelResult flushSingleLevel(int tailLength) {   // :183-222
        if (levels_ != 1) throw IllegalStateException("This instance is configured for levels=" + std::to_string(levels_) + ", expected=1");
        MultiLevelResult r = flushMultiLevel(tailLength);
        return {std::move(r.finalApprox), std::move(r.detailPerLevel), r.batch, r.n};
    }
    MultiLevelResult flushMultiLevel(int tailLength) {      // :231-276; the histories are not advanced
        if (mode_ == BoundaryMode::PERIODIC) throw UnsupportedOperationException("Flush is only applicable to ZERO_PADDING/SYMMETRIC");
        if (tailLength <= 0) return {{}, {}, levels_, 0, 0};
        if (!st_ || batch_ == 0) throw IllegalStateException("No prior blocks processed; cannot flush");
        if (tailLength > getMinFlushTailLength())
            throw IllegalArgumentException("tailLength (" + std::to_string(tailLength) + ") exceeds maximum allowed across levels (" +
                                           std::to_string(getMinFlushTailLength()) + ")");
        const int64_t b = batch_, t = tailLength;
        MultiLevelResult r{std::vector<double>((size_t)levels_ * b * t), std::vector<double>((size_t)b * t), levels_, (int)b, (int)t};
        Engine &e = Engine::get();
        e.check(vw_stream_flush(e.ctx(), st_, t, r.detailPerLevel.data(), t, b * t, r.finalApprox.data(), t, 0));
        return r;
    }
    int getMinFlushTailLength() const { return (int)hs_.size() - 1; }
    int getHistoryLengthForLevel(int level) const {
        if (level < 1 || level > levels_) throw IllegalArgumentException("level must be in [1," + std::to_string(levels_) + "]");
        return ((int)hs_.size() - 1) << (level - 1);
    }
    int suggestFlushTailLength() const { return getMinFlushTailLength(); }

private:
    BoundaryMode mode_;
    int levels_;
    std::vector<double> hs_, gs_;
    vw_stream_state *st_ = nullptr;
    int batch_ = 0;
};

// ---- BatchSIMDMODWT SoA statics (EXT/extensions/modwt/BatchSIMDMODWT.java:64-81,282-308,343-424) -----------------------
// flat arrays indexed t*batchSize + b; the engine runs on that layout directly (vw_modwt_forward_soa), no transposes
struct BatchSIMDMODWT {
    static void convertToSoA(const std::vector<std::vector<double>> &signals, std::vector<double> &soaOutput) {   // :282-297
        const size_t b = signals.size(), n = b ? signals[0].size() : 0;
        soaOutput.resize(b * n);
        for (size_t t = 0; t < n; t++) for (size_t i = 0; i < b; i++) soaOutput[t * b + i] = signals[i][t];
    }
    static void convertFromSoA(const std::vector<double> &soaData, std::vector<std::vector<double>> &output) {   // :299-314
        const size_t b = output.size(), n = b ? output[0].size() : 0;
        for (size_t t = 0; t < n; t++) for (size_t i = 0; i < b; i++) output[i][t] = soaData[t * b + i];
    }
    static void batchMultiLevelMODWTSoA(const std::vector<double> &soaSignals, std::vector<std::vector<double>> &soaDetailPerLevel,
                                        std::vector<double> &soaApproxOut, const Wavelet &w, int batchSize, int signalLength, int levels) {
        if ((int)soaDetailPerLevel.size() != levels) throw IllegalArgumentException("soaDetailPerLevel length must equal levels");
        const size_t tot = (size_t)batchSize * (size_t)signalLength;
        if (soaSignals.size() != tot) throw IllegalArgumentException("soaSignals length must be batchSize * signalLength");
        const std::vector<double> hs = detail::scaled(w.lowPassDecomposition()), gs = detail::scaled(w.highPassDecomposition());
        std::vector<double *> ptrs;
        for (auto &d : soaDetailPerLevel) { d.resize(tot); ptrs.push_back(d.data()); }
        soaApproxOut.resize(tot);
        Engine &e = Engine::get();
        e.check(vw_modwt_forward_soa(e.ctx(), soaSignals.data(), batchSize, signalLength, hs.data(), gs.data(), (int)hs.size(), levels,
                                     ptrs.data(), soaApproxOut.data(), 0));
    }
    static void batchMODWTSoA(const std::vector<double> &soaSignals, std::vector<double> &soaApprox, std::vector<double> &soaDetail,
                              const Wavelet &w, int batchSize, int signalLength) {   // :64-81
        const size_t tot = (size_t)batchSize * (size_t)signalLength;
        if (soaSignals.size() != tot) throw IllegalArgumentException("soaSignals length must be batchSize * signalLength");
        std::vector<double> hs = detail::scaled(w.lowPassDecomposition()), gs = detail::scaled(w.highPassDecomposition());
        if (w.id() == Wavelet::Id::HAAR) { hs = {0.5, 0.5}; gs = {0.5, -0.5}; }   // literal taps of haarBatchMODWTSoA (:90-93)
        soaApprox.resize(tot); soaDetail.resize(tot);
        double *wp = soaDetail.data();
        Engine &e = Engine::get();
        e.check(vw_modwt_forward_soa(e.ctx(), soaSignals.data(), batchSize, signalLength, hs.data(), gs.data(), (int)hs.size(), 1, &wp,
                                     soaApprox.data(), 0));
    }
};

}  // namespace vectorwave
