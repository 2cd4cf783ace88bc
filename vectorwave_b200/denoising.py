"""WaveletDenoiser over the native engine (CORE/denoising/WaveletDenoiser.java) -- SURVEY.md 8f row 4.

The reference's denoiser is a caller of the MODWT path: decompose, estimate sigma = median(|W_1|) / 0.6745, pick a
threshold per level from (W_j, sigma / sqrt(2^j)) with one of the selectors, threshold the details, reconstruct.  Here
every pass over the coefficients runs on the device (exact median select, mean / variance reductions, the SURE risk
scan, thresholding, the transforms); only the scalar selector formulas are evaluated on the host, exactly as written in
the reference.

SURE: the reference evaluates the risk of every candidate with an O(n^2) double loop (:441-492).  A sort + prefix-sum
evaluation would change the summation order enough to flip the arg-min between neighbouring candidates, so the device
kernel keeps the double loop -- one thread per candidate, the reference's coefficient order and roundings -- and returns
the JVM's threshold bit for bit (n = 65536 costs about a millisecond; the engine refuses batch * n^2 > 2^44).
"""
import enum
import math

import numpy as np

from . import _native
from ._native import ORDER_PAIR
from ._native import _is_torch
from .errors import (ErrorCode, IllegalArgumentException, InvalidArgumentException, InvalidSignalException,
                     NativeEngineError, NullPointerException)
from .modwt import MODWTTransform, MultiLevelMODWTTransform, _as_signal, multilevel_alignment
from .wavelets import BoundaryMode, Daubechies


class ThresholdMethod(enum.Enum):   # :602-632
    UNIVERSAL = "UNIVERSAL"
    SURE = "SURE"
    MINIMAX = "MINIMAX"
    BAYES = "BAYES"
    FIXED = "FIXED"


class ThresholdType(enum.Enum):     # :636-650
    SOFT = "SOFT"
    HARD = "HARD"


MAX_SAFE_LEVEL_FOR_SCALING = 31     # :57
BAYES_EPSILON = 1e-10               # :67

_METHOD_CODE = {ThresholdMethod.UNIVERSAL: _native.THR_UNIVERSAL, ThresholdMethod.SURE: _native.THR_SURE,
                ThresholdMethod.MINIMAX: _native.THR_MINIMAX, ThresholdMethod.BAYES: _native.THR_BAYES}


class WaveletDenoiser:
    ThresholdMethod = ThresholdMethod
    ThresholdType = ThresholdType

    def __init__(self, wavelet, boundaryMode, engine=None):
        if wavelet is None:
            raise InvalidArgumentException("wavelet cannot be null", ErrorCode.VAL_NULL_ARGUMENT)
        if boundaryMode is None:
            raise InvalidArgumentException("boundaryMode cannot be null", ErrorCode.VAL_NULL_ARGUMENT)
        self.wavelet, self.boundaryMode, self._engine = wavelet, boundaryMode, engine

    @staticmethod
    def forFinancialData():
        """:99-101"""
        return WaveletDenoiser(Daubechies.DB4, BoundaryMode.PERIODIC)

    # ---- selectors (:391-552), scalar formulas on the host, reductions on the device ---------------------------
    def _threshold(self, eng, coeffs, n, sigma, method):
        if method == ThresholdMethod.UNIVERSAL:
            return sigma * math.sqrt(2.0 * math.log(n))
        if method == ThresholdMethod.MINIMAX:                       # :497-509
            log_n = math.log(n)
            if n <= 32:
                return 0.0
            if n <= 64:
                return sigma * 0.3936 + 0.1829 * sigma * log_n
            return sigma * (0.4745 + 0.1148 * log_n)
        if method == ThresholdMethod.BAYES:                         # :521-552
            sigma2 = sigma * sigma
            _, variance = eng.mean_variance(coeffs)
            sigma_x = math.sqrt(max(0.0, variance - sigma2) + BAYES_EPSILON)
            return sigma2 / sigma_x
        if method == ThresholdMethod.SURE:                          # :441-472
            try:
                return eng.sure_threshold(coeffs, sigma)
            except NativeEngineError as e:                          # n^2 beyond the engine's bound
                raise InvalidArgumentException(str(e), ErrorCode.CFG_UNSUPPORTED_OPERATION) from e
        if method == ThresholdMethod.FIXED:                         # :414-425
            raise InvalidArgumentException("Fixed threshold method requires explicit threshold value",
                                           ErrorCode.CFG_UNSUPPORTED_OPERATION)
        raise InvalidArgumentException("Unknown threshold selection method", ErrorCode.CFG_UNSUPPORTED_OPERATION)

    def _sigma(self, eng, detail):
        """estimateNoiseSigma (:376-387): exact median of |detail| on the device, / 0.6745"""
        return eng.median_abs(detail) / 0.6745

    # ---- API ---------------------------------------------------------------------------------------------
    def denoise(self, signal, method, type=ThresholdType.SOFT):
        """:111-145 single level."""
        t = MODWTTransform(self.wavelet, self.boundaryMode, self._engine)
        eng = t._eng()
        x = _as_signal(signal)
        w, v = eng.forward(x, t._hs, t._gs, 1, self.boundaryMode.value, _native.FLAG_CHECK_FINITE)
        sigma = self._sigma(eng, w[0])
        thr = self._threshold(eng, w[0], w[0].shape[-1], sigma, method)
        return self._finish_single(t, eng, w, v, thr, type)

    def denoiseFixed(self, signal, threshold, type):
        """:354-366"""
        t = MODWTTransform(self.wavelet, self.boundaryMode, self._engine)
        eng = t._eng()
        w, v = eng.forward(_as_signal(signal), t._hs, t._gs, 1, self.boundaryMode.value, _native.FLAG_CHECK_FINITE)
        return self._finish_single(t, eng, w, v, float(threshold), type)

    def _finish_single(self, t, eng, w, v, thr, type):
        eng.threshold(w[0], thr, type == ThresholdType.SOFT)
        align = [(-1, 0, -1, 0)] if self.boundaryMode == BoundaryMode.SYMMETRIC else None   # MODWTTransform.inverse :277-295
        return eng.inverse(w, v, t._hrs, t._grs, self.boundaryMode.value, align, ORDER_PAIR)

    def denoiseMultiLevel(self, signal, levels, method, type):
        """:155-171 + DenoisedMultiLevelResult (:183-231): sigma from level 1, per-level sigma / sqrt(2^j)."""
        t = MultiLevelMODWTTransform(self.wavelet, self.boundaryMode, self._engine)
        res = t.decomposeMutable(signal, levels)
        eng = t._eng()
        if res.getLevels() > MAX_SAFE_LEVEL_FOR_SCALING:
            raise InvalidArgumentException("Decomposition level exceeds safe limit for scale-dependent thresholds",
                                           ErrorCode.VAL_TOO_LARGE)
        sigma = self._sigma(eng, res.getMutableDetailCoeffs(1))
        n = res.getSignalLength()
        self.lastThresholds = []
        for level in range(1, res.getLevels() + 1):
            d = res.getMutableDetailCoeffs(level)
            level_scale = math.sqrt(1 << level)                      # :221
            thr = self._threshold(eng, d, n, sigma / level_scale, method)
            self.lastThresholds.append(thr)
            eng.threshold(d, thr, type == ThresholdType.SOFT)
        return t.reconstruct(res)

    # ---- batches: [B][N] rows, each with its own noise level, in one engine call (vw_wavelet_denoise) ----------------
    # Row b gets what the single-signal method gives signals[b]; the selectors run on the device in the same arithmetic.
    @staticmethod
    def _batch(signals):
        if signals is None:
            raise NullPointerException("signals cannot be null")
        x = signals if _is_torch(signals) else np.asarray(signals, dtype=np.float64)
        if x.ndim != 2:
            raise IllegalArgumentException("batch methods take a [B][N] array of signals")
        if x.shape[1] == 0:
            raise InvalidSignalException("Signal cannot be empty", ErrorCode.VAL_EMPTY)
        return x

    @staticmethod
    def _method_code(method):
        if method == ThresholdMethod.FIXED:                         # :414-425
            raise InvalidArgumentException("Fixed threshold method requires explicit threshold value",
                                           ErrorCode.CFG_UNSUPPORTED_OPERATION)
        if method not in _METHOD_CODE:
            raise InvalidArgumentException("Unknown threshold selection method", ErrorCode.CFG_UNSUPPORTED_OPERATION)
        return _METHOD_CODE[method]

    def _denoise_batch(self, x, levels, multilevel, code, fixed, type, align, order):
        t = MODWTTransform(self.wavelet, self.boundaryMode, self._engine)
        try:
            return t._eng().wavelet_denoise(x, t._hs, t._gs, levels, self.boundaryMode.value, align, order, multilevel,
                                            code, fixed, type == ThresholdType.SOFT, _native.FLAG_CHECK_FINITE)
        except NativeEngineError as e:                              # SURE: levels * batch * n^2 beyond the engine's bound
            if code != _native.THR_SURE:
                raise
            raise InvalidArgumentException(str(e), ErrorCode.CFG_UNSUPPORTED_OPERATION) from e

    def _single_align(self):
        return [(-1, 0, -1, 0)] if self.boundaryMode == BoundaryMode.SYMMETRIC else None   # MODWTTransform.inverse

    def denoiseBatch(self, signals, method, type=ThresholdType.SOFT):
        """denoise() of every row of a [B][N] numpy array or CUDA tensor, returned as the same kind."""
        x = self._batch(signals)
        code = self._method_code(method)
        return self._denoise_batch(x, 1, False, code, 0.0, type, self._single_align(), ORDER_PAIR)[0]

    def denoiseFixedBatch(self, signals, threshold, type):
        """denoiseFixed() of every row with the one given threshold."""
        x = self._batch(signals)
        return self._denoise_batch(x, 1, False, _native.THR_FIXED, float(threshold), type, self._single_align(),
                                   ORDER_PAIR)[0]

    def denoiseMultiLevelBatch(self, signals, levels, method, type):
        """denoiseMultiLevel() of every row; lastThresholds becomes [B][J], row b as denoiseMultiLevel(signals[b])
        leaves it."""
        x = self._batch(signals)
        t = MultiLevelMODWTTransform(self.wavelet, self.boundaryMode, self._engine)
        n = int(x.shape[1])
        max_levels = t._calculate_max_levels(n)
        if levels is None:
            levels = max_levels
        if levels < 1 or levels > max_levels:
            raise InvalidArgumentException(
                f"Invalid number of decomposition levels: {levels} (maximum {max_levels} for signal length {n})",
                ErrorCode.CFG_INVALID_DECOMPOSITION_LEVEL)
        if levels > MAX_SAFE_LEVEL_FOR_SCALING:
            raise InvalidArgumentException("Decomposition level exceeds safe limit for scale-dependent thresholds",
                                           ErrorCode.VAL_TOO_LARGE)
        code = self._method_code(method)
        align, order = multilevel_alignment(self.wavelet, self.boundaryMode, levels)
        out, thr = self._denoise_batch(x, levels, True, code, 0.0, type, align, order)
        thr = thr.cpu().numpy() if _is_torch(thr) else thr
        self.lastThresholds = np.ascontiguousarray(thr.T)
        return out
