"""Host mirror of the reference's MODWT classes over the native engine.

Same class / method names, argument meaning and error behaviour as
CORE/modwt/MODWTTransform.java, MultiLevelMODWTTransform.java, MODWTResult(+Impl).java,
MultiLevelMODWTResult(+Impl).java, MutableMultiLevelMODWTResult(+Impl).java and
SymmetricAlignmentStrategy.java, so the parity tests read like the reference's own tests.
All arithmetic runs in libvwmodwt.so on the GPU; this file only validates, scales filters by
1/sqrt(2), builds the per-level alignment table and owns the result layout.

Signals may be numpy arrays (host path, staged by the shim) or float64 torch CUDA tensors
(device path, zero copy; results stay on the device).
"""
import math

import numpy as np

from . import _native
from ._native import Engine, ORDER_PAIR, ORDER_SPLIT
from .errors import (ErrorCode, IllegalArgumentException, InvalidArgumentException, InvalidSignalException,
                     NullPointerException)
from .wavelets import BoundaryMode, Coiflet, Daubechies, Haar, Symlet

SCALE = 1.0 / math.sqrt(2.0)  # 1.0 / Math.sqrt(2.0), CORE/modwt/MODWTTransform.java:139


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _copy(a):
    return a.clone() if _is_torch(a) else np.array(a, dtype=np.float64, copy=True)


def _all_finite(a):
    if _is_torch(a):
        import torch
        return bool(torch.isfinite(a).all().item())
    return bool(np.isfinite(a).all())


def _require_mode(wavelet, boundary_mode):
    if wavelet is None:
        raise NullPointerException("wavelet cannot be null")
    if boundary_mode is None:
        raise NullPointerException("boundaryMode cannot be null")
    if boundary_mode not in (BoundaryMode.PERIODIC, BoundaryMode.ZERO_PADDING, BoundaryMode.SYMMETRIC):
        # CORE/modwt/MODWTTransform.java:96-110
        raise InvalidArgumentException(
            "MODWT only supports PERIODIC, ZERO_PADDING, and SYMMETRIC boundary modes",
            ErrorCode.CFG_UNSUPPORTED_BOUNDARY_MODE)


def _as_signal(signal, what="signal"):
    if signal is None:
        raise NullPointerException(f"{what} cannot be null")
    if _is_torch(signal):
        return signal
    a = np.asarray(signal, dtype=np.float64)
    return a


def _length(a):
    return int(a.shape[-1]) if a.ndim else 0


# ---------------------------------------------------------------------------------------------
# results
# ---------------------------------------------------------------------------------------------
class MODWTResult:
    """CORE/modwt/MODWTResult.java:25-110 (+Impl :16-97): two same-length arrays, defensive copies."""

    def __init__(self, approximationCoeffs, detailCoeffs, _validate=True):
        if approximationCoeffs is None:
            raise NullPointerException("approximationCoeffs cannot be null")
        if detailCoeffs is None:
            raise NullPointerException("detailCoeffs cannot be null")
        a, d = _as_signal(approximationCoeffs), _as_signal(detailCoeffs)
        if _length(a) != _length(d):
            raise IllegalArgumentException(
                "Approximation and detail coefficients must have the same length. "
                f"Got approximation length: {_length(a)}, detail length: {_length(d)}")
        if _length(a) == 0:
            raise IllegalArgumentException("Coefficient arrays cannot be empty")
        if _validate and not (_all_finite(a) and _all_finite(d)):
            raise InvalidSignalException("coefficients contain NaN or Infinity", ErrorCode.VAL_NON_FINITE_VALUES)
        self._a, self._d = _copy(a), _copy(d)

    @staticmethod
    def create(approximationCoeffs, detailCoeffs):
        return MODWTResult(approximationCoeffs, detailCoeffs)

    def approximationCoeffs(self):
        return _copy(self._a)

    def detailCoeffs(self):
        return _copy(self._d)

    def getSignalLength(self):
        return _length(self._a)

    def isValid(self):
        return _length(self._a) == _length(self._d) and _all_finite(self._a) and _all_finite(self._d)


class MultiLevelMODWTResult:
    """CORE/modwt/MultiLevelMODWTResult.java:32-99 (+Impl): levels are 1-based, 1 = finest; every array has
    the signal length; getters return copies.  Storage is one [J][N] block plus V_J, host or device."""

    def __init__(self, details, approx, engine=None):
        self._w = details      # [J][N]
        self._v = approx       # [N]
        self._engine = engine

    def getLevels(self):
        return int(self._w.shape[0])

    def getSignalLength(self):
        return int(self._v.shape[-1])

    def _check_level(self, level):
        if level < 1 or level > self.getLevels():
            raise IllegalArgumentException(f"Level must be between 1 and {self.getLevels()}, got: {level}")

    def getDetailCoeffsAtLevel(self, level):
        self._check_level(level)
        return _copy(self._w[level - 1])

    def getApproximationCoeffs(self):
        return _copy(self._v)

    def _energy(self, a):
        # sum of squares on the device (CORE/modwt/MultiLevelMODWTResultImpl.java:91-139)
        return (self._engine or Engine.get()).energy(a)

    def getDetailEnergyAtLevel(self, level):
        self._check_level(level)
        return self._energy(self._w[level - 1])

    def getApproximationEnergy(self):
        return self._energy(self._v)

    def getTotalEnergy(self):
        return self.getApproximationEnergy() + sum(self.getDetailEnergyAtLevel(j) for j in range(1, self.getLevels() + 1))

    def getRelativeEnergyDistribution(self):
        total = self.getTotalEnergy()
        out = np.zeros(self.getLevels() + 1)
        if total != 0:
            out[0] = self.getApproximationEnergy() / total
            for j in range(1, self.getLevels() + 1):
                out[j] = self.getDetailEnergyAtLevel(j) / total
        return out

    def copy(self):
        return MultiLevelMODWTResult(_copy(self._w), _copy(self._v), self._engine)

    def isValid(self):
        return self._w.shape[-1] == self._v.shape[-1] and _all_finite(self._w) and _all_finite(self._v)


class MutableMultiLevelMODWTResult(MultiLevelMODWTResult):
    """CORE/modwt/MutableMultiLevelMODWTResult.java:30-123: live arrays + in-place thresholding."""

    def getMutableDetailCoeffs(self, level):
        self._check_level(level)
        return self._w[level - 1]

    def getMutableApproximationCoeffs(self):
        return self._v

    def setDetailCoeffs(self, level, coeffs):
        self._check_level(level)
        if coeffs is None:
            raise NullPointerException("coeffs cannot be null")
        if _length(_as_signal(coeffs)) != self.getSignalLength():
            raise IllegalArgumentException("Coefficient array length must match signal length")
        self._w[level - 1][...] = coeffs if _is_torch(coeffs) or not _is_torch(self._w) else self._to_dev(coeffs)

    def setApproximationCoeffs(self, coeffs):
        if coeffs is None:
            raise NullPointerException("coeffs cannot be null")
        if _length(_as_signal(coeffs)) != self.getSignalLength():
            raise IllegalArgumentException("Coefficient array length must match signal length")
        self._v[...] = coeffs if _is_torch(coeffs) or not _is_torch(self._v) else self._to_dev(coeffs)

    def _to_dev(self, a):
        import torch
        return torch.as_tensor(np.asarray(a, dtype=np.float64), device=self._v.device)

    def clearCaches(self):
        pass  # energies are computed on demand; nothing is cached

    def applyThreshold(self, level, threshold, soft):
        """:83-118; level 0 = approximation.  Runs the native threshold kernel in place."""
        eng = self._engine or Engine.get()
        if level == 0:
            eng.threshold(self._v, float(threshold), soft)
        else:
            self._check_level(level)
            eng.threshold(self._w[level - 1], float(threshold), soft)
        self.clearCaches()

    def toImmutable(self):
        return MultiLevelMODWTResult(_copy(self._w), _copy(self._v), self._engine)


# ---------------------------------------------------------------------------------------------
# SYMMETRIC alignment (host policy, passed to the engine as data)
# ---------------------------------------------------------------------------------------------
class SymmetricAlignmentStrategy:
    """CORE/modwt/SymmetricAlignmentStrategy.java:43-117 -- identity tests on the shared singletons."""

    @staticmethod
    def decide(wavelet, level):
        l0 = wavelet.lowPassReconstruction().size
        detail_plus = True
        if l0 <= 2:
            return True, (0 if level <= 1 else -1), True, 0
        approx_plus = False
        if wavelet is Daubechies.DB6:
            dh, dg = (0 if level <= 1 else -1), (1 if level >= 3 else 0)
        elif wavelet is Daubechies.DB8:
            dh, dg = (0 if level <= 1 else 1), (1 if level >= 2 else 0)
        elif wavelet is Symlet.SYM4:
            approx_plus, detail_plus, dh, dg = True, False, 0, 0
        elif wavelet is Symlet.SYM8:
            dh, dg = (0, 0) if level <= 1 else ((1, 0) if level == 2 else (1, 1))
        elif wavelet is Coiflet.COIF2:
            approx_plus, detail_plus, dh, dg = True, False, (0 if level <= 1 else 1), 0
        elif wavelet is Coiflet.COIF3:
            detail_plus = False
            dh, dg = (0, 0) if level <= 1 else (-1, 1)
        elif l0 >= 12:
            dh = dg = 0 if (level <= 1 or level % 2 == 0) else -1
        else:
            dh, dg = (0, 0) if level <= 1 else (-1, 0)
        return approx_plus, dh, detail_plus, dg


def compute_tau_j(base_filter_length, level):
    """CORE/modwt/MultiLevelMODWTTransform.java:795-806 computeTauJ."""
    lm1 = base_filter_length - 1
    if level <= 1:
        return max(0, lm1 // 2)
    return (lm1 * (1 << (level - 1))) // 2


def multilevel_alignment(wavelet, boundary_mode, levels):
    """Per-level (sigma_h, tau_h, sigma_g, tau_g) + summation order of MultiLevelMODWTTransform's inverse
    (:554-645): PERIODIC split order t+l; ZERO_PADDING pair order t+l; SYMMETRIC split order with the
    alignment table."""
    if boundary_mode == BoundaryMode.PERIODIC:
        return None, ORDER_SPLIT
    if boundary_mode == BoundaryMode.ZERO_PADDING:
        return None, ORDER_PAIR
    lh = wavelet.lowPassReconstruction().size
    lg = wavelet.highPassReconstruction().size
    table = []
    for level in range(1, levels + 1):
        ap, dh, dp, dg = SymmetricAlignmentStrategy.decide(wavelet, level)
        table.append((1 if ap else -1, compute_tau_j(lh, level) + dh, 1 if dp else -1, compute_tau_j(lg, level) + dg))
    return table, ORDER_SPLIT


# ---------------------------------------------------------------------------------------------
# transforms
# ---------------------------------------------------------------------------------------------
class MODWTTransform:
    """CORE/modwt/MODWTTransform.java: single-level forward / inverse and their batch forms."""

    def __init__(self, wavelet, boundaryMode, engine=None, flags=0):
        _require_mode(wavelet, boundaryMode)
        self.wavelet = wavelet
        self.boundaryMode = boundaryMode
        self._engine = engine
        self._flags = flags
        self._hs = wavelet.lowPassDecomposition() * SCALE     # :139-150
        self._gs = wavelet.highPassDecomposition() * SCALE
        self._hrs = wavelet.lowPassReconstruction() * SCALE   # :229-238
        self._grs = wavelet.highPassReconstruction() * SCALE

    def _eng(self):
        if self._engine is None:
            self._engine = Engine.get()
        return self._engine

    def getWavelet(self):
        return self.wavelet

    def getBoundaryMode(self):
        return self.boundaryMode

    def forward(self, signal):
        """:131-189.  Raises NullPointerException / InvalidSignalException(VAL_EMPTY | VAL_NON_FINITE_VALUES)."""
        x = _as_signal(signal)
        if x.ndim != 1:
            raise IllegalArgumentException("forward takes one 1-D signal; use forwardBatch for [B][N]")
        w, v = self._eng().forward(x, self._hs, self._gs, 1, self.boundaryMode.value,
                                   _native.FLAG_CHECK_FINITE | self._flags)
        return MODWTResult(v, w[0], _validate=False)

    def inverse(self, modwtResult):
        """:203-299: pair-added products; SYMMETRIC uses t-l."""
        if modwtResult is None:
            raise NullPointerException("modwtResult cannot be null")
        if not modwtResult.isValid():
            raise InvalidSignalException("MODWTResult contains invalid coefficients", ErrorCode.VAL_NON_FINITE_VALUES)
        v, w = modwtResult._a, modwtResult._d
        align = [(-1, 0, -1, 0)] if self.boundaryMode == BoundaryMode.SYMMETRIC else None
        return self._eng().inverse(w.reshape(1, -1), v, self._hrs, self._grs, self.boundaryMode.value, align,
                                   ORDER_PAIR, flags=self._flags)

    def forwardBatch(self, signals):
        """:486-515 (+ :564-631).  Same-length signals run as one [B][N] launch, mixed lengths as one packed launch."""
        if signals is None:
            raise NullPointerException("signals array cannot be null")
        if len(signals) == 0:
            return []
        if any(s is None for s in signals):
            raise NullPointerException("signal cannot be null")
        lengths = {_length(_as_signal(s)) for s in signals}
        if len(lengths) != 1:
            return self._forward_mixed(signals)
        if _is_torch(signals):
            x = signals
        elif _is_torch(signals[0]):
            import torch
            x = torch.stack(list(signals))
        else:
            x = np.asarray(signals, dtype=np.float64)
        w, v = self._eng().forward(x, self._hs, self._gs, 1, self.boundaryMode.value,
                                   _native.FLAG_CHECK_FINITE | self._flags)
        return [MODWTResult(v[b], w[0, b], _validate=False) for b in range(x.shape[0])]

    def inverseBatch(self, results):
        """:531-559 (+ :636-689).  With >= 4 same-length results of n >= 64 the reference's optimized body is
        taken, whose SYMMETRIC rule is t+l (:672-684) instead of inverse()'s t-l (SURVEY.md D4)."""
        if results is None:
            raise NullPointerException("results array cannot be null")
        if len(results) == 0:
            return []
        if any(r is None for r in results):
            raise NullPointerException("result cannot be null")
        lengths = {r.getSignalLength() for r in results}
        n = results[0].getSignalLength()
        if len(lengths) != 1:
            return self._inverse_mixed(results)
        optimized = len(results) >= 4 and n >= 64
        if not optimized:
            for r in results:
                if not r.isValid():
                    raise InvalidSignalException("MODWTResult contains invalid coefficients",
                                                 ErrorCode.VAL_NON_FINITE_VALUES)
        if _is_torch(results[0]._a):
            import torch
            v = torch.stack([r._a for r in results])
            w = torch.stack([r._d for r in results])
        else:
            v = np.stack([r._a for r in results])
            w = np.stack([r._d for r in results])
        align = None
        if self.boundaryMode == BoundaryMode.SYMMETRIC and not optimized:
            align = [(-1, 0, -1, 0)]
        out = self._eng().inverse(w.reshape(1, len(results), n), v, self._hrs, self._grs, self.boundaryMode.value,
                                  align, ORDER_PAIR, flags=self._flags)
        return [out[b] for b in range(len(results))]

    # -- mixed lengths: one packed call per direction (vw_modwt_forward_varlen / vw_modwt_inverse_varlen) ----------------
    @staticmethod
    def _pack(rows):
        """rows -> (packed buffer, offsets): torch.cat keeps CUDA tensors on the device, anything else packs on the host;
        None when the rows mix residencies (those keep the per-row path)."""
        offsets = np.zeros(len(rows) + 1, dtype=np.int64)
        np.cumsum([int(r.shape[-1]) for r in rows], out=offsets[1:])
        if all(_is_torch(r) and r.is_cuda for r in rows):
            import torch
            return torch.cat([r.reshape(-1) for r in rows]), offsets
        if any(_is_torch(r) for r in rows):
            return None, offsets
        return np.concatenate([np.asarray(r, dtype=np.float64).reshape(-1) for r in rows]), offsets

    def _forward_mixed(self, signals):
        """forward() per row, as one launch.  Rows are checked in index order like the reference's loop: the first row
        that is not 1-D raises here, after the rows before it ran (so an earlier empty or non-finite row still wins)."""
        rows = [_as_signal(s) for s in signals]
        bad = next((b for b, r in enumerate(rows) if r.ndim != 1), len(rows))
        good = rows[:bad]
        out = []
        if good:
            x, offsets = self._pack(good)
            if x is None:
                out = [self.forward(r) for r in good]
            else:
                w, v = self._eng().forward_varlen(x, offsets, self._hs, self._gs, self.boundaryMode.value,
                                                  _native.FLAG_CHECK_FINITE | self._flags)
                out = [MODWTResult(v[offsets[b]:offsets[b + 1]], w[offsets[b]:offsets[b + 1]], _validate=False)
                       for b in range(len(good))]
        if bad < len(rows):
            raise IllegalArgumentException("forward takes one 1-D signal; use forwardBatch for [B][N]")
        return out

    def _inverse_mixed(self, results):
        """inverse() per row (pair-added, SYMMETRIC t-l), as one launch; the lowest row with NaN / Inf raises."""
        w, offsets = self._pack([r._d for r in results])
        v, _ = self._pack([r._a for r in results])
        if w is None or v is None or _is_torch(w) != _is_torch(v):
            return [self.inverse(r) for r in results]
        x = self._eng().inverse_varlen(w, v, offsets, self._hrs, self._grs, self.boundaryMode.value,
                                       _native.FLAG_CHECK_FINITE | self._flags)
        return [x[offsets[b]:offsets[b + 1]] for b in range(len(results))]


class MultiLevelMODWTTransform:
    """CORE/modwt/MultiLevelMODWTTransform.java: cascade decompose / reconstruct and the partial variants."""

    MAX_DECOMPOSITION_LEVELS = 10  # :117 -- the effective cap is 9 (SURVEY.md D1)

    def __init__(self, wavelet, boundaryMode, engine=None, flags=0, enforce_level_cap=True):
        _require_mode(wavelet, boundaryMode)
        self.wavelet = wavelet
        self.boundaryMode = boundaryMode
        self._engine = engine
        self._flags = flags
        # the reference rejects J=10 (config #4); enforce_level_cap=False is the documented opt-out (SURVEY.md D1)
        self._enforce_cap = enforce_level_cap
        self._hs = wavelet.lowPassDecomposition() * SCALE      # ScalarOps.java:909-916 (one rounding per tap)
        self._gs = wavelet.highPassDecomposition() * SCALE
        self._hrs = wavelet.lowPassReconstruction() * SCALE
        self._grs = wavelet.highPassReconstruction() * SCALE

    def _eng(self):
        if self._engine is None:
            self._engine = Engine.get()
        return self._engine

    def getWavelet(self):
        return self.wavelet

    def getBoundaryMode(self):
        return self.boundaryMode

    @staticmethod
    def getMaxDecompositionLevels():
        return MultiLevelMODWTTransform.MAX_DECOMPOSITION_LEVELS

    def _calculate_max_levels(self, n):
        """:455-501 restated on the host (pure integer policy)."""
        l = self._hs.size
        if n <= l:
            return 0
        limit = self.MAX_DECOMPOSITION_LEVELS if self._enforce_cap else 62
        max_level = 1
        while max_level < limit:
            if (l - 1) * (1 << (max_level - 1)) + 1 > n:
                break
            max_level += 1
        return max_level - 1

    def getMaximumLevels(self, signalLength):
        return min(self._calculate_max_levels(signalLength), self.MAX_DECOMPOSITION_LEVELS if self._enforce_cap else 62)

    def _decompose(self, signal, levels, mutable):
        x = _as_signal(signal)
        if x.ndim != 1:
            raise IllegalArgumentException("decompose takes one 1-D signal")
        n = _length(x)
        if n == 0:
            raise InvalidSignalException("Signal cannot be empty for multi-level MODWT", ErrorCode.VAL_EMPTY)
        max_levels = self._calculate_max_levels(n)
        if levels is None:
            levels = max_levels
        if levels < 1 or levels > max_levels:
            raise InvalidArgumentException(
                f"Invalid number of decomposition levels: {levels} (maximum {max_levels} for signal length {n})",
                ErrorCode.CFG_INVALID_DECOMPOSITION_LEVEL)
        # ValidationUtils.validateFiniteValues (:211) runs on the device as part of the call
        w, v = self._eng().forward(x, self._hs, self._gs, levels, self.boundaryMode.value,
                                   _native.FLAG_CHECK_FINITE | self._flags)
        cls = MutableMultiLevelMODWTResult if mutable else MultiLevelMODWTResult
        return cls(w, v, self._eng())

    def decompose(self, signal, levels=None):
        """:195-255."""
        if signal is None:
            raise NullPointerException("signal cannot be null")
        return self._decompose(signal, levels, False)

    def decomposeMutable(self, signal, levels=None):
        """:267-330."""
        if signal is None:
            raise NullPointerException("signal cannot be null")
        return self._decompose(signal, levels, True)

    def decomposeResident(self, signal, levels=None, result=None):
        """decomposeMutable with the coefficients kept in HBM (vw_modwt_decompose_h): a ResidentMultiLevelMODWTResult
        copies a level to the host only when asked, thresholds / energies run on the device, `reconstruct()` moves 8
        B/sample back.  `result`: an earlier resident result of the same shape whose device storage is reused."""
        if signal is None:
            raise NullPointerException("signal cannot be null")
        x = _as_signal(signal)
        if x.ndim != 1:
            raise IllegalArgumentException("decompose takes one 1-D signal")
        n = _length(x)
        if n == 0:
            raise InvalidSignalException("Signal cannot be empty for multi-level MODWT", ErrorCode.VAL_EMPTY)
        max_levels = self._calculate_max_levels(n)
        if levels is None:
            levels = max_levels
        if levels < 1 or levels > max_levels:
            raise InvalidArgumentException(
                f"Invalid number of decomposition levels: {levels} (maximum {max_levels} for signal length {n})",
                ErrorCode.CFG_INVALID_DECOMPOSITION_LEVEL)
        handle = self._eng().decompose_resident(x, self._hs, self._gs, levels, self.boundaryMode.value,
                                                result=result._handle if result is not None else None,
                                                flags=_native.FLAG_CHECK_FINITE | self._flags)
        return ResidentMultiLevelMODWTResult(self, handle)

    def _reconstruct(self, result, detail_mask, use_approx):
        if isinstance(result, ResidentMultiLevelMODWTResult):
            align, order = multilevel_alignment(self.wavelet, self.boundaryMode, result.getLevels())
            return result._handle.reconstruct(self._hrs, self._grs, self.boundaryMode.value, align, order, detail_mask,
                                              use_approx)[0]
        align, order = multilevel_alignment(self.wavelet, self.boundaryMode, result.getLevels())
        return self._eng().inverse(result._w, result._v, self._hrs, self._grs, self.boundaryMode.value, align, order,
                                   detail_mask, use_approx, flags=self._flags)

    def reconstruct(self, result):
        """:339-349."""
        if result is None:
            raise NullPointerException("result cannot be null")
        return self._reconstruct(result, (1 << result.getLevels()) - 1, True)

    def reconstructFromLevel(self, result, startLevel):
        """:361-386: details finer than startLevel are replaced by zeros."""
        if result is None:
            raise NullPointerException("result cannot be null")
        levels = result.getLevels()
        if startLevel < 1 or startLevel > levels:
            raise InvalidArgumentException(f"Invalid start level: {startLevel}. Must be between 1 and {levels}")
        mask = ((1 << levels) - 1) & ~((1 << (startLevel - 1)) - 1)
        return self._reconstruct(result, mask, True)

    def reconstructLevels(self, result, minLevel, maxLevel):
        """:398-446: band-pass; the approximation enters only when the top level is inside the band."""
        if result is None:
            raise NullPointerException("result cannot be null")
        levels = result.getLevels()
        if minLevel < 1 or maxLevel > levels or minLevel > maxLevel:
            raise InvalidArgumentException("Invalid level range for partial reconstruction",
                                           ErrorCode.CFG_INVALID_DECOMPOSITION_LEVEL)
        mask = 0
        for level in range(minLevel, maxLevel + 1):
            mask |= 1 << (level - 1)
        return self._reconstruct(result, mask, levels <= maxLevel)


# ---------------------------------------------------------------------------------------------
# ParallelMultiLevelMODWT / MODWTTransformFactory (thin host classes over the same engine calls)
# ---------------------------------------------------------------------------------------------
class ResidentMultiLevelMODWTResult:
    """MutableMultiLevelMODWTResult (CORE/modwt/MutableMultiLevelMODWTResult.java:30-123) backed by a device-resident
    vw_result: the Python twin of java/.../modwt/GpuResidentResult.java."""

    def __init__(self, transform, handle):
        self._t, self._handle = transform, handle

    def getLevels(self):
        return self._handle.shape()[2]

    def getSignalLength(self):
        return self._handle.shape()[1]

    def _check(self, level):
        if level < 1 or level > self.getLevels():
            raise IllegalArgumentException(f"Level must be between 1 and {self.getLevels()}, got: {level}")

    def getDetailCoeffsAtLevel(self, level):
        self._check(level)
        return self._handle.get_level(level)[0]

    def getApproximationCoeffs(self):
        return self._handle.get_level(0)[0]

    def setDetailCoeffs(self, level, coeffs):
        self._check(level)
        self._handle.set_level(level, np.asarray(coeffs, dtype=np.float64).reshape(1, -1))

    def setApproximationCoeffs(self, coeffs):
        self._handle.set_level(0, np.asarray(coeffs, dtype=np.float64).reshape(1, -1))

    def applyThreshold(self, level, threshold, soft):
        if level == 0:                                        # the reference thresholds the approximation for level 0 (:84-86)
            v = self.getApproximationCoeffs()
            a = np.abs(v)
            self.setApproximationCoeffs(np.where(a > threshold, np.sign(v) * (a - threshold), 0.0) if soft
                                        else np.where(a <= threshold, 0.0, v))
            return
        self._check(level)
        self._handle.threshold(level, float(threshold), soft)

    def applyUniversalThreshold(self, soft=True):
        """VectorWaveSwtAdapter.applyUniversalThreshold (:505-520) on the resident coefficients; returns the threshold."""
        return float(self._handle.universal_threshold(soft)[0])

    def getDetailEnergyAtLevel(self, level):
        self._check(level)
        return float(self._handle.energy(level)[0])

    def getApproximationEnergy(self):
        return float(self._handle.energy(0)[0])

    def getTotalEnergy(self):
        return sum(self.getDetailEnergyAtLevel(j) for j in range(1, self.getLevels() + 1)) + self.getApproximationEnergy()

    def reconstruct(self):
        return self._t.reconstruct(self)

    def close(self):
        self._handle.free()


class ParallelMultiLevelMODWT:
    """CORE/modwt/ParallelMultiLevelMODWT.java:84-176.  The reference runs the h and g convolutions of a level on an
    executor; here the level is one kernel launch anyway, so only its observable quirks are mirrored: any
    non-PERIODIC mode -- SYMMETRIC included -- is computed as ZERO_PADDING (:125-129,156-162; SURVEY.md D6), and the
    level admissibility uses `n < L` instead of `n <= L` (:225)."""

    MAX_DECOMPOSITION_LEVELS = 10

    def __init__(self, parallelism=0, engine=None):
        self._engine = engine

    def _calculate_max_levels(self, n, l):
        if n < l:
            return 0
        max_level = 1
        while max_level < self.MAX_DECOMPOSITION_LEVELS:
            if (l - 1) * (1 << (max_level - 1)) + 1 > n:
                break
            max_level += 1
        return max_level - 1

    def decompose(self, signal, wavelet, mode, levels):
        if signal is None:
            raise NullPointerException("signal cannot be null")
        x = _as_signal(signal)
        if _length(x) == 0:
            raise InvalidSignalException("Signal cannot be empty", ErrorCode.VAL_EMPTY)
        hs, gs = wavelet.lowPassDecomposition() * SCALE, wavelet.highPassDecomposition() * SCALE
        max_levels = self._calculate_max_levels(_length(x), hs.size)
        if levels < 1 or levels > max_levels:
            raise InvalidArgumentException(f"Invalid number of levels: {levels}. Must be between 1 and {max_levels}",
                                           ErrorCode.CFG_INVALID_DECOMPOSITION_LEVEL)
        eng = self._engine or Engine.get()
        eff = BoundaryMode.PERIODIC if mode == BoundaryMode.PERIODIC else BoundaryMode.ZERO_PADDING
        w, v = eng.forward(x, hs, gs, levels, eff.value, _native.FLAG_CHECK_FINITE)
        return MultiLevelMODWTResult(w, v, eng)

    def shutdown(self):
        pass

    def close(self):
        pass


class MODWTTransformFactory:
    """CORE/modwt/MODWTTransformFactory.java:120-230: sugar over the two constructors (PERIODIC by default)."""

    @staticmethod
    def create(wavelet, boundaryMode=BoundaryMode.PERIODIC):
        return MODWTTransform(wavelet, boundaryMode)

    @staticmethod
    def createMultiLevel(wavelet, boundaryMode=BoundaryMode.PERIODIC):
        return MultiLevelMODWTTransform(wavelet, boundaryMode)
