"""BatchStreamingMODWT over the native engine (EXT/extensions/modwt/BatchStreamingMODWT.java).

Blockwise batch MODWT with a carried left history per level: every level keeps the last (L-1)*2^(j-1) samples of ITS
input, so consecutive blocks continue each other exactly (ZERO_PADDING: zeros before the stream; SYMMETRIC: the first
block reflected about its left edge, per level, :326-334).  PERIODIC has no state: each block is transformed on its own,
like the reference (:62-64,113-115).

The histories live in HBM behind one native stream state (vw_stream_state): a block's whole cascade, the first-block
initialisation, the batch-size restart and the flush tail all run below the C ABI, so this class only validates,
chooses the residency of the results and raises the reference's exceptions.
"""
import numpy as np

from ._native import Engine
from .batch import BatchMODWT, MultiLevelResult, SingleLevelResult, _validate_aos
from .errors import IllegalArgumentException
from .modwt import SCALE, _is_torch
from .wavelets import BoundaryMode


class UnsupportedOperationException(RuntimeError):
    pass


class IllegalStateException(RuntimeError):
    pass


class BatchStreamingMODWT:
    class Builder:
        def __init__(self):
            self._wavelet, self._mode, self._levels, self._engine = None, BoundaryMode.PERIODIC, 1, None

        def wavelet(self, w):
            self._wavelet = w
            return self

        def boundary(self, mode):
            self._mode = mode
            return self

        def levels(self, levels):
            self._levels = levels
            return self

        def engine(self, engine):
            self._engine = engine
            return self

        def build(self):
            if self._wavelet is None:
                raise IllegalArgumentException("wavelet must be set")
            return BatchStreamingMODWT(self)

    def __init__(self, b):
        self.wavelet, self.boundaryMode, self.levels = b._wavelet, b._mode, b._levels
        if self.levels < 1:
            raise IllegalArgumentException("levels must be >= 1")
        self._engine = b._engine
        self._hs = self.wavelet.lowPassDecomposition() * SCALE       # per-stage 1/sqrt(2), ScalarOps.java:909-916
        self._gs = self.wavelet.highPassDecomposition() * SCALE
        l = self._hs.size
        self._hist_len = [(l - 1) * (1 << j) for j in range(self.levels)]   # filterLen(level) - 1, :302-303
        self._state = None        # native stream state, created by the first block

    # ---- helpers ------------------------------------------------------------------------------------------
    def _eng(self):
        return self._engine or Engine.get()

    def _ensure_levels(self, expected):
        if self.levels != expected:
            raise IllegalStateException(f"This instance is configured for levels={self.levels}, expected={expected}")

    def _process(self, x):
        """x: validated [B][n] block (numpy or torch) -> (W [levels][B][n], V [B][n]) in the block's residency"""
        eng = self._eng()
        if _is_torch(x):
            import torch
            x = x.to(dtype=torch.float64, device=f"cuda:{eng.device}").contiguous()
        if self._state is None:
            self._state = eng.stream_create(self._hs, self._gs, self.levels, self.boundaryMode.value)
        return self._state.process(x)

    # ---- API ----------------------------------------------------------------------------------------------
    def processSingleLevel(self, block):
        """:55-103"""
        self._ensure_levels(1)
        x = _validate_aos(block)
        if self.boundaryMode == BoundaryMode.PERIODIC:
            return BatchMODWT.singleLevelAoS(self.wavelet, x, self._engine)
        w, v = self._process(x)
        return SingleLevelResult(v, w[0])

    def processMultiLevel(self, block):
        """:111-163"""
        x = _validate_aos(block)
        if self.boundaryMode == BoundaryMode.PERIODIC:
            return BatchMODWT.multiLevelAoS(self.wavelet, x, self.levels, self._engine)
        w, v = self._process(x)
        return MultiLevelResult(w, v)

    def _flush(self, tail_length):
        """the cascade over buildTailFromHistorySoA's tail (:358-372); the histories are not advanced (:205-222,252-274)"""
        if self.boundaryMode == BoundaryMode.PERIODIC:
            raise UnsupportedOperationException("Flush is only applicable to ZERO_PADDING/SYMMETRIC")
        if tail_length <= 0:
            return None
        if self._state is None or self._state.batch is None:
            raise IllegalStateException("No prior blocks processed; cannot flush")
        limit = min(self._hist_len)
        if tail_length > limit:
            raise IllegalArgumentException(
                f"tailLength ({tail_length}) exceeds maximum allowed across levels ({limit}). "
                "Use getMinFlushTailLength() to choose a valid tail length.")
        return self._state.flush(tail_length)

    def flushSingleLevel(self, tailLength):
        """:183-222"""
        self._ensure_levels(1)
        r = self._flush(tailLength)
        if r is None:
            return SingleLevelResult(np.zeros((0, 0)), np.zeros((0, 0)))
        w, v = r
        return SingleLevelResult(v, w[0])

    def flushMultiLevel(self, tailLength):
        """:231-276"""
        r = self._flush(tailLength)
        if r is None:
            return MultiLevelResult(np.zeros((self.levels, 0, 0)), np.zeros((0, 0)))
        w, v = r
        return MultiLevelResult(w, v)

    def getMinFlushTailLength(self):
        return min(self._hist_len)

    def getHistoryLengthForLevel(self, level):
        if level < 1 or level > self.levels:
            raise IllegalArgumentException(f"level must be in [1,{self.levels}]")
        return self._hist_len[level - 1]

    def suggestFlushTailLength(self):
        return self._hist_len[0] if self.levels == 1 else min(self._hist_len)

    def close(self):
        if self._state is not None:
            self._state.close()
            self._state = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False
