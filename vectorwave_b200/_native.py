"""ctypes binding of libvwmodwt.so (include/vw_modwt.h) -- the same C ABI the Java FFM binding uses.

There is no CPU compute path: if the shared library is missing or no CUDA device is present,
`Engine.get()` raises NativeEngineError.  Host numpy arrays are staged by the shim; torch CUDA
tensors are passed as device pointers (zero copy) and the work is enqueued on torch's current stream.
"""
import ctypes as C
import os
import threading

import numpy as np

from .errors import (ErrorCode, IllegalArgumentException, InvalidArgumentException, InvalidSignalException,
                     NativeEngineError, NullPointerException)

_HERE = os.path.dirname(os.path.abspath(__file__))
# VW_LIB_PATH: developer A/B builds of the same engine (csrc/Makefile TARGET=...); never a different implementation
LIB_PATH = os.environ.get("VW_LIB_PATH") or os.path.join(_HERE, "libvwmodwt.so")

FLAG_DEVICE_PTRS = 1 << 0
FLAG_CHECK_FINITE = 1 << 1
FLAG_BITEXACT = 1 << 2
FLAG_NO_FUSE = 1 << 3
FLAG_NO_SYNC = 1 << 4

ORDER_SPLIT, ORDER_PAIR = 0, 1

# vw_threshold_method: WaveletDenoiser.ThresholdMethod in declaration order
THR_UNIVERSAL, THR_SURE, THR_MINIMAX, THR_BAYES, THR_FIXED = 0, 1, 2, 3, 4

VW_OK = 0
_STATUS = {
    1: (NullPointerException, None),
    3: (InvalidSignalException, ErrorCode.VAL_NON_FINITE_VALUES),
    5: (InvalidArgumentException, ErrorCode.VAL_TOO_LARGE),
    6: (InvalidSignalException, ErrorCode.VAL_EMPTY),
    7: (IllegalArgumentException, None),
    103: (InvalidArgumentException, ErrorCode.CFG_UNSUPPORTED_BOUNDARY_MODE),
    104: (InvalidArgumentException, ErrorCode.CFG_INVALID_DECOMPOSITION_LEVEL),
    400: (IllegalArgumentException, None),
}


class VwAlign(C.Structure):
    _fields_ = [("sigma_h", C.c_int32), ("tau_h", C.c_int32), ("sigma_g", C.c_int32), ("tau_g", C.c_int32)]


SPAN_MAX_GROUPS = 16


class VwSpanPlan(C.Structure):
    """vw_span_plan of include/vw_modwt.h: the layout and launch groups of a span-sharded cascade."""
    _fields_ = [("l", C.c_int32), ("levels", C.c_int32), ("world", C.c_int32), ("reserved", C.c_int32),
                ("n_local", C.c_int64), ("ngroups_f", C.c_int32), ("ngroups_i", C.c_int32),
                ("first_f", C.c_int32 * SPAN_MAX_GROUPS), ("nlev_f", C.c_int32 * SPAN_MAX_GROUPS),
                ("first_i", C.c_int32 * SPAN_MAX_GROUPS), ("nlev_i", C.c_int32 * SPAN_MAX_GROUPS),
                ("halo_f", C.c_int64 * SPAN_MAX_GROUPS), ("halo_i", C.c_int64 * SPAN_MAX_GROUPS),
                ("lead", C.c_int64), ("lead_w", C.c_int64), ("pad", C.c_int64), ("inverse_msg", C.c_int64)]


class VwTiming(C.Structure):
    _fields_ = [("device_ms", C.c_float), ("host_ms", C.c_float), ("launches", C.c_int32), ("reserved", C.c_int32)]


_dp = C.POINTER(C.c_double)
_vp = C.c_void_p
_i64 = C.c_int64
_i32 = C.c_int32
_u32 = C.c_uint32

# name -> (restype, argtypes); also the list tests check against include/vw_modwt.h
SIGNATURES = {
    "vw_init": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "vw_destroy": (C.c_int, [_vp]),
    "vw_last_error": (C.c_char_p, [_vp]),
    "vw_status_name": (C.c_char_p, [C.c_int]),
    "vw_abi_version": (C.c_int, []),
    "vw_set_stream": (C.c_int, [_vp, _vp]),
    "vw_reset_stream": (C.c_int, [_vp]),
    "vw_synchronize": (C.c_int, [_vp]),
    "vw_device_index": (C.c_int, [_vp]),
    "vw_set_option": (C.c_int, [_vp, C.c_char_p, _i64]),
    "vw_launch_count": (_i64, [_vp]),
    "vw_plan_query": (C.c_int, [C.c_int, _i32, _i32, _i64, C.POINTER(_i32), C.POINTER(_i32), _i32]),
    "vw_describe_plan": (C.c_int, [C.c_int, _i32, _i32, _i64, _i64, _i32, C.c_char_p, C.c_size_t]),
    "vw_lattice_query": (C.c_int, [_dp, _dp, _i32, _dp, _i32, _dp]),
    "vw_alloc_pinned": (_vp, [C.c_size_t]),
    "vw_free_pinned": (None, [_vp]),
    "vw_device_alloc": (C.c_int, [_vp, C.c_size_t, C.POINTER(_vp)]),
    "vw_device_free": (C.c_int, [_vp, _vp]),
    "vw_copy_h2d": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "vw_copy_d2h": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "vw_max_levels": (C.c_int, [_i64, _i32, _i32]),
    "vw_conv_modwt": (C.c_int, [_vp, _vp, _i64, _vp, _i64, _i32, _vp, _u32]),
    "vw_modwt_forward": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _dp, _dp, _i32, _i32, _i32, _vp, _i64, _i64, _vp,
                                   _i64, _u32]),
    "vw_modwt_inverse": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _i64, _i64, _i64, _dp, _dp, _i32, _i32, _i32,
                                   C.POINTER(VwAlign), _i32, C.c_uint64, _i32, _vp, _i64, _u32]),
    "vw_modwt_forward_varlen": (C.c_int, [_vp, _vp, C.POINTER(_i64), _i64, _dp, _dp, _i32, _i32, _vp, _vp, _u32]),
    "vw_modwt_inverse_varlen": (C.c_int, [_vp, _vp, _vp, C.POINTER(_i64), _i64, _dp, _dp, _i32, _i32, _vp, _u32]),
    "vw_threshold": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _dp, _i32, _i32, _u32]),
    "vw_universal_threshold": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _dp, _u32]),
    "vw_swt_denoise": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _dp, _dp, _i32, _i32, _i32, C.POINTER(VwAlign), _i32,
                                 C.c_double, _i32, _vp, _i64, _dp, _u32]),
    "vw_wavelet_denoise": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _dp, _dp, _i32, _i32, _i32, C.POINTER(VwAlign), _i32,
                                     _i32, _i32, C.c_double, _i32, _vp, _i64, _dp, _u32]),
    "vw_energy": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _dp, _u32]),
    "vw_median_abs": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _dp, _u32]),
    "vw_mean_variance": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _dp, _dp, _u32]),
    "vw_modwt_forward_soa": (C.c_int, [_vp, _vp, _i64, _i64, _dp, _dp, C.c_int32, C.c_int32, C.POINTER(C.c_void_p), _vp, _u32]),
    "vw_sure_threshold": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _dp, _dp, _dp, _u32]),
    "vw_modwt_stream_level": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _dp, _dp, _i32, _i32, _vp, _i64, _vp, _i64, _u32]),
    "vw_stream_create": (C.c_int, [_vp, _dp, _dp, _i32, _i32, _i32, C.POINTER(_vp)]),
    "vw_stream_destroy": (C.c_int, [_vp, _vp]),
    "vw_stream_process": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _u32]),
    "vw_stream_flush": (C.c_int, [_vp, _vp, _i64, _vp, _i64, _i64, _vp, _i64, _u32]),
    "vw_stream_reset": (C.c_int, [_vp]),
    "vw_modwt_forward_span": (C.c_int, [_vp, _vp, _i64, _i64, _dp, _dp, _i32, _i32, _i32, _vp, _i64, _vp, _u32]),
    "vw_modwt_inverse_span": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _dp, _dp, _i32, _i32, _i32, _i32, _vp, _u32]),
    "vw_span_halo": (_i64, [_i32, _i32, _i32]),
    "vw_span_plan_query": (C.c_int, [_i32, _i32, _i64, _i32, C.POINTER(VwSpanPlan)]),
    "vw_modwt_forward_span_all": (C.c_int, [_vp, _vp, C.POINTER(VwSpanPlan), _dp, _dp, _vp, _i64, _vp, _u32]),
    "vw_span_pack_inverse": (C.c_int, [_vp, C.POINTER(VwSpanPlan), _vp, _i64, _vp, _vp, _u32]),
    "vw_span_unpack_inverse": (C.c_int, [_vp, C.POINTER(VwSpanPlan), _vp, _vp, _i64, _vp, _u32]),
    "vw_modwt_inverse_span_all": (C.c_int, [_vp, C.POINTER(VwSpanPlan), _vp, _i64, _vp, _dp, _dp, _i32, _vp, _u32]),
    "vw_modwt_inverse_span_all_thr": (C.c_int, [_vp, C.POINTER(VwSpanPlan), _vp, _i64, _vp, _dp, _dp, _i32, _vp, _i32, _vp,
                                                _u32]),
    "vw_span_median_bins": (_i32, [_i32]),
    "vw_span_median_state_bytes": (C.c_size_t, [_i64]),
    "vw_span_median_init": (C.c_int, [_vp, _vp, _i64]),
    "vw_span_median_hist": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _vp]),
    "vw_span_median_pick": (C.c_int, [_vp, _vp, _i32, _vp]),
    "vw_span_median_value": (C.c_int, [_vp, _vp, C.c_double, _vp]),
    "vw_init_multi": (C.c_int, [C.POINTER(C.c_int), _i32, C.POINTER(_vp)]),
    "vw_destroy_multi": (C.c_int, [_vp]),
    "vw_multi_size": (_i32, [_vp]),
    "vw_multi_ctx": (_vp, [_vp, _i32]),
    "vw_multi_last_error": (C.c_char_p, [_vp]),
    "vw_multi_synchronize": (C.c_int, [_vp]),
    "vw_modwt_forward_sharded": (C.c_int, [_vp, C.POINTER(VwSpanPlan), C.POINTER(_vp), _dp, _dp, _i32, C.POINTER(_vp), _i64,
                                           C.POINTER(_vp), C.POINTER(C.c_float), _u32]),
    "vw_modwt_inverse_sharded": (C.c_int, [_vp, C.POINTER(VwSpanPlan), C.POINTER(_vp), _i64, C.POINTER(_vp), _dp, _dp, _i32,
                                           _i32, C.POINTER(_vp), C.POINTER(C.c_float), _u32]),
    "vw_swt_denoise_sharded": (C.c_int, [_vp, C.POINTER(VwSpanPlan), C.POINTER(_vp), _dp, _dp, _i32, _i32, C.c_double, _i32,
                                         C.POINTER(_vp), _i64, C.POINTER(_vp), C.POINTER(_vp), _dp, _u32]),
    "vw_modwt_decompose_h": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _dp, _dp, _i32, _i32, _i32, C.POINTER(_vp), _u32]),
    "vw_result_shape": (C.c_int, [_vp, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i32)]),
    "vw_result_get_level": (C.c_int, [_vp, _vp, _i32, _vp, _i64, _u32]),
    "vw_result_set_level": (C.c_int, [_vp, _vp, _i32, _vp, _i64, _u32]),
    "vw_result_device_ptr": (_vp, [_vp, _i32]),
    "vw_result_threshold": (C.c_int, [_vp, _vp, _i32, _dp, _i32, _i32]),
    "vw_result_universal_threshold": (C.c_int, [_vp, _vp, _i32, _dp]),
    "vw_result_energy": (C.c_int, [_vp, _vp, _i32, _dp]),
    "vw_modwt_reconstruct_h": (C.c_int, [_vp, _vp, _dp, _dp, _i32, _i32, C.POINTER(VwAlign), _i32, C.c_uint64, _i32, _vp,
                                         _i64, _u32]),
    "vw_result_free": (C.c_int, [_vp, _vp]),
    "vw_graph_begin": (C.c_int, [_vp]),
    "vw_graph_end": (C.c_int, [_vp, C.POINTER(_vp)]),
    "vw_graph_launch": (C.c_int, [_vp, _vp, _u32]),
    "vw_graph_destroy": (C.c_int, [_vp, _vp]),
    "vw_last_timing": (C.c_int, [_vp, C.POINTER(VwTiming)]),
    "vw_probe_fp64": (C.c_int, [_vp, _dp, _dp]),
}

_lib = None
_lib_lock = threading.Lock()


def load_library():
    """dlopen libvwmodwt.so and declare every entry point.  Works without a GPU (symbol checks)."""
    global _lib
    with _lib_lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise NativeEngineError(
                    f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                    "(there is no CPU fallback for the MODWT engine)")
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def describe_plan(forward, l, levels, n, tile=0, fuse=0):
    """Text of the level schedule (host logic only; works without a GPU)."""
    buf = C.create_string_buffer(4096)
    rc = load_library().vw_describe_plan(int(bool(forward)), int(l), int(levels), int(n), int(tile), int(fuse), buf, 4096)
    if rc < 0:
        raise IllegalArgumentException(f"vw_describe_plan failed: {rc}")
    return buf.value.decode()


def lattice_query(hs, gs):
    """(coefficients or None, tap_err): the paraunitary lattice the column kernels of long filters would use for the
    scaled pair (hs, gs) -- t_1..t_{K-1} then the 2 x 2 base matrix -- or None when the pair keeps the direct form
    (host logic only; csrc/vw_lattice.cu)."""
    import numpy as np
    hs = np.ascontiguousarray(hs, dtype=np.float64)
    gs = np.ascontiguousarray(gs, dtype=np.float64)
    coef = np.zeros(64, dtype=np.float64)
    err = C.c_double(0.0)
    rc = load_library().vw_lattice_query(hs.ctypes.data_as(_dp), gs.ctypes.data_as(_dp), int(hs.size), coef.ctypes.data_as(_dp), 64,
                                          C.byref(err))
    if rc < 0:
        raise IllegalArgumentException(f"vw_lattice_query failed: {rc}")
    return (coef[:rc].copy() if rc > 0 else None), err.value


def plan_groups(forward, l, levels, n):
    """[(first_level, nlevels), ...] of the engine's launch schedule (host logic only)."""
    first = (_i32 * 64)()
    nlev = (_i32 * 64)()
    rc = load_library().vw_plan_query(int(bool(forward)), int(l), int(levels), int(n), first, nlev, 64)
    if rc < 0:
        raise IllegalArgumentException(f"vw_plan_query failed: {rc}")
    return [(int(first[i]), int(nlev[i])) for i in range(rc)]


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _np_rows(a, what="signal"):
    """host array -> (2-D float64 view with contiguous rows, was_1d)."""
    if a is None:
        raise NullPointerException(f"{what} cannot be null")
    a = np.asarray(a, dtype=np.float64)
    one_d = a.ndim == 1
    if one_d:
        a = a.reshape(1, -1)
    if a.ndim != 2:
        raise IllegalArgumentException(f"{what} must be 1-D or 2-D, got {a.ndim}-D")
    if a.shape[1] > 1 and a.strides[1] != 8 or (a.shape[0] > 1 and a.strides[0] % 8) or \
            (a.shape[0] > 1 and a.strides[0] < a.shape[1] * 8):
        a = np.ascontiguousarray(a)
    return a, one_d


def _ld(a):
    if _is_torch(a):
        return a.stride(0) if a.shape[0] > 1 else max(a.shape[1], 1)
    return a.strides[0] // 8 if a.shape[0] > 1 else max(a.shape[1], 1)


def _ptr(a):
    return a.data_ptr() if _is_torch(a) else a.ctypes.data


def _fp(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class Engine:
    """One native context (device + stream + scratch) per CUDA device, shared per process."""
    _engines = {}
    _lock = threading.Lock()

    def __init__(self, device):
        self.lib = load_library()
        ctx = _vp()
        rc = self.lib.vw_init(int(device), C.byref(ctx))
        if rc != VW_OK:
            raise NativeEngineError(
                f"vw_init(device={device}) failed with {self.lib.vw_status_name(rc).decode()}: the MODWT engine "
                "needs a CUDA device (no CPU fallback exists)")
        self.ctx = ctx
        self.device = self.lib.vw_device_index(ctx)
        self._call_lock = threading.Lock()

    @classmethod
    def get(cls, device=None):
        if device is None:
            try:
                import torch
                device = torch.cuda.current_device() if torch.cuda.is_available() else 0
            except Exception:
                device = 0
        with cls._lock:
            eng = cls._engines.get(device)
            if eng is None:
                eng = cls._engines[device] = Engine(device)
        return eng

    # -- plumbing ----------------------------------------------------------------------------
    def _check(self, rc):
        if rc == VW_OK:
            return
        msg = self.lib.vw_last_error(self.ctx).decode(errors="replace")
        name = self.lib.vw_status_name(rc).decode()
        exc, code = _STATUS.get(rc, (NativeEngineError, None))
        if code is not None:
            raise exc(f"[{code.value}] {msg}", code)
        raise exc(f"{name}: {msg}")

    def _bind_stream(self, *arrays):
        """device pointers => run on torch's current stream; returns the flag word.  Callers hold _call_lock across this and
        the ABI call that follows: vw_set_stream + the launch are two calls, and another thread rebinding the ctx in
        between would put the kernels on the wrong stream."""
        if any(_is_torch(a) for a in arrays if a is not None):
            import torch
            for a in arrays:
                if a is None:
                    continue
                if not _is_torch(a) or not a.is_cuda or a.dtype != torch.float64:
                    raise IllegalArgumentException("device calls need float64 CUDA tensors for every buffer")
                if a.device.index != self.device:
                    raise IllegalArgumentException(f"tensor on cuda:{a.device.index}, engine on cuda:{self.device}")
            self._check(self.lib.vw_set_stream(self.ctx, _vp(torch.cuda.current_stream(self.device).cuda_stream)))
            return FLAG_DEVICE_PTRS | FLAG_NO_SYNC
        self._check(self.lib.vw_reset_stream(self.ctx))
        return 0

    def pinned_empty(self, shape):
        """float64 numpy array over page-locked host memory (vw_alloc_pinned): the host side of asynchronous
        DMA, what the Java binding exposes as MemorySegment.reinterpret.  Freed when the array is collected."""
        count = int(np.prod(shape))
        ptr = self.lib.vw_alloc_pinned(max(count, 1) * 8)
        if not ptr:
            raise NativeEngineError("vw_alloc_pinned failed")
        buf = (C.c_double * max(count, 1)).from_address(ptr)
        arr = np.frombuffer(buf, dtype=np.float64, count=count).reshape(shape)
        lib = self.lib
        import weakref
        weakref.finalize(buf, lib.vw_free_pinned, ptr)
        return arr

    def set_option(self, name, value):
        self._check(self.lib.vw_set_option(self.ctx, name.encode(), int(value)))

    def launch_count(self):
        return int(self.lib.vw_launch_count(self.ctx))

    def synchronize(self):
        self._check(self.lib.vw_synchronize(self.ctx))

    def max_levels(self, n, l, cap=10):
        return int(self.lib.vw_max_levels(int(n), int(l), int(cap)))

    @staticmethod
    def _rows(x, what="signal"):
        if x is None:
            raise NullPointerException(f"{what} cannot be null")
        if _is_torch(x):
            one_d = x.dim() == 1
            x2 = x.reshape(1, -1) if one_d else x
            if x2.dim() != 2:
                raise IllegalArgumentException(f"{what} must be 1-D or 2-D")
            if x2.shape[1] > 1 and x2.stride(1) != 1:
                x2 = x2.contiguous()
            return x2, one_d
        return _np_rows(x, what)

    @staticmethod
    def _empty_like_rows(x, *shape):
        if _is_torch(x):
            import torch
            return torch.empty(shape, dtype=torch.float64, device=x.device)
        return np.empty(shape, dtype=np.float64)

    @staticmethod
    def _align_array(align, levels):
        if align is None:
            return None
        if len(align) != levels:
            raise IllegalArgumentException("alignment table must have one entry per level")
        arr = (VwAlign * levels)()
        for j, (sh, th, sg, tg) in enumerate(align):
            arr[j] = VwAlign(int(sh), int(th), int(sg), int(tg))
        return arr

    # -- primitives --------------------------------------------------------------------------
    def conv(self, x, filt, mode, out=None, flags=0):
        x2, _ = self._rows(x)
        if x2.shape[0] != 1:
            raise IllegalArgumentException("conv takes one signal")
        filt = _fp(filt)
        if _is_torch(x2):
            import torch
            fdev = torch.as_tensor(filt, device=x2.device)
            res = out if out is not None else torch.empty_like(x2[0])
            with self._call_lock:
                fl = self._bind_stream(x2, res) | flags
                self._check(self.lib.vw_conv_modwt(self.ctx, _vp(x2.data_ptr()), x2.shape[1], _vp(fdev.data_ptr()),
                                                   filt.size, mode, _vp(res.data_ptr()), fl))
            return res
        res = out if out is not None else np.empty(x2.shape[1])
        if res.dtype != np.float64 or not res.flags.c_contiguous or res.size != x2.shape[1]:
            raise IllegalArgumentException("output must be a contiguous float64 array of the signal's length")
        with self._call_lock:
            fl = self._bind_stream() | flags
            self._check(self.lib.vw_conv_modwt(self.ctx, _vp(x2.ctypes.data), x2.shape[1], _vp(filt.ctypes.data),
                                               filt.size, mode, _vp(res.ctypes.data), fl))
        return res

    def forward(self, x, hs, gs, levels, mode, flags=0, w_out=None, v_out=None):
        """x [B][N] (or [N]) -> (W [J][B][N], V_J [B][N]); same residency (numpy / torch.cuda) as x."""
        x2, one_d = self._rows(x)
        b, n = x2.shape
        hs, gs = _fp(hs), _fp(gs)
        if hs.size != gs.size:
            raise IllegalArgumentException("low-pass and high-pass filters must have the same length")
        lev = max(int(levels), 0)
        w = w_out if w_out is not None else self._empty_like_rows(x2, max(lev, 1), b, max(n, 1))
        v = v_out if v_out is not None else self._empty_like_rows(x2, b, max(n, 1))
        ldw = w.stride(1) if _is_torch(w) else w.strides[1] // 8
        lsw = w.stride(0) if _is_torch(w) else w.strides[0] // 8
        with self._call_lock:
            fl = self._bind_stream(x2, w, v) | flags
            self._check(self.lib.vw_modwt_forward(
                self.ctx, _vp(_ptr(x2)), b, n, _ld(x2), hs.ctypes.data_as(_dp), gs.ctypes.data_as(_dp), hs.size,
                int(levels), int(mode), _vp(_ptr(w)), ldw, lsw, _vp(_ptr(v)), _ld(v), fl))
        if one_d:
            return w[:, 0, :], v[0]
        return w, v

    def forward_soa(self, soa_x, batch, n, hs, gs, soa_w_levels, soa_v, flags=0):
        """BatchSIMDMODWT SoA layout ([t*batch + b], PERIODIC) in place: flat 1-D arrays, all numpy or all CUDA tensors;
        soa_w_levels = one flat output per level, soa_v = flat approximation output.  No transposes."""
        hs, gs = _fp(hs), _fp(gs)
        levels = len(soa_w_levels)
        tot = int(batch) * int(n)
        arrs = [soa_x, soa_v] + list(soa_w_levels)
        if any(_is_torch(a) for a in arrs) and not all(_is_torch(a) and a.is_cuda for a in arrs):
            raise IllegalArgumentException("SoA buffers must be all numpy or all CUDA tensors")
        for a in arrs:
            ok = (a.is_contiguous() and a.dtype.is_floating_point and a.element_size() == 8) if _is_torch(a) else \
                (isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags.c_contiguous)
            if not ok or (a.numel() if _is_torch(a) else a.size) != tot:
                raise IllegalArgumentException("SoA buffers must be contiguous float64 arrays of batchSize * signalLength")
        ptrs = (C.c_void_p * max(levels, 1))(*[_ptr(a) for a in soa_w_levels])
        with self._call_lock:
            fl = self._bind_stream(*arrs) | flags
            self._check(self.lib.vw_modwt_forward_soa(
                self.ctx, _vp(_ptr(soa_x)), int(batch), int(n), hs.ctypes.data_as(_dp), gs.ctypes.data_as(_dp), hs.size,
                levels, ptrs, _vp(_ptr(soa_v)), fl))

    def inverse(self, w, v, hs, gs, mode, align=None, order=ORDER_SPLIT, detail_mask=None, use_approx=True,
                flags=0, out=None):
        """W [J][B][N] (or [J][N]), V [B][N] (or [N]) -> x [B][N] (or [N])."""
        if w is None or v is None:
            raise NullPointerException("coefficients cannot be null")
        one_d = (v.dim() if _is_torch(v) else np.ndim(v)) == 1
        if not _is_torch(w):
            w = np.asarray(w, dtype=np.float64)
            v = np.asarray(v, dtype=np.float64)
        if one_d:
            w = w.reshape(w.shape[0], 1, -1)
            v = v.reshape(1, -1)
        if _is_torch(w):
            w, v = w.contiguous(), v.contiguous()
        else:
            w, v = np.ascontiguousarray(w), np.ascontiguousarray(v)
        levels, b, n = w.shape
        if tuple(v.shape) != (b, n):
            raise IllegalArgumentException("approximation and detail shapes must match")
        hs, gs = _fp(hs), _fp(gs)
        if detail_mask is None:
            detail_mask = (1 << levels) - 1
        res = out if out is not None else self._empty_like_rows(v, b, n)
        al = self._align_array(align, levels)
        with self._call_lock:
            fl = self._bind_stream(w, v, res) | flags
            self._check(self.lib.vw_modwt_inverse(
                self.ctx, _vp(_ptr(w)), n, b * n, _vp(_ptr(v)), n, b, n, hs.ctypes.data_as(_dp),
                gs.ctypes.data_as(_dp), hs.size, levels, int(mode), al, int(order), C.c_uint64(detail_mask),
                int(bool(use_approx)), _vp(_ptr(res)), _ld(res), fl))
        return res[0] if one_d else res

    @staticmethod
    def _packed(a, what):
        """1-D packed buffer: a contiguous float64 numpy array (pinned ones stay as they are) or CUDA tensor"""
        if a is None:
            raise NullPointerException(f"{what} cannot be null")
        if _is_torch(a):
            if a.dim() != 1:
                raise IllegalArgumentException(f"packed {what} must be 1-D")
            return a.contiguous()
        a = np.ascontiguousarray(a, dtype=np.float64)
        if a.ndim != 1:
            raise IllegalArgumentException(f"packed {what} must be 1-D")
        return a

    @staticmethod
    def _offsets(offsets, size):
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        if off.ndim != 1 or off.size < 2:
            raise IllegalArgumentException("offsets must hold batch + 1 row boundaries")
        if int(off[-1]) > size:
            raise IllegalArgumentException(f"offsets end at {int(off[-1])}, beyond the packed buffer of {size} samples")
        return off

    def forward_varlen(self, x, offsets, hs, gs, mode, flags=0, w_out=None, v_out=None):
        """Single-level forward of rows of different lengths in one launch: row b is x[offsets[b]:offsets[b+1]] of the
        packed 1-D x; returns packed (W, V) with the same layout and residency (numpy, pinned numpy or CUDA tensor)."""
        x = self._packed(x, "signal")
        size = x.numel() if _is_torch(x) else x.size
        off = self._offsets(offsets, size)
        hs, gs = _fp(hs), _fp(gs)
        if hs.size != gs.size:
            raise IllegalArgumentException("low-pass and high-pass filters must have the same length")
        w = w_out if w_out is not None else self._empty_like_rows(x, max(size, 1))
        v = v_out if v_out is not None else self._empty_like_rows(x, max(size, 1))
        with self._call_lock:
            fl = self._bind_stream(x, w, v) | flags
            self._check(self.lib.vw_modwt_forward_varlen(
                self.ctx, _vp(_ptr(x)), off.ctypes.data_as(C.POINTER(_i64)), off.size - 1, hs.ctypes.data_as(_dp),
                gs.ctypes.data_as(_dp), hs.size, int(mode), _vp(_ptr(w)), _vp(_ptr(v)), fl))
        return w[:size], v[:size]

    def inverse_varlen(self, w, v, offsets, hs, gs, mode, flags=0, out=None):
        """Single-level inverse (MODWTTransform.inverse per row: pair-added, SYMMETRIC t-l, else t+l) of packed rows of
        different lengths in one launch; returns the packed reconstruction."""
        w, v = self._packed(w, "detail coefficients"), self._packed(v, "approximation coefficients")
        size = w.numel() if _is_torch(w) else w.size
        if (v.numel() if _is_torch(v) else v.size) != size:
            raise IllegalArgumentException("approximation and detail buffers must have the same length")
        off = self._offsets(offsets, size)
        hs, gs = _fp(hs), _fp(gs)
        res = out if out is not None else self._empty_like_rows(v, max(size, 1))
        with self._call_lock:
            fl = self._bind_stream(w, v, res) | flags
            self._check(self.lib.vw_modwt_inverse_varlen(
                self.ctx, _vp(_ptr(w)), _vp(_ptr(v)), off.ctypes.data_as(C.POINTER(_i64)), off.size - 1,
                hs.ctypes.data_as(_dp), gs.ctypes.data_as(_dp), hs.size, int(mode), _vp(_ptr(res)), fl))
        return res[:size]

    def threshold(self, coeffs, thresholds, soft, flags=0):
        """In place on `coeffs` ([B][N] or [N]); thresholds: scalar or per-row host values."""
        c2, _ = self._rows(coeffs, "coefficients")
        thr = np.atleast_1d(np.asarray(thresholds, dtype=np.float64))
        per_row = int(thr.size > 1)
        if per_row and thr.size != c2.shape[0]:
            raise IllegalArgumentException("one threshold per row expected")
        if not _is_torch(c2) and not np.shares_memory(c2, coeffs):
            raise IllegalArgumentException("in-place thresholding needs a contiguous float64 array")
        with self._call_lock:
            fl = self._bind_stream(c2) | flags
            self._check(self.lib.vw_threshold(self.ctx, _vp(_ptr(c2)), c2.shape[0], c2.shape[1], _ld(c2),
                                              thr.ctypes.data_as(_dp), per_row, int(bool(soft)), fl))
        return coeffs

    def universal_threshold(self, w1, flags=0):
        w2, one_d = self._rows(w1, "coefficients")
        out = np.empty(w2.shape[0])
        with self._call_lock:
            fl = self._bind_stream(w2) | flags
            self._check(self.lib.vw_universal_threshold(self.ctx, _vp(_ptr(w2)), w2.shape[0], w2.shape[1], _ld(w2),
                                                        out.ctypes.data_as(_dp), fl))
        return float(out[0]) if one_d else out

    def denoise(self, x, hs, gs, levels, mode, align=None, order=ORDER_SPLIT, threshold=-1.0, soft=True, flags=0):
        x2, one_d = self._rows(x)
        b, n = x2.shape
        hs, gs = _fp(hs), _fp(gs)
        res = self._empty_like_rows(x2, b, max(n, 1))
        thr = np.empty(max(b, 1))
        al = self._align_array(align, int(levels)) if align is not None else None
        with self._call_lock:
            fl = self._bind_stream(x2, res) | flags
            self._check(self.lib.vw_swt_denoise(
                self.ctx, _vp(_ptr(x2)), b, n, _ld(x2), hs.ctypes.data_as(_dp), gs.ctypes.data_as(_dp), hs.size,
                int(levels), int(mode), al, int(order), float(threshold), int(bool(soft)), _vp(_ptr(res)), _ld(res),
                thr.ctypes.data_as(_dp), fl))
        return (res[0], float(thr[0])) if one_d else (res, thr)

    def wavelet_denoise(self, x, hs, gs, levels, mode, align=None, order=ORDER_SPLIT, multilevel=True,
                        method=THR_UNIVERSAL, fixed_threshold=0.0, soft=True, flags=0):
        """WaveletDenoiser over a [B][N] batch (or one [N] signal) in one call: x -> (denoised, thresholds [levels][B]),
        both in x's residency (numpy, or CUDA tensors whose rows may have a stride ld > n)."""
        x2, one_d = self._rows(x)
        b, n = x2.shape
        hs, gs = _fp(hs), _fp(gs)
        res = self._empty_like_rows(x2, b, max(n, 1))
        lev = max(int(levels), 1)
        thr = np.empty((lev, max(b, 1)))
        al = self._align_array(align, int(levels)) if align is not None else None
        with self._call_lock:
            fl = self._bind_stream(x2, res) | flags
            self._check(self.lib.vw_wavelet_denoise(
                self.ctx, _vp(_ptr(x2)), b, n, _ld(x2), hs.ctypes.data_as(_dp), gs.ctypes.data_as(_dp), hs.size,
                int(levels), int(mode), al, int(order), int(bool(multilevel)), int(method), float(fixed_threshold),
                int(bool(soft)), _vp(_ptr(res)), _ld(res), thr.ctypes.data_as(_dp), fl))
        thr = thr[:, :b]
        if _is_torch(x2):
            import torch
            thr = torch.as_tensor(thr, device=x2.device)
        return (res[0], thr[:, 0]) if one_d else (res, thr)

    def median_abs(self, c, flags=0):
        """exact median(|c|) per row (WaveletDenoiser.estimateNoiseSigma's order statistic)"""
        c2, one_d = self._rows(c, "coefficients")
        out = np.empty(c2.shape[0])
        with self._call_lock:
            fl = self._bind_stream(c2) | flags
            self._check(self.lib.vw_median_abs(self.ctx, _vp(_ptr(c2)), c2.shape[0], c2.shape[1], _ld(c2),
                                               out.ctypes.data_as(_dp), fl))
        return float(out[0]) if one_d else out

    def mean_variance(self, c, flags=0):
        """(mean, population variance about the mean) per row"""
        c2, one_d = self._rows(c, "coefficients")
        m, v = np.empty(c2.shape[0]), np.empty(c2.shape[0])
        with self._call_lock:
            fl = self._bind_stream(c2) | flags
            self._check(self.lib.vw_mean_variance(self.ctx, _vp(_ptr(c2)), c2.shape[0], c2.shape[1], _ld(c2),
                                                  m.ctypes.data_as(_dp), v.ctypes.data_as(_dp), fl))
        return (float(m[0]), float(v[0])) if one_d else (m, v)

    def sure_threshold(self, c, sigma, flags=0, with_risk=False):
        """WaveletDenoiser.calculateSUREThreshold per row (the reference's O(n^2) risk scan, bit for bit, on the device)"""
        c2, one_d = self._rows(c, "coefficients")
        sg = np.ascontiguousarray(np.broadcast_to(np.asarray(sigma, dtype=np.float64), (c2.shape[0],)))
        thr, risk = np.empty(c2.shape[0]), np.empty(c2.shape[0])
        with self._call_lock:
            fl = self._bind_stream(c2) | flags
            self._check(self.lib.vw_sure_threshold(self.ctx, _vp(_ptr(c2)), c2.shape[0], c2.shape[1], _ld(c2),
                                                   sg.ctypes.data_as(_dp), thr.ctypes.data_as(_dp),
                                                   risk.ctypes.data_as(_dp), fl))
        if with_risk:
            return (float(thr[0]), float(risk[0])) if one_d else (thr, risk)
        return float(thr[0]) if one_d else thr

    def energy(self, c, flags=0):
        c2, one_d = self._rows(c, "coefficients")
        out = np.empty(c2.shape[0])
        with self._call_lock:
            fl = self._bind_stream(c2) | flags
            self._check(self.lib.vw_energy(self.ctx, _vp(_ptr(c2)), c2.shape[0], c2.shape[1], _ld(c2),
                                           out.ctypes.data_as(_dp), fl))
        return float(out[0]) if one_d else out

    # -- span-sharded pieces (device tensors only) -----------------------------------------------
    def span_halo(self, l, first_level, nlevels):
        return int(self.lib.vw_span_halo(int(l), int(first_level), int(nlevels)))

    def forward_span(self, vin_ext, halo, hs, gs, first_level, nlevels, flags=0, w_out=None, v_out=None):
        """vin_ext: 1-D CUDA tensor [halo | span] -> (W [nlevels][n_local], V [n_local]).
        w_out: optional [nlevels][>= n_local] rows (row stride free), v_out: optional [n_local] (may be a slice)."""
        import torch
        n_local = vin_ext.numel() - halo
        hs, gs = _fp(hs), _fp(gs)
        w = w_out if w_out is not None else torch.empty((nlevels, max(n_local, 1)), dtype=torch.float64,
                                                        device=vin_ext.device)
        v = v_out if v_out is not None else torch.empty(max(n_local, 1), dtype=torch.float64, device=vin_ext.device)
        with self._call_lock:
            fl = self._bind_stream(vin_ext, w, v) | flags
            self._check(self.lib.vw_modwt_forward_span(
                self.ctx, _vp(vin_ext.data_ptr()), int(halo), int(n_local), hs.ctypes.data_as(_dp),
                gs.ctypes.data_as(_dp), hs.size, int(first_level), int(nlevels), _vp(w.data_ptr()), w.stride(0),
                _vp(v.data_ptr()), fl))
        return w, v

    def stream_level(self, ext, hist, hs, gs, level, w_out, v_out, flags=0):
        """One level of a streaming block: ext [B][hist + n] CUDA rows of [history | block] -> W, V [B][n] written into
        w_out / v_out (2-D CUDA views, unit inner stride; v_out may be the block part of the next level's ext)."""
        b, n = ext.shape[0], ext.shape[1] - hist
        hs, gs = _fp(hs), _fp(gs)
        assert ext.stride(1) == 1 and w_out.stride(1) == 1 and v_out.stride(1) == 1
        with self._call_lock:
            fl = self._bind_stream(ext, w_out, v_out) | flags
            self._check(self.lib.vw_modwt_stream_level(
                self.ctx, _vp(ext.data_ptr()), int(b), ext.stride(0), int(hist), int(n), hs.ctypes.data_as(_dp),
                gs.ctypes.data_as(_dp), hs.size, int(level), _vp(w_out.data_ptr()), w_out.stride(0),
                _vp(v_out.data_ptr()), v_out.stride(0), fl))
        return w_out, v_out

    def stream_create(self, hs, gs, levels, mode):
        """vw_stream_create: a StreamState keeping every level's history of a blockwise ZERO_PADDING / SYMMETRIC stream
        in HBM (BatchStreamingMODWT's state)."""
        hs, gs = _fp(hs), _fp(gs)
        if hs.size != gs.size:
            raise IllegalArgumentException("low-pass and high-pass filters must have the same length")
        st = StreamState(self, int(levels))
        with self._call_lock:
            self._check(self.lib.vw_stream_create(self.ctx, hs.ctypes.data_as(_dp), gs.ctypes.data_as(_dp), hs.size,
                                                  int(levels), int(mode), C.byref(st.handle)))
        return st

    def inverse_span(self, vin_ext, w_ext, halo, hs, gs, first_level, nlevels, order=ORDER_SPLIT, flags=0, out=None):
        """vin_ext [span | halo], w_ext [nlevels][span | halo] (CUDA) -> V_{first-1} [n_local]."""
        import torch
        n_local = vin_ext.numel() - halo
        hs, gs = _fp(hs), _fp(gs)
        if w_ext.stride(1) != 1:
            w_ext = w_ext.contiguous()
        out = out if out is not None else torch.empty(max(n_local, 1), dtype=torch.float64, device=vin_ext.device)
        with self._call_lock:
            fl = self._bind_stream(vin_ext, w_ext, out) | flags
            self._check(self.lib.vw_modwt_inverse_span(
                self.ctx, _vp(vin_ext.data_ptr()), _vp(w_ext.data_ptr()), w_ext.stride(0), int(halo), int(n_local),
                hs.ctypes.data_as(_dp), gs.ctypes.data_as(_dp), hs.size, int(first_level), int(nlevels), int(order),
                _vp(out.data_ptr()), fl))
        return out

    # -- span-sharded cascades, up-front halo schedule (one ABI call per direction) ------------------------
    def forward_span_all(self, xext, plan, hs, gs, w, v, flags=0):
        """xext [lead | n_local] (halo in place), w [levels][row_stride], v [n_local + pad]: CUDA tensors."""
        hs, gs = _fp(hs), _fp(gs)
        with self._call_lock:
            fl = self._bind_stream(xext, w, v) | flags
            self._check(self.lib.vw_modwt_forward_span_all(self.ctx, _vp(xext.data_ptr()), C.byref(plan), hs.ctypes.data_as(_dp),
                                                           gs.ctypes.data_as(_dp), _vp(w.data_ptr()), w.stride(0),
                                                           _vp(v.data_ptr()), fl))

    def span_pack_inverse(self, plan, w, v, msg):
        with self._call_lock:
            fl = self._bind_stream(w, v, msg)
            self._check(self.lib.vw_span_pack_inverse(self.ctx, C.byref(plan), _vp(w.data_ptr()), w.stride(0),
                                                      _vp(v.data_ptr()), _vp(msg.data_ptr()), fl))

    def span_unpack_inverse(self, plan, msg, w, v):
        """msg None: the open end of a ZERO_PADDING signal (zeros)."""
        with self._call_lock:
            fl = self._bind_stream(w, v, msg)
            self._check(self.lib.vw_span_unpack_inverse(self.ctx, C.byref(plan), _vp(msg.data_ptr() if msg is not None else None),
                                                        _vp(w.data_ptr()), w.stride(0), _vp(v.data_ptr()), fl))

    def inverse_span_all(self, plan, w, v, hs, gs, order, out, flags=0):
        hs, gs = _fp(hs), _fp(gs)
        with self._call_lock:
            fl = self._bind_stream(w, v, out) | flags
            self._check(self.lib.vw_modwt_inverse_span_all(self.ctx, C.byref(plan), _vp(w.data_ptr()), w.stride(0),
                                                           _vp(v.data_ptr()), hs.ctypes.data_as(_dp), gs.ctypes.data_as(_dp),
                                                           int(order), _vp(out.data_ptr()), fl))

    def inverse_span_all_thr(self, plan, w, v, hs, gs, order, thr, soft, out, flags=0):
        """inverse_span_all of the thresholded W: thr is a one-element float64 CUDA tensor (the threshold stays on the
        device), applied to every W sample as the kernels load it; W and V are left as they are."""
        hs, gs = _fp(hs), _fp(gs)
        with self._call_lock:
            fl = self._bind_stream(w, v, thr, out) | flags
            self._check(self.lib.vw_modwt_inverse_span_all_thr(self.ctx, C.byref(plan), _vp(w.data_ptr()), w.stride(0),
                                                               _vp(v.data_ptr()), hs.ctypes.data_as(_dp), gs.ctypes.data_as(_dp),
                                                               int(order), _vp(thr.data_ptr()), int(bool(soft)),
                                                               _vp(out.data_ptr()), fl))

    # -- exact median of |c| over spans on several ranks (vw_span_median_*; device tensors, nothing synchronises) -----
    def span_median_state(self, n_local):
        """a device state blob for the median rounds of a span of n_local samples (uint8 CUDA tensor)"""
        import torch
        return torch.empty(int(self.lib.vw_span_median_state_bytes(int(n_local))), dtype=torch.uint8,
                           device=torch.device("cuda", self.device))

    def span_median_init(self, state, n_total):
        with self._call_lock:
            self._bind_torch_stream()
            self._check(self.lib.vw_span_median_init(self.ctx, _vp(state.data_ptr()), int(n_total)))

    def span_median_hist(self, state, c, rnd, hist):
        """histogram of this rank's span c (float64 CUDA, contiguous) for round `rnd` into hist (int64 CUDA tensor of
        span_median_bins(rnd) entries; the counts are unsigned 64-bit, far below 2^63)"""
        with self._call_lock:
            self._bind_torch_stream()
            self._check(self.lib.vw_span_median_hist(self.ctx, _vp(state.data_ptr()), _vp(c.data_ptr()), int(c.numel()), int(rnd),
                                                     _vp(hist.data_ptr())))

    def span_median_pick(self, state, rnd, hist_sum):
        with self._call_lock:
            self._bind_torch_stream()
            self._check(self.lib.vw_span_median_pick(self.ctx, _vp(state.data_ptr()), int(rnd), _vp(hist_sum.data_ptr())))

    def span_median_value(self, state, factor, out):
        """out (one float64 CUDA element) = median / 0.6745 * factor, or the raw median for factor < 0"""
        with self._call_lock:
            self._bind_torch_stream()
            self._check(self.lib.vw_span_median_value(self.ctx, _vp(state.data_ptr()), float(factor), _vp(out.data_ptr())))

    def _bind_torch_stream(self):
        import torch
        self._check(self.lib.vw_set_stream(self.ctx, _vp(torch.cuda.current_stream(self.device).cuda_stream)))

    # -- timing record / graph replay ----------------------------------------------------------------------
    def last_timing(self):
        """(device_ms, host_ms, launches) of the last public call; needs set_option("timing", 1)."""
        t = VwTiming()
        self._check(self.lib.vw_last_timing(self.ctx, C.byref(t)))
        return float(t.device_ms), float(t.host_ms), int(t.launches)

    def probe_fp64(self):
        """(sustained FP64 FMA TFLOP/s measured now on this device, max SM MHz)"""
        t, m = C.c_double(0.0), C.c_double(0.0)
        with self._call_lock:
            self._check(self.lib.vw_reset_stream(self.ctx))
            self._check(self.lib.vw_probe_fp64(self.ctx, C.byref(t), C.byref(m)))
        return float(t.value), float(m.value)

    def capture(self):
        """`with eng.capture() as g: eng.forward(...)` records the calls into one CUDA graph; `g.launch()` replays them."""
        return _GraphCapture(self)

    # -- device-resident results -------------------------------------------------------------------------------
    def decompose_resident(self, x, hs, gs, levels, mode, result=None, flags=0):
        """vw_modwt_decompose_h: the coefficients stay in HBM behind a DeviceResult (reused when `result` has the shape)."""
        x2, _ = self._rows(x)
        b, n = x2.shape
        hs, gs = _fp(hs), _fp(gs)
        res = result if result is not None else DeviceResult(self)
        with self._call_lock:
            fl = self._bind_stream(x2) | flags
            self._check(self.lib.vw_modwt_decompose_h(self.ctx, _vp(_ptr(x2)), b, n, _ld(x2), hs.ctypes.data_as(_dp),
                                                      gs.ctypes.data_as(_dp), hs.size, int(levels), int(mode),
                                                      C.byref(res.handle), fl))
        return res


SPAN_MEDIAN_ROUNDS = 7      # VW_SPAN_MEDIAN_ROUNDS


def span_median_bins(rnd):
    """entries of round rnd's histogram (two tables: the lower and the upper middle order statistic)"""
    return int(load_library().vw_span_median_bins(int(rnd)))


def span_plan(l, levels, n_local, world):
    """vw_span_plan_query: layout + launch groups of the up-front span schedule (host logic only)."""
    plan = VwSpanPlan()
    rc = load_library().vw_span_plan_query(int(l), int(levels), int(n_local), int(world), C.byref(plan))
    if rc == 7:
        raise IllegalArgumentException("the total halo exceeds the per-rank span: use fewer ranks or levels")
    if rc == 5:
        raise InvalidArgumentException("upsampled filter longer than the signal", ErrorCode.VAL_TOO_LARGE)
    if rc != VW_OK:
        raise IllegalArgumentException(f"vw_span_plan_query failed: {rc}")
    return plan


class _GraphCapture:
    def __init__(self, eng):
        self.eng, self.handle = eng, _vp()

    def __enter__(self):
        with self.eng._call_lock:
            self.eng._check(self.eng.lib.vw_reset_stream(self.eng.ctx))
            self.eng._check(self.eng.lib.vw_graph_begin(self.eng.ctx))
        return self

    def __exit__(self, et, ev, tb):
        rc = self.eng.lib.vw_graph_end(self.eng.ctx, C.byref(self.handle))
        if et is None:
            self.eng._check(rc)
        return False

    def launch(self, flags=0):
        with self.eng._call_lock:
            self.eng._check(self.eng.lib.vw_reset_stream(self.eng.ctx))
            self.eng._check(self.eng.lib.vw_graph_launch(self.eng.ctx, self.handle, flags))

    def close(self):
        if self.handle:
            self.eng.lib.vw_graph_destroy(self.eng.ctx, self.handle)
            self.handle = _vp()


class DeviceResult:
    """A MultiLevelMODWTResult whose coefficients live in HBM (vw_result): levels come to the host only on request."""

    def __init__(self, eng):
        self.eng, self.handle = eng, _vp()

    def shape(self):
        b, n, j = _i64(), _i64(), _i32()
        self.eng._check(self.eng.lib.vw_result_shape(self.handle, C.byref(b), C.byref(n), C.byref(j)))
        return int(b.value), int(n.value), int(j.value)

    def get_level(self, level, out=None):
        """level 1..J: detail coefficients; 0: approximation -> [B][N] host array (or into a CUDA tensor `out`)."""
        b, n, _ = self.shape()
        res = out if out is not None else np.empty((b, n))
        with self.eng._call_lock:
            fl = self.eng._bind_stream(res)
            self.eng._check(self.eng.lib.vw_result_get_level(self.eng.ctx, self.handle, int(level), _vp(_ptr(res)), _ld(res), fl))
        return res

    def set_level(self, level, src):
        s2, _ = self.eng._rows(src, "coefficients")
        with self.eng._call_lock:
            fl = self.eng._bind_stream(s2)
            self.eng._check(self.eng.lib.vw_result_set_level(self.eng.ctx, self.handle, int(level), _vp(_ptr(s2)), _ld(s2), fl))

    def threshold(self, level, thresholds, soft):
        thr = np.atleast_1d(np.asarray(thresholds, dtype=np.float64))
        with self.eng._call_lock:
            self.eng._bind_stream()
            self.eng._check(self.eng.lib.vw_result_threshold(self.eng.ctx, self.handle, int(level), thr.ctypes.data_as(_dp),
                                                             int(thr.size > 1), int(bool(soft))))

    def universal_threshold(self, soft=True):
        b = self.shape()[0]
        thr = np.empty(b)
        with self.eng._call_lock:
            self.eng._bind_stream()
            self.eng._check(self.eng.lib.vw_result_universal_threshold(self.eng.ctx, self.handle, int(bool(soft)), thr.ctypes.data_as(_dp)))
        return thr

    def energy(self, level):
        out = np.empty(self.shape()[0])
        with self.eng._call_lock:
            self.eng._bind_stream()
            self.eng._check(self.eng.lib.vw_result_energy(self.eng.ctx, self.handle, int(level), out.ctypes.data_as(_dp)))
        return out

    def reconstruct(self, hs, gs, mode, align=None, order=ORDER_SPLIT, detail_mask=None, use_approx=True, out=None, flags=0):
        b, n, j = self.shape()
        hs, gs = _fp(hs), _fp(gs)
        res = out if out is not None else np.empty((b, n))
        if detail_mask is None:
            detail_mask = (1 << j) - 1
        al = Engine._align_array(align, j)
        with self.eng._call_lock:
            fl = self.eng._bind_stream(res) | flags
            self.eng._check(self.eng.lib.vw_modwt_reconstruct_h(self.eng.ctx, self.handle, hs.ctypes.data_as(_dp), gs.ctypes.data_as(_dp),
                                                                hs.size, int(mode), al, int(order), C.c_uint64(detail_mask),
                                                                int(bool(use_approx)), _vp(_ptr(res)), _ld(res), fl))
        return res

    def free(self):
        if self.handle:
            self.eng.lib.vw_result_free(self.eng.ctx, self.handle)
            self.handle = _vp()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class StreamState:
    """vw_stream_state: the histories of a blockwise stream live in HBM, and every block runs its whole cascade in one
    call.  Outputs follow the block's residency (numpy / pinned numpy: staged by the engine; CUDA tensor: zero copy)."""

    def __init__(self, eng, levels):
        self.eng, self.levels, self.handle = eng, levels, _vp()
        self.batch = None          # rows of the running stream (output shape of flush); None: no block since create / reset

    @staticmethod
    def _wv(w, v):
        ldw = w.stride(1) if _is_torch(w) else w.strides[1] // 8
        lsw = w.stride(0) if _is_torch(w) else w.strides[0] // 8
        return ldw, lsw, _ld(v)

    def process(self, x, flags=0, w_out=None, v_out=None):
        """block [B][n] -> (W [levels][B][n], V_J [B][n]); advances every level's history."""
        x2, _ = Engine._rows(x, "block")
        b, n = x2.shape
        w = w_out if w_out is not None else Engine._empty_like_rows(x2, self.levels, b, max(n, 1))
        v = v_out if v_out is not None else Engine._empty_like_rows(x2, b, max(n, 1))
        ldw, lsw, ldv = self._wv(w, v)
        with self.eng._call_lock:
            fl = self.eng._bind_stream(x2, w, v) | flags
            self.eng._check(self.eng.lib.vw_stream_process(self.eng.ctx, self.handle, _vp(_ptr(x2)), b, n, _ld(x2), _vp(_ptr(w)),
                                                           ldw, lsw, _vp(_ptr(v)), ldv, fl))
        self.batch = b
        return w, v

    def flush(self, tail_length, flags=0, w_out=None, v_out=None):
        """the cascade over the flush tail (histories not advanced) -> (W [levels][batch][tail], V_J [batch][tail]);
        host arrays unless CUDA tensors are given as outputs"""
        t, batch = max(int(tail_length), 1), self.batch or 1
        w = w_out if w_out is not None else np.empty((self.levels, batch, t))
        v = v_out if v_out is not None else np.empty((batch, t))
        ldw, lsw, ldv = self._wv(w, v)
        with self.eng._call_lock:
            fl = self.eng._bind_stream(w, v) | flags
            self.eng._check(self.eng.lib.vw_stream_flush(self.eng.ctx, self.handle, int(tail_length), _vp(_ptr(w)), ldw, lsw,
                                                         _vp(_ptr(v)), ldv, fl))
        return w, v

    def reset(self):
        self.eng._check(self.eng.lib.vw_stream_reset(self.handle))
        self.batch = None

    def close(self):
        if self.handle:
            with self.eng._call_lock:
                self.eng.lib.vw_stream_destroy(self.eng.ctx, self.handle)
            self.handle = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiEngine:
    """Several GPUs driven by ONE host thread (vw_init_multi): what a JVM caller uses for a span-sharded long signal.
    Buffers are torch CUDA tensors here, one list entry per device."""

    def __init__(self, devices):
        self.lib = load_library()
        self.devices = list(devices)
        arr = (C.c_int * len(self.devices))(*self.devices)
        self.handle = _vp()
        rc = self.lib.vw_init_multi(arr, len(self.devices), C.byref(self.handle))
        if rc != VW_OK:
            raise NativeEngineError(f"vw_init_multi({self.devices}) failed with {self.lib.vw_status_name(rc).decode()}")

    def _check(self, rc):
        if rc != VW_OK:
            msg = self.lib.vw_multi_last_error(self.handle).decode(errors="replace")
            exc, code = _STATUS.get(rc, (NativeEngineError, None))
            raise exc(f"[{code.value}] {msg}", code) if code is not None else exc(f"{self.lib.vw_status_name(rc).decode()}: {msg}")

    @staticmethod
    def _ptrs(tensors):
        return (_vp * len(tensors))(*[t.data_ptr() for t in tensors])

    def forward(self, plan, xext, hs, gs, mode, w, v, timed=False, flags=0):
        hs, gs = _fp(hs), _fp(gs)
        ms = C.c_float(0.0)
        self._check(self.lib.vw_modwt_forward_sharded(self.handle, C.byref(plan), self._ptrs(xext), hs.ctypes.data_as(_dp),
                                                      gs.ctypes.data_as(_dp), int(mode), self._ptrs(w), w[0].stride(0),
                                                      self._ptrs(v), C.byref(ms) if timed else None, flags))
        return float(ms.value) if timed else None

    def inverse(self, plan, w, v, hs, gs, mode, order, xout, timed=False, flags=0):
        hs, gs = _fp(hs), _fp(gs)
        ms = C.c_float(0.0)
        self._check(self.lib.vw_modwt_inverse_sharded(self.handle, C.byref(plan), self._ptrs(w), w[0].stride(0), self._ptrs(v),
                                                      hs.ctypes.data_as(_dp), gs.ctypes.data_as(_dp), int(mode), int(order),
                                                      self._ptrs(xout), C.byref(ms) if timed else None, flags))
        return float(ms.value) if timed else None

    def denoise(self, plan, xext, hs, gs, mode, order, w, v, xout, threshold=-1.0, soft=True, flags=0):
        """vw_swt_denoise_sharded: buffers as forward / inverse (xext filled behind the lead); returns the threshold, or
        None under FLAG_NO_SYNC (reading it back would wait for rank 0)"""
        hs, gs = _fp(hs), _fp(gs)
        thr = C.c_double(0.0)
        want = not (flags & FLAG_NO_SYNC)
        self._check(self.lib.vw_swt_denoise_sharded(self.handle, C.byref(plan), self._ptrs(xext), hs.ctypes.data_as(_dp),
                                                    gs.ctypes.data_as(_dp), int(mode), int(order), float(threshold), int(bool(soft)),
                                                    self._ptrs(w), w[0].stride(0), self._ptrs(v), self._ptrs(xout),
                                                    C.byref(thr) if want else None, flags))
        return float(thr.value) if want else None

    def synchronize(self):
        self._check(self.lib.vw_multi_synchronize(self.handle))

    def launch_count(self):
        return sum(int(self.lib.vw_launch_count(_vp(self.lib.vw_multi_ctx(self.handle, r)))) for r in range(len(self.devices)))

    def close(self):
        if self.handle:
            self.lib.vw_destroy_multi(self.handle)
            self.handle = _vp()
