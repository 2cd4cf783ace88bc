"""Mixed-length single-level batches (vw_modwt_forward_varlen / vw_modwt_inverse_varlen): every row against the CPU
oracle (1e-12 * max|x|, bit-identical under VW_FLAG_BITEXACT), against today's per-signal forward / inverse loop, the
reference's error order (lowest bad row wins), one launch per direction whatever the row count, and the C++ host."""
import os
import subprocess
import sys

import numpy as np
import pytest

import vectorwave_b200 as vw
from oracle import cref
from oracle.wavelets import filters
from vectorwave_b200 import _native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BM = vw.BoundaryMode
MODES = [BM.PERIODIC, BM.ZERO_PADDING, BM.SYMMETRIC]
WAVELETS = ["haar", "db2", "db4", "db6", "db8", "db10", "sym4", "sym8", "coif2", "coif3", "coif5"]
S = 1.0 / np.sqrt(2.0)
MIXED = [1, 2, 3, 5, 7, 1, 11, 13, 16, 31, 64, 97, 127, 1000, 1021, 4096, 4099, 3, 2, 1]


def _rows(lengths, seed):
    rng = np.random.default_rng(seed)
    return [rng.standard_normal(n) for n in lengths]


def _pack(rows):
    off = np.zeros(len(rows) + 1, dtype=np.int64)
    np.cumsum([r.size for r in rows], out=off[1:])
    return np.concatenate(rows), off


def _tol(x):
    return 1e-12 * max(1.0, float(np.max(np.abs(x))))


def _check_rows(x, off, w, v, xr, h, g, mode, exact):
    """forward rows against the oracle; the inverse of the ORACLE's coefficients against its inverse (t - l for SYMMETRIC)"""
    tol = _tol(x)
    for b in range(off.size - 1):
        s, e = off[b], off[b + 1]
        vo, wo = cref.forward_single(x[s:e], h, g, mode)
        xo = cref.inverse_single(vo, wo, h, g, mode)
        if exact:
            np.testing.assert_array_equal(v[s:e], vo, err_msg=f"row {b} V")
            np.testing.assert_array_equal(w[s:e], wo, err_msg=f"row {b} W")
            np.testing.assert_array_equal(xr[s:e], xo, err_msg=f"row {b} inverse")
        else:
            np.testing.assert_allclose(v[s:e], vo, rtol=0, atol=tol, err_msg=f"row {b} V")
            np.testing.assert_allclose(w[s:e], wo, rtol=0, atol=tol, err_msg=f"row {b} W")
            np.testing.assert_allclose(xr[s:e], xo, rtol=0, atol=tol, err_msg=f"row {b} inverse")


def _oracle_coeffs(x, off, h, g, mode):
    w, v = np.empty_like(x), np.empty_like(x)
    for b in range(off.size - 1):
        s, e = off[b], off[b + 1]
        v[s:e], w[s:e] = cref.forward_single(x[s:e], h, g, mode)
    return w, v


# ---- host-only checks ------------------------------------------------------------------------------------------
def test_offsets_are_checked_on_the_host():
    with pytest.raises(vw.IllegalArgumentException):
        _native.Engine._offsets([0], 4)
    with pytest.raises(vw.IllegalArgumentException):
        _native.Engine._offsets([0, 3, 9], 8)
    np.testing.assert_array_equal(_native.Engine._offsets([0, 3, 8], 8), [0, 3, 8])


# ---- GPU -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", WAVELETS)
def test_every_row_matches_the_oracle(name, mode):
    eng = vw.Engine.get()
    h, g, _ = filters(name)
    x, off = _pack(_rows(MIXED, 11))
    for flags, exact in ((0, False), (_native.FLAG_BITEXACT, True)):
        w, v = eng.forward_varlen(x, off, h * S, g * S, mode.value, flags)
        wo, vo = _oracle_coeffs(x, off, h, g, mode.value)
        xr = eng.inverse_varlen(wo, vo, off, h * S, g * S, mode.value, flags)
        _check_rows(x, off, w, v, xr, h, g, mode.value, exact)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", ["db4", "sym8", "coif5"])
def test_long_row_between_single_samples(name, mode):
    eng = vw.Engine.get()
    h, g, _ = filters(name)
    x, off = _pack(_rows([1, 1 << 20, 1, 1, 2, 1 << 12, 1], 12))
    for flags, exact in ((0, False), (_native.FLAG_BITEXACT, True)):
        w, v = eng.forward_varlen(x, off, h * S, g * S, mode.value, flags)
        wo, vo = _oracle_coeffs(x, off, h, g, mode.value)
        xr = eng.inverse_varlen(wo, vo, off, h * S, g * S, mode.value, flags)
        _check_rows(x, off, w, v, xr, h, g, mode.value, exact)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_ten_thousand_short_rows_bit_exact(mode):
    eng = vw.Engine.get()
    rng = np.random.default_rng(13)
    x, off = _pack(_rows(rng.integers(1, 65, size=12000), 14))
    for name in ("haar", "sym8", "coif5"):
        h, g, _ = filters(name)
        w, v = eng.forward_varlen(x, off, h * S, g * S, mode.value, _native.FLAG_BITEXACT)
        wo, vo = _oracle_coeffs(x, off, h, g, mode.value)
        np.testing.assert_array_equal(w, wo)
        np.testing.assert_array_equal(v, vo)
        xr = eng.inverse_varlen(wo, vo, off, h * S, g * S, mode.value, _native.FLAG_BITEXACT)
        for b in range(0, off.size - 1, 97):
            s, e = off[b], off[b + 1]
            np.testing.assert_array_equal(xr[s:e], cref.inverse_single(vo[s:e], wo[s:e], h, g, mode.value))
        wf, vf = eng.forward_varlen(x, off, h * S, g * S, mode.value)
        np.testing.assert_allclose(wf, wo, rtol=0, atol=_tol(x))
        np.testing.assert_allclose(vf, vo, rtol=0, atol=_tol(x))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_pageable_pinned_and_device_inputs_agree(mode):
    import torch
    eng = vw.Engine.get()
    h, g, _ = filters("db8")
    hs, gs = h * S, g * S
    for lengths in (MIXED, [700_001, 5, 1_300_003, 1, 999_983, 17]):     # small (zero-copy when pinned), large (pipelined)
        x, off = _pack(_rows(lengths, 15))
        wo, vo = _oracle_coeffs(x, off, h, g, mode.value)
        w0, v0 = eng.forward_varlen(x, off, hs, gs, mode.value)
        xp = eng.pinned_empty(x.shape)
        xp[...] = x
        wp, vp = eng.forward_varlen(xp, off, hs, gs, mode.value, w_out=eng.pinned_empty(x.shape), v_out=eng.pinned_empty(x.shape))
        wd, vd = eng.forward_varlen(torch.as_tensor(x, device="cuda"), off, hs, gs, mode.value)
        torch.cuda.synchronize()
        np.testing.assert_allclose(w0, wo, rtol=0, atol=_tol(x))
        np.testing.assert_allclose(v0, vo, rtol=0, atol=_tol(x))
        for w, v in ((wp, vp), (wd.cpu().numpy(), vd.cpu().numpy())):
            np.testing.assert_array_equal(w, w0)
            np.testing.assert_array_equal(v, v0)
        x0 = eng.inverse_varlen(wo, vo, off, hs, gs, mode.value)
        wpp, vpp = eng.pinned_empty(x.shape), eng.pinned_empty(x.shape)
        wpp[...], vpp[...] = wo, vo
        xpp = eng.inverse_varlen(wpp, vpp, off, hs, gs, mode.value, out=eng.pinned_empty(x.shape))
        xdd = eng.inverse_varlen(torch.as_tensor(wo, device="cuda"), torch.as_tensor(vo, device="cuda"), off, hs, gs, mode.value)
        torch.cuda.synchronize()
        for b in range(off.size - 1):
            s, e = off[b], off[b + 1]
            np.testing.assert_allclose(x0[s:e], cref.inverse_single(vo[s:e], wo[s:e], h, g, mode.value), rtol=0, atol=_tol(x))
        np.testing.assert_array_equal(xpp, x0)
        np.testing.assert_array_equal(xdd.cpu().numpy(), x0)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("flags", [0, _native.FLAG_BITEXACT])
def test_batch_api_equals_the_per_signal_loop(mode, flags):
    t = vw.MODWTTransform(vw.Daubechies.DB4, mode, flags=flags)
    rows = _rows(MIXED, 16)
    got = t.forwardBatch(rows)
    loop = [t.forward(r) for r in rows]
    tol = _tol(np.concatenate(rows))
    for a, b in zip(got, loop):
        if flags:
            np.testing.assert_array_equal(a.approximationCoeffs(), b.approximationCoeffs())
            np.testing.assert_array_equal(a.detailCoeffs(), b.detailCoeffs())
        else:
            np.testing.assert_allclose(a.approximationCoeffs(), b.approximationCoeffs(), rtol=0, atol=tol)
            np.testing.assert_allclose(a.detailCoeffs(), b.detailCoeffs(), rtol=0, atol=tol)
    back = t.inverseBatch(loop)
    for r, res in zip(back, loop):
        ref = t.inverse(res)
        if flags:
            np.testing.assert_array_equal(r, ref)
        else:
            np.testing.assert_allclose(r, ref, rtol=0, atol=tol)


@pytest.mark.gpu
def test_symmetric_inverse_batch_uses_the_minus_rule():
    # mixed lengths take inverse() per row (t - l), not the optimized equal-length body (t + l)
    h, g, _ = filters("sym4")
    t = vw.MODWTTransform(vw.Symlet.SYM4, BM.SYMMETRIC)
    rows = _rows([64, 100, 128, 5, 300], 17)
    res = t.forwardBatch(rows)
    for r, out in zip(res, t.inverseBatch(res)):
        v, w = r.approximationCoeffs(), r.detailCoeffs()
        minus = cref.inverse_single(v, w, h, g, 2, batch_variant=False)
        plus = cref.inverse_single(v, w, h, g, 2, batch_variant=True)
        np.testing.assert_allclose(out, minus, rtol=0, atol=_tol(v))
        assert v.size < 8 or np.max(np.abs(minus - plus)) > 1e-6    # the two rules really differ here


@pytest.mark.gpu
def test_device_tensor_lists_stay_on_the_device():
    import torch
    t = vw.MODWTTransform(vw.Coiflet.COIF5, BM.PERIODIC)
    rows = [torch.as_tensor(r, device="cuda") for r in _rows(MIXED, 18)]
    res = t.forwardBatch(rows)
    assert all(r.approximationCoeffs().is_cuda for r in res)
    back = t.inverseBatch(res)
    assert all(b.is_cuda for b in back)
    h, g, _ = filters("coif5")
    for x, r in zip(rows, res):
        vo, wo = cref.forward_single(x.cpu().numpy(), h, g, 0)
        np.testing.assert_allclose(r.approximationCoeffs().cpu().numpy(), vo, rtol=0, atol=_tol(vo))
        np.testing.assert_allclose(r.detailCoeffs().cpu().numpy(), wo, rtol=0, atol=_tol(vo))


@pytest.mark.gpu
def test_one_launch_per_direction_whatever_the_row_count():
    import torch
    eng = vw.Engine.get()
    h, g, _ = filters("sym8")
    deltas = []
    for batch in (10, 10_000):
        x, off = _pack(_rows(np.random.default_rng(batch).integers(1, 200, size=batch), 19))
        xd = torch.as_tensor(x, device="cuda")
        for flags in (0, _native.FLAG_CHECK_FINITE):
            n0 = eng.launch_count()
            w, v = eng.forward_varlen(xd, off, h * S, g * S, 2, flags)
            n1 = eng.launch_count()
            eng.inverse_varlen(w, v, off, h * S, g * S, 2, flags)
            deltas.append((flags, n1 - n0, eng.launch_count() - n1))
        torch.cuda.synchronize()
    assert deltas[:2] == deltas[2:]
    assert deltas[0][1:] == (1, 1)


@pytest.mark.gpu
def test_errors_name_the_lowest_bad_row_like_the_loop():
    t = vw.MODWTTransform(vw.Daubechies.DB4, BM.PERIODIC)
    ok, nan, empty = np.ones(9), np.array([1.0, np.nan, 2.0]), np.array([])
    for rows, code, row in (([ok, ok[:5], nan, empty, ok], vw.ErrorCode.VAL_NON_FINITE_VALUES, 2),
                            ([ok, empty, nan, ok[:4]], vw.ErrorCode.VAL_EMPTY, 1),
                            ([ok[:2], ok, np.array([np.inf]), nan], vw.ErrorCode.VAL_NON_FINITE_VALUES, 2)):
        with pytest.raises(vw.InvalidSignalException) as batch_err:
            t.forwardBatch(rows)
        assert batch_err.value.error_code == code and f"row {row}" in str(batch_err.value)
        with pytest.raises(vw.InvalidSignalException) as loop_err:
            [t.forward(r) for r in rows]
        assert loop_err.value.error_code == code
    with pytest.raises(vw.IllegalArgumentException):   # a 2-D row after a NaN row: the NaN row still wins
        t.forwardBatch([ok[:3], np.ones((2, 2))])
    with pytest.raises(vw.InvalidSignalException):
        t.forwardBatch([nan, np.ones((2, 2))])
    res = t.forwardBatch([ok, ok[:3], ok[:5], ok[:7]])
    res[1]._a[0] = np.nan
    res[3]._d[2] = np.inf
    with pytest.raises(vw.InvalidSignalException) as inv_err:
        t.inverseBatch(res)
    assert inv_err.value.error_code == vw.ErrorCode.VAL_NON_FINITE_VALUES and "row 1" in str(inv_err.value)


@pytest.mark.gpu
def test_bad_offsets_and_capture_are_rejected():
    import ctypes as C
    eng = vw.Engine.get()
    h, g, _ = filters("db4")
    hs, gs = np.ascontiguousarray(h * S), np.ascontiguousarray(g * S)
    x = np.ones(16)
    out = np.empty(16), np.empty(16)
    for bad in ([1, 8, 16], [0, 9, 8, 16], [0, 4, 2]):
        off = np.asarray(bad, dtype=np.int64)
        rc = eng.lib.vw_modwt_forward_varlen(eng.ctx, x.ctypes.data, off.ctypes.data_as(C.POINTER(C.c_int64)), off.size - 1,
                                             hs.ctypes.data_as(_native._dp), gs.ctypes.data_as(_native._dp), 8, 0,
                                             out[0].ctypes.data, out[1].ctypes.data, 0)
        assert rc == 7, bad
        rc = eng.lib.vw_modwt_inverse_varlen(eng.ctx, x.ctypes.data, x.ctypes.data, off.ctypes.data_as(C.POINTER(C.c_int64)),
                                             off.size - 1, hs.ctypes.data_as(_native._dp), gs.ctypes.data_as(_native._dp), 8, 0,
                                             out[0].ctypes.data, 0)
        assert rc == 7, bad
    with pytest.raises(vw.NativeEngineError):
        with eng.capture():
            eng.forward_varlen(eng.pinned_empty((16,)), [0, 8, 16], hs, gs, 0)


@pytest.mark.gpu
def test_cpp_host_mixed_length_forward_batch():
    sys.path.insert(0, ROOT)
    cref.build()
    exe = os.path.join(ROOT, "tests", "cpp", "_build", "varlen_host")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    lib, ora = os.path.join(ROOT, "vectorwave_b200"), os.path.join(ROOT, "oracle", "_build")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "varlen_host.cpp"), "-o", exe, "-L", lib, "-lvwmodwt", "-L", ora,
                           "-lvw_oracle", f"-Wl,-rpath,{lib}", f"-Wl,-rpath,{ora}", "-Wl,-rpath,/usr/local/cuda/lib64"])
    p = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and p.stdout.strip().endswith("ok"), p.stdout[-2000:] + p.stderr[-2000:]
