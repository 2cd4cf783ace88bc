"""Streaming MODWT state on the device (vw_stream_create / process / flush / reset / destroy): every level's history kept
in HBM and a block's whole cascade in one call.  Every block is compared with nptwin.StreamingOracle to 1e-12*max|x|,
and bit for bit under VW_FLAG_BITEXACT; the fused kernel and the per-level path (VW_FLAG_NO_FUSE, and shapes whose rows
do not fit one CTA) both run; the C++ host class runs against the C oracle; the Python facade keeps its exceptions."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import vectorwave_b200 as vw
from oracle import cref, nptwin
from oracle.wavelets import filters
from vectorwave_b200 import _native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
S = 1.0 / np.sqrt(2.0)
ZP, SYM = 1, 2
F = _native


def _taps(name):
    h, g, _ = filters(name)
    return h, g, np.ascontiguousarray(h * S), np.ascontiguousarray(g * S)


def _check(got, ref, tol, exact, what):
    w, v = (np.asarray(a.cpu() if hasattr(a, "cpu") else a) for a in got)
    wo, vo = ref
    if exact:
        assert np.array_equal(w, wo) and np.array_equal(v, vo), what
    else:
        err = max(float(np.max(np.abs(w - wo))), float(np.max(np.abs(v - vo))))
        assert err <= tol, f"{what}: {err:.3e} > {tol:.3e}"


# ---- CPU: the facade raises what it raised before, without touching a device ------------------------------------------
def test_facade_exceptions_need_no_device():
    from vectorwave_b200.streaming import IllegalStateException, UnsupportedOperationException
    BM = vw.BoundaryMode
    with pytest.raises(vw.IllegalArgumentException):
        vw.BatchStreamingMODWT.Builder().build()
    with pytest.raises(vw.IllegalArgumentException):
        vw.BatchStreamingMODWT.Builder().wavelet(vw.Daubechies.DB4).levels(0).build()
    st = vw.BatchStreamingMODWT.Builder().wavelet(vw.Daubechies.DB4).boundary(BM.SYMMETRIC).levels(2).build()
    with pytest.raises(IllegalStateException):
        st.processSingleLevel(np.ones((2, 8)))
    with pytest.raises(IllegalStateException):
        st.flushMultiLevel(3)
    with pytest.raises(vw.IllegalArgumentException):
        st.processMultiLevel([])
    with pytest.raises(vw.IllegalArgumentException):
        st.processMultiLevel([[1.0, 2.0], [3.0]])
    with pytest.raises(vw.IllegalArgumentException):
        st.getHistoryLengthForLevel(3)
    assert st.getHistoryLengthForLevel(2) == 14 and st.getMinFlushTailLength() == 7 == st.suggestFlushTailLength()
    assert np.asarray(st.flushMultiLevel(0).finalApprox()).shape == (0, 0)
    with pytest.raises(UnsupportedOperationException):
        vw.BatchStreamingMODWT.Builder().wavelet(vw.Daubechies.DB4).levels(2).build().flushMultiLevel(3)
    st.close()
    with pytest.raises(IllegalStateException):
        st.flushMultiLevel(3)


# ---- GPU: parity with the oracle, both paths, exact and fused arithmetic -------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("levels", [1, 2, 3, 4, 5, 6, 7])
@pytest.mark.parametrize("mode", [ZP, SYM])
@pytest.mark.parametrize("name", ["haar", "db4", "sym8", "db8", "coif5"])
def test_blocks_flush_restart_and_reset_match_the_oracle(name, mode, levels):
    eng = vw.Engine.get()
    h, g, hs, gs = _taps(name)
    rng = np.random.default_rng(levels * 10 + mode)
    b = 4
    x = rng.standard_normal((b, 3000))
    tol = 1e-12 * float(np.max(np.abs(x)))
    first = 1 if name == "haar" else 3        # shorter than every history: the SYMMETRIC first block wraps many times
    sizes = (first, 517, 2, 1001)
    tail = len(h) - 1
    ref = []
    so = nptwin.StreamingOracle(h, g, levels, mode)
    at = 0
    for s in sizes:
        ref.append(so.process(x[:, at:at + s]))
        at += s
    ref_flush = so.flush(tail)
    ref_next = so.process(x[:, at:at + 300])
    ref_restart = nptwin.StreamingOracle(h, g, levels, mode).process(x[:2, :64])   # batch 4 -> 2 restarts
    ref_reset = nptwin.StreamingOracle(h, g, levels, mode).process(x[:2, 64:100])
    for flags in (0, F.FLAG_NO_FUSE, F.FLAG_BITEXACT, F.FLAG_BITEXACT | F.FLAG_NO_FUSE):
        exact = bool(flags & F.FLAG_BITEXACT)
        st = eng.stream_create(hs, gs, levels, mode)
        try:
            at = 0
            for s, r in zip(sizes, ref):
                _check(st.process(x[:, at:at + s], flags), r, tol, exact, f"block {s} flags {flags}")
                at += s
            _check(st.flush(tail, flags), ref_flush, tol, exact, f"flush flags {flags}")
            _check(st.process(x[:, at:at + 300], flags), ref_next, tol, exact, f"after flush flags {flags}")
            _check(st.process(x[:2, :64], flags), ref_restart, tol, exact, f"batch change flags {flags}")
            st.reset()
            _check(st.process(x[:2, 64:100], flags), ref_reset, tol, exact, f"reset flags {flags}")
        finally:
            st.close()


@pytest.mark.gpu
def test_one_launch_per_block_and_flush_on_the_fused_path():
    import torch
    eng = vw.Engine.get()
    h, g, hs, gs = _taps("db4")
    x = torch.as_tensor(np.random.default_rng(3).standard_normal((64, 3 * 256)), device="cuda")
    for mode in (ZP, SYM):
        st = eng.stream_create(hs, gs, 4, mode)
        deltas = []
        for k in range(3):
            n0 = eng.launch_count()
            st.process(x[:, k * 256:(k + 1) * 256])
            deltas.append(eng.launch_count() - n0)
        w = torch.empty((4, 64, 7), dtype=torch.float64, device="cuda")
        v = torch.empty((64, 7), dtype=torch.float64, device="cuda")
        n0 = eng.launch_count()
        st.flush(7, w_out=w, v_out=v)
        deltas.append(eng.launch_count() - n0)
        torch.cuda.synchronize()
        st.close()
        assert deltas == [1, 1, 1, 1], deltas


@pytest.mark.gpu
@pytest.mark.parametrize("name,levels,n,mode", [("coif5", 10, 300, SYM), ("db4", 3, 20000, ZP), ("coif5", 8, 15000, ZP)])
def test_shapes_that_do_not_fit_a_cta_take_the_per_level_path(name, levels, n, mode):
    eng = vw.Engine.get()
    h, g, hs, gs = _taps(name)
    x = np.random.default_rng(n).standard_normal((3, 3 * n))
    tol = 1e-12 * float(np.max(np.abs(x)))
    so = nptwin.StreamingOracle(h, g, levels, mode)
    st = eng.stream_create(hs, gs, levels, mode)
    try:
        for k, s in enumerate((n, 7, n)):
            blk = x[:, k * n:k * n + s]
            n0 = eng.launch_count()
            got = st.process(blk)
            # the path is chosen per call: one launch exactly when the two level buffers fit one CTA (227 KB on sm_100)
            fits = 2 * (((len(h) - 1) << (levels - 1)) + s) * 8 <= 227 * 1024
            assert (eng.launch_count() - n0 == 1) == fits
            _check(got, so.process(blk), tol, False, f"{name} J={levels} block {s}")
        _check(st.flush(len(h) - 1), so.flush(len(h) - 1), tol, False, "flush")
    finally:
        st.close()


@pytest.mark.gpu
def test_fused_and_per_level_paths_agree_and_the_last_cta_is_covered():
    import torch
    eng = vw.Engine.get()
    h, g, hs, gs = _taps("sym8")
    x = torch.as_tensor(np.random.default_rng(5).standard_normal((4096, 2 * 1024)), device="cuda")
    tol = 1e-12 * float(torch.max(torch.abs(x)))
    a = eng.stream_create(hs, gs, 6, SYM)
    b = eng.stream_create(hs, gs, 6, SYM)
    rows = [0, 1, 2047, 4094, 4095]
    so = nptwin.StreamingOracle(h, g, 6, SYM)
    try:
        for k in range(2):
            blk = x[:, k * 1024:(k + 1) * 1024]
            wa, va = a.process(blk)
            wb, vb = b.process(blk, F.FLAG_NO_FUSE)
            torch.cuda.synchronize()
            assert float(torch.max(torch.abs(wa - wb))) <= tol and float(torch.max(torch.abs(va - vb))) <= tol
            wo, vo = so.process(blk[rows].cpu().numpy())
            _check((wa[:, rows], va[rows]), (wo, vo), tol, False, f"block {k}")
    finally:
        a.close()
        b.close()


# ---- GPU: residency, strides, independent handles --------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", [ZP, SYM])
def test_pageable_pinned_device_inputs_and_strided_outputs(mode):
    import torch
    eng = vw.Engine.get()
    h, g, hs, gs = _taps("db8")
    J, b, n = 3, 5, 333
    x = np.random.default_rng(mode).standard_normal((b, 4 * n))
    tol = 1e-12 * float(np.max(np.abs(x)))
    so = nptwin.StreamingOracle(h, g, J, mode)
    refs = [so.process(x[:, k * n:(k + 1) * n]) for k in range(4)]
    ref_flush = so.flush(9)
    st = eng.stream_create(hs, gs, J, mode)
    try:
        # pageable host block
        _check(st.process(x[:, :n]), refs[0], tol, False, "pageable")
        # pinned host block and pinned, strided outputs
        xp = eng.pinned_empty((b, n))
        xp[:] = x[:, n:2 * n]
        wbig, vbig = eng.pinned_empty((J, b + 1, n + 3)), eng.pinned_empty((b, n + 5))
        st.process(xp, w_out=wbig[:, :b, 1:n + 1], v_out=vbig[:, 2:n + 2])
        _check((wbig[:, :b, 1:n + 1], vbig[:, 2:n + 2]), refs[1], tol, False, "pinned")
        # device block of stride > n, strided device outputs
        xd = torch.as_tensor(x, device="cuda")[:, 2 * n:3 * n]
        wd = torch.full((J, b + 2, n + 7), 7.0, dtype=torch.float64, device="cuda")
        vd = torch.full((b, n + 9), 7.0, dtype=torch.float64, device="cuda")
        st.process(xd, w_out=wd[:, 1:b + 1, 3:n + 3], v_out=vd[:, 4:n + 4])
        torch.cuda.synchronize()
        _check((wd[:, 1:b + 1, 3:n + 3], vd[:, 4:n + 4]), refs[2], tol, False, "device")
        assert bool((wd[:, 0] == 7.0).all()) and bool((wd[:, :, :3] == 7.0).all()) and bool((vd[:, :4] == 7.0).all())
        assert bool((vd[:, n + 4:] == 7.0).all()) and bool((wd[:, :, n + 3:] == 7.0).all())
        _check(st.process(torch.as_tensor(x[:, 3 * n:], device="cuda")), refs[3], tol, False, "device contiguous")
        _check(st.flush(9), ref_flush, tol, False, "flush")
    finally:
        st.close()


@pytest.mark.gpu
def test_two_handles_on_one_ctx_stay_independent():
    eng = vw.Engine.get()
    h, g, hs, gs = _taps("db4")
    h2, g2, hs2, gs2 = _taps("haar")
    x = np.random.default_rng(8).standard_normal((3, 1200))
    tol = 1e-12 * float(np.max(np.abs(x)))
    s1, s2 = eng.stream_create(hs, gs, 3, ZP), eng.stream_create(hs2, gs2, 5, SYM)
    o1, o2 = nptwin.StreamingOracle(h, g, 3, ZP), nptwin.StreamingOracle(h2, g2, 5, SYM)
    try:
        for k in range(4):
            a, c = x[:, k * 300:(k + 1) * 300], x[::-1, k * 300:(k + 1) * 300].copy()
            _check(s1.process(a), o1.process(a), tol, False, f"first handle, block {k}")
            _check(s2.process(c), o2.process(c), tol, False, f"second handle, block {k}")
        _check(s1.flush(7), o1.flush(7), tol, False, "first handle flush")
        _check(s2.flush(1), o2.flush(1), tol, False, "second handle flush")
    finally:
        s1.close()
        s2.close()


# ---- GPU: errors return the documented status and leave the handle usable -------------------------------------------
@pytest.mark.gpu
def test_errors_leave_the_handle_usable():
    eng = vw.Engine.get()
    lib, ctx = eng.lib, eng.ctx
    h, g, hs, gs = _taps("db4")
    dp = lambda a: a.ctypes.data_as(F._dp)   # noqa: E731
    out = C.c_void_p()
    assert lib.vw_stream_create(ctx, dp(hs), dp(gs), 8, 3, 0, C.byref(out)) == 103      # PERIODIC
    assert lib.vw_stream_create(ctx, dp(hs), dp(gs), 8, 3, 3, C.byref(out)) == 103      # CONSTANT
    assert lib.vw_stream_create(ctx, dp(hs), dp(gs), 8, 0, 1, C.byref(out)) == 104
    assert lib.vw_stream_create(ctx, dp(hs), dp(gs), 8, 31, 1, C.byref(out)) == 104
    assert lib.vw_stream_create(ctx, None, dp(gs), 8, 3, 1, C.byref(out)) == 1
    assert lib.vw_stream_create(ctx, dp(hs), dp(gs), 8, 3, 1, None) == 1
    st = eng.stream_create(hs, gs, 3, SYM)
    x = np.random.default_rng(2).standard_normal((4, 900))
    tol = 1e-12 * float(np.max(np.abs(x)))
    so = nptwin.StreamingOracle(h, g, 3, SYM)
    w, v = np.empty((3, 4, 300)), np.empty((4, 300))
    try:
        assert lib.vw_stream_flush(ctx, st.handle, 3, dp(w), 300, 1200, dp(v), 300, 0) == 301   # before any block
        _check(st.process(x[:, :300]), so.process(x[:, :300]), tol, False, "first block")
        xb = np.ascontiguousarray(x[:, 300:600])
        proc = lambda xp, b, n, ldx, wp, vp: lib.vw_stream_process(ctx, st.handle, xp, b, n, ldx, wp, n, b * n, vp, n, 0)  # noqa: E731
        assert proc(None, 4, 300, 300, dp(w), dp(v)) == 1
        assert proc(dp(xb), 4, 300, 300, None, dp(v)) == 1
        assert proc(dp(xb), 4, 300, 300, dp(w), None) == 1
        assert lib.vw_stream_process(ctx, None, dp(xb), 4, 300, 300, dp(w), 300, 1200, dp(v), 300, 0) == 1
        assert proc(dp(xb), 4, 0, 300, dp(w), dp(v)) == 6          # n < 1
        assert proc(dp(xb), 0, 300, 300, dp(w), dp(v)) == 7        # batch < 1
        assert proc(dp(xb), 4, 300, 299, dp(w), dp(v)) == 7        # ldx < n
        assert lib.vw_stream_flush(ctx, st.handle, 8, dp(w), 8, 32, dp(v), 8, 0) == 7           # tail > l - 1
        assert lib.vw_stream_flush(ctx, st.handle, 0, dp(w), 8, 32, dp(v), 8, 0) == 6
        assert lib.vw_stream_flush(ctx, st.handle, 3, None, 8, 32, dp(v), 8, 0) == 1
        bad = np.array(xb)
        bad[2, 17] = np.nan
        assert lib.vw_stream_process(ctx, st.handle, dp(bad), 4, 300, 300, dp(w), 300, 1200, dp(v), 300, F.FLAG_CHECK_FINITE) == 3
        # none of the failures advanced or restarted the stream
        _check(st.process(xb), so.process(xb), tol, False, "block after the errors")
        _check(st.flush(7), so.flush(7), tol, False, "flush after the errors")
    finally:
        st.close()


@pytest.mark.gpu
def test_a_handle_of_another_device_is_refused():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    e0, e1 = vw.Engine.get(0), vw.Engine.get(1)
    h, g, hs, gs = _taps("db4")
    st = e0.stream_create(hs, gs, 2, ZP)
    x = np.ones((2, 64))
    w, v = np.empty((2, 2, 64)), np.empty((2, 64))
    try:
        rc = e1.lib.vw_stream_process(e1.ctx, st.handle, x.ctypes.data, 2, 64, 64, w.ctypes.data, 64, 128, v.ctypes.data, 64, 0)
        assert rc == 400
        assert e1.lib.vw_stream_destroy(e1.ctx, st.handle) == 400
        so = nptwin.StreamingOracle(h, g, 2, ZP)
        _check(st.process(x), so.process(x), 1e-12, False, "after the refusal")
    finally:
        st.close()


# ---- GPU: the facade on the handle, and the C++ host class -----------------------------------------------------------
@pytest.mark.gpu
def test_facade_tensor_blocks_stay_on_the_device():
    import torch
    BM = vw.BoundaryMode
    h, g, _, _ = _taps("sym8")
    x = np.random.default_rng(4).standard_normal((6, 900))
    tol = 1e-12 * float(np.max(np.abs(x)))
    so = nptwin.StreamingOracle(h, g, 3, SYM)
    with vw.BatchStreamingMODWT.Builder().wavelet(vw.get_wavelet("sym8")).boundary(BM.SYMMETRIC).levels(3).build() as st:
        for k in range(3):
            r = st.processMultiLevel(torch.as_tensor(x[:, k * 300:(k + 1) * 300], device="cuda"))
            assert r.detailPerLevel().is_cuda and r.finalApprox().is_cuda
            _check((r.detailPerLevel(), r.finalApprox()), so.process(x[:, k * 300:(k + 1) * 300]), tol, False, f"block {k}")
        f = st.flushMultiLevel(15)
        _check((f.detailPerLevel(), f.finalApprox()), so.flush(15), tol, False, "flush")


@pytest.mark.gpu
def test_cpp_host_streaming_class():
    sys.path.insert(0, ROOT)
    cref.build()
    exe = os.path.join(ROOT, "tests", "cpp", "_build", "stream_host")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    lib, ora = os.path.join(ROOT, "vectorwave_b200"), os.path.join(ROOT, "oracle", "_build")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "stream_host.cpp"), "-o", exe, "-L", lib, "-lvwmodwt", "-L", ora,
                           "-lvw_oracle", f"-Wl,-rpath,{lib}", f"-Wl,-rpath,{ora}", "-Wl,-rpath,/usr/local/cuda/lib64"])
    p = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and p.stdout.strip().endswith("ok"), p.stdout[-2000:] + p.stderr[-2000:]
