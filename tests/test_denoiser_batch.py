"""Batched WaveletDenoiser (vw_wavelet_denoise, WaveletDenoiser.denoise*Batch): per-(level, row) thresholds selected on
the device in the reference's arithmetic, and level-indexed thresholds applied as every synthesis path loads W."""
import math
import os
import subprocess

import numpy as np
import pytest

import vectorwave_b200 as vw
from oracle import nptwin
from oracle.wavelets import filters
from vectorwave_b200 import _native
from vectorwave_b200.denoising import ThresholdMethod as M, ThresholdType as T, WaveletDenoiser
from vectorwave_b200.modwt import multilevel_alignment
from vectorwave_b200.errors import (ErrorCode, IllegalArgumentException, InvalidArgumentException,
                                    InvalidSignalException)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
S = 1.0 / math.sqrt(2.0)
MODES = [vw.BoundaryMode.PERIODIC, vw.BoundaryMode.ZERO_PADDING, vw.BoundaryMode.SYMMETRIC]
METHODS = [M.UNIVERSAL, M.MINIMAX, M.BAYES, M.SURE]
NP_METHOD = {M.UNIVERSAL: "UNIVERSAL", M.MINIMAX: "MINIMAX", M.BAYES: "BAYES", M.SURE: "SURE"}


def noisy_rows(b, n, seed):
    """rows whose noise levels differ by orders of magnitude (1e-3 .. 1e3), on a shared smooth signal"""
    rng = np.random.default_rng(seed)
    t = np.arange(n) / max(n, 1)
    scale = 10.0 ** np.linspace(-3, 3, b)
    return np.sin(2 * np.pi * 5 * t)[None, :] * 2.0 + scale[:, None] * rng.standard_normal((b, n))


# ---- CPU: the host scalars and the validation that needs no device ---------------------------------------------------

SCALARS_SRC = r"""
#include <cstdio>
#include <cstdlib>
#include "vw_internal.cuh"
int main(int argc, char **argv) {
    for (int i = 1; i < argc; i++) {
        VwDenoiseSel a;
        const long long n = atoll(argv[i]);
        vw_denoise_scalars(n, 31, a);
        printf("%lld %a %a %a", n, a.root, a.log_n, a.minimax_c);
        for (int j = 0; j < 31; j++) printf(" %a", a.level_scale[j]);
        printf("\n");
    }
    return 0;
}
"""


def test_host_scalars_are_the_denoising_py_formulas(tmp_path):
    src = tmp_path / "scalars.cpp"
    src.write_text(SCALARS_SRC)
    exe = tmp_path / "scalars"
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"),
                           "-I", os.path.join(ROOT, "vectorwave_b200", "csrc"), "-I", "/usr/local/cuda/include",
                           str(src), "-o", str(exe)])
    ns = [1, 2, 7, 32, 33, 64, 65, 1000, 4096, 12345, 1 << 20, (1 << 22) + 2]
    out = subprocess.run([str(exe)] + [str(n) for n in ns], capture_output=True, text=True, check=True).stdout
    for line, n in zip(out.splitlines(), ns):
        f = [float.fromhex(v) for v in line.split()[1:]]
        log_n = math.log(n)
        assert f[0] == math.sqrt(2.0 * math.log(n))                 # UNIVERSAL (and the SURE cap)
        assert f[1] == log_n                                        # MINIMAX n <= 64
        assert f[2] == 0.4745 + 0.1148 * log_n                      # MINIMAX n > 64: sigma * (0.4745 + 0.1148 * log_n)
        assert f[3:] == [math.sqrt(1 << j) for j in range(1, 32)]   # level_scale = math.sqrt(1 << level)


def test_batch_methods_validate_before_touching_the_device():
    den = WaveletDenoiser(vw.Daubechies.DB4, vw.BoundaryMode.PERIODIC)
    x = np.ones((3, 256))
    with pytest.raises(InvalidArgumentException) as e:
        den.denoiseBatch(x, M.FIXED)
    assert e.value.getErrorCode() == ErrorCode.CFG_UNSUPPORTED_OPERATION
    with pytest.raises(InvalidArgumentException) as e:
        den.denoiseMultiLevelBatch(x, 2, M.FIXED, T.SOFT)
    assert e.value.getErrorCode() == ErrorCode.CFG_UNSUPPORTED_OPERATION
    with pytest.raises(InvalidArgumentException) as e:
        den.denoiseMultiLevelBatch(x, 7, M.UNIVERSAL, T.SOFT)       # max 6 for db4 at n = 256
    assert e.value.getErrorCode() == ErrorCode.CFG_INVALID_DECOMPOSITION_LEVEL
    with pytest.raises(InvalidSignalException) as e:
        den.denoiseMultiLevelBatch(np.ones((3, 0)), 1, M.UNIVERSAL, T.SOFT)
    assert e.value.getErrorCode() == ErrorCode.VAL_EMPTY
    with pytest.raises(InvalidSignalException) as e:
        den.denoiseBatch(np.ones((3, 0)), M.UNIVERSAL)
    assert e.value.getErrorCode() == ErrorCode.VAL_EMPTY
    with pytest.raises(IllegalArgumentException):
        den.denoiseBatch(np.ones(256), M.UNIVERSAL)


# ---- GPU -------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def eng():
    e = vw.Engine.get()
    yield e
    e.set_option("lattice", 15)


def host_thresholds(eng, den, w, n, levels, method, multilevel):
    """denoising.py's selectors, per (level, row), on the engine's own coefficients and statistics"""
    b = w.shape[1]
    thr = np.empty((levels, b))
    for r in range(b):
        sigma = den._sigma(eng, np.ascontiguousarray(w[0, r]))
        for j in range(1, levels + 1):
            s = sigma / math.sqrt(1 << j) if multilevel else sigma
            thr[j - 1, r] = den._threshold(eng, np.ascontiguousarray(w[j - 1, r]), n, s, method)
    return thr


@pytest.mark.gpu
@pytest.mark.parametrize("soft", [True, False], ids=["soft", "hard"])
@pytest.mark.parametrize("method", METHODS, ids=[m.value for m in METHODS])
@pytest.mark.parametrize("mode", MODES, ids=[m.name for m in MODES])
def test_multilevel_thresholds_exact_and_rows_match_the_single_signal_path(eng, mode, method, soft):
    levels, n = 4, 1000
    x = noisy_rows(5, n, seed=7)
    den = WaveletDenoiser(vw.Daubechies.DB4, mode)
    typ = T.SOFT if soft else T.HARD
    out = den.denoiseMultiLevelBatch(x, levels, method, typ)
    t = vw.MultiLevelMODWTTransform(vw.Daubechies.DB4, mode)
    w, _ = eng.forward(x, t._hs, t._gs, levels, mode.value)
    ref = host_thresholds(eng, den, np.asarray(w), n, levels, method, True)
    assert np.array_equal(den.lastThresholds, ref.T), (den.lastThresholds, ref.T)
    assert den.lastThresholds.shape == (5, levels)
    h, g, wid = filters("db4")
    for r in range(5):
        one = WaveletDenoiser(vw.Daubechies.DB4, mode)
        single = one.denoiseMultiLevel(x[r], levels, method, typ)
        tol = 1e-12 * float(np.max(np.abs(x[r])))
        assert one.lastThresholds == list(den.lastThresholds[r])
        assert np.max(np.abs(out[r] - single)) <= tol
        wn, vn = nptwin.decompose(x[r], h, g, levels, mode.value)
        wd = np.stack([nptwin.threshold(np.asarray(w)[j, r], ref[j, r], soft) for j in range(levels)])
        assert np.max(np.abs(out[r] - nptwin.reconstruct(wd, vn, h, g, mode.value, wid))) <= tol


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 5, 32, 33, 64, 65, 1000])
@pytest.mark.parametrize("mode", MODES, ids=[m.name for m in MODES])
def test_single_level_thresholds_exact_including_short_rows(eng, mode, n):
    x = noisy_rows(4, n, seed=n)
    den = WaveletDenoiser(vw.Daubechies.DB4, mode)
    t = vw.MODWTTransform(vw.Daubechies.DB4, mode)
    w, _ = eng.forward(x, t._hs, t._gs, 1, mode.value)
    for method in METHODS:
        out, thr = eng.wavelet_denoise(x, t._hs, t._gs, 1, mode.value, den._single_align(), _native.ORDER_PAIR, False,
                                       _native.__dict__["THR_" + method.value], 0.0, True)
        assert np.array_equal(thr, host_thresholds(eng, den, np.asarray(w), n, 1, method, False)), method
        batch = den.denoiseBatch(x, method, T.SOFT)
        for r in range(4):
            tol = 1e-12 * float(np.max(np.abs(x[r])))
            assert np.max(np.abs(batch[r] - den.denoise(x[r], method, T.SOFT))) <= tol, (method, r)
    fixed = den.denoiseFixedBatch(x, 0.25, T.HARD)
    for r in range(4):
        assert np.max(np.abs(fixed[r] - den.denoiseFixed(x[r], 0.25, T.HARD))) <= 1e-12 * float(np.max(np.abs(x[r])))


# the shapes of tests/test_synthesis_paths.py: (id, wavelet, n, J, "lattice" option, flags)
CASES = [
    ("db4-4096-J4-lean-tile", "db4", 4096, 4, 15, 0),
    ("haar-20000-J9-tile-column", "haar", 20000, 9, 15, 0),
    ("sym8-40000-J8-dirpairs", "sym8", 40000, 8, 15, 0),
    ("sym8-40000-J8-dirsingles", "sym8", 40000, 8, 11, 0),
    ("db10-40000-J8-dirpairs", "db10", 40000, 8, 15, 0),
    ("coif3-40000-J8-dirsingles", "coif3", 40000, 8, 11, 0),
    ("coif5-65536-J8-latpairs", "coif5", 65536, 8, 15, 0),
    ("coif5-65536-J8-latsingles", "coif5", 65536, 8, 1, 0),
    ("coif5-65536-J8-direct", "coif5", 65536, 8, 0, 0),
    ("db6-9000-J7-colsingle", "db6", 9000, 7, 15, 0),
    ("db4-12345-J4-oddn", "db4", 12345, 4, 15, 0),
    ("db4-4096-J4-nofuse-generic", "db4", 4096, 4, 15, _native.FLAG_NO_FUSE),
]


@pytest.mark.gpu
@pytest.mark.parametrize("method", [_native.THR_UNIVERSAL, _native.THR_MINIMAX], ids=["UNIVERSAL", "MINIMAX"])
@pytest.mark.parametrize("mode", [0, 1], ids=["PERIODIC", "ZERO_PADDING"])
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_every_synthesis_path_thresholds_by_level(eng, case, mode, method):
    cid, name, n, levels, lattice, flags = case
    h, g, wid = filters(name)
    hs, gs = h * S, g * S
    order = _native.ORDER_SPLIT if mode == 0 else _native.ORDER_PAIR
    x = noisy_rows(3, n, seed=levels)
    eng.set_option("lattice", lattice)
    try:
        eng.denoise(x, hs, gs, levels, mode, None, order, -1.0, True, flags)
        eng.wavelet_denoise(x, hs, gs, levels, mode, None, order, True, method, 0.0, True, flags)
        l0 = eng.launch_count()
        eng.denoise(x, hs, gs, levels, mode, None, order, -1.0, True, flags)
        swt = eng.launch_count() - l0
        l0 = eng.launch_count()
        out, thr = eng.wavelet_denoise(x, hs, gs, levels, mode, None, order, True, method, 0.0, True, flags)
        ours = eng.launch_count() - l0
        w, v = eng.forward(x, hs, gs, levels, mode, flags)
    finally:
        eng.set_option("lattice", 15)
    # no extra thresholding pass: the level-indexed table rides on the same stages as vw_swt_denoise's single table
    assert ours <= swt + 1, (cid, ours, swt)
    assert len(set(thr[:, 0])) == levels                       # every level has its own threshold
    w, v = np.asarray(w), np.asarray(v)
    for r in range(3):
        wd = np.stack([nptwin.threshold(w[j, r], thr[j, r], True) for j in range(levels)])
        ref = nptwin.reconstruct(wd, v[r], h, g, mode, wid)
        err = float(np.max(np.abs(out[r] - ref)))
        assert err <= 1e-12 * float(np.max(np.abs(x[r]))), (cid, r, err)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=[m.name for m in MODES])
def test_bitexact_flag_matches_the_numpy_pipeline_bit_for_bit(eng, mode):
    h, g, wid = filters("db4")
    x = noisy_rows(4, 777, seed=3)
    ml = vw.MultiLevelMODWTTransform(vw.Daubechies.DB4, mode)
    den = WaveletDenoiser(vw.Daubechies.DB4, mode)
    align, order = multilevel_alignment(vw.Daubechies.DB4, mode, 3)
    for method in (M.UNIVERSAL, M.MINIMAX):
        out, thr = eng.wavelet_denoise(x, ml._hs, ml._gs, 3, mode.value, align, order, True,
                                       _native.__dict__["THR_" + method.value], 0.0, True, _native.FLAG_BITEXACT)
        for r in range(4):
            ref, rthr = nptwin.denoiser_multilevel(x[r], h, g, 3, mode.value, wid, NP_METHOD[method], True)
            assert list(thr[:, r]) == rthr, method
            assert np.array_equal(out[r], ref), method
    out, _ = eng.wavelet_denoise(x, ml._hs, ml._gs, 1, mode.value, den._single_align(), _native.ORDER_PAIR, False,
                                 _native.THR_FIXED, 0.3, False, _native.FLAG_BITEXACT)
    for r in range(4):
        ref, _ = nptwin.denoiser_single(x[r], h, g, mode.value, "FIXED", False, fixed=0.3)
        assert np.array_equal(out[r], ref)


@pytest.mark.gpu
def test_residency_and_row_strides(eng):
    import torch
    x = noisy_rows(6, 4096, seed=11)
    den = WaveletDenoiser(vw.Daubechies.DB4, vw.BoundaryMode.PERIODIC)
    ref = den.denoiseMultiLevelBatch(x, 4, M.BAYES, T.SOFT)
    assert isinstance(ref, np.ndarray) and ref.shape == x.shape
    host_thr = den.lastThresholds.copy()
    for pad in (0, 7, 64):
        buf = torch.zeros((6, 4096 + pad), dtype=torch.float64, device="cuda")
        view = buf[:, :4096]
        view.copy_(torch.as_tensor(x))
        out = den.denoiseMultiLevelBatch(view, 4, M.BAYES, T.SOFT)
        assert torch.is_tensor(out) and out.is_cuda
        assert np.max(np.abs(out.cpu().numpy() - ref)) <= 1e-12 * float(np.max(np.abs(x)))
        assert np.array_equal(den.lastThresholds, host_thr)
        one = den.denoiseBatch(view, M.UNIVERSAL)
        assert torch.is_tensor(one) and one.is_cuda
        t = vw.MODWTTransform(vw.Daubechies.DB4, vw.BoundaryMode.PERIODIC)
        _, thr = eng.wavelet_denoise(view, t._hs, t._gs, 1, 0, None, _native.ORDER_PAIR, False, _native.THR_UNIVERSAL)
        assert torch.is_tensor(thr) and thr.is_cuda and tuple(thr.shape) == (1, 6)


def _code(excinfo):
    return type(excinfo.value), excinfo.value.getErrorCode()


@pytest.mark.gpu
def test_errors_match_the_single_signal_path(eng):
    den = WaveletDenoiser(vw.Daubechies.DB4, vw.BoundaryMode.PERIODIC)
    x = noisy_rows(4, 512, seed=5)
    x[2, 100] = np.nan
    with pytest.raises(InvalidSignalException) as eb:
        den.denoiseMultiLevelBatch(x, 3, M.UNIVERSAL, T.SOFT)
    with pytest.raises(InvalidSignalException) as es:
        den.denoiseMultiLevel(x[2], 3, M.UNIVERSAL, T.SOFT)
    assert _code(eb) == _code(es) and eb.value.getErrorCode() == ErrorCode.VAL_NON_FINITE_VALUES
    with pytest.raises(InvalidSignalException) as eb:
        den.denoiseBatch(x, M.BAYES)
    with pytest.raises(InvalidSignalException) as es:
        den.denoise(x[2], M.BAYES)
    assert _code(eb) == _code(es)
    x[2, 100] = 0.0
    for call_b, call_s in ((lambda: den.denoiseMultiLevelBatch(x, 9, M.UNIVERSAL, T.SOFT),
                            lambda: den.denoiseMultiLevel(x[0], 9, M.UNIVERSAL, T.SOFT)),
                           (lambda: den.denoiseMultiLevelBatch(x, 2, M.FIXED, T.SOFT),
                            lambda: den.denoiseMultiLevel(x[0], 2, M.FIXED, T.SOFT)),
                           (lambda: den.denoiseBatch(x, M.FIXED), lambda: den.denoise(x[0], M.FIXED)),
                           (lambda: den.denoiseMultiLevelBatch(np.ones((2, 0)), 1, M.SURE, T.SOFT),
                            lambda: den.denoiseMultiLevel(np.ones(0), 1, M.SURE, T.SOFT))):
        with pytest.raises(Exception) as eb:
            call_b()
        with pytest.raises(Exception) as es:
            call_s()
        assert _code(eb) == _code(es)
    # SURE scores n candidates against n coefficients: refused beyond levels * batch * n^2 = 2^44
    big = np.random.default_rng(1).standard_normal((4, 1 << 21))
    with pytest.raises(InvalidArgumentException) as eb:
        den.denoiseMultiLevelBatch(big, 2, M.SURE, T.SOFT)
    with pytest.raises(InvalidArgumentException) as es:
        den.denoise(np.random.default_rng(2).standard_normal((1 << 22) + 2), M.SURE)
    assert _code(eb) == _code(es) and eb.value.getErrorCode() == ErrorCode.CFG_UNSUPPORTED_OPERATION
    # the engine itself: the scaling cap, and single level takes levels = 1
    t = vw.MODWTTransform(vw.Haar(), vw.BoundaryMode.PERIODIC)
    with pytest.raises(InvalidArgumentException) as e:
        eng.wavelet_denoise(np.ones((1, 1 << 12)), t._hs, t._gs, 32, 0, None, _native.ORDER_SPLIT, True,
                            _native.THR_UNIVERSAL)
    assert e.value.getErrorCode() == ErrorCode.VAL_TOO_LARGE
    with pytest.raises(IllegalArgumentException):
        eng.wavelet_denoise(np.ones((1, 4096)), t._hs, t._gs, 2, 0, None, _native.ORDER_SPLIT, False,
                            _native.THR_UNIVERSAL)
