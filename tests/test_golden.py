"""Golden vectors (tests/golden/modwt_golden.npz, made by tests/golden/make_golden.py from the reference's own seeded
fixtures): the CPU oracle and its independent numpy twin must reproduce them bit for bit (drift guard, no GPU), and
the CUDA engine must match them through the C ABI to 1e-12 * max|x| per level (GPU).

The file pins each array by a SHA-256 digest of all of its values plus a stored sample of them (make_golden.py says
why); the inputs are regenerated from their seeds, and the full expected arrays are the oracle's, accepted only once
they reproduce the golden digests."""
import importlib.util
import os

import numpy as np
import pytest

from oracle import nptwin
from oracle.wavelets import filters

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLD = os.path.join(HERE, "modwt_golden.npz")
REL = 1e-12   # north_star: every coefficient within 1e-12 * max|x| per level

_spec = importlib.util.spec_from_file_location("make_golden", os.path.join(HERE, "make_golden.py"))
make_golden = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(make_golden)


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def _cases(gold):
    keys = sorted({k.split("/")[0] for k in gold.files})
    for key in keys:
        parts = key.split("_")
        name = parts[1]
        levels = int([p for p in parts if p[0] == "j" and p[1:].isdigit()][0][1:])
        m = [p for p in parts if p[0] == "m" and p[1:].isdigit()]
        mode = int(m[0][1:]) if m else 0
        yield key, name, mode, levels


def _inputs():
    return {key: x for key, _, _, _, x in make_golden.cases()}


def _check(gold, name, a):
    """`a` is the golden array `name` bit for bit: its stored sample (a readable failure), then the digest of every value"""
    a = np.ascontiguousarray(a, dtype=np.float64)
    np.testing.assert_array_equal(a.ravel()[gold[name + "/idx"]], gold[name + "/val"], err_msg=name)
    assert np.array_equal(make_golden.digest(a), gold[name + "/sha256"]), f"{name}: digest differs"


def _expected(gold, key, name, mode, levels, x):
    """the oracle's arrays of one case, each checked against the golden file"""
    arrays, thresholds = make_golden.outputs(key, name, mode, levels, x)
    for k, a in arrays.items():
        _check(gold, f"{key}/{k}", a)
    for k, t in thresholds.items():
        assert np.array_equal(np.array([t]), gold[f"{key}/{k}"]), f"{key}/{k}"
    return arrays


def test_fixture_inventory(gold):
    cases = list(_cases(gold))
    assert len(cases) >= 40
    assert {m for _, _, m, _ in cases} == {0, 1, 2}
    assert {"haar", "db4", "db8", "sym8", "coif5"} <= {n for _, n, _, _ in cases}
    assert {key for key, _, _, _ in cases} == set(_inputs())
    for key, _, _, _ in cases:
        names = {"x", "w", "v", "xr"} | ({"denoise_soft1", "denoise_soft0"} if key.startswith("swt_") else set())
        for n in names:
            assert {f"{key}/{n}/sha256", f"{key}/{n}/idx", f"{key}/{n}/val"} <= set(gold.files), f"{key}/{n}"


def test_oracle_and_numpy_twin_reproduce_the_golden_vectors_bit_for_bit(gold):
    xs = _inputs()
    for key, name, mode, levels in _cases(gold):
        h, g, wid = filters(name)
        x = xs[key]
        _check(gold, key + "/x", x)
        exp = _expected(gold, key, name, mode, levels, x)   # the C oracle, row by row
        if x.shape[1] > 512:   # the numpy twin is slow: small cases only
            continue
        for i in range(x.shape[0]):
            w, v = exp["w"][:, i, :], exp["v"][i]
            w2, v2 = nptwin.decompose(x[i], h, g, levels, mode)
            assert np.array_equal(w2, w) and np.array_equal(v2, v), key
            assert np.array_equal(nptwin.reconstruct(w, v, h, g, mode, wid), exp["xr"][i]), key


def test_periodic_golden_round_trips_where_the_table_permits(gold):
    # ModwtPeriodicRoundTripTest.java:37 (1e-9); absolute 1e-10 only for tables accurate enough (SURVEY.md D2)
    xs = _inputs()
    for key, name, mode, levels in _cases(gold):
        if mode != 0:
            continue
        x = xs[key]
        _check(gold, key + "/x", x)
        xr = _expected(gold, key, name, mode, levels, x)["xr"]
        tol = 1e-10 if name in ("haar", "db2", "db6", "db8", "coif5") else (1e-9 if name in ("db4",) else 1e-2)
        assert float(np.max(np.abs(x - xr))) <= tol, key


@pytest.mark.gpu
def test_engine_matches_golden_vectors(gold):
    import vectorwave_b200 as vw
    from vectorwave_b200.modwt import multilevel_alignment
    eng = vw.Engine.get()
    s = nptwin.S
    bms = [vw.BoundaryMode.PERIODIC, vw.BoundaryMode.ZERO_PADDING, vw.BoundaryMode.SYMMETRIC]
    xs = _inputs()
    for key, name, mode, levels in _cases(gold):
        h, g, wid = filters(name)
        x = np.ascontiguousarray(xs[key])
        _check(gold, key + "/x", x)
        exp = _expected(gold, key, name, mode, levels, x)
        tol = REL * float(np.max(np.abs(x)))
        for flags in (0, vw._native.FLAG_BITEXACT):
            w, v = eng.forward(x, h * s, g * s, levels, mode, flags)
            w = np.asarray(w).reshape(levels, x.shape[0], -1)
            v = np.asarray(v).reshape(x.shape[0], -1)
            if flags:   # separate multiply / add in Java's tap order: identical bits
                _check(gold, key + "/w", w)
                _check(gold, key + "/v", v)
            else:
                assert float(np.max(np.abs(w - exp["w"]))) <= tol, key
                assert float(np.max(np.abs(v - exp["v"]))) <= tol, key
            align, order = multilevel_alignment(vw.get_wavelet(name), bms[mode], levels)
            xr = np.asarray(eng.inverse(exp["w"], exp["v"], h * s, g * s, mode, align, order, flags=flags))
            assert float(np.max(np.abs(xr.reshape(x.shape) - exp["xr"]))) <= tol, key
        if key.startswith("swt_"):
            swt = vw.VectorWaveSwtAdapter(vw.get_wavelet(name), bms[mode])
            for soft in (True, False):
                den = np.asarray(swt.denoise(x[0], levels, -1.0, soft))
                assert float(np.max(np.abs(den - exp[f"denoise_soft{int(soft)}"]))) <= tol, key
