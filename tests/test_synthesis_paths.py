"""Partial reconstruction and caller strides on every synthesis path, against an extended-precision reference.

Reference.  A `np.longdouble` (64-bit significand) restatement of the synthesis cascade of `oracle/nptwin.synth_level`,
with the same double taps hs = h*S, gs = g*S the engine gets, the index rules of PERIODIC, ZERO_PADDING and SYMMETRIC,
the SYMMETRIC (sigma, tau) table `multilevel_alignment` hands the engine, and `detail_mask` / `use_approx` handled as in
`nptwin.reconstruct`.  An analysis cascade built the same way serves the stride tests.

Bound.  A running-error bound per output sample, u = 2^-53, gamma_m = m*u / (1 - m*u), L taps:
    A_J = |V_J| [use_approx],   A_{j-1} = |H| * A_j + |G| * (|W_j| mask_j)
    E_J = 0,                    E_{j-1} = (1 + gamma_2L) |H| * E_j + gamma_2L A_{j-1}
(`*` is the level's own index rule evaluated with |taps|).  A level sums 2L products of computed inputs; whatever the
order (FMA chains, separate multiply and add, ORDER_SPLIT or ORDER_PAIR), each product meets at most 2L roundings, so the
sum is off by <= gamma_2L times the sum of |products| <= gamma_2L (A_{j-1} + |H| * E_j).  E is evaluated in longdouble,
rounded up by (1 + 8u), and a check is |x_hat - x_ref| <= E_0 + 2^-60 |x_ref|.  Every term is linear in the inputs, so
the reference and the bound of a mask are sums of per-level components, which the GPU tests compute once per case.

Lattice levels.  The coif5 column kernels in lattice form compute with the rotation coefficients vw_lattice_query
returns, not with the taps.  Their taps are off from hs, gs by at most tap_err (which this file recomputes in
longdouble and takes the larger of), and each output passes through K - 1 rotation stages, the 2 x 2 base matrix and one
final add: at most 2K + 4 roundings on any path even without FMA, each relative to the |.|-evaluation of the lattice.
That evaluation is <= c_lat times the unit-tap sum U_{j-1} = 1 * (A_j + E_j) + 1 * |W_j|, with c_lat the largest output
of the |t_k|, |b| lattice on a unit impulse.  So a coif5 level adds kappa U_{j-1}, kappa = tap_err + gamma_{2K+4} c_lat,
to its E (for every level, so the bound holds whichever form ran).  `test_lattice_term_bounds_the_numpy_lattice_model`
checks the term on the numpy model of `tests/test_lattice.py`.  It is looser than the direct-form bound: kappa U is
about 31x gamma_2L A of a coif5 level (median over samples of mixed-scale inputs; kappa = 5.5e-15 against
gamma_60 = 6.7e-15, and U is about 38x A).  It is needed all the same: on those inputs the lattice model's error reaches
4x gamma_2L A, and 2% of kappa U.
"""
import fractions
import functools

import numpy as np
import pytest

import vectorwave_b200 as vw
from oracle import cref, nptwin
from oracle.wavelets import TABLES, filters
from vectorwave_b200 import _native
from vectorwave_b200.modwt import multilevel_alignment

from test_lattice import _analysis_rows, _expand, _synthesis_rows

LD = np.longdouble
assert np.finfo(LD).nmant >= 63, "the reference needs an extended longdouble (64-bit significand)"
U = 2.0 ** -53
S = nptwin.S
BMODE = [vw.BoundaryMode.PERIODIC, vw.BoundaryMode.ZERO_PADDING, vw.BoundaryMode.SYMMETRIC]
MODE_ID = ["per", "zero", "sym"]
PLAIN = (1, 0, 1, 0)


def gamma(m, u=U):
    return LD(m) * LD(u) / (LD(1) - LD(m) * LD(u))


def taps(name):
    h, g, _ = filters(name)
    return h * S, g * S


def alignment(name, mode, levels):
    """per-level (sigma_h, tau_h, sigma_g, tau_g) and summation order, exactly as the engine is given them"""
    table, order = multilevel_alignment(vw.get_wavelet(name), BMODE[mode], levels)
    return (list(table) if table is not None else [PLAIN] * levels), order


# ---- the longdouble cascades --------------------------------------------------------------------------------------------

@functools.lru_cache(maxsize=4096)
def _index(n, d, k, sigma, tau, mode, shift):
    t = np.arange(n)
    idx = (t + k * d - tau if sigma > 0 else t - k * d + tau) + shift
    if mode == 0:
        return np.mod(idx, n), None
    if mode == 2:
        return nptwin.mirror(idx, n), None
    valid = (idx >= 0) & (idx < n)
    return np.clip(idx, 0, n - 1), valid


def _stage(n, a, dj, fh, fg, level, mode, al, dtype=LD, shift=0):
    """one synthesis level: out[t] = sum_k fh[k] a[ix_h(t, k)] + fg[k] dj[ix_g(t, k)]; None stands for zeros"""
    d = 1 << (level - 1)
    acc = np.zeros(n, dtype)
    for src, f, sig, tau in ((a, fh, al[0], al[1]), (dj, fg, al[2], al[3])):
        if src is None:
            continue
        for k in range(len(f)):
            idx, valid = _index(n, d, k, int(sig), int(tau), mode, shift)
            term = f[k] * src[idx]
            acc += term if valid is None else np.where(valid, term, dtype(0))
    return acc


def synth_ld(w, v, hs, gs, mode, align, detail_mask, use_approx, dtype=LD, shift_level=0):
    """the synthesis cascade of nptwin.reconstruct in `dtype` (default longdouble); w [J][n], v [n]"""
    levels, n = w.shape
    fh, fg = np.asarray(hs).astype(dtype), np.asarray(gs).astype(dtype)
    cur = np.asarray(v).astype(dtype) if use_approx else None
    for level in range(levels, 0, -1):
        dj = np.asarray(w[level - 1]).astype(dtype) if (detail_mask >> (level - 1)) & 1 else None
        if cur is None and dj is None:
            continue
        cur = _stage(n, cur, dj, fh, fg, level, mode, align[level - 1], dtype, 1 if level == shift_level else 0)
    return cur if cur is not None else np.zeros(n, dtype)


def synth_bound(w, v, hs, gs, mode, align, detail_mask, use_approx, kappa=0.0, u=U):
    """E_0 of the running-error bound (module docstring), rounded up"""
    levels, n = w.shape
    ah, ag = np.abs(hs).astype(LD), np.abs(gs).astype(LD)
    one = np.ones(len(hs), LD)
    g2 = gamma(2 * len(hs), u)
    a = np.abs(v).astype(LD) if use_approx else None
    e = None
    for level in range(levels, 0, -1):
        al = align[level - 1]
        dj = np.abs(w[level - 1]).astype(LD) if (detail_mask >> (level - 1)) & 1 else None
        if a is None and dj is None:
            continue
        a_new = _stage(n, a, dj, ah, ag, level, mode, al)
        e_new = g2 * a_new
        if e is not None:
            e_new += (1 + g2) * _stage(n, e, None, ah, ag, level, mode, al)
        if kappa:
            ae = a if e is None else a + e
            e_new += LD(kappa) * _stage(n, ae, dj, one, one, level, mode, al)
        a, e = a_new, e_new
    return e * LD(1 + 8 * u) if e is not None else np.zeros(n, LD)


def _conv(n, x, f, d, mode):
    """analysis: out[t] = sum_k f[k] x[ext(t - k d)] (nptwin.conv)"""
    return _stage(n, x, None, f, f, d.bit_length(), mode, (-1, 0, -1, 0))


def analysis_ld(x, hs, gs, levels, mode, kappa=0.0):
    """(W [J][n], V_J, E_W [J][n], E_V): the analysis cascade in longdouble and its running-error bound (L-term sums)"""
    n = x.shape[-1]
    fh, fg = np.asarray(hs).astype(LD), np.asarray(gs).astype(LD)
    ah, ag, one = np.abs(fh), np.abs(fg), np.ones(len(hs), LD)
    gl = gamma(len(hs))
    cur, a, e = np.asarray(x).astype(LD), np.abs(x).astype(LD), np.zeros(n, LD)
    ws, ews = [], []
    for level in range(1, levels + 1):
        d = 1 << (level - 1)
        ws.append(_conv(n, cur, fg, d, mode))
        cur = _conv(n, cur, fh, d, mode)
        ew = (1 + gl) * _conv(n, e, ag, d, mode) + gl * _conv(n, a, ag, d, mode)
        a_new = _conv(n, a, ah, d, mode)
        ev = (1 + gl) * _conv(n, e, ah, d, mode) + gl * a_new
        if kappa:
            unit = LD(kappa) * _conv(n, a + e, one, d, mode)
            ew, ev = ew + unit, ev + unit
        ews.append(ew * LD(1 + 8 * U))
        a, e = a_new, ev * LD(1 + 8 * U)
    return np.stack(ws), cur, np.stack(ews), e


def within(out, ref, bound):
    """(ok, worst |err| / limit, where): |out - ref| <= bound + 2^-60 |ref| on every sample"""
    err = np.abs(np.asarray(out, dtype=np.float64).astype(LD) - ref)
    lim = bound + LD(2.0 ** -60) * np.abs(ref)
    ratio = np.where(lim > 0, err / np.where(lim > 0, lim, 1), np.where(err > 0, np.inf, 0))
    i = int(np.argmax(ratio))
    return bool(np.all(err <= lim)), float(ratio[i]), i


# ---- the lattice term -----------------------------------------------------------------------------------------------------

def _abs_synthesis_rows(v, w, coef):
    """_synthesis_rows of tests/test_lattice.py evaluated with |coefficients| and every subtraction turned into an
    addition: bounds the magnitude of every intermediate of the lattice synthesis on inputs |v|, |w|"""
    k = coef.size - 3
    t, b = np.abs(coef[:k - 1]), np.abs(coef[k - 1:])
    n, l = v.size, 2 * k
    out = np.zeros(n)
    dl = np.zeros((k - 1, 2))
    y0prev = 0.0
    for m in range(n + l - 1):
        aa, bb = abs(v[m % n]), abs(w[m % n])
        for s in range(k - 2, -1, -1):
            an, bb = aa + t[s] * bb, bb + t[s] * aa
            aa = dl[s, m & 1]
            dl[s, m & 1] = an
        y0 = b[0] * aa + b[2] * bb
        y1 = b[1] * aa + b[3] * bb
        if m - (l - 1) >= 0:
            out[m - (l - 1)] = y0prev + y1
        y0prev = y0
    return out


def _abs_analysis_rows(u, coef):
    """_analysis_rows of tests/test_lattice.py with |coefficients| and additions only"""
    k = coef.size - 3
    t, b = np.abs(coef[:k - 1]), np.abs(coef[k - 1:])
    n = u.size
    v, w = np.zeros(n), np.zeros(n)
    dl = np.zeros((k - 1, 2))
    uprev = 0.0
    for q in range(-30, n):
        x = abs(u[q % n])
        aa = b[0] * x + b[1] * uprev
        bb = b[2] * x + b[3] * uprev
        uprev = x
        for s in range(k - 1):
            bd = dl[s, q & 1]
            dl[s, q & 1] = bb
            aa, bb = aa + t[s] * bd, bd + t[s] * aa
        if q >= 0:
            v[q], w[q] = aa, bb
    return v, w


@functools.lru_cache(maxsize=None)
def lattice_kappa(name, forward=False):
    """kappa of the module docstring for the pair the lattice column kernels would use (0 when the pair keeps the
    direct form): tap_err + gamma_{2K+4} c_lat"""
    hs, gs = taps(name)
    if hs.size < 24:                       # the lattice form exists for long pairs only (vw_lattice_query rejects short ones)
        return 0.0
    coef, tap_err = _native.lattice_query(hs, gs)
    if coef is None:
        return 0.0
    k = coef.size - 3
    hh, gg = _expand(coef)
    tap = max(float(tap_err), float(np.max(np.abs(hh - hs.astype(LD)))), float(np.max(np.abs(gg - gs.astype(LD)))))
    n = 4 * coef.size
    imp = np.zeros(n)
    imp[0] = 1.0
    if forward:
        c_lat = max(float(np.max(r)) for r in _abs_analysis_rows(imp, coef))
    else:
        c_lat = max(float(np.max(_abs_synthesis_rows(imp, 0 * imp, coef))), float(np.max(_abs_synthesis_rows(0 * imp, imp, coef))))
    return float(LD(tap) + gamma(2 * k + 4) * LD(c_lat)) * (1 + 8 * U)


# ---- test data ------------------------------------------------------------------------------------------------------------

def coefficients(levels, n, batch=2, seed=0, spike_row=None):
    """independent W_j, V_J: every level and every row at its own scale 10^s, s in -6..6; a 1e12 spike in W_1 of one row"""
    rng = np.random.default_rng(seed)
    s = rng.integers(-6, 7, size=(batch, levels + 1))
    w = rng.standard_normal((levels, batch, n)) * (10.0 ** s[:, :levels].T)[:, :, None]
    v = rng.standard_normal((batch, n)) * (10.0 ** s[:, levels])[:, None]
    if spike_row is not None:
        w[0, spike_row, n // 3] = 1e12
    return w, v


# ---- CPU: the reference and the bound ---------------------------------------------------------------------------------

def test_alignment_table_given_to_the_engine_matches_the_oracle_rule():
    for name in TABLES:
        h, _, wid = filters(name)
        table, _ = alignment(name, 2, 9)
        for level in range(1, 10):
            ap, dh, dp, dg = nptwin.alignment(wid, h.size, level)
            tau = nptwin.tau_j(h.size, level)
            assert table[level - 1] == (1 if ap else -1, tau + dh, 1 if dp else -1, tau + dg), (name, level)


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("name", ["haar", "db4", "sym8", "coif5"])
def test_float64_oracle_passes_the_bound_for_every_kind_of_mask(name, mode):
    h, g, wid = filters(name)
    hs, gs = h * S, g * S
    levels, n = 4, 700
    align, _ = alignment(name, mode, levels)
    w, v = coefficients(levels, n, 1, seed=len(name) + mode, spike_row=0)
    w, v = w[:, 0], v[0]
    kappa = lattice_kappa(name)
    for mask in (0b1111, 0b0001, 0b1000, 0b0110, 0b0101, 0b1010, 0):
        for approx in (True, False):
            out = cref.reconstruct(w, v, h, g, mode, wid, detail_mask=mask, use_approx=approx)
            ref = synth_ld(w, v, hs, gs, mode, align, mask, approx)
            ok, r, i = within(out, ref, synth_bound(w, v, hs, gs, mode, align, mask, approx, kappa))
            assert ok, (mask, approx, r, i)


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_longdouble_reference_agrees_with_exact_fraction_sums(mode):
    """the whole cascade in Fractions on a short signal; the longdouble reference must sit inside the same bound
    evaluated with the longdouble unit roundoff 2^-64"""
    name, levels, n = "db2", 3, 40
    hs, gs = taps(name)
    align, _ = alignment(name, mode, levels)
    w, v = coefficients(levels, n, 1, seed=3 + mode)
    w, v = w[:, 0], v[0]
    F = fractions.Fraction
    fh, fg = [F(x) for x in hs], [F(x) for x in gs]
    for mask, approx in ((0b111, True), (0b010, False), (0b101, True)):
        cur = [F(x) for x in v] if approx else [F(0)] * n
        for level in range(levels, 0, -1):
            d = 1 << (level - 1)
            dj = [F(x) for x in w[level - 1]] if (mask >> (level - 1)) & 1 else [F(0)] * n
            nxt = []
            for t in range(n):
                acc = F(0)
                for src, f, sig, tau in ((cur, fh, align[level - 1][0], align[level - 1][1]),
                                         (dj, fg, align[level - 1][2], align[level - 1][3])):
                    for k in range(len(f)):
                        idx, valid = _index(n, d, k, sig, tau, mode, 0)
                        if valid is None or valid[t]:
                            acc += f[k] * src[int(idx[t])]
                nxt.append(acc)
            cur = nxt
        ref = synth_ld(w, v, hs, gs, mode, align, mask, approx)
        bnd = synth_bound(w, v, hs, gs, mode, align, mask, approx, u=2.0 ** -64)
        for t in (0, 1, n // 2, n - 2, n - 1):
            err = abs(F(*ref[t].as_integer_ratio()) - cur[t])
            assert err <= F(*bnd[t].as_integer_ratio()) + F(1, 1 << 80), (mask, approx, t)


def _leak_case(mode):
    """db4, J = 4: W_2 alone extracted (use_approx = 0) while the masked-out W_1 makes max|x| about 1e8 and V is ~1e-7"""
    name, levels, n = "db4", 4, 512
    h, g, wid = filters(name)
    hs, gs = h * S, g * S
    rng = np.random.default_rng(40 + mode)
    w = rng.standard_normal((levels, n)) * np.array([1e8, 1.0, 1e2, 1e-2])[:, None]
    v = rng.standard_normal(n) * 1e-7
    mask = 0b0010
    align, _ = alignment(name, mode, levels)
    xmax = float(np.max(np.abs(cref.reconstruct(w, v, h, g, mode, wid))))
    good = cref.reconstruct(w, v, h, g, mode, wid, detail_mask=mask, use_approx=False)
    ref = synth_ld(w, v, hs, gs, mode, align, mask, False)
    bnd = synth_bound(w, v, hs, gs, mode, align, mask, False)
    return name, h, g, wid, w, v, mask, align, xmax, good, ref, bnd


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_broken_variants_fail_the_bound_where_the_old_tolerance_passes_them(mode):
    name, h, g, wid, w, v, mask, align, xmax, good, ref, bnd = _leak_case(mode)
    hs, gs = h * S, g * S
    assert within(good, ref, bnd)[0]
    old_tol = 1e-12 * xmax
    out_max = float(np.max(np.abs(good)))
    assert out_max < 1e-6 * xmax                                   # a small band next to a large signal
    leak_w1 = synth_ld(w, v, hs, gs, mode, align, 0b0001, False).astype(np.float64)
    h2 = h.copy()
    h2[int(np.argmax(np.abs(h2)))] *= 1 + 1e-13
    variants = {
        "masked-out W_1 leaked at 1e-6 of the output": good + 1e-6 * out_max * leak_w1 / float(np.max(np.abs(leak_w1))),
        "V leaked with use_approx = 0": good + synth_ld(w, v, hs, gs, mode, align, 0, True).astype(np.float64),
        "one tap perturbed by 1e-13 relative": cref.reconstruct(w, v, h2, g, mode, wid, detail_mask=mask, use_approx=False),
    }
    for what, bad in variants.items():
        assert not within(bad, ref, bnd)[0], what
        assert float(np.max(np.abs(bad - good))) <= old_tol, what    # ... which 1e-12 * max|x| does not see
    shifted = synth_ld(w, v, hs, gs, mode, align, mask, False, dtype=np.float64, shift_level=1)
    assert not within(shifted, ref, bnd)[0]
    assert float(np.max(np.abs(shifted - good))) > old_tol


def test_lattice_term_bounds_the_numpy_lattice_model():
    """the float64 lattice recurrences of tests/test_lattice.py on one periodic level, at mixed scales: inside
    kappa U alone (synthesis) and inside the analysis bound (both forms' terms)"""
    hs, gs = taps("coif5")
    coef, _ = _native.lattice_query(hs, gs)
    assert coef is not None
    kappa = lattice_kappa("coif5")
    n = 1024
    rng = np.random.default_rng(9)
    scale = 10.0 ** rng.integers(-6, 7, size=n)
    v, w = rng.standard_normal(n) * scale, rng.standard_normal(n) * scale[::-1]
    ref = _stage(n, v.astype(LD), w.astype(LD), hs.astype(LD), gs.astype(LD), 1, 0, PLAIN)
    unit = _stage(n, np.abs(v).astype(LD), np.abs(w).astype(LD), np.ones(30, LD), np.ones(30, LD), 1, 0, PLAIN)
    direct = gamma(60) * _stage(n, np.abs(v).astype(LD), np.abs(w).astype(LD), np.abs(hs).astype(LD), np.abs(gs).astype(LD), 1, 0, PLAIN)
    out = _synthesis_rows(v, w, coef)
    assert within(out, ref, LD(kappa) * unit)[0]
    assert not within(out, ref, direct)[0]              # the direct-form term alone does not cover the lattice
    ratio = float(np.median(LD(kappa) * unit / direct))
    assert 20 < ratio < 45, ratio                       # the docstring's "about 31x"
    x = rng.standard_normal(n) * scale
    wr, vr, ew, ev = analysis_ld(x, hs, gs, 1, 0, lattice_kappa("coif5", True))
    va, wa = _analysis_rows(x, coef)
    assert within(va, vr, ev)[0] and within(wa, wr[0], ew[0])[0]
    # and the model is really off the direct sums by more than the longdouble reference is
    assert float(np.max(np.abs(out.astype(LD) - ref))) > 0


# ---- GPU: every synthesis path, with masks --------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def eng():
    e = vw.Engine.get()
    yield e
    e.set_option("lattice", 15)


def _plan(l, levels, n):
    """[(first, nlev, kind)] of the default synthesis plan; kind is 'fused', 'column' or 'per-level'"""
    out = []
    for line in _native.describe_plan(False, l, levels, n).splitlines():
        lv, rest = line.split(": ", 1)
        a, b = (int(x) for x in lv.split()[1].split("-"))
        out.append((a, b - a + 1, rest.split()[0]))
    return out


def _plan_text(plan):
    return " | ".join(f"L{a}-{a + k - 1} {kind}" for a, k, kind in plan)


def _masks(levels, plan, extra=()):
    full = (1 << levels) - 1
    half = levels // 2
    ms = {0, full, (1 << half) - 1, full & ~((1 << half) - 1), 0b11, full & ~(full >> 2),
          0x5555555555 & full, 0xAAAAAAAAAA & full}
    ms |= {1 << j for j in range(levels)}
    for a, k, _ in plan:                   # every mask that splits a planned group: a proper subset of its levels
        if k >= 2:
            grp = ((1 << k) - 1) << (a - 1)
            for sub in range(1, (1 << k) - 1):
                ms.add((full & ~grp) | (sub << (a - 1)))
    ms |= set(extra)
    return sorted(ms)


_REF_CACHE = {}


class Reference:
    """per-component longdouble reference and bound of one row; a mask's are sums of components"""

    def __init__(self, name, mode, w, v, lattice_term=True):
        self.name, self.mode, self.w, self.v = name, mode, w, v
        self.hs, self.gs = taps(name)
        self.align, self.order = alignment(name, mode, w.shape[0])
        self.kappa = lattice_kappa(name) if lattice_term else 0.0
        self.comp = {}

    def _component(self, j):
        if j not in self.comp:
            mask, approx = (0, True) if j == 0 else (1 << (j - 1), False)
            args = (self.w, self.v, self.hs, self.gs, self.mode, self.align, mask, approx)
            self.comp[j] = (synth_ld(*args), synth_bound(*args, kappa=self.kappa))
        return self.comp[j]

    def of(self, mask, approx):
        n = self.v.size
        x, e = np.zeros(n, LD), np.zeros(n, LD)
        for j in ([0] if approx else []) + [j for j in range(1, self.w.shape[0] + 1) if (mask >> (j - 1)) & 1]:
            cx, ce = self._component(j)
            x, e = x + cx, e + ce
        return x, e

    def check(self, out, mask, approx, what):
        x, e = self.of(mask, approx)
        ok, r, i = within(out, x, e)
        assert ok, f"{what}: mask={mask:#b} use_approx={approx}: |err| / bound = {r:.3g} at t = {i}"


def _reference(name, mode, n, levels, seed):
    key = (name, mode, n, levels, seed)
    if key not in _REF_CACHE:
        w, v = coefficients(levels, n, 2, seed, spike_row=1)
        _REF_CACHE.clear()
        _REF_CACHE[key] = (w, v, Reference(name, mode, w[:, -1], v[-1]))
    return _REF_CACHE[key]


def _pairs_on(l, lattice):
    return (l == 30 and lattice & 2 and lattice & 1) or (l in (16, 18, 20) and lattice & 4)


# (id, wavelet, n, J, "lattice" option, flags); the id names what the default plan / the option makes run
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
@pytest.mark.parametrize("mode", [0, 1, 2], ids=MODE_ID)
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_every_synthesis_path_with_masks_within_the_bound(eng, case, mode):
    cid, name, n, levels, lattice, flags = case
    hs, gs = taps(name)
    l = hs.size
    w, v, ref = _reference(name, mode, n, levels, seed=n + levels)
    plan = _plan(l, levels, n)
    full = (1 << levels) - 1
    if mode == 2:
        path = f"SYMMETRIC: aligned tile stage for levels 1-2, column kernels from level 3 ({cid})"
    elif flags & _native.FLAG_NO_FUSE:
        path = f"generic per-level kernels ({cid})"
    else:
        path = f"plan {_plan_text(plan)}, lattice option {lattice} ({cid})"
    tile_levels = [a for a, k, kind in plan if kind == "fused"]
    pairs = [a for a, k, kind in plan if kind == "column" and k == 2]
    extra = []
    if tile_levels and pairs:
        ref_mask = full & ~(1 << (tile_levels[0] - 1))
        extra = [ref_mask] + [ref_mask & ~(1 << (a - 1)) for a in pairs]
    eng.set_option("lattice", lattice)
    try:
        eng.inverse(w, v, hs, gs, mode, ref.align, ref.order, full, True, flags)
        counts = {}
        for mask in _masks(levels, plan, extra):
            for approx in (True, False):
                l0 = eng.launch_count()
                out = np.asarray(eng.inverse(w, v, hs, gs, mode, ref.align, ref.order, mask, approx, flags))
                counts[(mask, approx)] = k = eng.launch_count() - l0
                what = f"{path}, {k} launches"
                if mask == 0 and not approx:
                    assert not np.any(out), what
                ref.check(out[-1], mask, approx, what)
    finally:
        eng.set_option("lattice", 15)
    if mode == 2 or flags & _native.FLAG_NO_FUSE:
        assert set(counts.values()) == {levels}, (path, counts)             # one launch per level, whatever the mask
        return
    if lattice == 15:
        expect = sum(1 if kind == "fused" or (kind == "column" and k == 2) else k for a, k, kind in plan)
        assert counts[(full, True)] == expect, (path, counts[(full, True)])
    if extra:
        # splitting a pair's mask runs its two levels as single column kernels: one launch more than with the pair whole
        # (both masks are partial, so both calls plan alike); with the pairs off it costs nothing
        for m in extra[1:]:
            assert counts[(m, True)] - counts[(extra[0], True)] == (1 if _pairs_on(l, lattice) else 0), (path, m)
        # no V (use_approx = 0): the top pair declines too
        top = plan[-1]
        declines = 1 if _pairs_on(l, lattice) and top[2] == "column" and top[1] == 2 else 0
        assert counts[(extra[0], False)] - counts[(extra[0], True)] == declines, path


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2], ids=MODE_ID)
@pytest.mark.parametrize("name,n,levels", [("db4", 4096, 4), ("sym8", 6000, 6), ("coif5", 9000, 5)])
def test_bitexact_partial_reconstruction_equals_the_java_order_oracle(eng, name, n, levels, mode):
    """VW_FLAG_BITEXACT: the per-level kernels in the reference's order, bit for bit.  The only freedom is the sign of an
    empty sum's zero: the oracle starts every sum from +0.0 and adds +-0.0 products of the zeroed level, a kernel that
    skips a masked-out level starts from its first product; -0.0 == +0.0 compares equal, every other value bit for bit."""
    h, g, wid = filters(name)
    hs, gs = h * S, g * S
    align, order = alignment(name, mode, levels)
    w, v = coefficients(levels, n, 2, seed=n + mode, spike_row=0)
    for mask in _masks(levels, []):
        for approx in (True, False):
            out = np.asarray(eng.inverse(w, v, hs, gs, mode, align, order, mask, approx, _native.FLAG_BITEXACT))
            for i in range(2):
                exp = cref.reconstruct(w[:, i], v[i], h, g, mode, wid, detail_mask=mask, use_approx=approx)
                assert np.array_equal(out[i], exp), (mask, approx, i)
                nz = exp != 0
                assert np.array_equal(out[i][nz].view(np.int64), exp[nz].view(np.int64)), (mask, approx, i)


# ---- GPU: public entry points at deep shapes ------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2], ids=MODE_ID)
@pytest.mark.parametrize("name,n,levels", [("coif5", 65536, 8), ("sym8", 40000, 8)])
def test_public_partial_reconstructions_within_the_bound(eng, name, n, levels, mode):
    import torch
    rng = np.random.default_rng(n + mode)
    x = rng.standard_normal(n) * 10.0 ** rng.integers(-3, 4, size=n)
    x[n // 5] = 1e9
    wav = vw.get_wavelet(name)
    t = vw.MultiLevelMODWTTransform(wav, BMODE[mode])
    res = t.decompose(x, levels)
    w = np.stack([np.asarray(res.getDetailCoeffsAtLevel(j)) for j in range(1, levels + 1)])
    v = np.asarray(res.getApproximationCoeffs())
    ref = Reference(name, mode, w, v)
    full = (1 << levels) - 1
    for start in (1, 2, levels // 2, levels):
        mask = full & ~((1 << (start - 1)) - 1)
        ref.check(np.asarray(t.reconstructFromLevel(res, start)), mask, True, f"reconstructFromLevel({start})")
    for lo, hi in ((1, 1), (2, 5), (3, 3), (levels - 1, levels), (1, levels)):
        mask = ((1 << hi) - 1) & ~((1 << (lo - 1)) - 1)
        ref.check(np.asarray(t.reconstructLevels(res, lo, hi)), mask, hi == levels, f"reconstructLevels({lo}, {hi})")
    swt = vw.VectorWaveSwtAdapter(wav, BMODE[mode])
    for target in (0, 1, levels // 2, levels):
        mask = 0 if target == 0 else 1 << (target - 1)
        ref.check(np.asarray(swt.extractLevel(x, levels, target)), mask, target == 0, f"extractLevel({target})")
    # the resident result (vw_modwt_reconstruct_h), into host and device outputs
    rr = t.decomposeResident(x, levels)
    try:
        assert np.array_equal(np.asarray(rr.getDetailCoeffsAtLevel(levels)), w[-1])
        ref.check(np.asarray(t.reconstructFromLevel(rr, 3)), full & ~0b11, True, "resident reconstructFromLevel(3)")
        align, order = alignment(name, mode, levels)
        hrs, grs = taps(name)
        for mask, approx in ((0b1, False), (0b10100, True), (0, True), (full, False), (0, False)):
            host = rr._handle.reconstruct(hrs, grs, mode, align, order, mask, approx)
            ref.check(host[0], mask, approx, "DeviceResult.reconstruct -> host")
            dev = torch.full((1, n), 7.0, dtype=torch.float64, device="cuda")
            rr._handle.reconstruct(hrs, grs, mode, align, order, mask, approx, out=dev)
            torch.cuda.synchronize()
            ref.check(dev.cpu().numpy()[0], mask, approx, "DeviceResult.reconstruct -> device")
            if mask == 0 and not approx:
                assert not np.any(host) and not torch.any(dev)
    finally:
        rr.close()


# ---- GPU: caller strides and misaligned buffers through the C ABI ---------------------------------------------------------

SENTINEL = -3.5e300

# (id, base offset in elements, extra ld of x / w / v / out, extra gap between W levels)
STRIDES = [
    ("contiguous", 0, (0, 0, 0, 0), 0),
    ("off16B-even", 2, (2, 2, 2, 2), 2),
    ("off8B-odd", 1, (1, 3, 1, 3), 1),
    ("off0-odd-ld", 0, (3, 1, 3, 1), 3),
    ("off16B-odd-gap", 2, (2, 2, 2, 2), 1),
    ("off8B-even", 1, (2, 2, 2, 2), 2),
]


def _tma_ok(cfg):
    _, off, ex, gap = cfg
    return off % 2 == 0 and all(e % 2 == 0 for e in ex) and gap % 2 == 0


class _Buf:
    """rows [..][b][n] placed at `off + level * lsw + row * ld` inside a sentinel-filled flat allocation"""

    def __init__(self, eng, layout, shape, off, ld, lsw=0):
        *lead, b, n = shape
        nl = lead[0] if lead else 1
        self.shape, self.ld, self.lsw, self.layout = shape, ld, lsw, layout
        total = off + (nl - 1) * lsw + (b - 1) * ld + n + 5
        pos = off + np.arange(nl)[:, None, None] * lsw + np.arange(b)[None, :, None] * ld + np.arange(n)[None, None, :]
        self.pos = pos.reshape(shape)
        if layout == "device":
            import torch
            self.flat = torch.full((total,), SENTINEL, dtype=torch.float64, device="cuda")
            self.ptr = self.flat.data_ptr() + 8 * off
        else:
            self.flat = eng.pinned_empty((total,)) if layout == "pinned" else np.empty(total)
            self.flat[:] = SENTINEL
            self.ptr = self.flat.ctypes.data + 8 * off

    def put(self, data):
        if self.layout == "device":
            import torch
            self.flat[torch.as_tensor(self.pos.reshape(-1), device="cuda")] = torch.as_tensor(data.reshape(-1), device="cuda")
        else:
            self.flat[self.pos] = data

    def host(self):
        return self.flat.cpu().numpy() if self.layout == "device" else np.array(self.flat)

    def rows(self):
        return self.host()[self.pos]

    def sentinels_intact(self):
        h = self.host()
        outside = np.ones(h.size, bool)
        outside[self.pos.reshape(-1)] = False
        return bool(np.all(h[outside].view(np.int64) == np.float64(SENTINEL).view(np.int64)))


def _abi_roundtrip(eng, layout, cfg, name, n, levels, x, w, v):
    """vw_modwt_forward of x and vw_modwt_inverse of (w, v) with the strides of cfg -> (W, V, x_hat)"""
    import ctypes as C
    import torch
    _, off, (ex_x, ex_w, ex_v, ex_o), gap = cfg
    hs, gs = taps(name)
    b = x.shape[0]
    ldw = n + ex_w
    lsw = b * ldw + gap
    bx = _Buf(eng, layout, (b, n), off, n + ex_x)
    bw = _Buf(eng, layout, (levels, b, n), off, ldw, lsw)
    bv = _Buf(eng, layout, (b, n), off, n + ex_v)
    bx.put(x)
    flags = _native.FLAG_DEVICE_PTRS if layout == "device" else 0
    if layout == "device":
        torch.cuda.synchronize()
    lib, ctx = eng.lib, eng.ctx
    dp = C.POINTER(C.c_double)
    with eng._call_lock:
        eng._check(lib.vw_reset_stream(ctx))
        eng._check(lib.vw_modwt_forward(ctx, C.c_void_p(bx.ptr), b, n, bx.ld, hs.ctypes.data_as(dp), gs.ctypes.data_as(dp),
                                        hs.size, levels, 0, C.c_void_p(bw.ptr), bw.ld, bw.lsw, C.c_void_p(bv.ptr), bv.ld, flags))
    fw, fv = bw.rows(), bv.rows()
    assert bx.sentinels_intact() and bw.sentinels_intact() and bv.sentinels_intact(), "forward wrote outside its rows"
    bw.put(w)
    bv.put(v)
    bo = _Buf(eng, layout, (b, n), off, n + ex_o)
    if layout == "device":
        torch.cuda.synchronize()
    with eng._call_lock:
        eng._check(lib.vw_reset_stream(ctx))
        eng._check(lib.vw_modwt_inverse(ctx, C.c_void_p(bw.ptr), bw.ld, bw.lsw, C.c_void_p(bv.ptr), bv.ld, b, n,
                                        hs.ctypes.data_as(dp), gs.ctypes.data_as(dp), hs.size, levels, 0, None,
                                        _native.ORDER_SPLIT, C.c_uint64((1 << levels) - 1), 1, C.c_void_p(bo.ptr), bo.ld, flags))
    xo = bo.rows()
    assert bo.sentinels_intact() and bw.sentinels_intact() and bv.sentinels_intact(), "inverse wrote outside its rows"
    assert np.array_equal(bw.rows(), w) and np.array_equal(bv.rows(), v), "inverse changed its inputs"
    return fw, fv, xo


_STRIDE_REF = {}


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["device", "pageable", "pinned"])
@pytest.mark.parametrize("name,n,levels", [("db4", 4096, 4), ("sym8", 40000, 8), ("coif5", 65536, 8)],
                         ids=["db4-lean-tile", "sym8-tile-dirpair", "coif5-tile-latpair"])
def test_caller_strides_and_misaligned_buffers_through_the_abi(eng, name, n, levels, layout):
    key = (name, n, levels)
    if key not in _STRIDE_REF:
        rng = np.random.default_rng(n)
        x = rng.standard_normal((2, n)) * np.array([[1e-3], [1e4]])
        w, v = coefficients(levels, n, 2, seed=levels, spike_row=1)
        hs, gs = taps(name)
        fwd = analysis_ld(x[-1], hs, gs, levels, 0, lattice_kappa(name, True))
        _STRIDE_REF.clear()
        _STRIDE_REF[key] = (x, w, v, fwd, Reference(name, 0, w[:, -1], v[-1]))
    x, w, v, (wr, vr, ewr, evr), ref = _STRIDE_REF[key]
    base = None
    for cfg in STRIDES:
        fw, fv, xo = _abi_roundtrip(eng, layout, cfg, name, n, levels, x, w, v)
        what = f"{layout} {cfg[0]}"
        for j in range(levels):
            ok, r, i = within(fw[j, -1], wr[j], ewr[j])
            assert ok, f"{what}: W_{j + 1} |err| / bound = {r:.3g} at {i}"
        ok, r, i = within(fv[-1], vr, evr)
        assert ok, f"{what}: V |err| / bound = {r:.3g} at {i}"
        ref.check(xo[-1], (1 << levels) - 1, True, what)
        if base is None:
            base = (fw, fv, xo)
        elif _tma_ok(cfg):
            assert all(np.array_equal(a.view(np.int64), c.view(np.int64)) for a, c in zip((fw, fv, xo), base)), \
                f"{what}: not bit-identical to the contiguous call"
