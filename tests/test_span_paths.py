"""The span-sharded long signal, rank by rank on one device, against an extended-precision reference.

Reference.  `synth_ld_from` is the synthesis twin of `test_analysis_paths.analysis_ld_from`: levels first + nlev - 1 ..
first of the `t + k d` synthesis rule with the plain alignment (+1, 0, +1, 0), PERIODIC or ZERO_PADDING, in
`np.longdouble`, with the running-error bound of `test_synthesis_paths` (gamma_2L per level, plus kappa U on every level
when the coif5 lattice kernels may run).  Started at level 1 it is `synth_ld` term for term (checked below).

Signal.  One long signal of `world` spans: rank r's span is the mixed-scale row of `test_analysis_paths.mixed_row` scaled by
1, 2^-300, 2^+300 or all zero (r mod 4), with +-1e8 spikes (at the span's scale) at every seam and halo edge,
r n_local + {0, 1, -1, lead - 1, lead, pad - 1, pad}.  A halo taken from the wrong neighbour, at the wrong offset or of the
wrong length puts 2^+300 samples next to 2^-300 ones, or moves a spike, far outside the bound; the all-zero span gives
exact zeros outside the reach of its neighbours' halos.  The reference of rank r is the window [r n_local, (r + 1) n_local)
of the whole-signal reference in the signal's mode.

What is pinned.  `vw_modwt_inverse_span` group by group (the kernel each group reaches, by its launch count; odd spans with
the exact halo on 8-byte-offset buffers and odd level strides; spans of whole 256-byte rows with the halo rounded up to 32
as the plan does; `FLAG_BITEXACT` bit for bit against a float64 window in `nptwin.synth_level`'s order, both orders); the
whole-cascade calls `forward_span_all`, `span_pack_inverse`, `span_unpack_inverse` and `inverse_span_all` rank by rank on
one context (NaN-filled buffers with slack, message layout, launch counts); the one-thread multi-device driver on a
repeated device, bit for bit equal to the one-context exchange and, under `FLAG_BITEXACT`, to the C oracle; the
asynchronous return of that driver; and the packed variable-length inverse.  Every check prints its worst |err| / bound.
"""
import fractions

import numpy as np
import pytest

from oracle import cref, nptwin
from oracle.wavelets import filters
from vectorwave_b200 import _native
from vectorwave_b200.errors import IllegalArgumentException

from test_analysis_paths import LATTICE_FROM, analysis_ld_from, lattice_term, mixed_row, perturbed_pair
from test_synthesis_paths import PLAIN, gamma, lattice_kappa, synth_bound, synth_ld, taps, within

LD = np.longdouble
U = 2.0 ** -53
S = nptwin.S
MODE_ID = ["per", "zero"]
FNO = _native.FLAG_NO_FUSE
FBX = _native.FLAG_BITEXACT
SENTINEL = -3.5e300
SCALES = [0, -300, 300, None]       # rank r's span is scaled by 2^SCALES[r % 4]; None: all zeros


# ---- reference ---------------------------------------------------------------------------------------------------------

def _ahead(x, reach, mode):
    """x followed by the `reach` samples the t + k d rule reads past its end (ring wrap, or zeros)"""
    n = x.shape[-1]
    if mode == 0:
        return x[np.mod(np.arange(n + reach), n)]
    return np.concatenate([x, np.zeros(reach, x.dtype)])


def _level(n, a, dj, fh, fg, d, mode, dtype):
    """one synthesis level, out[t] = sum_k fh[k] a[t + k d] + sum_k fg[k] dj[t + k d]: the order of
    test_synthesis_paths._stage (every low-pass product, then every high-pass one); None stands for zeros.  It reads
    slices of one extended copy instead of _stage's cached per-tap index arrays, which at 2^18 samples and 30 taps would
    hold hundreds of MB"""
    acc = np.zeros(n, dtype)
    reach = (len(fh) - 1) * d
    for src, f in ((a, fh), (dj, fg)):
        if src is None:
            continue
        ext = _ahead(src, reach, mode)
        for k in range(len(f)):
            acc += f[k] * ext[k * d:k * d + n]
    return acc


def synth_ld_from(v, w_rows, first, nlev, hs, gs, mode, kappa=0.0, u=U):
    """(V_{first-1}, E): levels first + nlev - 1 .. first of the synthesis cascade of the exact inputs v (= V of the top
    level) and w_rows[i] (= W_{first+i}) in longdouble, and the running-error bound of the module docstring"""
    n = np.asarray(v).shape[-1]
    fh, fg = np.asarray(hs).astype(LD), np.asarray(gs).astype(LD)
    ah, ag, one = np.abs(fh), np.abs(fg), np.ones(len(hs), LD)
    g2 = gamma(2 * len(hs), u)
    cur = np.asarray(v).astype(LD)
    a, e = np.abs(cur), None
    for i in range(nlev - 1, -1, -1):
        d = 1 << (first + i - 1)
        dj = np.asarray(w_rows[i]).astype(LD)
        adj = np.abs(dj)
        cur = _level(n, cur, dj, fh, fg, d, mode, LD)
        a_new = _level(n, a, adj, ah, ag, d, mode, LD)
        e_new = g2 * a_new
        if e is not None:
            e_new += (1 + g2) * _level(n, e, None, ah, ag, d, mode, LD)
        if kappa:
            e_new += LD(kappa) * _level(n, a if e is None else a + e, adj, one, one, d, mode, LD)
        a, e = a_new, e_new
    return cur, e * LD(1 + 8 * u)


def synth_f64_from(v, w_rows, first, nlev, hs, gs, mode, order=_native.ORDER_SPLIT, reverse=False):
    """the same cascade in float64 without FMA: ORDER_SPLIT adds every low-pass product, then every high-pass one
    (nptwin.synth_level's PERIODIC order); ORDER_PAIR adds h[k] a + g[k] w pair by pair (its ZERO_PADDING order);
    reverse=True runs k = L-1 .. 0 and the high-pass products first (another order)"""
    n = np.asarray(v).shape[-1]
    cur = np.asarray(v, dtype=np.float64)
    ks = list(range(len(hs)))[::-1] if reverse else list(range(len(hs)))
    for i in range(nlev - 1, -1, -1):
        d = 1 << (first + i - 1)
        reach = (len(hs) - 1) * d
        a, dj = _ahead(cur, reach, mode), _ahead(np.asarray(w_rows[i], dtype=np.float64), reach, mode)
        acc = np.zeros(n)
        if order == _native.ORDER_PAIR:
            for k in ks:
                acc = acc + (hs[k] * a[k * d:k * d + n] + gs[k] * dj[k * d:k * d + n])
        else:
            for src, f in (((dj, gs), (a, hs)) if reverse else ((a, hs), (dj, gs))):
                for k in ks:
                    acc = acc + f[k] * src[k * d:k * d + n]
        cur = acc
    return cur


def synth_f64_linear(vin, w_ext, first, nlev, hs, gs, n_local, order):
    """what the per-level span kernels compute on [span | halo] rows (LINEAR), in float64 in nptwin.synth_level's order:
    level j covers [0, n_local + the halo of the levels below) and reads its inputs t + k d"""
    cur = np.asarray(vin, dtype=np.float64)
    for i in range(nlev - 1, -1, -1):
        d = 1 << (first + i - 1)
        m = n_local + (_native.load_library().vw_span_halo(hs.size, first, i) if i > 0 else 0)
        a, dj = cur, np.asarray(w_ext[i], dtype=np.float64)
        acc = np.zeros(m)
        if order == _native.ORDER_PAIR:
            for k in range(hs.size):
                acc = acc + (hs[k] * a[k * d:k * d + m] + gs[k] * dj[k * d:k * d + m])
        else:
            for k in range(hs.size):
                acc = acc + hs[k] * a[k * d:k * d + m]
            for k in range(gs.size):
                acc = acc + gs[k] * dj[k * d:k * d + m]
        cur = acc
    return cur


def span_signal(n_local, world, lead, pad, seed):
    """the long signal of the module docstring"""
    x = mixed_row(n_local * world, seed)
    offs = sorted(p for p in {0, 1, lead - 1, lead, pad - 1, pad, n_local - 1} if 0 <= p < n_local)
    spikes = 1e8 * np.where(np.arange(len(offs)) % 2 == 0, 1.0, -0.75)
    for r in range(world):
        seg = x[r * n_local:(r + 1) * n_local]
        s = SCALES[r % 4]
        if s is None:
            seg[:] = 0.0
            continue
        seg[offs] = spikes
        seg[:] = np.ldexp(seg, s)
    return x


class Worst:
    """the worst |err| / bound of one check, with where it was"""

    def __init__(self, path):
        self.path, self.ratio, self.where = path, 0.0, None

    def check(self, out, ref, bnd, where):
        ok, r, t = within(out, ref, bnd)
        assert ok, f"{self.path}: {where} t={t}: |err| / bound = {r:.3g}"
        if r > self.ratio:
            self.ratio, self.where = r, f"{where} t={t}"

    def report(self):
        print(f"\nWORST {self.path}: {self.ratio:.3g} of the bound at {self.where}")


# ---- CPU: the reference and the bound -------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", [0, 1], ids=MODE_ID)
@pytest.mark.parametrize("name", ["db4", "coif5"])
def test_synth_ld_from_level_1_is_synth_ld(name, mode):
    hs, gs = taps(name)
    levels, n = 3, 400
    rng = np.random.default_rng(3 + mode)
    w, v = rng.standard_normal((levels, n)) * 1e3, rng.standard_normal(n)
    kappa = lattice_kappa(name)
    x, e = synth_ld_from(v, w, 1, levels, hs, gs, mode, kappa)
    full = (1 << levels) - 1
    assert np.array_equal(x, synth_ld(w, v, hs, gs, mode, [PLAIN] * levels, full, True))
    assert np.array_equal(e, synth_bound(w, v, hs, gs, mode, [PLAIN] * levels, full, True, kappa))


@pytest.mark.parametrize("mode", [0, 1], ids=MODE_ID)
def test_synth_ld_from_agrees_with_exact_fraction_sums(mode):
    """levels 3-2 of db4 on a short row in Fractions: the longdouble reference sits inside the bound evaluated with the
    longdouble unit roundoff 2^-64"""
    hs, gs = taps("db4")
    n, first, nlev = 60, 2, 2
    rng = np.random.default_rng(11 + mode)
    w = rng.standard_normal((nlev, n)) * np.array([[1e6], [1e-3]])
    v = rng.standard_normal(n)
    v[n - 1] = 1e9
    x, e = synth_ld_from(v, w, first, nlev, hs, gs, mode, u=2.0 ** -64)
    F = fractions.Fraction
    fh, fg = [F(c) for c in hs], [F(c) for c in gs]
    cur = [F(c) for c in v]
    for i in range(nlev - 1, -1, -1):
        d = 1 << (first + i - 1)
        dj = [F(c) for c in w[i]]

        def at(src, p):
            return src[p % n] if mode == 0 else (src[p] if p < n else F(0))
        cur = [sum((fh[k] * at(cur, t + k * d) + fg[k] * at(dj, t + k * d) for k in range(hs.size)), F(0)) for t in range(n)]
    for t in range(n):
        assert abs(F(*x[t].as_integer_ratio()) - cur[t]) <= F(*e[t].as_integer_ratio()) + F(1, 1 << 80), t


@pytest.mark.parametrize("mode", [0, 1], ids=MODE_ID)
@pytest.mark.parametrize("name,first,nlev", [("db4", 1, 4), ("sym8", 3, 2), ("coif5", 3, 2), ("haar", 5, 4)])
def test_float64_oracle_and_a_reordered_sum_are_within_the_bound(name, first, nlev, mode):
    h, g, wid = filters(name)
    hs, gs = h * S, g * S
    n = 5000
    x = span_signal(n // 4, 4, 300, 600, n + first)
    w = np.stack([x * (10.0 ** (i - 1)) for i in range(nlev)])
    v = np.roll(x, 77)
    ref, bnd = synth_ld_from(v, w, first, nlev, hs, gs, mode, lattice_kappa(name))
    for order in (_native.ORDER_SPLIT, _native.ORDER_PAIR):
        assert within(synth_f64_from(v, w, first, nlev, hs, gs, mode, order), ref, bnd)[0], order
    assert within(synth_f64_from(v, w, first, nlev, hs, gs, mode, reverse=True), ref, bnd)[0]
    if first == 1:      # from level 1 the oracle itself: its PERIODIC and ZERO_PADDING rules are the plain alignment
        wz = np.zeros((nlev, n))
        wz[:] = w
        ok, r, _ = within(cref.reconstruct(wz, v, h, g, mode, wid), ref, bnd)
        assert ok and r > 1e-3, r           # and the bound is not loose by orders of magnitude


@pytest.mark.parametrize("mode", [0, 1], ids=MODE_ID)
def test_broken_variants_fail_the_bound_where_the_old_tolerance_passes_them(mode):
    """db4 levels 1-3 over three spans scaled 1, 2^-300, 2^-300: a tap off by 1e-13, and the halo of the middle span
    taken one sample too far right (it moves 2^-300 samples only), both pass 1e-12 max|x| and fail the bound"""
    h, g, _ = filters("db4")
    hs, gs = h * S, g * S
    n_local, first, nlev = 2000, 1, 3
    halo = int(_native.load_library().vw_span_halo(hs.size, first, nlev))
    rng = np.random.default_rng(5 + mode)
    scale = np.repeat([1.0, 2.0 ** -300, 2.0 ** -300], n_local)
    w = np.stack([mixed_row(3 * n_local, 40 + i) * scale for i in range(nlev)])
    v = (mixed_row(3 * n_local, 50) + rng.standard_normal(3 * n_local)) * scale
    ref, bnd = synth_ld_from(v, w, first, nlev, hs, gs, mode)
    good = synth_f64_from(v, w, first, nlev, hs, gs, mode)
    assert within(good, ref, bnd)[0]
    old_tol = 1e-12 * float(np.max(np.abs(good)))
    h2, g2 = perturbed_pair(hs, gs)
    bad_tap = synth_f64_from(v, w, first, nlev, h2, g2, mode)
    assert float(np.max(np.abs(bad_tap - good))) <= old_tol
    assert not within(bad_tap, ref, bnd)[0]
    # the middle span computed from [span | halo] rows whose halo starts one sample late
    lo, hi = n_local, 2 * n_local
    sl = np.r_[lo:hi, hi + 1:hi + 1 + halo]
    vin, wext = v[sl], w[:, sl]
    shifted = synth_f64_linear(vin, wext, first, nlev, hs, gs, n_local, _native.ORDER_SPLIT)
    right = synth_f64_linear(v[lo:hi + halo], w[:, lo:hi + halo], first, nlev, hs, gs, n_local, _native.ORDER_SPLIT)
    assert float(np.max(np.abs(shifted - right))) <= old_tol
    assert within(right, ref[lo:hi], bnd[lo:hi])[0]
    assert not within(shifted, ref[lo:hi], bnd[lo:hi])[0]


def test_span_signal_layout():
    lead, pad, n_local = 300, 512, 1000
    x = span_signal(n_local, 5, lead, pad, 1)
    assert not np.any(x[3 * n_local:4 * n_local])
    for r, s in enumerate([0, -300, 300, None, 0]):
        if s is None:
            continue
        seg = np.ldexp(x[r * n_local:(r + 1) * n_local], -s)
        for p in (0, 1, lead - 1, lead, pad - 1, pad, n_local - 1):
            assert abs(seg[p]) >= 7.5e7, (r, p)
        assert float(np.max(np.abs(np.delete(seg, [0, 1, lead - 1, lead, pad - 1, pad, n_local - 1])))) < 1.1e6


@pytest.mark.parametrize("mode", [0, 1, 2], ids=["per", "zero", "sym"])
def test_varlen_alignment_is_the_single_level_inverse(mode):
    """the (sigma, tau) the varlen test uses for each mode: nptwin's single-level inverse lies within its bound"""
    for name in ("haar", "db4", "coif5"):
        h, g, _ = filters(name)
        hs, gs = h * S, g * S
        for n in (1, 2, 7, 64, 301):
            rng = np.random.default_rng(n + mode)
            w, v = rng.standard_normal((1, n)) * 1e4, rng.standard_normal(n)
            al = [VARLEN_ALIGN[mode]]
            ref = synth_ld(w, v, hs, gs, mode, al, 1, True)
            bnd = synth_bound(w, v, hs, gs, mode, al, 1, True)
            assert within(nptwin.inverse_single(v, w[0], h, g, mode), ref, bnd)[0], (name, n)


# ---- CPU: the span plans of the tested shapes -------------------------------------------------------------------------

# (wavelet, J, world, n_local, lead, pad, forward groups, inverse groups)
SHAPES = [
    ("coif5", 10, 2, 131075, 29696, 29696, [(1, 1), (2, 1), (3, 2), (5, 2), (7, 2), (9, 2)], None),
    ("db4", 5, 3, 256, 256, 256, [(1, 4), (5, 1)], None),
    ("sym8", 7, 1, 40001, 1952, 1952, [(1, 1), (2, 2), (4, 2), (6, 2)], [(1, 3), (4, 2), (6, 2)]),
    ("haar", 9, 4, 4097, 544, 544, [(1, 1), (2, 4), (6, 4)], [(1, 4), (5, 4), (9, 1)]),
    ("db10", 8, 2, 65531, 4896, 4896, [(1, 2), (3, 2), (5, 2), (7, 2)], None),
    ("coif5", 6, 2, 32768, 1856, 1856, [(1, 1), (2, 1), (3, 2), (5, 2)], None),
]
SHAPE_ID = [f"{s[0]}-J{s[1]}-w{s[2]}-n{s[3]}" for s in SHAPES]


def _groups(plan, forward):
    if forward:
        return [(plan.first_f[g], plan.nlev_f[g]) for g in range(plan.ngroups_f)]
    return [(plan.first_i[g], plan.nlev_i[g]) for g in range(plan.ngroups_i)]


@pytest.mark.parametrize("shape", SHAPES, ids=SHAPE_ID)
def test_span_plans_of_the_tested_shapes(shape):
    name, levels, world, n_local, lead, pad, gf, gi = shape
    hs, _ = taps(name)
    plan = _native.span_plan(hs.size, levels, n_local, world)
    assert (plan.lead, plan.pad) == (lead, pad)
    assert _groups(plan, True) == gf
    assert _groups(plan, False) == (gi if gi is not None else gf)
    lib = _native.load_library()
    for g in range(plan.ngroups_i):         # every halo is the exact one rounded up to 32 samples
        need = lib.vw_span_halo(hs.size, plan.first_i[g], plan.nlev_i[g])
        assert plan.halo_i[g] == (need + 31) // 32 * 32
    if name == "db4":
        assert lead == pad == n_local                   # the smallest legal span: a neighbour hands over all of it
        with pytest.raises(IllegalArgumentException):
            _native.span_plan(hs.size, levels, n_local - 1, world)


# ---- GPU helpers ------------------------------------------------------------------------------------------------------

def _colmin(l):
    return 3 if l >= 24 else 6           # vw_column_min_level


def _pair_kernel(l, lattice):
    """the column pair kernel the engine has for this filter length and `lattice` option, or None"""
    if l == 30 and lattice & 2 and lattice & 1:
        return "lattice pair"
    if l in (16, 18, 20) and lattice & 4:
        return "direct-form column pair"
    return None


def inverse_span_kernel(l, first, nlev, flags=0, lattice=15):
    """(kernel, launches) of one vw_modwt_inverse_span group, following its dispatch: a column pair for two levels from
    the column threshold on, a column single for one level there, the tile synthesis otherwise; per-level kernels (one
    launch per level) under NO_FUSE or BITEXACT"""
    if flags & (FNO | FBX):
        return ("per-level exact" if flags & FBX else "per-level"), nlev
    if first >= _colmin(l):
        if nlev == 2 and _pair_kernel(l, lattice):
            return _pair_kernel(l, lattice), 1
        if nlev == 1:
            return ("lattice single" if l == 30 and lattice & 1 else "column single"), 1
    return "tile", 1


def forward_span_launches(nlev, flags=0):
    """launches of one vw_modwt_forward_span group: one (analysis pair, column single or tile kernel), or two for every
    per-level level but the last (V and W of a level the group goes on from are two launches)"""
    if flags & (FNO | FBX):
        return 2 * nlev - 1
    return 1


def _lattice_in_plan(plan, l, lattice, flags, forward):
    """whether some group of the plan runs on a coif5 lattice column kernel (its levels then carry the kappa term)"""
    if l != 30 or flags & (FNO | FBX) or not lattice & 1:
        return False
    groups = _groups(plan, forward)
    if forward:
        return any(a >= LATTICE_FROM and (k == 1 or lattice & 2) for a, k in groups)
    return any(inverse_span_kernel(l, a, k, flags, lattice)[0].startswith("lattice") for a, k in groups)


@pytest.fixture
def eng():
    import vectorwave_b200 as vw
    e = vw.Engine.get()
    try:
        yield e
    finally:
        e.set_option("lattice", 15)


def _sync():
    import torch
    torch.cuda.synchronize()


def _bits(t):
    """a tensor's values as int64 bit patterns on the host (NaN payloads and -0.0 included)"""
    return t.detach().cpu().numpy().view(np.int64)


# ---- GPU: vw_modwt_inverse_span, one launch group -----------------------------------------------------------------------

# (wavelet, first level, levels, flags, lattice option, summation order); the kernel is inverse_span_kernel's
INV_SPANS = [
    ("db4", 1, 3, 0, 15, 0),        # tile group from level 1
    ("db4", 3, 2, 0, 15, 0),        # tile group from dilation 4
    ("db4", 6, 1, 0, 15, 0),        # column single
    ("db6", 7, 1, 0, 15, 0),        # column single
    ("sym8", 6, 2, 0, 15, 0),       # direct-form column pair
    ("db10", 7, 2, 0, 15, 0),       # direct-form column pair
    ("coif5", 3, 2, 0, 15, 0),      # lattice pair
    ("coif5", 4, 1, 0, 15, 0),      # lattice single
    ("coif5", 3, 2, 0, 0, 0),       # lattice option 0: no pair, the tile synthesis in direct form
    ("coif5", 3, 2, 0, 1, 0),       # lattice option 1: lattice singles allowed, pairs off: the tile synthesis again
    ("coif5", 4, 1, 0, 0, 0),       # lattice option 0: direct-form column single
    ("sym8", 2, 3, FNO, 15, 0),     # per-level, ORDER_SPLIT
    ("sym8", 2, 3, FNO, 15, 1),     # per-level, ORDER_PAIR
    ("coif5", 3, 2, FNO, 15, 0),
    ("coif5", 3, 2, FNO, 15, 1),
]


def _inv_id(c):
    name, first, nlev, flags, lattice, order = c
    return (f"{name}-L{first}x{nlev}" + ("-nofuse" if flags else "") + (f"-lat{lattice}" if lattice != 15 else "") +
            ("-pair" if order else ""))


def _span_rows(x, n_in, layout):
    """x [..][n_in] as CUDA rows: "odd" puts row 0 8 bytes past a 16-byte boundary with an odd row stride, "plain" is
    contiguous; returns (rows, flat buffer)"""
    import torch
    x = np.atleast_2d(x)
    b = x.shape[0]
    if layout == "plain":
        flat = torch.as_tensor(np.ascontiguousarray(x), device="cuda").reshape(-1)
        return flat.view(b, n_in), flat
    ld = n_in + 1 if n_in % 2 == 0 else n_in
    flat = torch.full((1 + b * ld + 8,), SENTINEL, dtype=torch.float64, device="cuda")
    rows = flat[1:1 + b * ld].view(b, ld)[:, :n_in]
    rows.copy_(torch.as_tensor(x, device="cuda"))
    assert rows.data_ptr() % 16 == 8 and (b == 1 or rows.stride(0) % 2 == 1)
    return rows, flat


@pytest.mark.gpu
@pytest.mark.parametrize("case", INV_SPANS, ids=[_inv_id(c) for c in INV_SPANS])
def test_inverse_span_is_the_window_of_the_whole_synthesis(eng, case):
    """[span | halo] rows of V and of every W row of the group, cut from a whole PERIODIC coefficient set, against the
    span window of the whole-set reference; once with an odd span, the exact halo and 8-byte-offset rows of odd stride,
    once with a span of whole 256-byte rows and the halo rounded up to 32 samples"""
    import torch
    from test_synthesis_paths import coefficients
    name, first, nlev, flags, lattice, order = case
    hs, gs = taps(name)
    l = hs.size
    kernel, launches = inverse_span_kernel(l, first, nlev, flags, lattice)
    kappa = lattice_kappa(name) if kernel.startswith("lattice") else 0.0
    need = eng.span_halo(l, first, nlev)
    eng.set_option("lattice", lattice)
    for n_local, halo, layout in ((6001, need, "odd"), (6144, (need + 31) // 32 * 32, "plain")):
        n_in = n_local + halo
        whole = n_in + 37
        w, v = coefficients(nlev, whole, 1, seed=first * 10 + nlev + n_local, spike_row=0)
        w, v = w[:, 0].copy(), v[0].copy()
        for p in (n_local - 1, n_local, n_local + 1, n_local + need - 1, n_local + halo - 1):
            v[p] = 1e9 * (-1) ** p
            w[:, p] = -2e9 * (-1) ** p
        ref, bnd = synth_ld_from(v, w, first, nlev, hs, gs, 0, kappa)
        ref, bnd = ref[:n_local], bnd[:n_local]
        vin, vflat = _span_rows(v[:n_in], n_in, layout)
        wext, wflat = _span_rows(w[:, :n_in], n_in, layout)
        out, oflat = _span_rows(np.zeros(n_local), n_local, layout)
        oflat.fill_(SENTINEL)
        _sync()
        path = (f"inverse_span {name} levels {first}-{first + nlev - 1} {kernel}, {launches} launches, lattice {lattice}, "
                f"order {order}, n_local {n_local}, halo {halo}, {layout}")
        l0 = eng.launch_count()
        eng.inverse_span(vin[0], wext, halo, hs, gs, first, nlev, order, flags, out=out[0])
        k = eng.launch_count() - l0
        _sync()
        assert k == launches, (path, k)
        res = out[0].cpu().numpy()
        worst = Worst(path)
        worst.check(res, ref, bnd, "V_%d" % (first - 1))
        worst.report()
        o = oflat.cpu().numpy()
        assert np.count_nonzero(o == SENTINEL) == o.size - n_local, f"{path}: wrote outside its {n_local} outputs"
        # negative control: the same call with taps off by 1e-13
        eng.inverse_span(vin[0], wext, halo, *perturbed_pair(hs, gs), first, nlev, order, flags, out=out[0])
        _sync()
        bad = not within(out[0].cpu().numpy(), ref, bnd)[0]
        print(f"NEGATIVE {path}: a 1e-13 tap error {'leaves' if bad else 'stays inside'} the bound")
        if not kappa:                       # a lattice level's bound is wider than a 1e-13 tap error
            assert bad, path
        # FLAG_BITEXACT: the per-level exact kernels, bit for bit a float64 window in nptwin.synth_level's order
        for o_ in (_native.ORDER_SPLIT, _native.ORDER_PAIR):
            l0 = eng.launch_count()
            eng.inverse_span(vin[0], wext, halo, hs, gs, first, nlev, o_, FBX, out=out[0])
            assert eng.launch_count() - l0 == nlev
            _sync()
            exp = synth_f64_linear(v[:n_in], w[:, :n_in], first, nlev, hs, gs, n_local, o_)
            got = out[0].cpu().numpy()
            assert np.array_equal(got.view(np.int64), exp.view(np.int64)), \
                f"{path}: BITEXACT order {o_}: {np.count_nonzero(got != exp)} samples differ"
        assert np.array_equal(_bits(vin), v[None, :n_in].view(np.int64)) and \
            np.array_equal(_bits(wext), w[:, :n_in].view(np.int64)), f"{path}: the call changed its inputs"


# ---- GPU: whole-cascade calls, rank by rank on one context ----------------------------------------------------------

SLACK = 37

_REFS = {}


def _forward_reference(shape, mode, kappa):
    """(x, plan, W ref, V ref, E_W, E_V) of a shape's whole signal, cached across flags and tests"""
    name, levels, world, n_local = shape[:4]
    key = (name, levels, world, n_local, mode, kappa)
    if key not in _REFS:
        hs, gs = taps(name)
        plan = _native.span_plan(hs.size, levels, n_local, world)
        x = span_signal(n_local, world, int(plan.lead), int(plan.pad), n_local + levels + world)
        if len(_REFS) >= 2:
            _REFS.pop(next(iter(_REFS)))
        _REFS[key] = (x, plan) + tuple(analysis_ld_from(x, 1, levels, hs, gs, mode, kappa))
    return _REFS[key]


def _reach_f(l, levels):
    return (l - 1) * ((1 << levels) - 1)


def _check_forward(path, shape, plan, x, refs, wg, vg):
    """W_1..W_J and V_J of every rank against the whole-signal analysis bound; exact zeros in an all-zero span past the
    reach of its left neighbour"""
    name, levels, world, n_local = shape[:4]
    wr, vr, ewr, evr = refs
    worst = Worst(path + " forward")
    for r in range(world):
        win = slice(r * n_local, (r + 1) * n_local)
        for j in range(levels):
            worst.check(wg[j, win], wr[j, win], ewr[j, win], f"rank {r} W_{j + 1}")
        worst.check(vg[win], vr[win], evr[win], f"rank {r} V_{levels}")
        if SCALES[r % 4] is None:
            reach = _reach_f(taps(name)[0].size, levels)
            assert not np.any(wg[:, r * n_local + reach:(r + 1) * n_local]) and not np.any(vg[r * n_local + reach:(r + 1) * n_local])
    worst.report()


def _check_inverse(path, shape, mode, wg, vg, xg, kappa):
    """each rank's reconstruction against synth_ld of the device's own concatenated W and V"""
    name, levels, world, n_local = shape[:4]
    hs, gs = taps(name)
    ref, bnd = synth_ld_from(vg, wg, 1, levels, hs, gs, mode, kappa)
    worst = Worst(path + " inverse")
    for r in range(world):
        win = slice(r * n_local, (r + 1) * n_local)
        worst.check(xg[win], ref[win], bnd[win], f"rank {r} x")
    worst.report()


def _host_message(plan, w, v):
    """the synthesis halo message of one rank, gathered on the host by the layout of vw_span_pack_inverse: V_J[0 .. si_in
    of the top group), then for every inverse group g (ascending) its rows W_j[0 .. si_in[g])"""
    lead_w = int(plan.lead_w)
    si = np.cumsum([int(plan.halo_i[g]) for g in range(plan.ngroups_i)])
    parts = [v[:si[-1]]]
    for g, (first, nlev) in enumerate(_groups(plan, False)):
        for j in range(first, first + nlev):
            parts.append(w[j - 1, lead_w:lead_w + si[g]])
    msg = np.concatenate(parts)
    assert msg.size == plan.inverse_msg
    return msg


def _one_context(eng, shape, mode, flags, lattice, x, plan):
    """forward_span_all, pack, unpack and inverse_span_all of every rank on one engine, with the halo exchanges done on
    the host side; checks buffers and launch counts, returns (W [world][J][stride], V [world][n_local + pad], xout)"""
    import torch
    name, levels, world, n_local = shape[:4]
    hs, gs = taps(name)
    l = hs.size
    lead, lead_w, pad = int(plan.lead), int(plan.lead_w), int(plan.pad)
    row = lead_w + n_local + pad
    fwd_k = sum(forward_span_launches(k, flags) for _, k in _groups(plan, True))
    inv_k = sum(inverse_span_kernel(l, a, k, flags, lattice)[1] for a, k in _groups(plan, False))
    ws, vs, xexts = [], [], []
    for r in range(world):
        left = (r - 1) % world
        if mode == 1 and r == 0:
            lead_part = np.zeros(lead)
        else:
            lead_part = x[(left + 1) * n_local - lead:(left + 1) * n_local]
        xext = torch.as_tensor(np.concatenate([lead_part, x[r * n_local:(r + 1) * n_local]]), device="cuda")
        w = torch.full((levels, row + SLACK), float("nan"), dtype=torch.float64, device="cuda")
        v = torch.full((n_local + pad,), float("nan"), dtype=torch.float64, device="cuda")
        xexts.append(xext)
        ws.append(w)
        vs.append(v)
    _sync()
    x_bits = [_bits(e) for e in xexts]
    for r in range(world):
        l0 = eng.launch_count()
        eng.forward_span_all(xexts[r], plan, hs, gs, ws[r], vs[r], flags)
        assert eng.launch_count() - l0 == fwd_k, (shape, flags, eng.launch_count() - l0, fwd_k)
    _sync()
    for r in range(world):
        assert np.array_equal(_bits(xexts[r]), x_bits[r]), f"rank {r}: forward_span_all changed xext"
        w = ws[r].cpu().numpy()
        assert np.all(np.isnan(w[:, row:])), f"rank {r}: forward_span_all wrote into the slack past the W rows"
        assert np.all(np.isnan(w[:, lead_w + n_local:row])) and np.all(np.isnan(vs[r].cpu().numpy()[n_local:])), \
            f"rank {r}: forward_span_all wrote into the pad areas"
    msgs = []
    for r in range(world):
        msg = torch.full((int(plan.inverse_msg),), float("nan"), dtype=torch.float64, device="cuda")
        l0 = eng.launch_count()
        eng.span_pack_inverse(plan, ws[r], vs[r], msg)
        assert eng.launch_count() - l0 == 1
        msgs.append(msg)
    _sync()
    for r in range(world):
        exp = _host_message(plan, ws[r].cpu().numpy(), vs[r].cpu().numpy())
        assert np.array_equal(msgs[r].cpu().numpy().view(np.int64), exp.view(np.int64)), f"rank {r}: message layout"
    for r in range(world):
        right = (r + 1) % world
        msg = None if (mode == 1 and r == world - 1) else msgs[right]
        l0 = eng.launch_count()
        eng.span_unpack_inverse(plan, msg, ws[r], vs[r])
        assert eng.launch_count() - l0 == 1
    _sync()
    si = np.cumsum([int(plan.halo_i[g]) for g in range(plan.ngroups_i)])
    for r in range(world):                  # the pad areas hold the right neighbour's first samples, or zeros
        right = (r + 1) % world
        zero = mode == 1 and r == world - 1
        v, vn = vs[r].cpu().numpy(), vs[right].cpu().numpy()
        assert np.array_equal(v[n_local:n_local + si[-1]], np.zeros(si[-1]) if zero else vn[:si[-1]]), f"rank {r} V pad"
        w, wn = ws[r].cpu().numpy(), ws[right].cpu().numpy()
        for g, (first, nlev) in enumerate(_groups(plan, False)):
            for j in range(first - 1, first - 1 + nlev):
                got = w[j, lead_w + n_local:lead_w + n_local + si[g]]
                assert np.array_equal(got, np.zeros(si[g]) if zero else wn[j, lead_w:lead_w + si[g]]), f"rank {r} W_{j + 1} pad"
    before = [(_bits(ws[r]), _bits(vs[r])) for r in range(world)]
    order = _native.ORDER_PAIR if mode == 1 else _native.ORDER_SPLIT
    outs = []
    for r in range(world):
        out = torch.full((n_local + 1,), SENTINEL, dtype=torch.float64, device="cuda")
        l0 = eng.launch_count()
        eng.inverse_span_all(plan, ws[r], vs[r], hs, gs, order, out[:n_local], flags)
        assert eng.launch_count() - l0 == inv_k, (shape, flags, eng.launch_count() - l0, inv_k)
        outs.append(out)
    _sync()
    for r in range(world):
        assert np.array_equal(_bits(ws[r]), before[r][0]) and np.array_equal(_bits(vs[r]), before[r][1]), \
            f"rank {r}: inverse_span_all changed W or V"
        assert float(outs[r][n_local].item()) == SENTINEL, f"rank {r}: inverse_span_all wrote past xout[n_local]"
    return ([w.cpu().numpy() for w in ws], [v.cpu().numpy() for v in vs], [o[:n_local].cpu().numpy() for o in outs])


def _gather_w_v(plan, shape, ws, vs):
    lead_w, n_local = int(plan.lead_w), shape[3]
    return (np.concatenate([w[:, lead_w:lead_w + n_local] for w in ws], axis=1),
            np.concatenate([v[:n_local] for v in vs]))


def _sharded(shape, mode, flags, lattice, x, plan, devices=None):
    """vw_modwt_forward_sharded + vw_modwt_inverse_sharded over `devices` (default: device 0 once per rank), with NaN
    leads the engine must fill; returns W, V, xout per rank as host arrays"""
    import torch
    name, levels, world, n_local = shape[:4]
    devices = devices or [0] * world
    hs, gs = taps(name)
    lead, lead_w, pad = int(plan.lead), int(plan.lead_w), int(plan.pad)
    row = lead_w + n_local + pad
    me = _native.MultiEngine(devices)
    try:
        for r in range(world):
            me.lib.vw_set_option(me.lib.vw_multi_ctx(me.handle, r), b"lattice", int(lattice))
        xext, ws, vs, xo = [], [], [], []
        for r, d in enumerate(devices):
            dev = torch.device("cuda", d)
            e = torch.full((lead + n_local,), float("nan"), dtype=torch.float64, device=dev)
            e[lead:] = torch.as_tensor(x[r * n_local:(r + 1) * n_local], device=dev)
            xext.append(e)
            ws.append(torch.full((levels, row + SLACK), float("nan"), dtype=torch.float64, device=dev))
            vs.append(torch.full((n_local + pad,), float("nan"), dtype=torch.float64, device=dev))
            xo.append(torch.full((n_local,), SENTINEL, dtype=torch.float64, device=dev))
        for d in set(devices):
            torch.cuda.synchronize(d)
        me.forward(plan, xext, hs, gs, mode, ws, vs, flags=flags)
        order = _native.ORDER_PAIR if mode == 1 else _native.ORDER_SPLIT
        me.inverse(plan, ws, vs, hs, gs, mode, order, xo, flags=flags)
        return [w.cpu().numpy() for w in ws], [v.cpu().numpy() for v in vs], [o.cpu().numpy() for o in xo]
    finally:
        me.close()


def _same_bits(a, b):
    return np.array_equal(np.asarray(a).view(np.int64), np.asarray(b).view(np.int64))


def _oracle_equal(got, exp):
    """equal to the oracle, every non-zero value bit for bit.  The only freedom is the sign of a zero: the oracle starts
    every sum from +0.0 and skips a ZERO_PADDING term past the end, a kernel starts from its first product and adds the
    +-0.0 product of a zero it reads"""
    got, exp = np.asarray(got), np.asarray(exp)
    nz = exp != 0
    return np.array_equal(got, exp) and np.array_equal(got[nz].view(np.int64), exp[nz].view(np.int64))


# (shape index, lattice options): every shape with the default engine; coif5 J = 6 also with the lattice option at 0 and 1
CASCADES = [(i, 15) for i in range(len(SHAPES))] + [(5, 0), (5, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1], ids=MODE_ID)
@pytest.mark.parametrize("si,lattice", CASCADES,
                         ids=[SHAPE_ID[i] + ("" if lat == 15 else f"-lat{lat}") for i, lat in CASCADES])
def test_whole_cascades_rank_by_rank_and_the_sharded_driver(eng, si, lattice, mode):
    """section by section for flags 0, NO_FUSE and BITEXACT: the one-context span calls with host-side exchanges within
    the bounds (forward against the whole-signal analysis, inverse against synth_ld of the device's own W and V); the
    one-thread multi-device driver on device 0 repeated, bit for bit the same; under BITEXACT both bit for bit the C
    oracle's decompose and reconstruct"""
    shape = SHAPES[si]
    name, levels, world, n_local = shape[:4]
    h, g, wid = filters(name)
    hs, gs = h * S, g * S
    l = hs.size
    eng.set_option("lattice", lattice)
    plan = _native.span_plan(l, levels, n_local, world)
    for flags in (0, FNO, FBX):
        kf = lattice_term(name, lattice) if _lattice_in_plan(plan, l, lattice, flags, True) else 0.0
        ki = lattice_kappa(name) if _lattice_in_plan(plan, l, lattice, flags, False) else 0.0
        x, plan, *refs = _forward_reference(shape, mode, kf)
        path = f"{SHAPE_ID[si]} {MODE_ID[mode]} lattice {lattice} flags {flags}"
        ws, vs, xs = _one_context(eng, shape, mode, flags, lattice, x, plan)
        wg, vg = _gather_w_v(plan, shape, ws, vs)
        xg = np.concatenate(xs)
        _check_forward(path + " one context", shape, plan, x, refs, wg, vg)
        _check_inverse(path + " one context", shape, mode, wg, vg, xg, ki)
        if flags & FBX:
            wo, vo = cref.decompose(x, h, g, levels, mode)
            assert _oracle_equal(wg, wo) and _oracle_equal(vg, vo), f"{path}: BITEXACT forward differs from cref.decompose"
            assert _oracle_equal(xg, cref.reconstruct(wg, vg, h, g, mode, wid)), f"{path}: BITEXACT differs from cref.reconstruct"
        sw, sv, sx = _sharded(shape, mode, flags, lattice, x, plan)
        swg, svg = _gather_w_v(plan, shape, sw, sv)
        assert _same_bits(swg, wg) and _same_bits(svg, vg), f"{path}: the sharded driver's W, V differ from the one-context calls"
        assert _same_bits(np.concatenate(sx), xg), f"{path}: the sharded driver's xout differs from the one-context calls"
        print(f"SHARDED {path}: W, V and xout bit for bit the one-context calls")


@pytest.mark.gpu
def test_sharded_driver_asynchronous_return():
    """VW_FLAG_NO_SYNC: two forward + inverse steps of two signals into separate buffers, one vw_multi_synchronize at the
    end.  The second inverse's pack must wait until the left neighbour has read the first message (ev_ready ordering);
    a message overwritten early puts the second signal's halo into the first reconstruction"""
    import torch
    shape = SHAPES[3]                       # haar J = 9 over four spans, one of them all zeros
    name, levels, world, n_local = shape[:4]
    hs, gs = taps(name)
    mode = 0
    plan = _native.span_plan(hs.size, levels, n_local, world)
    lead, lead_w, pad = int(plan.lead), int(plan.lead_w), int(plan.pad)
    row = lead_w + n_local + pad
    # the second signal is a negated one of another seed: a message of one step read in the other is off by ~2e6
    signals = [span_signal(n_local, world, lead, pad, 990), -span_signal(n_local, world, lead, pad, 991)]
    me = _native.MultiEngine([0] * world)
    try:
        bufs = []
        for x in signals:
            xext = [torch.full((lead + n_local,), float("nan"), dtype=torch.float64, device="cuda") for _ in range(world)]
            for r in range(world):
                xext[r][lead:] = torch.as_tensor(x[r * n_local:(r + 1) * n_local], device="cuda")
            bufs.append((xext, [torch.full((levels, row + SLACK), float("nan"), dtype=torch.float64, device="cuda") for _ in range(world)],
                         [torch.full((n_local + pad,), float("nan"), dtype=torch.float64, device="cuda") for _ in range(world)],
                         [torch.full((n_local,), SENTINEL, dtype=torch.float64, device="cuda") for _ in range(world)]))
        torch.cuda.synchronize()
        for xext, w, v, xo in bufs:
            me.forward(plan, xext, hs, gs, mode, w, v, flags=_native.FLAG_NO_SYNC)
            me.inverse(plan, w, v, hs, gs, mode, _native.ORDER_SPLIT, xo, flags=_native.FLAG_NO_SYNC)
        me.synchronize()
        results = [([t.cpu().numpy() for t in w], [t.cpu().numpy() for t in v], [t.cpu().numpy() for t in xo]) for _, w, v, xo in bufs]
    finally:
        me.close()
    for i, (x, (ws, vs, xs)) in enumerate(zip(signals, results)):
        wr, vr, ewr, evr = analysis_ld_from(x, 1, levels, hs, gs, mode)
        wg, vg = _gather_w_v(plan, shape, ws, vs)
        path = f"NO_SYNC step {i + 1} {SHAPE_ID[3]}"
        _check_forward(path, shape, plan, x, (wr, vr, ewr, evr), wg, vg)
        _check_inverse(path, shape, mode, wg, vg, np.concatenate(xs), 0.0)


@pytest.mark.gpu
def test_sharded_driver_over_real_devices():
    import torch
    count = torch.cuda.device_count()
    if count < 2:
        pytest.skip("needs at least two GPUs")
    world = min(count, 8)
    shape = ("coif5", 10, world, 131075)
    h, g, _ = filters("coif5")
    hs, gs = h * S, g * S
    plan = _native.span_plan(hs.size, 10, 131075, world)
    kf, ki = lattice_term("coif5"), lattice_kappa("coif5")
    x = span_signal(131075, world, int(plan.lead), int(plan.pad), 4242)
    refs = analysis_ld_from(x, 1, 10, hs, gs, 0, kf)
    ws, vs, xs = _sharded(shape, 0, 0, 15, x, plan, devices=list(range(world)))
    wg, vg = _gather_w_v(plan, shape, ws, vs)
    path = f"coif5 J10 over {world} devices"
    _check_forward(path, shape, plan, x, refs, wg, vg)
    _check_inverse(path, shape, 0, wg, vg, np.concatenate(xs), ki)


# ---- GPU: the packed variable-length inverse ---------------------------------------------------------------------------

# the single-level rule of vw_modwt_inverse_varlen (MODWTTransform.inverse): t + l, and t - l under SYMMETRIC
VARLEN_ALIGN = [PLAIN, PLAIN, (-1, 0, -1, 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2], ids=["per", "zero", "sym"])
@pytest.mark.parametrize("name", ["haar", "db4", "sym8", "coif5"])
def test_inverse_varlen_rows_within_the_bound(eng, name, mode):
    import torch
    hs, gs = taps(name)
    lengths = [1, 2, 7, 64, 1001, 4096, 9000]
    ws, vs = [], []
    for i, m in enumerate(lengths):
        rng = np.random.default_rng(17 * i + m + mode)
        sc = 300 if i % 2 == 0 else -300
        w = np.ldexp(rng.standard_normal(m) * 10.0 ** rng.integers(-6, 7, size=m), sc)
        v = np.ldexp(mixed_row(m, i) if m > 2 else rng.standard_normal(m), sc)
        ws.append(w)
        vs.append(v)
    offsets = np.concatenate([[0], np.cumsum(lengths)])
    l0 = eng.launch_count()
    out = eng.inverse_varlen(torch.as_tensor(np.concatenate(ws), device="cuda"), torch.as_tensor(np.concatenate(vs), device="cuda"),
                             offsets, hs, gs, mode)
    assert eng.launch_count() - l0 == 1                     # every row in one launch
    _sync()
    out = out.cpu().numpy()
    worst = Worst(f"inverse varlen {name} {['per', 'zero', 'sym'][mode]}")
    al = [VARLEN_ALIGN[mode]]
    for i, m in enumerate(lengths):
        w, v = ws[i][None], vs[i]
        ref = synth_ld(w, v, hs, gs, mode, al, 1, True)
        bnd = synth_bound(w, v, hs, gs, mode, al, 1, True)
        worst.check(out[offsets[i]:offsets[i + 1]], ref, bnd, f"row {i} n={m}")
    worst.report()
