"""Every analysis path, level by level, against an extended-precision reference, with the kernel that ran pinned.

Reference.  `analysis_ld_from` is the analysis cascade of `oracle/nptwin.decompose` in `np.longdouble` (64-bit
significand), started at any level: level j reads V_{j-1} at t - k 2^(j-1) under the PERIODIC, ZERO_PADDING or
SYMMETRIC index rule, with the double taps hs = h*S, gs = g*S the engine gets.  Started at level 1 it is
`test_synthesis_paths.analysis_ld` term for term (checked below); started deeper it is the reference of the span calls.

Bound.  A running-error bound per output sample, u = 2^-53, gamma_L = L u / (1 - L u), L taps:
    A_0 = |x|,  E_0 = 0
    A_j = |h| * A_{j-1},  E^V_j = (1 + gamma_L) |h| * E_{j-1} + gamma_L A_j,  E^W_j = (1 + gamma_L) |g| * E_{j-1} + gamma_L |g| * A_{j-1}
(`*` is the level's dilated convolution under the mode's index rule).  Every output sample is one L-term sum of
products of a tap and a computed input.  However the kernel orders that sum -- the tile kernels' item loops with FMA
chains, the transposed direct-form pair kernels that carry a partial sum from input row to input row, or a plain loop
without FMA -- each product meets at most L roundings (its multiply, or none under FMA, and at most L - 1 additions), so
the computed sum is off by at most gamma_L times the sum of |products|.  The transposed form still adds each output's
own L products, only the order of the additions differs; keeping V of the first level of a pair in registers rounds it
exactly as a store to memory does.  The bound is evaluated in longdouble and rounded up by (1 + 8u); a check is
|y_hat - y_ref| <= E + 2^-60 |y_ref|.  There is no underflow term: the inputs stay within 2^+-600.

Lattice levels.  The coif5 column kernels in lattice form compute with rotation coefficients, not the taps; those levels
add kappa U_j, kappa = tap_err + gamma_{2K+4} c_lat (`test_synthesis_paths.lattice_kappa(.., forward=True)`),
U_j = 1 * (A_{j-1} + E_{j-1}), to both E^V_j and E^W_j.  Only the column kernels have a lattice form, and they take a
level from dilation 4 on (level 3, `vw_column_min_level` of a 30-tap pair), so levels 1-2 keep the direct-form bound.

Inputs.  Each batch holds a mixed-scale row 1e6 sin(2 pi t / n) + N(0, 1) + 1e-6 N(0, 1), the same row scaled by 2^-300,
a row of spikes at both ends and at tile boundaries scaled by 2^+300 (next to the 2^-300 row, so that any leak of it into
that row would be seen), and an all-zero row whose outputs must be exact zeros.  The reference of a row scaled by a power of
two is the unscaled one, scaled.  Each check reports the worst |err| / bound with its row, level and t.

Launch counts pin the path.  A full default plan (`describe_plan(True, ..)`) costs one launch per fused or column group
and one per level for the rest; under SYMMETRIC every planned pair declines (two launches) and a fused group declines
when the row is shorter than its even halo htot; FLAG_NO_FUSE costs one launch per level.
"""
import fractions
import functools

import numpy as np
import pytest

import vectorwave_b200 as vw
from oracle import cref, nptwin
from oracle.wavelets import filters
from vectorwave_b200 import _native

from test_synthesis_paths import analysis_ld, gamma, lattice_kappa, taps, within

LD = np.longdouble
U = 2.0 ** -53
S = nptwin.S
MODE_ID = ["per", "zero", "sym"]
LATTICE_FROM = 3        # first level a 30-tap pair may run in lattice form (vw_column_min_level)


# ---- reference ---------------------------------------------------------------------------------------------------------

@functools.lru_cache(maxsize=512)
def _ext_index(n, reach, mode):
    """source index of positions -reach .. n-1 under the mode's index rule; n stands for a zero (ZERO_PADDING)"""
    pos = np.arange(-reach, n)
    if mode == 0:
        return np.mod(pos, n)
    if mode == 2:
        return nptwin.mirror(pos, n)
    return np.where(pos < 0, n, pos)


def _conv(x, f, d, mode):
    """out[.., t] = sum_k f[k] x[.., ext(t - k d)], accumulated k = 0, 1, .. (the order of test_synthesis_paths._stage)"""
    n = x.shape[-1]
    reach = (len(f) - 1) * d
    src = np.concatenate([x, np.zeros(x.shape[:-1] + (1,), x.dtype)], axis=-1) if mode == 1 else x
    ext = src[..., _ext_index(n, reach, mode)]
    acc = np.zeros(x.shape, x.dtype)
    for k in range(len(f)):
        acc += f[k] * ext[..., reach - k * d:reach - k * d + n]
    return acc


def analysis_ld_from(v, first_level, nlevels, hs, gs, mode, kappa=0.0, kappa_from=LATTICE_FROM, u=U):
    """(W [nlevels][.., n], V, E_W [nlevels][.., n], E_V): levels first_level .. first_level + nlevels - 1 of the
    analysis cascade of the exact input v (= V_{first_level - 1}) in longdouble, and the running-error bound of the
    module docstring; kappa is added from level kappa_from on"""
    fh, fg = np.asarray(hs).astype(LD), np.asarray(gs).astype(LD)
    ah, ag, one = np.abs(fh), np.abs(fg), np.ones(len(hs), LD)
    gl = gamma(len(hs), u)
    up = LD(1 + 8 * u)
    cur = np.asarray(v).astype(LD)
    a, e = np.abs(cur), np.zeros(cur.shape, LD)
    ws, ews = [], []
    for level in range(first_level, first_level + nlevels):
        d = 1 << (level - 1)
        ws.append(_conv(cur, fg, d, mode))
        cur = _conv(cur, fh, d, mode)
        ew = (1 + gl) * _conv(e, ag, d, mode) + gl * _conv(a, ag, d, mode)
        a_new = _conv(a, ah, d, mode)
        ev = (1 + gl) * _conv(e, ah, d, mode) + gl * a_new
        if kappa and level >= kappa_from:
            unit = LD(kappa) * _conv(a + e, one, d, mode)
            ew, ev = ew + unit, ev + unit
        ews.append(ew * up)
        a, e = a_new, ev * up
    return np.stack(ws), cur, np.stack(ews), e


def float_cascade(x, hs, gs, first_level, nlevels, mode, reverse=False):
    """the cascade in float64 without FMA; reverse=True adds the products k = L-1 .. 0 and splits each sum into two
    halves added at the end (another order than the oracle's)"""
    cur = np.asarray(x, dtype=np.float64)
    ws = []
    for level in range(first_level, first_level + nlevels):
        d = 1 << (level - 1)
        n = cur.shape[-1]
        reach = (len(hs) - 1) * d
        src = np.concatenate([cur, np.zeros(cur.shape[:-1] + (1,))], axis=-1) if mode == 1 else cur
        ext = src[..., _ext_index(n, reach, mode)]
        out = []
        for f in (gs, hs):
            ks = list(range(len(f)))[::-1] if reverse else list(range(len(f)))
            half = len(ks) // 2 if reverse else len(ks)
            parts = []
            for chunk in (ks[:half], ks[half:]):
                acc = np.zeros(cur.shape)
                for k in chunk:
                    acc = acc + f[k] * ext[..., reach - k * d:reach - k * d + n]
                parts.append(acc)
            out.append(parts[0] + parts[1])
        ws.append(out[0])
        cur = out[1]
    return np.stack(ws), cur


def lattice_term(name, lattice=15):
    """kappa of the bound for `name` when the engine's `lattice` option is `lattice` (bit 0: lattice form)"""
    return lattice_kappa(name, True) if lattice & 1 else 0.0


# ---- inputs ------------------------------------------------------------------------------------------------------------

def mixed_row(n, seed):
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    return 1e6 * np.sin(2 * np.pi * t / n) + rng.standard_normal(n) + 1e-6 * rng.standard_normal(n)


def spike_row(n, seed, tiles=()):
    """small noise with +-1e8 spikes at both ends and on both sides of every multiple of each tile size"""
    rng = np.random.default_rng(seed + 1)
    x = 1e-3 * rng.standard_normal(n)
    at = {0, 1, 2, n - 3, n - 2, n - 1}
    for tl in tiles:
        if tl > 0:
            for m in range(tl, n, tl):
                at |= {m - 1, m, m + 1}
    at = sorted(p for p in at if 0 <= p < n)
    x[at] = 1e8 * np.where(np.arange(len(at)) % 2 == 0, 1.0, -0.75)
    return x


# row r of a batch is 2^scale * base[row]; None is the all-zero row
RECIPE = [(0, 0), (0, -300), (1, 300), (None, 0)]


def make_batch(n, seed, tiles=()):
    base = np.stack([mixed_row(n, seed), spike_row(n, seed, tiles)])
    x = np.stack([np.ldexp(base[i], s) if i is not None else np.zeros(n) for i, s in RECIPE])
    return base, x


class Reference:
    """reference and bound of every row of a make_batch batch (computed once per distinct row)"""

    def __init__(self, base, hs, gs, mode, first_level, nlevels, kappa=0.0, window=None):
        w, v, ew, ev = analysis_ld_from(base, first_level, nlevels, hs, gs, mode, kappa)
        sl = slice(None) if window is None else slice(window, None)
        self.first = first_level
        self.w, self.v, self.ew, self.ev = w[..., sl], v[..., sl], ew[..., sl], ev[..., sl]

    def check(self, w, v, path, rows=RECIPE, report=True):
        """w [nlevels][B][n], v [B][n] for the rows of `rows`: all within the bound; returns the worst ratio"""
        worst = (0.0, None)
        for r, (i, s) in enumerate(rows):
            if i is None:
                assert not np.any(w[:, r]) and not np.any(v[r]), f"{path}: the all-zero row gave non-zero outputs"
                continue
            sc = LD(2) ** s
            for j in range(w.shape[0] + 1):
                out, ref, bnd = (w[j, r], self.w[j, i], self.ew[j, i]) if j < w.shape[0] else (v[r], self.v[i], self.ev[i])
                ok, ratio, t = within(out, ref * sc, bnd * sc)
                where = f"row {r} {'W_%d' % (self.first + j) if j < w.shape[0] else 'V'} t={t}"
                assert ok, f"{path}: {where}: |err| / bound = {ratio:.3g}"
                if ratio > worst[0]:
                    worst = (ratio, where)
        if report:
            print(f"\nWORST {path}: {worst[0]:.3g} of the bound at {worst[1]}")
        return worst[0]

    def failures(self, w, v, rows=RECIPE):
        """the levels (first .. , 0 for V) on which some row is outside the bound"""
        bad = set()
        for r, (i, s) in enumerate(rows):
            if i is None:
                continue
            sc = LD(2) ** s
            for j in range(w.shape[0]):
                if not within(w[j, r], self.w[j, i] * sc, self.ew[j, i] * sc)[0]:
                    bad.add(self.first + j)
            if not within(v[r], self.v[i] * sc, self.ev[i] * sc)[0]:
                bad.add(0)
        return bad


def perturbed(f):
    """f with its largest tap off by 1e-13 relative"""
    f = np.array(f, dtype=np.float64)
    k = int(np.argmax(np.abs(f)))
    f[k] *= 1 + 1e-13
    return f


def perturbed_pair(hs, gs):
    """the largest high-pass tap and its low-pass mirror image both off by 1e-13 relative: a quadrature-mirror pair
    stays one (vw_is_qmf), so the engine picks the same kernels as for the true taps"""
    hs, gs = np.array(hs, dtype=np.float64), np.array(gs, dtype=np.float64)
    k = int(np.argmax(np.abs(gs)))
    gs[k] *= 1 + 1e-13
    hs[hs.size - 1 - k] *= 1 + 1e-13
    return hs, gs


# ---- CPU: the reference and the bound -------------------------------------------------------------------------------

def test_analysis_ld_from_level_1_is_analysis_ld():
    hs, gs = taps("sym8")
    x = mixed_row(300, 1)
    for mode in (0, 1, 2):
        a = analysis_ld(x, hs, gs, 3, mode)
        b = analysis_ld_from(x, 1, 3, hs, gs, mode)
        for p, q in zip(a, b):
            assert np.array_equal(p, q), mode


def _oracle_cases():
    out = [(name, n, j) for name, n, j in (("haar", 4096, 6), ("db4", 4096, 4), ("sym8", 6000, 6), ("db10", 3000, 5),
                                           ("coif3", 3000, 5))]
    try:
        _native.load_library()
        out.append(("coif5", 3000, 5))
    except Exception:
        pass
    return out


@pytest.mark.parametrize("mode", [0, 1, 2], ids=MODE_ID)
@pytest.mark.parametrize("name,n,levels", _oracle_cases())
def test_float64_oracle_and_a_reordered_sum_are_within_the_bound(name, n, levels, mode):
    """the oracle's order and another one (reversed, split in halves, no FMA): the bound does not depend on the order"""
    h, g, _ = filters(name)
    hs, gs = h * S, g * S
    base, x = make_batch(n, n + levels, tiles=(1000, 1024))
    ref = Reference(base, hs, gs, mode, 1, levels, lattice_term(name) if hs.size == 30 else 0.0)
    wo = np.stack([np.stack(cref.decompose(x[r], h, g, levels, mode)[0]) for r in range(len(x))], axis=1)
    vo = np.stack([cref.decompose(x[r], h, g, levels, mode)[1] for r in range(len(x))])
    worst = ref.check(wo, vo, f"oracle {name} {MODE_ID[mode]}", report=False)
    assert worst > 1e-3, worst                      # and the bound is not loose by orders of magnitude
    wr, vr = float_cascade(x, hs, gs, 1, levels, mode, reverse=True)
    ref.check(wr, vr, f"reordered {name} {MODE_ID[mode]}", report=False)


@pytest.mark.parametrize("mode", [0, 1, 2], ids=MODE_ID)
def test_longdouble_reference_agrees_with_exact_fraction_sums(mode):
    """the cascade in Fractions on a short row; the longdouble reference sits inside the bound evaluated with the
    longdouble unit roundoff 2^-64"""
    name, n, levels = "db4", 40, 3
    hs, gs = taps(name)
    x = mixed_row(n, 5 + mode)
    x[0], x[-1] = 1e8, -3e7
    F = fractions.Fraction
    fh, fg = [F(c) for c in hs], [F(c) for c in gs]
    w, v, ew, ev = analysis_ld_from(x, 1, levels, hs, gs, mode, u=2.0 ** -64)
    cur = [F(c) for c in x]
    for j in range(levels):
        d = 1 << j
        idx = _ext_index(n, (hs.size - 1) * d, mode)
        reach = (hs.size - 1) * d
        src = cur + [F(0)]
        nw, nv = [], []
        for t in range(n):
            nw.append(sum((fg[k] * src[idx[reach + t - k * d]] for k in range(hs.size)), F(0)))
            nv.append(sum((fh[k] * src[idx[reach + t - k * d]] for k in range(hs.size)), F(0)))
        for t in range(n):
            assert abs(F(*w[j, t].as_integer_ratio()) - nw[t]) <= F(*ew[j, t].as_integer_ratio()) + F(1, 1 << 80), (j, t)
        cur = nv
    for t in range(n):
        assert abs(F(*v[t].as_integer_ratio()) - cur[t]) <= F(*ev[t].as_integer_ratio()) + F(1, 1 << 80), t


@pytest.mark.parametrize("mode", [0, 1, 2], ids=MODE_ID)
def test_broken_variants_fail_the_bound_where_the_old_tolerance_passes_them(mode):
    """db4 n = 4096 J = 4: a tap off by 1e-13 relative, and 1e-9 of a neighbouring row's W_1 leaked into W_1 of a row
    1e-6 its scale, both pass the batch-wide 1e-12 max|x| of the older tests and fail the bound"""
    name, n, levels = "db4", 4096, 4
    h, g, _ = filters(name)
    hs, gs = h * S, g * S
    big = mixed_row(n, 77)
    small = 1e-6 * mixed_row(n, 78)
    x = np.stack([big, small])
    old_tol = 1e-12 * float(np.max(np.abs(x)))
    rows = [(0, 0), (1, 0)]
    ref = Reference(x, hs, gs, mode, 1, levels)
    good = [cref.decompose(x[r], h, g, levels, mode) for r in range(2)]
    gw = np.stack([np.stack(good[r][0]) for r in range(2)], axis=1)
    gv = np.stack([good[r][1] for r in range(2)])
    ref.check(gw, gv, "oracle", rows, report=False)
    for what, fh, fg in (("low-pass", perturbed(h), g), ("high-pass", h, perturbed(g))):
        bad = [cref.decompose(x[r], fh, fg, levels, mode) for r in range(2)]
        bw = np.stack([np.stack(bad[r][0]) for r in range(2)], axis=1)
        bv = np.stack([bad[r][1] for r in range(2)])
        assert float(max(np.max(np.abs(bw - gw)), np.max(np.abs(bv - gv)))) <= old_tol, what
        fails = ref.failures(bw, bv, rows)
        assert fails, what
        if what == "high-pass":
            assert 1 in fails and 2 in fails, fails            # the high-pass tap shows on W_1 directly
    leak = gw.copy()
    leak[0, 1] += 1e-9 * gw[0, 0]                              # W_1: the big row's details are its noise, not its 1e6
    assert float(np.max(np.abs(leak - gw))) <= old_tol
    assert ref.failures(leak, gv, rows)


# ---- GPU --------------------------------------------------------------------------------------------------------------

@pytest.fixture
def eng():
    e = vw.Engine.get()
    try:
        yield e
    finally:
        for name, value in (("lattice", 15), ("lean", 3), ("tile", 0), ("fuse", 0)):
            e.set_option(name, value)


def _plan(l, levels, n, tile=0, fuse=0):
    """[(first, nlev, kind, hexact)] of the forward plan"""
    out = []
    for line in _native.describe_plan(True, l, levels, n, tile, fuse).splitlines():
        lv, rest = line.split(": ", 1)
        a, b = (int(z) for z in lv.split()[1].split("-"))
        out.append((a, b - a + 1, rest.split()[0], int(rest.split("halo=")[1].split()[0])))
    return out


def _plan_text(plan):
    return " | ".join(f"L{a}-{a + k - 1} {kind}" for a, k, kind, _ in plan)


def _expected_launches(plan, mode, n, flags, levels):
    if flags & _native.FLAG_NO_FUSE:
        return levels
    k = 0
    for _, nl, kind, hexact in plan:
        if kind == "fused":
            k += nl if mode == 2 and n < ((hexact + 1) & ~1) else 1
        elif kind == "column":
            k += 2 if nl == 2 and mode == 2 else 1
        else:
            k += nl
    return k


def _plan_tiles(l, levels, n, tile=0, fuse=0):
    """tile sizes of the plan's groups, and the lean kernels' 1024: where the spike row puts spikes"""
    text = _native.describe_plan(True, l, levels, n, tile, fuse)
    return tuple(sorted({int(line.split("tile=")[1].split()[0]) for line in text.splitlines()} | {1024}))


def _device_rows(x, layout):
    """x as CUDA rows: "plain" contiguous, or "odd": odd row stride and a base address 8 bytes past a 16-byte boundary"""
    import torch
    b, n = x.shape
    if layout == "plain":
        return torch.as_tensor(x, device="cuda")
    ld = n + 1 if n % 2 == 0 else n + 2
    flat = torch.full((1 + b * ld + 8,), -3.5e300, dtype=torch.float64, device="cuda")
    rows = flat[1:1 + b * ld].view(b, ld)[:, :n]
    rows.copy_(torch.as_tensor(x, device="cuda"))
    assert rows.stride(0) % 2 == 1 and rows.data_ptr() % 16 == 8
    return rows


def _forward(eng, xd, hs, gs, levels, mode, flags):
    import torch
    l0 = eng.launch_count()
    w, v = eng.forward(xd, hs, gs, levels, mode, flags)
    k = eng.launch_count() - l0
    torch.cuda.synchronize()
    return w.cpu().numpy(), v.cpu().numpy(), k


def _negative_control(eng, ref, xd, hs, gs, levels, mode, flags, path):
    """the same call with the engine given taps off by 1e-13 (perturbed_pair): some level must fail the bound, W_1 among
    them (its bound is the direct-form one on every path)"""
    w, v, _ = _forward(eng, xd, *perturbed_pair(hs, gs), levels, mode, flags)
    bad = ref.failures(w, v)
    assert bad, f"{path}: a 1e-13 tap error went unnoticed"
    assert 1 in bad or ref.first > 1, (path, bad)
    return bad


FNO = _native.FLAG_NO_FUSE
# (id, wavelet, n, J, engine options, flags, row layout, launches: None = from the default plan).  With the analysis
# pairs off (lattice bit 3 cleared) the planner runs levels 7-8 of sym8 as one tile group, and those of db10 and coif3
# as two single-level launches; with the lattice pairs off every coif5 level is a launch of its own.
CASES = [
    ("db4-4096-J4-lean-tile", "db4", 4096, 4, {}, 0, "plain", None),
    ("haar-20000-J9-tile-groups", "haar", 20000, 9, {}, 0, "plain", None),
    ("db6-20000-J8-tiles-colsingle", "db6", 20000, 8, {}, 0, "plain", None),
    ("db4-9000-J9-tiles-colsingle", "db4", 9000, 9, {}, 0, "plain", None),
    ("sym8-40000-J8-dirpair", "sym8", 40000, 8, {}, 0, "plain", None),
    ("sym8-40000-J8-nopair", "sym8", 40000, 8, {"lattice": 7}, 0, "plain", 4),
    ("db10-40000-J8-dirpair", "db10", 40000, 8, {}, 0, "plain", None),
    ("db10-40000-J8-nopair", "db10", 40000, 8, {"lattice": 7}, 0, "plain", 5),
    ("coif3-40000-J8-singles", "coif3", 40000, 8, {"lattice": 7}, 0, "plain", 5),
    ("coif5-65536-J8-latpair", "coif5", 65536, 8, {"lattice": 15}, 0, "plain", None),
    ("coif5-65536-J8-latsingles", "coif5", 65536, 8, {"lattice": 1}, 0, "plain", 8),
    ("coif5-65536-J8-direct", "coif5", 65536, 8, {"lattice": 0}, 0, "plain", 8),
    ("db4-12345-J4-nontma-oddld-off8", "db4", 12345, 4, {}, 0, "odd", None),
    ("sym8-9001-J6-nontma-oddld-off8", "sym8", 9001, 6, {}, 0, "odd", None),
    ("db4-4096-J4-general-tile", "db4", 4096, 4, {"lean": 0}, 0, "plain", 1),
    ("sym8-40000-J8-general-tile", "sym8", 40000, 8, {"lean": 0}, 0, "plain", None),
    ("db4-4096-J3-tile-eq-htot", "db4", 4096, 3, {"tile": 50}, 0, "plain", None),      # htot of levels 1-3: 50
    ("db6-9000-J6-fuse2-tile3000", "db6", 9000, 6, {"fuse": 2, "tile": 3000}, 0, "plain", None),
    ("haar-20000-J9-fuse6", "haar", 20000, 9, {"fuse": 6}, 0, "plain", None),
    ("db4-4096-J4-nofuse", "db4", 4096, 4, {}, FNO, "plain", None),
    ("coif5-9000-J5-nofuse", "coif5", 9000, 5, {}, FNO, "plain", None),
]


def _case_taps(name):
    if name == "rt14":
        rng = np.random.default_rng(14)
        return rng.standard_normal(14) * 0.3, rng.standard_normal(14) * 0.3
    return taps(name)


CASES.append(("rt14-nonqmf-9000-J5", "rt14", 9000, 5, {}, 0, "plain", None))

_REF = {}


def _reference(name, n, levels, mode, kappa, tiles):
    key = (name, n, levels, mode, kappa, tiles)
    if key not in _REF:
        hs, gs = _case_taps(name)
        base, x = make_batch(n, n + levels, tiles)
        if len(_REF) >= 6:
            _REF.pop(next(iter(_REF)))
        _REF[key] = (x, Reference(base, hs, gs, mode, 1, levels, kappa))
    return _REF[key]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2], ids=MODE_ID)
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_every_analysis_path_within_the_bound(eng, case, mode):
    cid, name, n, levels, opts, flags, layout, launches = case
    hs, gs = _case_taps(name)
    l = hs.size
    plan = _plan(l, levels, n, opts.get("tile", 0), opts.get("fuse", 0))
    tiles = _plan_tiles(l, levels, n, opts.get("tile", 0), opts.get("fuse", 0))
    kappa = lattice_term(name, opts.get("lattice", 15)) if l == 30 and not flags & FNO else 0.0
    x, ref = _reference(name, n, levels, mode, kappa, tiles)
    for k, val in opts.items():
        eng.set_option(k, val)
    xd = _device_rows(x, layout)
    w, v, k = _forward(eng, xd, hs, gs, levels, mode, flags)
    path = f"{cid} {MODE_ID[mode]}: plan {_plan_text(plan)}, {k} launches"
    ref.check(w, v, path)
    expect = launches if launches is not None else _expected_launches(plan, mode, n, flags, levels)
    assert k == expect, (path, expect)
    bad = _negative_control(eng, ref, xd, hs, gs, levels, mode, flags, path)
    print(f"NEGATIVE {cid} {MODE_ID[mode]}: levels outside the bound with a 1e-13 tap error: {sorted(bad)}")


# ---- GPU: SYMMETRIC edges ---------------------------------------------------------------------------------------------

EDGES = [("db2", 4), ("db4", 3), ("haar", 4)]       # J levels in one group from level 1: an odd hexact, htot = hexact + 1


@pytest.mark.gpu
@pytest.mark.parametrize("force_tile", [False, True], ids=["tile-auto", "tile-htot"])
@pytest.mark.parametrize("name,levels", EDGES, ids=[f"{e[0]}-J{e[1]}" for e in EDGES])
def test_symmetric_rows_around_the_halo(eng, name, levels, force_tile):
    """rows of hexact - 1, hexact and htot samples for the group of levels 1..J: the planner drops the group below
    hexact, the SYMMETRIC mirror patch (which needs its sources inside the row and the tile) declines it below htot and
    runs from htot on; with the tile forced to htot, also on a long row of many htot tiles"""
    hs, gs = taps(name)
    l = hs.size
    hexact = (l - 1) * ((1 << levels) - 1)
    htot = hexact + 1
    tile = htot if force_tile else 0
    eng.set_option("tile", tile)
    for n in [hexact - 1, hexact, htot] + ([4096] if force_tile else []):
        plan = _plan(l, levels, n, tile)
        base, x = make_batch(n, n, (htot,))
        ref = Reference(base, hs, gs, 2, 1, levels)
        xd = _device_rows(x, "plain")
        w, v, k = _forward(eng, xd, hs, gs, levels, 2, 0)
        path = f"SYMMETRIC {name} J{levels} n={n} tile={tile or 'auto'}: plan {_plan_text(plan)}, {k} launches"
        ref.check(w, v, path)
        whole = plan[0][1] == levels
        assert whole == (n >= hexact), path                    # the planner keeps the group iff its halo fits the row
        assert k == _expected_launches(plan, 2, n, 0, levels), path
        assert (k == 1) == (n >= htot), path                   # ... and the kernel takes it iff the row holds htot
        _negative_control(eng, ref, xd, hs, gs, levels, 2, 0, path)


# ---- GPU: offset entry points -------------------------------------------------------------------------------------------

# (wavelet, first level, levels, flags, launches): the kernel each group reaches is in the comment
SPANS = [
    ("db4", 1, 1, 0, 1),          # tile kernel, one level
    ("db4", 1, 3, 0, 1),          # tile kernel, three levels
    ("db4", 3, 2, 0, 1),          # tile kernel from dilation 4
    ("db4", 6, 1, 0, 1),          # column single
    ("db6", 7, 1, 0, 1),          # column single
    ("sym8", 6, 2, 0, 1),         # direct-form column pair
    ("db10", 7, 2, 0, 1),         # direct-form column pair
    ("coif5", 3, 2, 0, 1),        # lattice column pair
    ("coif5", 4, 1, 0, 1),        # lattice column single
    ("sym8", 2, 3, FNO, 5),       # per-level kernels: two launches for every level but the last
    ("coif5", 3, 2, FNO, 3),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,first,nlev,flags,launches", SPANS,
                         ids=[f"{s[0]}-L{s[1]}x{s[2]}{'-nofuse' if s[3] else ''}" for s in SPANS])
def test_forward_span_is_the_window_of_the_whole_row(eng, name, first, nlev, flags, launches):
    """[halo | span] rows (LINEAR offset calls, t0 = halo) against the span window of the whole-row reference.  The
    input is exact here, so a 1e-13 tap error must show on the group's first level -- except on a lattice level,
    whose kappa term (5.5e-15 per unit-tap sum) is wider than that error"""
    import torch
    hs, gs = taps(name)
    halo = eng.span_halo(hs.size, first, nlev)
    n_local = 6000 + 2 * halo
    kappa = lattice_term(name) if hs.size == 30 and not flags else 0.0
    base, x = make_batch(halo + n_local, first * 100 + nlev, (halo, 1024))
    ref = Reference(base, hs, gs, 1, first, nlev, kappa, window=halo)
    ws, vs = [], []
    for row in x:
        vin = torch.as_tensor(row, device="cuda")
        l0 = eng.launch_count()
        w, v = eng.forward_span(vin, halo, hs, gs, first, nlev, flags)
        k = eng.launch_count() - l0
        torch.cuda.synchronize()
        assert k == launches, (name, first, nlev, k)
        ws.append(w.cpu().numpy())
        vs.append(v.cpu().numpy())
    path = f"span {name} levels {first}-{first + nlev - 1}{' NO_FUSE' if flags else ''}, {launches} launches"
    ref.check(np.stack(ws, axis=1), np.stack(vs), path)
    w, v = eng.forward_span(torch.as_tensor(x[0], device="cuda"), halo, *perturbed_pair(hs, gs), first, nlev, flags)
    torch.cuda.synchronize()
    bad = ref.failures(w.cpu().numpy()[:, None], v.cpu().numpy()[None], [RECIPE[0]])
    print(f"NEGATIVE {path}: levels outside the bound with a 1e-13 tap error: {sorted(bad)}")
    if not (kappa and first >= LATTICE_FROM):       # a lattice level's bound is wider than a 1e-13 tap error
        assert first in bad, (path, bad)


@pytest.mark.gpu
@pytest.mark.parametrize("name,levels,blocks", [
    ("db4", 6, (3, 1001, 5, 4000, 27, 2964)),
    ("coif5", 4, (3, 777, 3, 2000, 1, 1216)),
    ("haar", 9, (3, 511, 2, 3000, 484)),
])
def test_zero_padding_stream_equals_the_whole_signal_reference(eng, name, levels, blocks):
    """blocks of 3 samples, odd and long ones: a block shorter than a level's halo sends that level to the column
    kernel (dilation >= 4) or the per-level kernel; the concatenated blocks are the whole-signal ZERO_PADDING analysis"""
    n = sum(blocks)
    hs, gs = taps(name)
    base, x = make_batch(n, n + levels, (1024,))
    ref = Reference(base, hs, gs, 1, 1, levels, lattice_term(name) if hs.size == 30 else 0.0)
    st = vw.BatchStreamingMODWT.Builder().wavelet(vw.get_wavelet(name)).boundary(vw.BoundaryMode.ZERO_PADDING) \
        .levels(levels).engine(eng).build()
    ws, vs, at = [], [], 0
    for b in blocks:
        r = st.processMultiLevel(x[:, at:at + b])
        ws.append(np.asarray(r.detailPerLevel()))
        vs.append(np.asarray(r.finalApprox()))
        at += b
    st.close()
    ref.check(np.concatenate(ws, axis=2), np.concatenate(vs, axis=1), f"stream ZERO {name} J{levels} blocks {blocks}")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2], ids=MODE_ID)
@pytest.mark.parametrize("name", ["haar", "db4", "sym8", "coif5"])
def test_forward_varlen_rows_within_the_bound(eng, name, mode):
    hs, gs = taps(name)
    lengths = [1, 2, 7, 4096, 3, 1001, 64, 9000, 5]
    rows = [make_batch(m, 31 * i + m, (1024,)) for i, m in enumerate(lengths)]
    packed = np.concatenate([x.reshape(-1) for _, x in rows])
    offsets = [0]
    for m in lengths:
        for _ in RECIPE:
            offsets.append(offsets[-1] + m)
    import torch
    l0 = eng.launch_count()
    w, v = eng.forward_varlen(torch.as_tensor(packed, device="cuda"), offsets, hs, gs, mode)
    assert eng.launch_count() - l0 == 1                     # every row in one launch
    torch.cuda.synchronize()
    w, v = w.cpu().numpy(), v.cpu().numpy()
    at = 0
    for (base, x), m in zip(rows, lengths):
        ref = Reference(base, hs, gs, mode, 1, 1)
        b = len(RECIPE)
        ref.check(w[at:at + b * m].reshape(1, b, m), v[at:at + b * m].reshape(b, m), f"varlen {name} {MODE_ID[mode]} n={m}")
        at += b * m


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2], ids=MODE_ID)
@pytest.mark.parametrize("name,n,levels", [("db4", 4096, 4), ("sym8", 40000, 8), ("coif5", 65536, 8)])
def test_decompose_resident_rows_within_the_bound(eng, name, n, levels, mode):
    hs, gs = taps(name)
    plan = _plan(hs.size, levels, n)
    x, ref = _reference(name, n, levels, mode, lattice_term(name) if hs.size == 30 else 0.0, _plan_tiles(hs.size, levels, n))
    l0 = eng.launch_count()
    res = eng.decompose_resident(x, hs, gs, levels, mode)
    try:
        k = eng.launch_count() - l0
        assert k == _expected_launches(plan, mode, n, 0, levels), (plan, k)
        assert res.shape() == (len(RECIPE), n, levels)
        w = np.stack([res.get_level(j) for j in range(1, levels + 1)])
        ref.check(w, res.get_level(0), f"resident {name} n={n} J{levels} {MODE_ID[mode]}: plan {_plan_text(plan)}")
    finally:
        res.free()
