"""The statistics kernels behind the denoising API against exact references.

vw_select.cu selects the exact median of |c| per row (radix select on the IEEE bit pattern) for the universal
threshold and scores SURE candidates; vw_generic.cu reduces rows to energy / mean / variance with a fixed tree and
applies thresholds in place.  Order statistics and thresholds are compared bit for bit with the reference's
arithmetic; the reductions are held to forward error bounds of their own tree, checked against sums that are
computed exactly and rounded once.  The CPU tests check the references and show, on a model of the reduction tree,
that the bounds reject a row with one thread partial missing.
"""
import math
from fractions import Fraction

import numpy as np
import pytest

from oracle import cref, nptwin
from oracle.wavelets import filters

gpu = pytest.mark.gpu

U = Fraction(1, 2 ** 53)            # unit roundoff of binary64
ETA = Fraction(1, 2 ** 1074)        # smallest subnormal: at most one per underflowing rounding
THREADS = 512                       # blockDim of k_energy / k_row_moment
S = 1.0 / math.sqrt(2.0)


# ---- exact references ----------------------------------------------------------------------------------------------
def median_abs_ref(row):
    """median of |row| as the reference computes it: Arrays.sort puts NaN last; even n averages the middle pair"""
    a = np.sort(np.abs(np.asarray(row, dtype=np.float64)))
    n = a.size
    return (float(a[n // 2 - 1]) + float(a[n // 2])) / 2.0 if n % 2 == 0 else float(a[n // 2])


def same(a, b):
    """bitwise equality of two doubles, any NaN equal to any NaN (the payload of a NaN median is not specified)"""
    a, b = float(a), float(b)
    if math.isnan(a) or math.isnan(b):
        return math.isnan(a) and math.isnan(b)
    return a == b and math.copysign(1.0, a) == math.copysign(1.0, b)


def to_float(q):
    """round an exact rational once (to nearest even); beyond the largest double -> inf"""
    try:
        return float(q)
    except OverflowError:
        return math.inf if q > 0 else -math.inf


def _split(x):
    c = 134217729.0 * x                 # Veltkamp: 2^27 + 1
    hi = c - (c - x)
    return hi, x - hi


def two_prod(a, b):
    """a * b == p + e exactly (Dekker), provided nothing overflows or underflows"""
    p = a * b
    ah, al = _split(a)
    bh, bl = _split(b)
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def two_sum(a, b):
    """a + b == s + e exactly (Knuth), provided nothing overflows"""
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def _dekker_safe(*arrays):
    """every nonzero magnitude in [2^-480, 2^500]: split products of these neither underflow nor overflow"""
    a = np.abs(np.concatenate([np.ravel(v) for v in arrays]))
    a = a[a != 0]
    return a.size == 0 or (float(a.min()) >= 2.0 ** -480 and float(a.max()) <= 2.0 ** 500)


def exact_sum(a):
    """the exact sum of finite doubles as a Fraction.  Each value is M * 2^(e - 53) with an integer |M| < 2^53; M is cut
    into three 18-bit limbs, and per exponent the limb sums of fewer than 2^35 values stay below 2^53, so the float64
    bincount adds integers without rounding."""
    a = np.asarray(a, dtype=np.float64).ravel()
    assert a.size < 1 << 35 and np.all(np.isfinite(a))
    mant, e = np.frexp(a)
    m = np.ldexp(np.abs(mant), 53).astype(np.int64)
    sign = np.sign(mant)
    e0 = int(e.min()) if a.size else 0
    idx = e - e0
    total = [0] * (int(idx.max()) + 1 if a.size else 0)
    for shift in (0, 18, 36):
        limb = ((m >> shift) & 0x3FFFF).astype(np.float64) * sign
        for k, v in enumerate(np.bincount(idx, weights=limb, minlength=len(total))):
            total[k] += int(v) << shift
    return sum((Fraction(t) * Fraction(2) ** (k + e0 - 53) for k, t in enumerate(total) if t), Fraction(0))


def _fraction_sum(values, f):
    vals, counts = np.unique(values, return_counts=True)
    return sum((f(Fraction(float(v))) * int(c) for v, c in zip(vals, counts)), Fraction(0))


SMALL = 8192   # outside the Dekker range, rows this short (or constant) are summed value by value in Fractions


def exact_sum_sq(x):
    """sum x^2 as an exact Fraction"""
    x = np.asarray(x, dtype=np.float64).ravel()
    if _dekker_safe(x):
        return exact_sum(np.concatenate(two_prod(x, x)))
    assert x.size <= SMALL or np.all(x == x[0])
    return _fraction_sum(x, lambda q: q * q)


def exact_sum_sq_dev(x, m):
    """sum (x - m)^2 as an exact Fraction"""
    x = np.asarray(x, dtype=np.float64).ravel()
    d, r = two_sum(x, -m)               # x - m == d + r;  (d + r)^2 = d^2 + 2dr + r^2
    if _dekker_safe(x, [m], d, r):
        return exact_sum(np.concatenate([*two_prod(d, d), *two_prod(2.0 * d, r), *two_prod(r, r)]))
    assert x.size <= SMALL or np.all(x == x[0])
    mq = Fraction(m)
    return _fraction_sum(x, lambda q: (q - mq) * (q - mq))


# ---- error bounds of the reduction tree -----------------------------------------------------------------------------
# k_energy / k_row_moment: 512 threads, thread t folds x[t], x[t + 512], ... (fma, or one add), then a 5-level shuffle
# tree inside each warp and a 4-level tree over the 16 warp sums.  Every term passes through at most m roundings.
def depth(n):
    return -(-n // THREADS) + 9


def gamma(k):
    return k * U / (1 - k * U)


def energy_ok(got, x):
    """|s^ - s| <= gamma_m * s, plus at most eta / 2 for each of the n fma results that lands in the subnormal range.
    An exact sum beyond the largest double must come back as +inf, as the reference's loop overflows."""
    x = np.asarray(x, dtype=np.float64).ravel()
    s = exact_sum_sq(x)
    if math.isinf(to_float(s)):
        return got == math.inf
    if not math.isfinite(got):
        return False
    return abs(Fraction(got) - s) <= gamma(depth(x.size)) * s + x.size * ETA


def mean_ok(got, x):
    """|m^ - sum x / n| <= gamma_(m+2) * sum|x| / n: the tree, then fl(1/n) and the product"""
    x = np.asarray(x, dtype=np.float64).ravel()
    n = x.size
    if not math.isfinite(got):
        return False
    return abs(Fraction(got) - exact_sum(x) / n) <= gamma(depth(n) + 2) * exact_sum(np.abs(x)) / n + ETA


def variance_ok(got, x, mean):
    """variance about the engine's own mean m^, so that the mean's error stays out: fl(x - m^) enters the fma squared
    (two roundings), then the tree (m) and the scaling (two): gamma_(m+4) * Q / n, plus eta per subnormal rounding"""
    x = np.asarray(x, dtype=np.float64).ravel()
    n = x.size
    q = exact_sum_sq_dev(x, mean)
    if math.isinf(to_float(q)):
        return got == math.inf
    if not math.isfinite(got):
        return False
    return abs(Fraction(got) - q / n) <= gamma(depth(n) + 4) * q / n + (n + 2) * ETA


def tree_model(x, step, drop=None):
    """k_energy / k_row_moment restated: thread t folds x[t], x[t + 512], ... with `step`, each warp sums its lanes with
    shfl_down 16..1, lane 0 of warp 0 sums the 16 warp partials with shfl_down 8..1.  drop: a thread partial to lose."""
    x = np.asarray(x, dtype=np.float64)
    s = np.zeros(THREADS)
    for t0 in range(0, x.size, THREADS):
        c = x[t0:t0 + THREADS]
        s[:c.size] = step(s[:c.size], c)
    if drop is not None:
        s[drop] = 0.0
    warps = s.reshape(THREADS // 32, 32)
    for o in (16, 8, 4, 2, 1):
        warps[:, :32 - o] = warps[:, :32 - o] + warps[:, o:]
    part = np.zeros(32)
    part[:THREADS // 32] = warps[:, 0]
    for o in (8, 4, 2, 1):
        part[:32 - o] = part[:32 - o] + part[o:]
    return float(part[0])


def fma_sq_step(s, c):
    """fma(c, c, s) per lane: the exact c^2 = p + e and s summed once, correctly rounded"""
    p, e = two_prod(c, c)
    return np.array([math.fsum(t) for t in zip(p, e, s)])


# ---- CPU: the references and the power of the assertions ------------------------------------------------------------
def test_exact_sums_agree_with_fractions():
    rng = np.random.default_rng(1)
    for scale in (1.0, 1e-100, 1e100, 1e140):
        for n in (1, 7, 100, 1000):
            x = rng.standard_normal(n) * scale
            assert exact_sum(x) == sum((Fraction(float(v)) for v in x), Fraction(0))
            assert exact_sum_sq(x) == sum((Fraction(float(v)) ** 2 for v in x), Fraction(0))
            m = float(x.mean()) * (1 + 1e-9)
            assert exact_sum_sq_dev(x, m) == sum(((Fraction(float(v)) - Fraction(m)) ** 2 for v in x), Fraction(0))
    sub = np.array([5e-324, -3e-320, 2.0 ** -1022, 1e300, -1e300])         # subnormals and large values sum exactly too
    assert exact_sum(sub) == sum((Fraction(float(v)) for v in sub), Fraction(0))
    # outside the Dekker range: subnormal squares, an overflowing sum
    assert exact_sum_sq(np.full(3, 1e-160)) == 3 * Fraction(1e-160) ** 2 and 0 < to_float(3 * Fraction(1e-160) ** 2) < 2.0 ** -1022
    assert to_float(exact_sum_sq(np.full(2, 1e154))) == math.inf and math.isfinite(to_float(exact_sum_sq(np.full(1, 1e154))))


def test_median_reference_is_java_order():
    rng = np.random.default_rng(2)
    for n in (1, 2, 3, 10, 11):
        x = rng.standard_normal(n)
        x[rng.random(n) < 0.3] = np.nan
        srt = sorted((abs(float(v)) for v in x), key=lambda v: (math.isnan(v), v))   # Double.compare: NaN last
        want = (srt[n // 2 - 1] + srt[n // 2]) / 2.0 if n % 2 == 0 else srt[n // 2]
        assert same(median_abs_ref(x), want)
    w = rng.standard_normal(501)
    assert same(nptwin.universal_threshold(w), median_abs_ref(w) / 0.6745 * math.sqrt(2 * math.log(501)))
    assert same(nptwin.universal_threshold(w), cref.universal_threshold(w))


def test_bounds_accept_the_tree_and_reject_a_dropped_partial():
    rng = np.random.default_rng(3)
    for n in (513, 5000):
        x = rng.standard_normal(n)
        model = tree_model(x, fma_sq_step)
        assert energy_ok(model, x)
        for drop in (0, 31, 32, 511):
            assert not energy_ok(tree_model(x, fma_sq_step, drop), x), (n, drop)
        mean = tree_model(x, lambda s, c: s + c) * (1.0 / n)
        assert mean_ok(mean, x)
        assert not mean_ok(tree_model(x, lambda s, c: s + c, drop=7) * (1.0 / n), x)
        var = tree_model(x - mean, fma_sq_step) * (1.0 / n)
        assert variance_ok(var, x, mean)
        assert not variance_ok(tree_model(x - mean, fma_sq_step, drop=300) * (1.0 / n), x, mean)
        # a relative tolerance of 1e-12 accepts answers the bound rejects
        good = to_float(exact_sum_sq(x))
        bad = good * (1 + 2e-13)
        assert energy_ok(good, x) and bad == pytest.approx(good, rel=1e-12) and not energy_ok(bad, x)


def test_neighbouring_rank_fails_exact_comparison():
    rng = np.random.default_rng(4)
    for row in (last_bit_row(rng), rng.standard_normal(1000)):
        a = np.sort(np.abs(row))
        n = a.size
        want = median_abs_ref(row)
        for lo in (n // 2 - 2, n // 2):                   # the pair one rank below / above
            assert not same((float(a[lo]) + float(a[lo + 1])) / 2.0, want)
    # upper middle rank taken twice on the last-bit row: one ulp off, which a relative tolerance of 1e-14 accepts
    row = last_bit_row(rng)
    wrong = float(np.sort(np.abs(row))[row.size // 2])
    assert wrong == pytest.approx(median_abs_ref(row), rel=1e-14) and not same(wrong, median_abs_ref(row))


# ---- edge rows for the selection -----------------------------------------------------------------------------------
def signs(rng, a):
    return np.where(rng.random(a.size) < 0.5, -a, a)


def cap_of(n):
    return int(min(max(n // 64, 1024), 1 << 20))


def in_bucket(rng, base, k):
    """k keys sharing base's top 24 bits (sign, exponent, top 12 mantissa bits); base has them all clear below"""
    ulp = math.ulp(base)
    return base + ulp * rng.integers(0, 1 << 40, k).astype(np.float64)


def bucket_row(rng, n, k):
    """the median ranks fall among k keys of one 24-bit bucket, [1, 1 + 2^-12)"""
    below = n // 2 - k // 2
    parts = [rng.uniform(0.1, 0.9, below), in_bucket(rng, 1.0, k), rng.uniform(2.0, 3.0, n - below - k)]
    return rng.permutation(signs(rng, np.concatenate(parts)))


def split_bucket_row(rng, n, k, upper):
    """even n; one middle rank alone in [1.5, 1.5 + 2^-12), the other among k keys of its own bucket"""
    if upper:      # rank n/2 - 1 is 1.5, rank n/2 is the smallest key of [2, 2 + 2^-11)
        parts = [rng.uniform(0.1, 0.9, n // 2 - 1), [1.5], in_bucket(rng, 2.0, k), rng.uniform(4.0, 5.0, n // 2 - k)]
    else:          # rank n/2 - 1 is the largest key of [1, 1 + 2^-12), rank n/2 is 1.5
        parts = [rng.uniform(0.1, 0.9, n // 2 - k), in_bucket(rng, 1.0, k), [1.5], rng.uniform(4.0, 5.0, n // 2 - 1)]
    return rng.permutation(signs(rng, np.concatenate(parts)))


def last_bit_row(rng, n=4096):
    """even n; the middle pair a, nextafter(a) share all bits but the last: only the final 8-bit pass splits them"""
    a = 1.0 + 2.0 ** -20
    b = np.nextafter(a, 2.0)
    k = 500
    low = a - math.ulp(1.0) * rng.integers(1, 1 << 30, k)          # same bucket, below a
    high = b + math.ulp(1.0) * rng.integers(1, 1 << 30, k)         # same bucket, above b
    rest = n // 2 - 1 - k
    row = np.concatenate([rng.uniform(0.1, 0.9, rest), low, [a, b], high, rng.uniform(2.0, 3.0, rest)])
    return rng.permutation(signs(rng, row))


def edge_rows():
    rng = np.random.default_rng(20261020)
    nan, inf = math.nan, math.inf
    neg_nan = -np.float64(nan)
    payload_nan = np.array([0x7FF0000000000001, 0xFFF80000000000AB], dtype=np.uint64).view(np.float64)
    sub = np.arange(1, 1000, dtype=np.float64) * 2.0 ** -1074 * rng.integers(1, 1 << 40, 999)
    rows = {
        "n1": [-2.5], "n1_zero": [-0.0], "n1_nan": [nan], "n1_inf": [-inf],
        "n2": [3.0, -1.0], "n3": [0.5, -7.0, 2.0],
        "last_bit": last_bit_row(rng),
        "exponent_buckets": rng.permutation(np.concatenate([rng.uniform(0.1, 0.5, 2047), [0.75, -1.5],
                                                            rng.uniform(2.0, 3.0, 2047)])),
        "nan_fewer_than_half": np.concatenate([rng.standard_normal(701), np.full(200, nan), np.full(50, neg_nan),
                                               np.tile(payload_nan, 25)]),
        "nan_half_even": np.concatenate([rng.standard_normal(500), np.full(500, nan)]),
        "nan_more_than_half": np.concatenate([rng.standard_normal(400), np.full(601, nan)]),
        "inf_below_median": np.concatenate([rng.standard_normal(601), np.full(200, inf), np.full(200, -inf)]),
        "inf_upper_middle": np.concatenate([rng.standard_normal(500), np.full(250, inf), np.full(250, -inf)]),
        "inf_and_nan": np.concatenate([np.full(3, inf), np.full(3, nan), [1.0, -2.0]]),
        "signed_zeros": rng.permutation(np.concatenate([np.full(400, -0.0), np.full(400, 0.0),
                                                        rng.standard_normal(200)])),
        "all_signed_zeros": [-0.0, 0.0, -0.0, 0.0],
        "subnormals": signs(rng, sub),
        "subnormal_pair_rounds_to_even": [0.0, -5e-324],
        "subnormal_and_normal": rng.permutation(np.concatenate([signs(rng, sub[:500]), rng.standard_normal(500)])),
        "middle_pair_overflows": [1e308, -1.7e308],
        "huge_and_tiny": rng.permutation(np.concatenate([rng.standard_normal(300) * 1e300, rng.standard_normal(301) * 1e-300])),
    }
    for n in (4096, 100001, 100002):
        cap = cap_of(n)
        rows[f"bucket_cap_{n}"] = bucket_row(rng, n, cap)
        rows[f"bucket_cap_plus_1_{n}"] = bucket_row(rng, n, cap + 1)
    for n in (4096, 100002):
        cap = cap_of(n)
        rows[f"upper_rank_overflows_{n}"] = split_bucket_row(rng, n, cap + 1, upper=True)
        rows[f"lower_rank_overflows_{n}"] = split_bucket_row(rng, n, cap + 1, upper=False)
        rows[f"upper_rank_at_cap_{n}"] = split_bucket_row(rng, n, cap, upper=True)
    return {k: np.asarray(v, dtype=np.float64) for k, v in rows.items()}


def test_edge_rows_are_what_they_claim():
    rows = edge_rows()
    key = lambda v: np.abs(v).view(np.uint64)            # noqa: E731

    def bucket_count(row, rank):
        k = np.sort(key(row))
        return int(np.sum((k >> 40) == (k[rank] >> 40)))

    for name, row in rows.items():
        n = row.size
        if name.startswith("bucket_cap_plus_1_"):
            assert bucket_count(row, n // 2) == cap_of(n) + 1, name
        elif name.startswith("bucket_cap_"):
            assert bucket_count(row, n // 2) == cap_of(n), name
        elif name.startswith(("upper_rank", "lower_rank")):
            k = cap_of(n) + (0 if "at_cap" in name else 1)
            lo, hi = bucket_count(row, n // 2 - 1), bucket_count(row, n // 2)
            assert (lo, hi) == ((1, k) if name.startswith("upper") else (k, 1)), name
    k = np.sort(key(rows["last_bit"]))
    n = k.size
    assert k[n // 2] - k[n // 2 - 1] == 1 and (k[n // 2] >> 8) == (k[n // 2 - 1] >> 8)
    k = np.sort(key(rows["exponent_buckets"]))
    n = k.size
    assert (k[n // 2] >> 52) != (k[n // 2 - 1] >> 52)


# ---- GPU: median and universal threshold ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng():
    import vectorwave_b200 as vw
    return vw.Engine.get()


EDGE_NAMES = sorted(edge_rows())


@gpu
@pytest.mark.parametrize("name", EDGE_NAMES)
def test_median_and_universal_threshold_edge_rows(eng, name):
    row = edge_rows()[name]
    with np.errstate(over="ignore", invalid="ignore"):          # inf and NaN medians are expected results here
        want = nptwin.universal_threshold(row)
    assert same(eng.median_abs(row), median_abs_ref(row)), name
    assert same(eng.universal_threshold(row), want), name


@gpu
def test_median_mixed_batch_in_one_call(eng):
    rng = np.random.default_rng(5)
    n = 4096
    cap = cap_of(n)
    rows = [rng.standard_normal(n), bucket_row(rng, n, cap), bucket_row(rng, n, cap + 1),
            split_bucket_row(rng, n, cap + 1, upper=True), split_bucket_row(rng, n, cap + 1, upper=False),
            last_bit_row(rng, n), np.full(n, -1.25), rng.standard_normal(n) * 1e-200, np.repeat(rng.standard_normal(4), n // 4),
            np.where(rng.random(n) < 0.3, np.nan, rng.standard_normal(n)), rng.standard_normal(n)]
    x = np.stack(rows)
    med = eng.median_abs(x)
    thr = eng.universal_threshold(x)
    for i, row in enumerate(rows):
        assert same(med[i], median_abs_ref(row)), i
        assert same(thr[i], nptwin.universal_threshold(row)), i


def _layouts(x):
    """the same rows as host pageable, host strided (ld > n), device contiguous, device strided"""
    import torch
    b, n = x.shape
    wide = np.full((b, n + 37), np.nan)
    wide[:, 5:5 + n] = x
    dwide = torch.as_tensor(wide, device="cuda")
    return {"host": x, "host_strided": wide[:, 5:5 + n], "device": torch.as_tensor(x, device="cuda"),
            "device_strided": dwide[:, 5:5 + n]}


@gpu
def test_median_on_every_layout(eng):
    rng = np.random.default_rng(6)
    n = 3001
    x = np.stack([rng.standard_normal(n), bucket_row(rng, n, cap_of(n) + 1), np.full(n, 0.3),
                  rng.standard_normal(n) * 1e5, bucket_row(rng, n, cap_of(n))])
    for layout, v in _layouts(x).items():
        assert tuple(v.shape) == x.shape
        med = eng.median_abs(v)
        thr = eng.universal_threshold(v)
        for i in range(x.shape[0]):
            assert same(med[i], median_abs_ref(x[i])), (layout, i)
            assert same(thr[i], nptwin.universal_threshold(x[i])), (layout, i)


# ---- GPU: more rows than one grid dimension ------------------------------------------------------------------------
BIG_B, BIG_N = 70000, 64


def _check_rows(b):
    """the rows either side of the 32768 (grid loop) and 65535 (gridDim.y) boundaries, the last row, a seeded sample"""
    fixed = [0, 32767, 32768, 65534, 65535, 65536, b - 1]
    return sorted(set(fixed) | set(np.random.default_rng(7).choice(b, 200, replace=False).tolist()))


@pytest.fixture(scope="module")
def big():
    rng = np.random.default_rng(8)
    x = rng.standard_normal((BIG_B, BIG_N)) * rng.uniform(0.1, 10.0, (BIG_B, 1))
    x[32768] = np.repeat([0.5, -2.0, 3.0, -0.5], BIG_N // 4)        # ties
    x[65535] = 1.0 + 2.0 ** -52 * np.arange(BIG_N)                # one bucket, differences in the last bits
    x[65536, ::2] *= 1e-3
    return x


@gpu
def test_median_universal_threshold_beyond_one_grid_dimension(eng, big):
    med = eng.median_abs(big)
    thr = eng.universal_threshold(big)
    for i in _check_rows(BIG_B):
        assert same(med[i], median_abs_ref(big[i])), i
        assert same(thr[i], nptwin.universal_threshold(big[i])), i


@gpu
def test_swt_denoise_beyond_one_grid_dimension(eng, big):
    name, levels, mode = "db4", 3, 0
    h, g, wid = filters(name)
    import torch
    den, thr = eng.denoise(big, h * S, g * S, levels, mode, threshold=-1.0, soft=True)
    # the engine's own W_1 (same plan, same kernels as inside the denoise): its selected threshold must be exact.  Against
    # the oracle's W_1 the median is only as close as the coefficients, which can be cancellation residue (the piecewise
    # constant row 32768 has |W_1| ~ 1e-11 away from its jumps), so there the bound is the 1e-12 * max|x| of the
    # transform, carried through the 1-Lipschitz order statistic and the factor sqrt(2 ln n) / 0.6745
    w1 = eng.forward(torch.as_tensor(big, device="cuda"), h * S, g * S, levels, mode)[0][0].cpu().numpy()
    factor = math.sqrt(2.0 * math.log(BIG_N)) / 0.6745
    for i in _check_rows(BIG_B):
        tol = 1e-12 * float(np.max(np.abs(big[i])))
        assert same(thr[i], nptwin.universal_threshold(w1[i])), i
        _, tref = cref.swt_denoise(big[i], h, g, levels, mode, wid, -1.0, True)
        assert abs(thr[i] - tref) <= tol * factor, i
        ref, _ = cref.swt_denoise(big[i], h, g, levels, mode, wid, float(thr[i]), True)   # the oracle at that threshold
        assert float(np.max(np.abs(den[i] - ref))) <= tol, i


@gpu
def test_resident_thresholds_beyond_one_grid_dimension(eng, big):
    name, levels, mode = "db4", 3, 0
    h, g, _ = filters(name)
    res = eng.decompose_resident(big, h * S, g * S, levels, mode)
    try:
        w = [res.get_level(j) for j in range(1, levels + 1)]
        rows = _check_rows(BIG_B)
        for j in range(1, levels + 1):
            e = res.energy(j)
            for i in rows:
                assert energy_ok(e[i], w[j - 1][i]), (j, i)
        thr = res.universal_threshold(True)
        for i in rows:
            assert same(thr[i], nptwin.universal_threshold(w[0][i])), i
        for j in range(1, levels + 1):
            got = res.get_level(j)
            assert np.array_equal(got.view(np.uint64), nptwin.threshold(w[j - 1], thr[:, None], True).view(np.uint64)), j
        # per-row host thresholds on one level: every row, bit for bit
        per_row = np.abs(np.random.default_rng(9).standard_normal(BIG_B))
        before = res.get_level(2)
        res.threshold(2, per_row, False)
        assert np.array_equal(res.get_level(2).view(np.uint64), nptwin.threshold(before, per_row[:, None], False).view(np.uint64))
    finally:
        res.free()


@gpu
def test_sure_threshold_energy_mean_variance_beyond_one_grid_dimension(eng, big):
    rows = _check_rows(BIG_B)
    sigma = np.array([nptwin.denoiser_sigma(r) for r in big])
    thr, risk = eng.sure_threshold(big, sigma, with_risk=True)
    for i in rows:
        assert (thr[i], risk[i]) == nptwin.sure_threshold(big[i], float(sigma[i])), i
    e = eng.energy(big)
    m, v = eng.mean_variance(big)
    for i in rows:
        assert energy_ok(e[i], big[i]), i
        assert mean_ok(m[i], big[i]), i
        assert variance_ok(v[i], big[i], m[i]), i


@gpu
def test_threshold_per_row_beyond_one_grid_dimension(eng, big):
    import torch
    per_row = np.abs(np.random.default_rng(10).standard_normal(BIG_B))
    for soft in (True, False):
        want = nptwin.threshold(big, per_row[:, None], soft).view(np.uint64)
        c = big.copy()
        eng.threshold(c, per_row, soft)
        assert np.array_equal(c.view(np.uint64), want), soft
        cd = torch.as_tensor(big, device="cuda")
        eng.threshold(cd, per_row, soft)
        assert np.array_equal(cd.cpu().numpy().view(np.uint64), want), soft


# ---- GPU: energy, mean and variance against the bounds -------------------------------------------------------------
@gpu
@pytest.mark.parametrize("n", [1, 2, 3, 100, 511, 512, 513, 1000, 4096, 5000, 65537, 1 << 20, 1 << 24])
def test_energy_mean_variance_within_bounds(eng, n):
    rng = np.random.default_rng(n)
    x = rng.standard_normal((2, n)) * np.array([[1e-3], [1.0]]) + np.array([[3.0], [0.0]])
    e = eng.energy(x)
    m, v = eng.mean_variance(x)
    for i in range(1 if n > 1 << 20 else 2):                  # the exact references of a 2^24 row take seconds
        assert energy_ok(e[i], x[i]), (n, i)
        assert mean_ok(m[i], x[i]), (n, i)
        assert variance_ok(v[i], x[i], m[i]), (n, i)


def _special_rows():
    rng = np.random.default_rng(11)
    return {
        "huge": rng.standard_normal(4096) * 1e150,
        "energy_overflows": np.full(4096, 1e154),
        "energy_overflows_mixed": np.concatenate([rng.standard_normal(3000), [1e154, -1e154], rng.standard_normal(1000)]),
        "subnormal_squares": rng.standard_normal(4096) * 1e-160,
        "subnormal_squares_long": np.full(1 << 20, -1e-160),
        "offset": 1e8 + rng.standard_normal(100000),
        "constant": np.full(100003, 0.1),
        "constant_short": np.full(777, -3.3),
        "zeros": np.zeros(1000),
    }


@gpu
@pytest.mark.parametrize("name", sorted(_special_rows()))
def test_energy_mean_variance_special_rows(eng, name):
    x = _special_rows()[name]
    e = eng.energy(x)
    assert energy_ok(e, x), name
    m, v = eng.mean_variance(x)
    assert mean_ok(m, x), name
    assert variance_ok(v, x, m), name
    if name == "offset":                              # two passes: the variance about the mean stays near 1
        assert abs(v - float(np.var(x))) <= 1e-9


@gpu
def test_reductions_are_deterministic_and_layout_independent(eng):
    rng = np.random.default_rng(12)
    n = 100003
    x = rng.standard_normal((4, n)) * np.array([[1.0], [1e-5], [1e5], [1.0]]) + np.array([[0.0], [0.0], [0.0], [1e6]])
    ref_e = eng.energy(x)
    ref_m, ref_v = eng.mean_variance(x)
    for i in range(4):
        assert energy_ok(ref_e[i], x[i]) and mean_ok(ref_m[i], x[i]) and variance_ok(ref_v[i], x[i], ref_m[i]), i
    for layout, view in _layouts(x).items():
        for _ in range(2):
            e = eng.energy(view)
            m, v = eng.mean_variance(view)
            assert np.array_equal(e.view(np.uint64), ref_e.view(np.uint64)), layout
            assert np.array_equal(m.view(np.uint64), ref_m.view(np.uint64)), layout
            assert np.array_equal(v.view(np.uint64), ref_v.view(np.uint64)), layout


# ---- GPU: threshold ------------------------------------------------------------------------------------------------
def _threshold_rows():
    rng = np.random.default_rng(13)
    t = 0.75
    edge = np.array([t, -t, np.nextafter(t, 0), -np.nextafter(t, 2), 0.0, -0.0, np.nan, -np.float64(np.nan),
                     np.inf, -np.inf, 5e-324, -5e-324, 1e308, -1e-308])
    rows = np.stack([rng.permutation(np.concatenate([edge, rng.standard_normal(2000 - edge.size)])) for _ in range(5)])
    rows[3, :edge.size] = edge * 0.0              # a row of signed zeros (and NaN) for t = 0
    return rows, np.array([t, 0.0, t, 0.0, np.inf])


def _writable_layouts(x):
    """(layout, rows to threshold in place, the whole buffer when the rows are a strided view of it)"""
    import torch
    b, n = x.shape
    wide = np.full((b, n + 37), np.nan)
    wide[:, 5:5 + n] = x
    dwide = torch.as_tensor(wide, device="cuda")
    return [("host", x.copy(), None), ("host_strided", wide[:, 5:5 + n], wide),
            ("device", torch.as_tensor(x, device="cuda"), None), ("device_strided", dwide[:, 5:5 + n], dwide)]


@gpu
@pytest.mark.parametrize("soft", [True, False])
def test_threshold_bitwise_on_edge_values(eng, soft):
    x, per_row = _threshold_rows()
    n = x.shape[1]
    for thr in (per_row, 0.75, 0.0):
        want = nptwin.threshold(x, thr[:, None] if np.ndim(thr) else thr, soft).view(np.uint64)
        for layout, c, buf in _writable_layouts(x):
            eng.threshold(c, thr, soft)
            got = c.cpu().numpy() if hasattr(c, "cpu") else c
            assert np.array_equal(np.ascontiguousarray(got).view(np.uint64), want), (layout, np.ndim(thr))
            if buf is not None:                                              # the gaps between rows are untouched
                w = buf.cpu().numpy() if hasattr(buf, "cpu") else buf
                assert np.all(np.isnan(w[:, :5])) and np.all(np.isnan(w[:, 5 + n:])), layout
