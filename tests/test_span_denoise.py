"""SWT denoise of one span-sharded long signal: the exact cross-rank median and the thresholded span synthesis.

CPU.  `np_span_median` restates the round protocol of the vw_span_median_* calls over `world` split arrays: seven digit
rounds on the bit pattern of |c| (two 12-bit rounds over the full spans, a rank-local candidate compaction before round 2,
five 8-bit rounds over the candidates or, where a rank's candidates overflowed, over its full span), every rank's
histogram summed before the pick.  It must give np.partition's median bit for bit on odd and even lengths, ties, +-0,
subnormals, 2^+-300 scales, middle order statistics in different ranks, one rank overflowing its candidates, and
world in {1, 2, 3, 8}.  A world-2 gloo run drives `SpanShardedMODWT.denoise` with a numpy stand-in engine.

GPU (one device).  Every rank runs on one context, the exchanges and the histogram sums done on the host: the threshold
equals, bit for bit, numpy's median-based threshold of the W_1 spans the device wrote; each rank's
`inverse_span_all_thr` output is within the extended-precision bound (`test_span_paths.synth_ld_from`) of the synthesis
of the gathered W / V thresholded with that value, on every synthesis path, with W and V untouched and nothing written
past xout[n_local]; `vw_swt_denoise_sharded` on device 0 repeated gives the same bits; the whole-signal `vw_swt_denoise`
agrees; error cases leave the objects usable.
"""
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import cref
from oracle.wavelets import filters
from vectorwave_b200 import BoundaryMode, _native, get_wavelet
from vectorwave_b200.errors import IllegalArgumentException, InvalidArgumentException, InvalidSignalException
from vectorwave_b200.sharded import SpanShardedMODWT

from test_dist_gloo import NumpySpanEngine
from test_span_paths import (FBX, FNO, MODE_ID, SENTINEL, Worst, _bits, _groups, _lattice_in_plan, _sync,
                             inverse_span_kernel, span_signal, synth_ld_from)
from test_synthesis_paths import lattice_kappa, taps

ROUNDS = 7
BIG = 12


# ---- the round protocol in numpy ---------------------------------------------------------------------------------------

def span_cap(n_local):
    return int(min(max(n_local // 64, 1024), 1 << 20))


def round_bits(rnd):
    return BIG if rnd < 2 else 8


def round_shift(rnd):
    return 64 - BIG * (rnd + 1) if rnd < 2 else 64 - 2 * BIG - 8 * (rnd - 1)


def _keys(c):
    return np.abs(np.asarray(c, dtype=np.float64)).view(np.uint64)


class NpSpanState:
    """one rank's state: the two tracked prefixes / remaining ranks and the rank-local candidate buffers"""

    def __init__(self, n_total, cap):
        self.n_total, self.cap = int(n_total), int(cap)
        self.prefix = [0, 0]
        self.rank = [(n_total - 1) // 2 if n_total % 2 == 0 else n_total // 2, n_total // 2]
        self.cand, self.count = [None, None], [0, 0]

    def hist(self, c, rnd):
        bits, shift = round_bits(rnd), round_shift(rnd)
        keys = _keys(c)
        if rnd == 2:                                   # compaction of the keys sharing the 24 decided bits
            for which in (0, 1):
                sel = keys[(keys >> np.uint64(40)) == np.uint64(self.prefix[which])]
                self.count[which] = sel.size
                self.cand[which] = sel[:self.cap]
        use_cand = rnd >= 2 and self.count[0] <= self.cap and self.count[1] <= self.cap
        out = np.zeros(2 << bits, dtype=np.uint64)
        for which in (0, 1):
            src = self.cand[which] if use_cand else keys
            hi = src >> np.uint64(shift + bits) if shift + bits < 64 else np.zeros_like(src)
            dg = (src >> np.uint64(shift)) & np.uint64((1 << bits) - 1)
            out[which << bits:(which + 1) << bits] = np.bincount(dg[hi == np.uint64(self.prefix[which])].astype(np.int64),
                                                                minlength=1 << bits).astype(np.uint64)
        return out

    def pick(self, rnd, hist_sum):
        bits = round_bits(rnd)
        for which in (0, 1):
            h = hist_sum[which << bits:(which + 1) << bits].astype(np.int64)
            cum = np.cumsum(h)
            b = int(np.searchsorted(cum, self.rank[which], side="right"))
            self.rank[which] -= int(cum[b - 1]) if b > 0 else 0
            self.prefix[which] = (self.prefix[which] << bits) | b

    def value(self, factor):
        lo, hi = (np.array([p], dtype=np.uint64).view(np.float64)[0] for p in self.prefix)
        med = (lo + hi) / 2.0 if self.n_total % 2 == 0 else hi
        return med if factor < 0 else (med / 0.6745) * factor


def np_span_median(spans, cap=None, states=None):
    """the raw median of |concat(spans)| by the round protocol; `states` (optional list) receives the rank states"""
    n_total = sum(int(np.asarray(s).size) for s in spans)
    st = [NpSpanState(n_total, cap if cap is not None else span_cap(np.asarray(s).size)) for s in spans]
    for rnd in range(ROUNDS):
        total = sum(s.hist(c, rnd) for s, c in zip(st, spans))
        for s in st:
            s.pick(rnd, total)
    if states is not None:
        states.extend(st)
    vals = {float(s.value(-1.0)) for s in st}
    assert len(vals) == 1 or all(math.isnan(v) for v in vals)
    return st[0].value(-1.0)


def np_median_abs(c):
    a = np.abs(np.asarray(c, dtype=np.float64))
    n = a.size
    p = np.partition(a, [(n - 1) // 2, n // 2])
    return (p[(n - 1) // 2] + p[n // 2]) / 2.0 if n % 2 == 0 else p[n // 2]


def universal(med, n_total):
    return (med / 0.6745) * math.sqrt(2.0 * math.log(float(n_total)))


def np_threshold(c, lam, soft):
    """vw_threshold_nonneg (lam >= 0) in float64"""
    a = np.abs(c)
    if soft:
        return np.where(a > lam, np.copysign(a - lam, c), 0.0)
    return np.where(a <= lam, 0.0, c)


def _same(a, b):
    return np.asarray(a, dtype=np.float64).view(np.int64) == np.asarray(b, dtype=np.float64).view(np.int64)


def _protocol_cases():
    rng = np.random.default_rng(11)
    cases = []
    for world in (1, 2, 3, 8):
        for n_total in (8 * 3 * 97, 8 * 3 * 97 + 1):          # even and odd
            x = rng.standard_normal(n_total)
            cases.append((f"normal-w{world}-n{n_total}", np.array_split(x, world), None))
    x = np.round(rng.standard_normal(5001) * 3.0)              # ties everywhere, +-0 among them
    x[::7] = -0.0
    cases.append(("ties-w3", np.array_split(x, 3), None))
    for world in (2, 3, 8):
        spans = [rng.standard_normal(300 + 7 * r) for r in range(world)]
        spans[1] = np.full(400 * world, 0.015625)             # a constant span holding the median: it alone overflows
        cases.append((f"constant-overflow-w{world}", spans, 16))
    sub = np.ldexp(rng.standard_normal(2000), -1060)           # subnormals
    big = np.ldexp(rng.standard_normal(2000), 300)
    small = np.ldexp(rng.standard_normal(2000), -300)
    cases.append(("subnormal-w2", [sub[:1000], sub[1000:]], None))
    cases.append(("scales-w3", [big, small, np.concatenate([sub[:999], [0.0, -0.0]])], None))
    # the two middle order statistics in different ranks: rank 0 holds the lower half, rank 1 the upper half
    v = np.sort(np.abs(rng.standard_normal(4000)))
    cases.append(("middle-split-w2", [-v[:2000], v[2000:]], None))
    cases.append(("middle-split-w8", [v[i::8][::-1] for i in range(8)], None))
    cases.append(("zeros-w8", [np.zeros(17) for _ in range(8)], 4))
    return cases


PROTO = _protocol_cases()


@pytest.mark.parametrize("case", PROTO, ids=[c[0] for c in PROTO])
def test_round_protocol_is_the_exact_median(case):
    _, spans, cap = case
    states = []
    got = np_span_median(spans, cap, states)
    whole = np.concatenate(spans)
    exp = np_median_abs(whole)
    assert _same(got, exp), (got, exp)
    if cap is not None and "overflow" in case[0]:
        over = [max(s.count) > s.cap for s in states]
        assert over[1] and not all(over), over            # rank 1 overflowed its candidates, some rank did not
    n = whole.size
    assert _same(universal(got, n), universal(exp, n))


def test_protocol_constants_match_the_library():
    lib = _native.load_library()
    assert _native.SPAN_MEDIAN_ROUNDS == ROUNDS
    for rnd in range(ROUNDS):
        assert lib.vw_span_median_bins(rnd) == 2 << round_bits(rnd) == _native.span_median_bins(rnd)
    assert lib.vw_span_median_bins(-1) == 0 and lib.vw_span_median_bins(ROUNDS) == 0
    # the digits cover the 64 key bits exactly once, most significant first
    assert [round_shift(r) for r in range(ROUNDS)] == [52, 40, 32, 24, 16, 8, 0]
    assert sum(round_bits(r) for r in range(ROUNDS)) == 64
    for n in (1, 64 * 1024, 64 * 4096 + 5, 1 << 27):
        assert lib.vw_span_median_state_bytes(n) == 256 + 16 * span_cap(n)
    assert lib.vw_span_median_state_bytes(0) == 0


# ---- the facade over gloo with a numpy stand-in engine --------------------------------------------------------------

class NumpyDenoiseEngine(NumpySpanEngine):
    """NumpySpanEngine plus the median rounds (NpSpanState) and the thresholded span synthesis"""

    def span_median_state(self, n_local):
        return {"n_local": int(n_local)}

    def span_median_init(self, state, n_total):
        state["st"] = NpSpanState(n_total, span_cap(state["n_local"]))

    def span_median_hist(self, state, c, rnd, hist):
        hist.copy_(torch.from_numpy(state["st"].hist(c.numpy(), rnd).astype(np.int64)))

    def span_median_pick(self, state, rnd, hist_sum):
        state["st"].pick(rnd, hist_sum.numpy().astype(np.uint64))

    def span_median_value(self, state, factor, out):
        out[0] = float(state["st"].value(factor))

    def inverse_span_all_thr(self, plan, w, v, hs, gs, order, thr, soft, out, flags=0):
        wt = torch.from_numpy(np_threshold(w.numpy(), float(thr[0]), soft))
        self.inverse_span_all(plan, wt, v, hs, gs, order, out, flags)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, name, n_total, levels, mode_value, threshold, soft, poison, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        x = np.random.default_rng(17).standard_normal(n_total) + np.sin(np.arange(n_total) / 50.0) * 4.0
        nl = n_total // world
        part = x[rank * nl:(rank + 1) * nl].copy()
        if poison and rank == 1:
            part[5] = np.nan
        sh = SpanShardedMODWT(get_wavelet(name), levels, nl, BoundaryMode(mode_value), engine=NumpyDenoiseEngine())
        try:
            out, lam = sh.denoise(torch.from_numpy(part), threshold=threshold, soft=soft)
        except InvalidSignalException:
            ret[rank] = "nonfinite"
        else:
            res = sh.forward(torch.from_numpy(part))
            ret[rank] = (out.numpy().copy(), lam, res.details()[0].numpy().copy())
        dist.barrier()
    finally:
        dist.destroy_process_group()


def _run_world2(*args):
    port = _free_port()
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, port) + args + (ret,), nprocs=2, join=True)
    return ret


@pytest.mark.parametrize("threshold,soft", [(-1.0, True), (-1.0, False), (0.75, True)], ids=["universal-soft", "universal-hard", "fixed"])
@pytest.mark.parametrize("mode", [BoundaryMode.PERIODIC, BoundaryMode.ZERO_PADDING])
def test_facade_two_ranks_equals_the_unsharded_denoise(mode, threshold, soft):
    name, n_total, levels = "sym8", 4096, 4
    ret = _run_world2(name, n_total, levels, mode.value, threshold, soft, False)
    h, g, wid = filters(name)
    x = np.random.default_rng(17).standard_normal(n_total) + np.sin(np.arange(n_total) / 50.0) * 4.0
    w1 = np.concatenate([ret[r][2] for r in range(2)])
    lam = ret[0][1]
    assert ret[1][1] == lam
    if threshold < 0:
        assert _same(lam, universal(np_median_abs(w1), n_total))      # from the W_1 spans the ranks hold
    else:
        assert lam == threshold
    wo, vo = cref.decompose(x, h, g, levels, mode.value)
    lam_ref = universal(np_median_abs(wo[0]), n_total) if threshold < 0 else threshold
    assert abs(lam - lam_ref) <= 1e-12 * lam_ref
    ref = cref.reconstruct(np_threshold(wo, lam, soft), vo, h, g, mode.value, wid)
    np.testing.assert_allclose(np.concatenate([ret[r][0] for r in range(2)]), ref, rtol=0, atol=1e-11)


def test_facade_rejects_a_nonfinite_span_on_every_rank():
    ret = _run_world2("db4", 2048, 3, BoundaryMode.PERIODIC.value, -1.0, True, True)
    assert ret[0] == "nonfinite" and ret[1] == "nonfinite"


def test_facade_single_rank_and_per_group_schedule():
    x = np.random.default_rng(3).standard_normal(2048)
    sh = SpanShardedMODWT(get_wavelet("db4"), 4, 2048, BoundaryMode.PERIODIC, engine=NumpyDenoiseEngine(), rank=0, world=1)
    out, lam = sh.denoise(torch.from_numpy(x.copy()))
    h, g, wid = filters("db4")
    ref, used = cref.swt_denoise(x, h, g, 4, 0, wid, -1.0, True)
    assert abs(lam - used) <= 1e-13 * used
    np.testing.assert_allclose(out.numpy(), ref, rtol=0, atol=1e-11)
    per_group = SpanShardedMODWT(get_wavelet("db4"), 4, 2048, BoundaryMode.PERIODIC, engine=NumpyDenoiseEngine(), rank=0,
                                 world=1, upfront=False)
    with pytest.raises(IllegalArgumentException):
        per_group.denoise(torch.from_numpy(x.copy()))
    chosen = SpanShardedMODWT(get_wavelet("db4"), 4, 2048, BoundaryMode.PERIODIC, engine=NumpyDenoiseEngine(), rank=0,
                              world=1, groups_forward=[(1, 4)], groups_inverse=[(1, 4)])
    with pytest.raises(IllegalArgumentException):
        chosen.denoise(torch.from_numpy(x.copy()))


# ---- GPU: rank by rank on one context -------------------------------------------------------------------------------

# (wavelet, J, world, n_local): haar / db4 / sym8 / coif5 over 2, 3 and 8 ranks
DEN_SHAPES = [
    ("haar", 6, 8, 4096),
    ("db4", 5, 3, 256),
    ("sym8", 7, 3, 8192),
    ("coif5", 6, 2, 32768),
    ("coif5", 5, 8, 4096),
]
DEN_ID = [f"{s[0]}-J{s[1]}-w{s[2]}-n{s[3]}" for s in DEN_SHAPES]
SIGNALS = ["mixed", "constant"]


@pytest.fixture
def eng():
    import vectorwave_b200 as vw
    e = vw.Engine.get()
    try:
        yield e
    finally:
        e.set_option("lattice", 15)


def _signal(shape, plan, kind):
    name, levels, world, n_local = shape
    x = span_signal(n_local, world, int(plan.lead), int(plan.pad), n_local + levels + world)
    if kind == "constant":
        x[(world - 1) * n_local:] = 3.0                 # the last span constant: W_1 ~ 0 there, ties galore
    return x


def _forward_ranks(eng, shape, mode, x, plan):
    """forward_span_all of every rank with the host-side analysis exchange, then the synthesis exchange (pack / unpack):
    device (W rows, V) per rank, pads filled"""
    name, levels, world, n_local = shape
    hs, gs = taps(name)
    lead, lead_w, pad = int(plan.lead), int(plan.lead_w), int(plan.pad)
    row = lead_w + n_local + pad
    ws, vs = [], []
    for r in range(world):
        left = (r - 1) % world
        lead_part = np.zeros(lead) if (mode == 1 and r == 0) else x[(left + 1) * n_local - lead:(left + 1) * n_local]
        xext = torch.as_tensor(np.concatenate([lead_part, x[r * n_local:(r + 1) * n_local]]), device="cuda")
        w = torch.full((levels, row), float("nan"), dtype=torch.float64, device="cuda")
        v = torch.full((n_local + pad,), float("nan"), dtype=torch.float64, device="cuda")
        eng.forward_span_all(xext, plan, hs, gs, w, v)
        ws.append(w)
        vs.append(v)
    msgs = []
    for r in range(world):
        msg = torch.empty(int(plan.inverse_msg), dtype=torch.float64, device="cuda")
        eng.span_pack_inverse(plan, ws[r], vs[r], msg)
        msgs.append(msg)
    for r in range(world):
        eng.span_unpack_inverse(plan, None if (mode == 1 and r == world - 1) else msgs[(r + 1) % world], ws[r], vs[r])
    _sync()
    return ws, vs


def _device_threshold(eng, plan, ws, n_total):
    """the seven rounds with the histograms summed on the host; returns every rank's threshold and raw median"""
    n_local, lead_w = int(plan.n_local), int(plan.lead_w)
    world = len(ws)
    states = [eng.span_median_state(n_local) for _ in range(world)]
    for st in states:
        eng.span_median_init(st, n_total)
    for rnd in range(ROUNDS):
        hists = [torch.empty(_native.span_median_bins(rnd), dtype=torch.int64, device="cuda") for _ in range(world)]
        for r in range(world):
            eng.span_median_hist(states[r], ws[r][0, lead_w:lead_w + n_local], rnd, hists[r])
        total = sum(h.cpu() for h in hists).cuda()
        for r in range(world):
            eng.span_median_pick(states[r], rnd, total)
    thr = torch.empty(world, dtype=torch.float64, device="cuda")
    med = torch.empty(world, dtype=torch.float64, device="cuda")
    factor = math.sqrt(2.0 * math.log(float(n_total)))
    for r in range(world):
        eng.span_median_value(states[r], factor, thr[r:r + 1])
        eng.span_median_value(states[r], -1.0, med[r:r + 1])
    _sync()
    return thr.cpu().numpy(), med.cpu().numpy()


def _gather(plan, ws, vs):
    n_local, lead_w = int(plan.n_local), int(plan.lead_w)
    return (np.concatenate([w.cpu().numpy()[:, lead_w:lead_w + n_local] for w in ws], axis=1),
            np.concatenate([v.cpu().numpy()[:n_local] for v in vs]))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", SIGNALS)
@pytest.mark.parametrize("mode", [0, 1], ids=MODE_ID)
@pytest.mark.parametrize("shape", DEN_SHAPES, ids=DEN_ID)
def test_threshold_rank_by_rank_is_numpys(eng, shape, mode, kind):
    name, levels, world, n_local = shape
    hs, _ = taps(name)
    plan = _native.span_plan(hs.size, levels, n_local, world)
    x = _signal(shape, plan, kind)
    ws, vs = _forward_ranks(eng, shape, mode, x, plan)
    wg, _ = _gather(plan, ws, vs)
    n_total = n_local * world
    thr, med = _device_threshold(eng, plan, ws, n_total)
    exp_med = np_median_abs(wg[0])
    assert np.all(_same(med, exp_med)), (med, exp_med)
    assert np.all(_same(thr, universal(exp_med, n_total))), (thr, universal(exp_med, n_total))
    print(f"THRESHOLD {name} J{levels} w{world} {MODE_ID[mode]} {kind}: median {exp_med!r} bit for bit on every rank")


# (shape index, flags, lattice option, soft, universal?) -- the synthesis paths the plans reach: lean / general tile
# (haar, db4, sym8), direct-form pairs (sym8 J = 7), lattice pairs and singles (coif5), per-level under NO_FUSE / BITEXACT
OUT_CASES = [
    (0, 0, 15, True, True), (0, FNO, 15, False, True),
    (1, 0, 15, True, True), (1, FBX, 15, True, False),
    (2, 0, 15, True, True), (2, 0, 15, False, False), (2, FNO, 15, True, True), (2, FBX, 15, False, True),
    (3, 0, 15, True, True), (3, 0, 15, False, True), (3, 0, 0, True, False), (3, FNO, 15, True, True),
    (4, 0, 15, False, True), (4, FBX, 15, True, True),
]


def _out_id(c):
    si, flags, lattice, soft, uni = c
    return (DEN_ID[si] + ("-nofuse" if flags == FNO else "-bitexact" if flags == FBX else "") +
            (f"-lat{lattice}" if lattice != 15 else "") + ("-soft" if soft else "-hard") + ("-universal" if uni else "-fixed"))


def _inv_launches(l, plan, flags, lattice):
    """inverse_span_all_thr's launches: the kernels of inverse_span_all (threshold on load) plus one threshold launch per
    level where the per-level kernels run"""
    k = 0
    for a, nlev in _groups(plan, False):
        kern, launches = inverse_span_kernel(l, a, nlev, flags, lattice)
        k += launches + (nlev if kern.startswith("per-level") else 0)
    return k


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1], ids=MODE_ID)
@pytest.mark.parametrize("case", OUT_CASES, ids=[_out_id(c) for c in OUT_CASES])
def test_thresholded_synthesis_rank_by_rank_within_the_bound(eng, case, mode):
    si, flags, lattice, soft, uni = case
    shape = DEN_SHAPES[si]
    name, levels, world, n_local = shape
    hs, gs = taps(name)
    l = hs.size
    eng.set_option("lattice", lattice)
    plan = _native.span_plan(l, levels, n_local, world)
    x = _signal(shape, plan, "mixed")
    ws, vs = _forward_ranks(eng, shape, mode, x, plan)
    wg, vg = _gather(plan, ws, vs)
    n_total = n_local * world
    if uni:
        lam = float(_device_threshold(eng, plan, ws, n_total)[0][0])
    else:
        lam = float(np.max(np.abs(wg[0]))) * 0.01            # a fixed value that zeroes some coefficients and keeps others
    thr = torch.tensor([lam], dtype=torch.float64, device="cuda")
    before = [(_bits(w), _bits(v)) for w, v in zip(ws, vs)]
    order = _native.ORDER_PAIR if mode == 1 else _native.ORDER_SPLIT
    outs = []
    for r in range(world):
        out = torch.full((n_local + 1,), SENTINEL, dtype=torch.float64, device="cuda")
        l0 = eng.launch_count()
        eng.inverse_span_all_thr(plan, ws[r], vs[r], hs, gs, order, thr, soft, out[:n_local], flags)
        assert eng.launch_count() - l0 == _inv_launches(l, plan, flags, lattice)
        outs.append(out)
    _sync()
    for r in range(world):
        assert np.array_equal(_bits(ws[r]), before[r][0]) and np.array_equal(_bits(vs[r]), before[r][1]), \
            f"rank {r}: inverse_span_all_thr changed W or V"
        assert float(outs[r][n_local].item()) == SENTINEL, f"rank {r}: wrote past xout[n_local]"
    kappa = lattice_kappa(name) if _lattice_in_plan(plan, l, lattice, flags, False) else 0.0
    wt = np_threshold(wg, lam, soft)
    ref, bnd = synth_ld_from(vg, wt, 1, levels, hs, gs, mode, kappa)
    worst = Worst(f"{_out_id(case)} {MODE_ID[mode]} thresholded synthesis")
    xg = np.concatenate([o[:n_local].cpu().numpy() for o in outs])
    for r in range(world):
        win = slice(r * n_local, (r + 1) * n_local)
        worst.check(xg[win], ref[win], bnd[win], f"rank {r} x")
    worst.report()
    zeroed = int(np.count_nonzero(wt == 0.0) - np.count_nonzero(wg == 0.0))
    assert zeroed > 0, "the threshold zeroed nothing: the case does not exercise thresholding"


def _multi_buffers(shape, plan, x, devices):
    name, levels, world, n_local = shape
    lead, lead_w, pad = int(plan.lead), int(plan.lead_w), int(plan.pad)
    row = lead_w + n_local + pad
    xext, ws, vs, xo = [], [], [], []
    for r, d in enumerate(devices):
        dev = torch.device("cuda", d)
        e = torch.full((lead + n_local,), float("nan"), dtype=torch.float64, device=dev)
        e[lead:] = torch.as_tensor(x[r * n_local:(r + 1) * n_local], device=dev)
        xext.append(e)
        ws.append(torch.full((levels, row), float("nan"), dtype=torch.float64, device=dev))
        vs.append(torch.full((n_local + pad,), float("nan"), dtype=torch.float64, device=dev))
        xo.append(torch.full((n_local + 1,), SENTINEL, dtype=torch.float64, device=dev))
    torch.cuda.synchronize()
    return xext, ws, vs, xo


@pytest.mark.gpu
@pytest.mark.parametrize("soft", [True, False], ids=["soft", "hard"])
@pytest.mark.parametrize("mode", [0, 1], ids=MODE_ID)
@pytest.mark.parametrize("si", [0, 2, 3, 4], ids=[DEN_ID[i] for i in (0, 2, 3, 4)])
def test_sharded_driver_is_the_rank_by_rank_path(eng, si, mode, soft):
    shape = DEN_SHAPES[si]
    name, levels, world, n_local = shape
    hs, gs = taps(name)
    plan = _native.span_plan(hs.size, levels, n_local, world)
    x = _signal(shape, plan, "mixed")
    order = _native.ORDER_PAIR if mode == 1 else _native.ORDER_SPLIT
    ws, vs = _forward_ranks(eng, shape, mode, x, plan)
    lam = float(_device_threshold(eng, plan, ws, n_local * world)[0][0])
    thr = torch.tensor([lam], dtype=torch.float64, device="cuda")
    ref = []
    for r in range(world):
        out = torch.empty(n_local, dtype=torch.float64, device="cuda")
        eng.inverse_span_all_thr(plan, ws[r], vs[r], hs, gs, order, thr, soft, out)
        ref.append(out)
    _sync()
    ref = np.concatenate([o.cpu().numpy() for o in ref])
    me = _native.MultiEngine([0] * world)
    try:
        xext, mw, mv, xo = _multi_buffers(shape, plan, x, [0] * world)
        l0 = me.launch_count()
        got_lam = me.denoise(plan, xext, hs, gs, mode, order, mw, mv, [o[:n_local] for o in xo], -1.0, soft)
        assert got_lam == lam or _same(got_lam, lam)
        got = np.concatenate([o[:n_local].cpu().numpy() for o in xo])
        assert np.array_equal(got.view(np.int64), ref.view(np.int64)), "driver output differs from the rank-by-rank path"
        assert all(float(o[n_local].item()) == SENTINEL for o in xo)
        launches = me.launch_count() - l0
        # NO_SYNC: a second signal (negated), then one vw_multi_synchronize
        xext2, mw2, mv2, xo2 = _multi_buffers(shape, plan, -x, [0] * world)
        assert me.denoise(plan, xext, hs, gs, mode, order, mw, mv, [o[:n_local] for o in xo], -1.0, soft,
                          flags=_native.FLAG_NO_SYNC) is None
        assert me.denoise(plan, xext2, hs, gs, mode, order, mw2, mv2, [o[:n_local] for o in xo2], -1.0, soft,
                          flags=_native.FLAG_NO_SYNC) is None
        me.synchronize()
        got1 = np.concatenate([o[:n_local].cpu().numpy() for o in xo])
        got2 = np.concatenate([o[:n_local].cpu().numpy() for o in xo2])
        assert np.array_equal(got1.view(np.int64), ref.view(np.int64))
        assert np.array_equal(got2, -ref), "the negated signal's denoise is not the negated result"
    finally:
        me.close()
    per_device_median = 1 + ROUNDS * 3 + 2 + 1          # init, (hist, sum, pick) per round, collect + mirror, value
    print(f"DRIVER {DEN_ID[si]} {MODE_ID[mode]}: {launches} launches, {per_device_median * world} in the median phase")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1], ids=MODE_ID)
@pytest.mark.parametrize("name,levels,world,n_local", [("db4", 6, 4, 16384), ("coif5", 6, 2, 32768), ("sym8", 5, 8, 8192)])
def test_sharded_driver_against_the_single_device_denoise(eng, name, levels, world, n_local, mode):
    hs, gs = taps(name)
    plan = _native.span_plan(hs.size, levels, n_local, world)
    n_total = n_local * world
    rng = np.random.default_rng(n_total + levels)
    x = np.sin(np.arange(n_total) * (2 * np.pi / 977.0)) * 5.0 + rng.standard_normal(n_total)
    order = _native.ORDER_PAIR if mode == 1 else _native.ORDER_SPLIT
    xd = torch.as_tensor(x, device="cuda")
    whole, whole_lam = eng.denoise(xd, hs, gs, levels, mode, None, order, -1.0, True)
    w_whole, _ = eng.forward(xd, hs, gs, levels, mode)
    _sync()
    me = _native.MultiEngine([0] * world)
    try:
        xext, mw, mv, xo = _multi_buffers((name, levels, world, n_local), plan, x, [0] * world)
        lam = me.denoise(plan, xext, hs, gs, mode, order, mw, mv, [o[:n_local] for o in xo], -1.0, True)
        got = np.concatenate([o[:n_local].cpu().numpy() for o in xo])
        wg, _ = _gather(plan, mw, mv)
    finally:
        me.close()
    w_whole = w_whole[:, 0, :].cpu().numpy() if w_whole.dim() == 3 else w_whole.cpu().numpy()
    if np.array_equal(wg[0].view(np.int64), w_whole[0].view(np.int64)):
        assert _same(lam, whole_lam)
    else:
        assert abs(lam - whole_lam) <= 1e-13 * whole_lam
    # coefficients within rounding of the threshold may be zeroed on one side only: count them (none expected)
    near = int(np.count_nonzero(np.abs(np.abs(wg) - lam) <= 8 * np.spacing(lam)) +
               np.count_nonzero(np.abs(np.abs(w_whole) - whole_lam) <= 8 * np.spacing(whole_lam)))
    assert near == 0, f"{near} coefficients within rounding of the threshold"
    whole = whole.cpu().numpy()
    err = float(np.max(np.abs(got - whole)))
    assert err <= 1e-12 * float(np.max(np.abs(x))), err
    print(f"VS WHOLE {name} J{levels} w{world} {MODE_ID[mode]}: lambda {lam!r} vs {whole_lam!r}, max |diff| {err:.3g}")


@pytest.mark.gpu
def test_sharded_driver_errors_leave_the_objects_usable(eng):
    shape = DEN_SHAPES[1]
    name, levels, world, n_local = shape
    hs, gs = taps(name)
    plan = _native.span_plan(hs.size, levels, n_local, world)
    x = _signal(shape, plan, "mixed")
    me = _native.MultiEngine([0] * world)
    try:
        xext, mw, mv, xo = _multi_buffers(shape, plan, x, [0] * world)
        outs = [o[:n_local] for o in xo]
        with pytest.raises(InvalidArgumentException):          # VW_EBOUNDARY
            me.denoise(plan, xext, hs, gs, 2, 0, mw, mv, outs)
        other = _native.span_plan(hs.size, levels, n_local, world + 1)
        with pytest.raises(IllegalArgumentException):          # VW_EINVAL: plan for another world
            me.denoise(other, xext, hs, gs, 0, 0, mw, mv, outs)
        bad = [e.clone() for e in xext]
        bad[1][int(plan.lead) + 7] = float("nan")
        with pytest.raises(InvalidSignalException) as ei:      # VW_ENONFINITE, names the rank
            me.denoise(plan, bad, hs, gs, 0, 0, mw, mv, outs, flags=_native.FLAG_CHECK_FINITE)
        assert "rank 1" in str(ei.value)
        torch.cuda.synchronize()
        assert all(np.all(o.cpu().numpy() == SENTINEL) for o in xo), "xout written by a rejected call"
        lam = me.denoise(plan, xext, hs, gs, 0, 0, mw, mv, outs, flags=_native.FLAG_CHECK_FINITE)
        assert np.isfinite(lam) and lam > 0
        assert all(float(o[n_local].item()) == SENTINEL for o in xo)
    finally:
        me.close()


@pytest.mark.gpu
def test_single_device_threshold_paths_keep_their_launch_counts(eng):
    x = np.random.default_rng(5).standard_normal((4, 1 << 14))
    xd = torch.as_tensor(x, device="cuda")
    hs, gs = taps("db4")
    l0 = eng.launch_count()
    eng.universal_threshold(xd)
    assert eng.launch_count() - l0 == 18             # init, 2 x (hist, pick), collect, mirror, 5 x (hist, pick), finish
    l0 = eng.launch_count()
    eng.forward(xd, hs, gs, 4, 0)
    fwd = eng.launch_count() - l0
    w, v = eng.forward(xd, hs, gs, 4, 0)
    l0 = eng.launch_count()
    eng.inverse(w, v, hs, gs, 0)
    inv = eng.launch_count() - l0
    l0 = eng.launch_count()
    eng.denoise(xd, hs, gs, 4, 0)
    assert eng.launch_count() - l0 == fwd + 18 + inv
