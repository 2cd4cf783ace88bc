"""Multi-GPU sharding of the MODWT path: one process per GPU (torch.distributed; NCCL over NVLink on the box).

* Batches shard by signal: contiguous blocks of signals per rank, no data-path communication (`shard_batch`).
* One long signal shards by contiguous span: rank r owns samples [r*N/P, (r+1)*N/P).  Analysis needs a LEFT halo
  (indices t - k*2^(j-1)), synthesis a RIGHT halo (t + k*2^(j-1)), ring-wrapped between the last and the first rank for
  PERIODIC, zeros at the open ends for ZERO_PADDING.  Two schedules:
    - up front (default whenever the total halo (L-1)*(2^J-1) fits the span): ONE exchange per direction -- the last
      H samples of x from the left neighbour before the analysis, the first samples of V_J and of every W_j from the
      right neighbour before the synthesis -- and every level is computed on a region that shrinks by its own halo
      (redundant recompute of <= H samples per level: 0.02 % at 2^27 samples per rank).  No per-level synchronisation.
    - per launch group (fallback when the span is shorter than the total halo): the group's dilated halo
      (L-1)*2^(first-1)*(2^nlev-1) is exchanged before every group.
  Messages are <= a few hundred KB, i.e. latency bound: NCCL send/recv inside one batch_isend_irecv group.
  The result equals the unsharded transform bit for bit of the same kernels (SURVEY.md D8: the reference's
  forwardChunked has no halo and is NOT the semantics implemented here).

Reference precedent for the halo semantics: EXT/extensions/modwt/BatchSIMDMODWT.java:447-507 (left history of
L_j-1 samples) and BatchStreamingMODWT.java:326-357.
"""
import math

import torch
import torch.distributed as dist

from . import _native
from ._native import Engine, ORDER_PAIR, ORDER_SPLIT, SPAN_MEDIAN_ROUNDS, span_median_bins
from .errors import ErrorCode, IllegalArgumentException, InvalidSignalException
from .wavelets import BoundaryMode

SCALE = 1.0 / math.sqrt(2.0)


def shard_batch(batch, rank, world):
    """Contiguous block [lo, hi) of `batch` signals owned by `rank` (remainder spread over the first ranks)."""
    base, extra = divmod(batch, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def _even_up(v):
    return (v + 1) & ~1


def _halo_up(v):
    """Halos are rounded up to 32 samples (256 B): every buffer offset the kernels see then keeps whole 32-byte
    sectors and 256-byte warp rows aligned (a halo of 58 samples made each warp access straddle an extra sector and
    turned stores into partial-sector writes: the span kernels ran 39 % slower than the unsharded ones)."""
    return (v + 31) & ~31


class SpanResult:
    """Per-rank slice of a multi-level decomposition.  Rows carry `pad` spare samples on the right so the inverse can
    receive the neighbour's halo in place (no repacking): w [J][n_local + pad], v [n_local + pad]."""

    def __init__(self, w, v, n_local, pad, storage=None):
        self.w, self.v, self.n_local, self.pad = w, v, n_local, pad
        self.storage = storage      # the full W allocation `w` is a view of (reused by forward(..., result=...))

    def details(self):
        return self.w[:, :self.n_local]

    def approximation(self):
        return self.v[:self.n_local]


class SpanShardedMODWT:
    """decompose / reconstruct of one long signal spread over the ranks of `group` (PERIODIC or ZERO_PADDING)."""

    def __init__(self, wavelet, levels, n_local, boundaryMode=BoundaryMode.PERIODIC, group=None, engine=None,
                 rank=None, world=None, groups_forward=None, groups_inverse=None, upfront=None):
        if boundaryMode not in (BoundaryMode.PERIODIC, BoundaryMode.ZERO_PADDING):
            raise IllegalArgumentException("span sharding supports PERIODIC and ZERO_PADDING (SYMMETRIC synthesis is "
                                           "two-sided per level; shard those by signal instead)")
        self.group = group
        self.rank = dist.get_rank(group) if rank is None and dist.is_initialized() else (rank or 0)
        self.world = dist.get_world_size(group) if world is None and dist.is_initialized() else (world or 1)
        self.engine = engine
        self.mode = boundaryMode
        self.levels = int(levels)
        self.n_local = int(n_local)
        self.hs = wavelet.lowPassDecomposition() * SCALE
        self.gs = wavelet.highPassDecomposition() * SCALE
        self.hrs = wavelet.lowPassReconstruction() * SCALE
        self.grs = wavelet.highPassReconstruction() * SCALE
        self.l = int(self.hs.size)
        n_total = self.n_local * self.world
        if (self.l - 1) * (1 << (self.levels - 1)) + 1 > n_total:
            raise IllegalArgumentException("upsampled filter longer than the signal")
        self.gf = groups_forward or _native.plan_groups(True, self.l, self.levels, n_total)
        self.gi = groups_inverse or _native.plan_groups(False, self.l, self.levels, n_total)
        self.halo_f = [_halo_up(self._halo(f, k)) for f, k in self.gf]
        self.halo_i = [_halo_up(self._halo(f, k)) for f, k in self.gi]
        if max(self.halo_f + self.halo_i) > self.n_local:
            raise IllegalArgumentException("a level group's halo exceeds the per-rank span; use fewer ranks or levels")
        # up-front schedule: cumulative (even-rounded) halos.  rf[g] = left halo still needed AFTER forward group g
        # (by the later groups); si[g] = right halo the inverse needs on the INPUTS of group g (its own + the lower groups')
        self.rf = [sum(self.halo_f[g + 1:]) for g in range(len(self.gf))]
        self.si_out = [sum(self.halo_i[:g]) for g in range(len(self.gi))]
        self.si_in = [self.si_out[g] + self.halo_i[g] for g in range(len(self.gi))]
        total_f, total_i = sum(self.halo_f), sum(self.halo_i)
        self.upfront = (max(total_f, total_i) <= self.n_local) if upfront is None else bool(upfront)
        if self.upfront and max(total_f, total_i) > self.n_local:
            raise IllegalArgumentException("the total halo exceeds the per-rank span: use the per-group schedule")
        self.pad = total_i if self.upfront else max(self.halo_i)
        self.lead = total_f if self.upfront else max(self.halo_f)
        self.lead_w = self.rf[0] if self.upfront else 0     # W rows carry the not-yet-final left part of each level
        # Default case (the engine's own launch groups, up-front schedule): layout and cascades live below the C ABI
        # (vw_span_plan_query + vw_modwt_{forward,inverse}_span_all); this class only moves the halos between ranks.
        # Caller-chosen groups and the per-group schedule keep the Python schedules below.
        self.plan = None
        if self.upfront and groups_forward is None and groups_inverse is None:
            self.plan = _native.span_plan(self.l, self.levels, self.n_local, self.world)
            self.lead, self.lead_w, self.pad = int(self.plan.lead), int(self.plan.lead_w), int(self.plan.pad)

    def _eng(self):
        if self.engine is None:
            self.engine = Engine.get()
        return self.engine

    def _halo(self, first, nlev):
        return (self.l - 1) * (1 << (first - 1)) * ((1 << nlev) - 1)

    # -- ring exchange --------------------------------------------------------------------------------------
    def _exchange(self, send, recv, to_right):
        """send -> right neighbour (to_right) or left neighbour; recv <- the opposite side.  PERIODIC wraps around the
        ring; ZERO_PADDING leaves the open end's halo at zero."""
        left, right = (self.rank - 1) % self.world, (self.rank + 1) % self.world
        dst, src = (right, left) if to_right else (left, right)
        periodic = self.mode == BoundaryMode.PERIODIC
        i_send = periodic or (self.rank != self.world - 1 if to_right else self.rank != 0)
        i_recv = periodic or (self.rank != 0 if to_right else self.rank != self.world - 1)
        if self.world == 1:
            if periodic:
                recv.copy_(send)
            else:
                recv.zero_()
            return
        ops = []
        if i_send:
            ops.append(dist.P2POp(dist.isend, send, dst, self.group))
        if i_recv:
            ops.append(dist.P2POp(dist.irecv, recv, src, self.group))
        else:
            recv.zero_()
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()

    # -- analysis -------------------------------------------------------------------------------------------
    def _scratch(self, key, count, length, dev):
        """Work buffers live with the object: multi-GB torch.empty calls per transform cost more than the kernels."""
        cache = self.__dict__.setdefault("_scratch_cache", {})
        bufs = cache.get(key)
        if bufs is None or bufs[0].numel() != length or bufs[0].device != dev or len(bufs) != count:
            bufs = [torch.empty(length, dtype=torch.float64, device=dev) for _ in range(count)]
            cache[key] = bufs
        return bufs

    # -- default path: one ABI call per direction around one exchange ------------------------------------------
    def _forward_plan(self, x_local, result=None):
        n, dev, p = self.n_local, x_local.device, self.plan
        row = self.lead_w + n + self.pad
        if result is not None and result.storage is not None and tuple(result.storage.shape) == (self.levels, row):
            wfull, vstore = result.storage, result.v
        else:
            wfull = torch.empty((self.levels, row), dtype=torch.float64, device=dev)
            vstore = torch.empty(n + self.pad, dtype=torch.float64, device=dev)
        (xext,) = self._scratch("xext", 1, self.lead + n, dev)
        xext[self.lead:].copy_(x_local)
        self.exchange_forward(xext)
        self._eng().forward_span_all(xext, p, self.hs, self.gs, wfull, vstore)
        return SpanResult(wfull[:, self.lead_w:], vstore, n, self.pad, storage=wfull)

    def exchange_forward(self, xext):
        """The analysis halo: my last `lead` samples -> right neighbour's lead area (ring wrap / zeros at the open end)."""
        if self.lead > 0:
            self._exchange(xext[self.n_local:].contiguous(), xext[:self.lead], to_right=True)

    def exchange_inverse(self, result):
        """The synthesis halo: the first samples of V_J and of every W_j row -> left neighbour's pad areas."""
        p, dev = self.plan, result.v.device
        if int(p.inverse_msg) == 0:
            return
        send, recv = self._scratch("msg", 2, int(p.inverse_msg), dev)
        eng = self._eng()
        eng.span_pack_inverse(p, result.storage, result.v, send)
        self._exchange(send, recv, to_right=False)
        eng.span_unpack_inverse(p, recv, result.storage, result.v)

    def exchange_only(self, result):
        """Both directions' halo exchanges without the cascades (bench.py times this separately)."""
        if self.plan is None:
            raise IllegalArgumentException("exchange_only needs the default (plan) schedule")
        (xext,) = self._scratch("xext", 1, self.lead + self.n_local, result.v.device)
        self.exchange_forward(xext)
        self.exchange_inverse(result)

    def _inverse_plan(self, result, order):
        self.exchange_inverse(result)
        out = torch.empty(self.n_local, dtype=torch.float64, device=result.v.device)
        self._eng().inverse_span_all(self.plan, result.storage, result.v, self.hrs, self.grs, order, out)
        return out

    def _forward_upfront(self, x_local, result=None):
        """One exchange of the total left halo, then every group on [-(halo still needed later), n)."""
        n, dev = self.n_local, x_local.device
        eng = self._eng()
        lead, lw = self.lead, self.lead_w
        if result is not None and result.storage is not None and tuple(result.storage.shape) == (self.levels, lw + n + self.pad):
            wfull, vstore = result.storage, result.v
        else:
            wfull = torch.empty((self.levels, lw + n + self.pad), dtype=torch.float64, device=dev)
            vstore = torch.empty(n + self.pad, dtype=torch.float64, device=dev)
        bufs = self._scratch("fwd", 2, lead + n, dev)
        bufs[0][lead:].copy_(x_local)
        if lead > 0:
            self._exchange(bufs[0][n:].contiguous(), bufs[0][:lead], to_right=True)   # my last `lead` samples -> right neighbour
        cur, have = 0, lead                        # bufs[cur][lead - have:] holds V_{first-1} on [-have, n)
        for g, (first, nlev) in enumerate(self.gf):
            keep = self.rf[g]                      # left halo the later groups still need
            last = g + 1 == len(self.gf)
            vout = vstore[:n] if last else bufs[cur ^ 1][lead - keep:]
            eng.forward_span(bufs[cur][lead - have:], have - keep, self.hs, self.gs, first, nlev,
                             w_out=wfull[first - 1:first - 1 + nlev, lw - keep:], v_out=vout)
            cur ^= 1
            have = keep
        return SpanResult(wfull[:, lw:], vstore, n, self.pad, storage=wfull)

    def _inverse_upfront(self, result, order):
        """One exchange of the right halos of V_J and of every W_j, then every group on [0, n + halo needed below)."""
        n, dev = self.n_local, result.v.device
        eng = self._eng()
        w, vtop = result.w, result.v
        ng = len(self.gi)
        # message: my first si_in[top] samples of V_J, and for every group the first si_in[g] samples of its W rows
        pieces = [vtop[:self.si_in[ng - 1]]]
        for g in range(ng):
            first, nlev = self.gi[g]
            pieces += [w[first - 1 + i, :self.si_in[g]] for i in range(nlev)]
        send = torch.cat(pieces).contiguous()
        recv = torch.empty_like(send)
        if send.numel() > 0:
            self._exchange(send, recv, to_right=False)
        at = self.si_in[ng - 1]
        vtop[n:n + at].copy_(recv[:at])
        for g in range(ng):
            first, nlev = self.gi[g]
            for i in range(nlev):
                w[first - 1 + i, n:n + self.si_in[g]].copy_(recv[at:at + self.si_in[g]])
                at += self.si_in[g]
        work = self._scratch("inv", 2, n + self.pad, dev)
        vext, cur, out = vtop, 0, None
        for g in range(ng - 1, -1, -1):
            first, nlev = self.gi[g]
            s_in, s_out = self.si_in[g], self.si_out[g]
            dst = torch.empty(n, dtype=torch.float64, device=dev) if g == 0 else work[cur][:n + s_out]
            eng.inverse_span(vext[:n + s_in], w[first - 1:first - 1 + nlev, :n + s_in], s_in - s_out, self.hrs, self.grs,
                             first, nlev, order, out=dst)
            out, vext = dst, work[cur]
            cur ^= 1
        return out

    def forward(self, x_local, result=None):
        """x_local: this rank's [n_local] span (float64, on the engine's device) -> SpanResult.  `result`: an earlier
        SpanResult of this object whose storage is overwritten instead of allocating 8*(J+1)*n_local fresh bytes."""
        n, dev = self.n_local, x_local.device
        if x_local.numel() != n:
            raise IllegalArgumentException(f"expected a span of {n} samples, got {x_local.numel()}")
        if self.plan is not None:
            return self._forward_plan(x_local, result)
        if self.upfront:
            return self._forward_upfront(x_local, result)
        eng = self._eng()
        w = torch.empty((self.levels, n + self.pad), dtype=torch.float64, device=dev)
        vstore = torch.empty(n + self.pad, dtype=torch.float64, device=dev)
        # two [lead | span] work buffers: each group reads one and writes its V into the other, right after the slot
        # where the next group's halo will land
        bufs = [torch.empty(self.lead + n, dtype=torch.float64, device=dev) for _ in range(2)]
        bufs[0][self.lead:].copy_(x_local)
        cur = 0
        for gi, (first, nlev) in enumerate(self.gf):
            halo = self.halo_f[gi]
            ext = bufs[cur]
            span = ext[self.lead:]
            if halo > 0:
                send = span[n - halo:].contiguous()
                self._exchange(send, ext[self.lead - halo:self.lead], to_right=True)
            last = gi + 1 == len(self.gf)
            vout = vstore[:n] if last else bufs[cur ^ 1][self.lead:]
            eng.forward_span(ext[self.lead - halo:], halo, self.hs, self.gs, first, nlev,
                             w_out=w[first - 1:first - 1 + nlev], v_out=vout)
            cur ^= 1
        return SpanResult(w, vstore, n, self.pad)

    # -- synthesis ------------------------------------------------------------------------------------------
    def inverse(self, result, order=ORDER_SPLIT):
        if self.plan is not None:
            return self._inverse_plan(result, order)
        if self.upfront:
            return self._inverse_upfront(result, order)
        n, dev = self.n_local, result.v.device
        eng = self._eng()
        w, pad = result.w, result.pad
        work = [torch.empty(n + pad, dtype=torch.float64, device=dev) for _ in range(2)]
        vext = result.v          # only its spare tail is written (the received halo); the coefficients stay intact
        cur = 0
        out = None
        for gi in range(len(self.gi) - 1, -1, -1):
            first, nlev = self.gi[gi]
            halo = self.halo_i[gi]
            rows = w[first - 1:first - 1 + nlev]
            if halo > 0:
                # one message: my first `halo` samples of V and of every W row of the group -> left neighbour
                send = torch.cat([vext[:halo].reshape(1, -1), rows[:, :halo]], dim=0).contiguous()
                recv = torch.empty_like(send)
                self._exchange(send, recv, to_right=False)
                vext[n:n + halo].copy_(recv[0])
                rows[:, n:n + halo].copy_(recv[1:])
            last = gi == 0
            dst = torch.empty(n, dtype=torch.float64, device=dev) if last else work[cur][:n]
            eng.inverse_span(vext[:n + halo], rows[:, :n + halo], halo, self.hrs, self.grs, first, nlev, order, out=dst)
            out = dst
            vext = work[cur]
            cur ^= 1
        return out

    # -- SWT denoise of the whole signal ----------------------------------------------------------------------
    def denoise(self, x_local, threshold=-1.0, soft=True):
        """VectorWaveSwtAdapter.denoise of the whole signal (vw_swt_denoise with batch = 1 on all world * n_local samples),
        computed span by span: decompose, threshold every detail level, reconstruct.  threshold < 0: the universal
        threshold median(|W_1|) / 0.6745 * sqrt(2 ln N) with the exact median over every rank's W_1 (seven histogram
        rounds, one all_reduce(SUM) of an int64 table per round over this object's group); otherwise the given value.
        V_J is not thresholded.  Returns (this rank's denoised span, the threshold).  Every rank must call it.  Needs the
        default (plan) schedule."""
        if self.plan is None:
            raise IllegalArgumentException("denoise needs the default schedule (engine launch groups, up-front halo exchange)")
        n, dev = self.n_local, x_local.device
        if x_local.numel() != n:
            raise IllegalArgumentException(f"expected a span of {n} samples, got {x_local.numel()}")
        # collective validation: every rank reaches the same decision before any other collective, so a NaN on one rank
        # cannot leave the others waiting in an all_reduce
        bad = torch.tensor([0 if bool(torch.isfinite(x_local).all()) else 1], dtype=torch.int64, device=dev)
        if self.world > 1:
            dist.all_reduce(bad, op=dist.ReduceOp.SUM, group=self.group)
        if int(bad.item()):
            raise InvalidSignalException(f"{int(bad.item())} rank(s) hold non-finite values (NaN or Infinity)",
                                         ErrorCode.VAL_NON_FINITE_VALUES)
        res = self._forward_plan(x_local)
        eng = self._eng()
        n_total = n * self.world
        if threshold < 0:
            w1 = res.storage[0, self.lead_w:self.lead_w + n]
            state = eng.span_median_state(n)
            eng.span_median_init(state, n_total)
            for rnd in range(SPAN_MEDIAN_ROUNDS):
                hist = torch.empty(span_median_bins(rnd), dtype=torch.int64, device=dev)
                eng.span_median_hist(state, w1, rnd, hist)
                if self.world > 1:
                    dist.all_reduce(hist, op=dist.ReduceOp.SUM, group=self.group)
                eng.span_median_pick(state, rnd, hist)
            thr = torch.empty(1, dtype=torch.float64, device=dev)
            eng.span_median_value(state, math.sqrt(2.0 * math.log(float(n_total))), thr)
        else:
            thr = torch.full((1,), float(threshold), dtype=torch.float64, device=dev)
        self.exchange_inverse(res)
        out = torch.empty(n, dtype=torch.float64, device=dev)
        order = ORDER_PAIR if self.mode == BoundaryMode.ZERO_PADDING else ORDER_SPLIT   # MultiLevelMODWTTransform.reconstruct
        eng.inverse_span_all_thr(self.plan, res.storage, res.v, self.hrs, self.grs, order, thr, soft, out)
        return out, float(thr.item())
