"""Span-sharded SWT denoise of config #4's shape (coif5, J = 10, one signal of 2^28 samples split over the job's GPUs) through
vw_swt_denoise_sharded, against the transform alone (vw_modwt_forward_sharded + vw_modwt_inverse_sharded).

Reports per step (wall time around a call that ends in a device synchronise, median of --steps after --warmup):
  transform_ms   forward_sharded + inverse_sharded
  denoise_ms     vw_swt_denoise_sharded with the universal soft threshold (exact cross-rank median)
  fixed_ms       vw_swt_denoise_sharded with a fixed threshold (no median phase)
  median_ms      denoise_ms - fixed_ms: the seven histogram rounds, their peer exchanges and sums
  median_rounds_rank0_ms  rank 0's seven median rounds on its own W_1 span timed with CUDA events (no exchange; with
                 one GPU this is the whole median phase)
  launches       kernels launched by one universal-threshold call, over all devices
and, with one GPU, whole_ms: vw_swt_denoise on the whole signal on that device.  The card name and power limit are read
in the same run (nvidia-smi).  Writes one JSON line to stdout (and to --out when given).

    python tools/span_denoise_bench.py [--gpus G] [--n-total 268435456] [--steps 10] [--warmup 3] [--out FILE]
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=0, help="devices to use (0: all)")
    ap.add_argument("--n-total", type=int, default=1 << 28)
    ap.add_argument("--levels", type=int, default=10)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    from oracle.wavelets import filters
    from vectorwave_b200 import _native

    if not torch.cuda.is_available():
        raise SystemExit("span_denoise_bench needs CUDA devices (nothing is measured without one)")
    world = args.gpus or torch.cuda.device_count()
    devices = list(range(world))
    n_local = args.n_total // world
    h, g, _ = filters("coif5")
    s = 1.0 / math.sqrt(2.0)
    hs, gs = h * s, g * s
    levels = args.levels
    plan = _native.span_plan(hs.size, levels, n_local, world)
    lead, lead_w, pad = int(plan.lead), int(plan.lead_w), int(plan.pad)
    row = lead_w + n_local + pad
    me = _native.MultiEngine(devices)
    xext, w, v, xo = [], [], [], []
    for r, d in enumerate(devices):
        dev = torch.device("cuda", d)
        gen = torch.Generator(device=dev).manual_seed(1234 + r)
        e = torch.empty(lead + n_local, dtype=torch.float64, device=dev)
        e[lead:] = torch.randn(n_local, dtype=torch.float64, device=dev, generator=gen)
        xext.append(e)
        w.append(torch.empty((levels, row), dtype=torch.float64, device=dev))
        v.append(torch.empty(n_local + pad, dtype=torch.float64, device=dev))
        xo.append(torch.empty(n_local, dtype=torch.float64, device=dev))
    for d in devices:
        torch.cuda.synchronize(d)

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        ts = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            fn()                       # every call below ends in a synchronise of all devices
            ts.append((time.perf_counter() - t0) * 1e3)
        return statistics.median(ts), min(ts)

    def transform():
        me.forward(plan, xext, hs, gs, 0, w, v)
        me.inverse(plan, w, v, hs, gs, 0, _native.ORDER_SPLIT, xo)

    lam = {}

    def denoise():
        lam["u"] = me.denoise(plan, xext, hs, gs, 0, _native.ORDER_SPLIT, w, v, xo, -1.0, True)

    def fixed():
        me.denoise(plan, xext, hs, gs, 0, _native.ORDER_SPLIT, w, v, xo, 0.5, True)

    res = {"tool": "span_denoise_bench", "card": card_info(), "gpus": world, "wavelet": "coif5", "levels": levels,
           "n_total": n_local * world, "n_local": n_local, "steps": args.steps, "warmup": args.warmup,
           "timing": "wall time around calls that end in a synchronise of every device; median (min) over steps"}
    res["transform_ms"], res["transform_min_ms"] = timed(transform)
    res["denoise_ms"], res["denoise_min_ms"] = timed(denoise)
    res["fixed_ms"], res["fixed_min_ms"] = timed(fixed)
    res["median_ms"] = res["denoise_ms"] - res["fixed_ms"]
    l0 = me.launch_count()
    denoise()
    res["launches"] = me.launch_count() - l0
    l0 = me.launch_count()
    transform()
    res["transform_launches"] = me.launch_count() - l0
    res["threshold"] = lam["u"]
    res["denoise_gsamples_s"] = n_local * world / (res["denoise_ms"] * 1e6)
    # the seven median rounds of rank 0 alone on its W_1 span (CUDA events, no exchange; with one GPU this is the whole
    # median phase): vw_span_median_init, 7 x (hist, pick), value
    eng0 = _native.Engine.get(0)
    w1 = w[0][0, lead_w:lead_w + n_local]
    state = eng0.span_median_state(n_local)
    hists = [torch.empty(_native.span_median_bins(r), dtype=torch.int64, device="cuda:0") for r in range(_native.SPAN_MEDIAN_ROUNDS)]
    thr = torch.empty(1, dtype=torch.float64, device="cuda:0")
    factor = math.sqrt(2.0 * math.log(float(n_local * world)))

    def rounds():
        eng0.span_median_init(state, n_local * world)
        for r in range(_native.SPAN_MEDIAN_ROUNDS):
            eng0.span_median_hist(state, w1, r, hists[r])
            eng0.span_median_pick(state, r, hists[r])
        eng0.span_median_value(state, factor, thr)

    with torch.cuda.device(0):
        for _ in range(args.warmup):
            rounds()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for a, b in ev:
            a.record()
            rounds()
            b.record()
        torch.cuda.synchronize(0)
    res["median_rounds_rank0_ms"] = statistics.median(a.elapsed_time(b) for a, b in ev)
    if world == 1:
        res["median_rounds_threshold"] = float(thr.item())
    me.close()
    del xext, w, v, xo
    if world == 1:
        torch.cuda.empty_cache()
        eng = _native.Engine.get(0)
        x = torch.randn(args.n_total, dtype=torch.float64, device="cuda:0",
                        generator=torch.Generator(device="cuda:0").manual_seed(1234))
        holder = {}

        def whole():
            holder["out"], holder["lam"] = eng.denoise(x, hs, gs, levels, 0, None, _native.ORDER_SPLIT, -1.0, True)
            torch.cuda.synchronize(0)

        res["whole_ms"], res["whole_min_ms"] = timed(whole)
        res["whole_threshold"] = holder["lam"]
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
