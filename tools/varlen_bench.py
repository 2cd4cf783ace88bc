"""Mixed-length single-level batches on one GPU: vw_modwt_forward_varlen / vw_modwt_inverse_varlen next to the
equal-length path (vw_modwt_forward / vw_modwt_inverse) on the same number of samples, the per-signal loop the
mixed-length batch API ran before, and the host-buffer end-to-end rate.

    python tools/varlen_bench.py [--out results.json] [--reps 10]

Device times are CUDA events around `reps` calls after warm-up; every timed working set exceeds the 126 MB L2 (the
short-row case cycles through enough copies).  HBM fraction: 24 B per sample and direction (read 8, write 16 forward;
read 16, write 8 inverse) over the peak of bench.measured_peaks().  The card's name and power limit are printed first.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
import vectorwave_b200 as vw  # noqa: E402
from oracle.wavelets import filters  # noqa: E402

S = 1.0 / np.sqrt(2.0)
MODES = {"PERIODIC": 0, "ZERO_PADDING": 1, "SYMMETRIC": 2}


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                                       text=True).strip()
    except Exception as e:   # the numbers below still stand, but unlabelled: say so
        return f"unknown ({e})"


def timed(fn, reps, warm=3):
    import torch
    for _ in range(warm):
        fn(0)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(reps):
        fn(i)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps   # ms per call


def lengths_for(case, rng):
    if case == "a":      # uniform in [1024, 65536], >= 2^28 samples
        out, tot = [], 0
        while tot < 1 << 28:
            out.append(int(rng.integers(1024, 65537)))
            tot += out[-1]
        return np.array(out)
    if case == "b":      # log-uniform in [16, 2^20], >= 2^28 samples
        out, tot = [], 0
        while tot < 1 << 28:
            out.append(int(round(np.exp(rng.uniform(np.log(16), np.log(1 << 20))))))
            tot += out[-1]
        return np.array(out)
    return rng.integers(1, 65, size=100_000)   # c: 10^5 rows of 1..64


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--loop-rows", type=int, default=2000)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "varlen_bench needs a CUDA device"
    eng = vw.Engine.get(0)
    peak, peak_src = bench.measured_peaks()
    info = {"card": card(), "hbm_peak_gbs": peak, "hbm_peak_source": peak_src, "rows": []}
    print(f"card: {info['card']}   HBM peak {peak:.0f} GB/s ({peak_src})", flush=True)
    rng = np.random.default_rng(2026)
    results = info["rows"]

    def report(case, wav, mode, path, direction, total, ms, extra=None):
        gs = total / ms / 1e6
        frac = total * 24.0 / (ms * 1e-3) / (peak * 1e9)
        row = {"case": case, "wavelet": wav, "mode": mode, "path": path, "direction": direction, "samples": int(total),
               "ms": round(ms, 4), "gsamples_s": round(gs, 2), "hbm_fraction": round(frac, 3)}
        row.update(extra or {})
        results.append(row)
        print(f"{case:3s} {wav:6s} {mode:12s} {path:9s} {direction:7s} {total:>11d} samples {ms:9.3f} ms "
              f"{gs:7.2f} GSamples/s  {frac:5.3f} of HBM", flush=True)

    for case in ("a", "b", "c"):
        lens = lengths_for(case, rng)
        off = np.zeros(lens.size + 1, dtype=np.int64)
        np.cumsum(lens, out=off[1:])
        total = int(off[-1])
        copies = 1 if total * 24 > 4 * (126 << 20) else int(np.ceil(4 * (126 << 20) / (total * 24)))
        xs = [torch.randn(total, dtype=torch.float64, device="cuda") for _ in range(copies)]
        print(f"case {case}: {lens.size} rows, {total} samples, lengths {lens.min()}..{lens.max()}, {copies} copies in rotation",
              flush=True)
        wavs = ("db4", "sym8") if case == "a" else ("db4",)
        for wav in wavs:
            h, g, _ = filters(wav)
            hs, gs = h * S, g * S
            for mname, mode in MODES.items():
                outs = [eng.forward_varlen(x, off, hs, gs, mode) for x in xs]
                ms = timed(lambda i: eng.forward_varlen(xs[i % copies], off, hs, gs, mode, w_out=outs[i % copies][0],
                                                        v_out=outs[i % copies][1]), args.reps)
                report(case, wav, mname, "varlen", "forward", total, ms)
                recon = [torch.empty_like(x) for x in xs]
                ms = timed(lambda i: eng.inverse_varlen(outs[i % copies][0], outs[i % copies][1], off, hs, gs, mode,
                                                        out=recon[i % copies]), args.reps)
                report(case, wav, mname, "varlen", "inverse", total, ms)
                if case == "a":   # the equal-length batch of the same total through vw_modwt_forward / vw_modwt_inverse
                    n = 32768
                    b = total // n
                    x2 = xs[0][:b * n].view(b, n)
                    w2, v2 = eng.forward(x2, hs, gs, 1, mode)
                    ms = timed(lambda i: eng.forward(x2, hs, gs, 1, mode, w_out=w2, v_out=v2), args.reps)
                    report(case, wav, mname, "equal", "forward", b * n, ms, {"rows_equal": b, "n_equal": n})
                    align = [(-1, 0, -1, 0)] if mode == 2 else None
                    r2 = torch.empty_like(v2)
                    ms = timed(lambda i: eng.inverse(w2, v2, hs, gs, mode, align, vw.modwt.ORDER_PAIR, out=r2), args.reps)
                    report(case, wav, mname, "equal", "inverse", b * n, ms, {"rows_equal": b, "n_equal": n})
                del outs, recon
                torch.cuda.empty_cache()

        if case == "a":
            # today's path for mixed lengths: one MODWTTransform.forward per row (host arrays), on the first rows only
            t = vw.MODWTTransform(vw.Daubechies.DB4, vw.BoundaryMode.PERIODIC)
            k = min(args.loop_rows, lens.size)
            host = xs[0][:int(off[k])].cpu().numpy()
            rows = [host[off[i]:off[i + 1]] for i in range(k)]
            t.forward(rows[0])
            t0 = time.perf_counter()
            for r in rows:
                t.forward(r)
            loop_s = time.perf_counter() - t0
            t.forwardBatch(rows)
            t0 = time.perf_counter()
            t.forwardBatch(rows)
            batch_s = time.perf_counter() - t0
            info["per_signal_loop"] = {"rows": k, "samples": int(off[k]), "loop_rows_s": round(k / loop_s, 1),
                                       "forwardBatch_rows_s": round(k / batch_s, 1), "loop_s": round(loop_s, 4),
                                       "forwardBatch_s": round(batch_s, 4)}
            print(f"per-signal loop (db4 PERIODIC, host arrays, {k} rows of case a): {k / loop_s:.0f} rows/s; "
                  f"forwardBatch on the same rows (one varlen call): {k / batch_s:.0f} rows/s", flush=True)
            # end-to-end host buffers (pinned): H2D + kernel + D2H of the whole of case a, chunked on row boundaries
            try:
                h, g, _ = filters("db4")
                xp = eng.pinned_empty((total,))
                xp[...] = xs[0].cpu().numpy()
                wp, vp = eng.pinned_empty((total,)), eng.pinned_empty((total,))
                eng.forward_varlen(xp, off, h * S, g * S, 0, w_out=wp, v_out=vp)
                t0 = time.perf_counter()
                reps = 3
                for _ in range(reps):
                    eng.forward_varlen(xp, off, h * S, g * S, 0, w_out=wp, v_out=vp)
                e2e = (time.perf_counter() - t0) / reps
                info["e2e_host_pinned_forward"] = {"case": "a", "wavelet": "db4", "mode": "PERIODIC", "samples": total,
                                                   "s": round(e2e, 4), "gsamples_s": round(total / e2e / 1e9, 3)}
                print(f"end-to-end host (pinned) forward, case a db4 PERIODIC: {e2e * 1e3:.1f} ms, "
                      f"{total / e2e / 1e9:.3f} GSamples/s", flush=True)
                del xp, wp, vp
            except Exception as e:
                info["e2e_host_pinned_forward"] = {"error": str(e)}
                print(f"end-to-end host run failed: {e}", flush=True)
        del xs
        torch.cuda.empty_cache()

    # varlen over equal-length, case a, per direction
    ratios = {}
    for r in results:
        if r["case"] == "a" and r["path"] == "varlen":
            eq = next(q for q in results if q["case"] == "a" and q["path"] == "equal" and q["wavelet"] == r["wavelet"]
                      and q["mode"] == r["mode"] and q["direction"] == r["direction"])
            key = f"{r['wavelet']} {r['mode']} {r['direction']}"
            ratios[key] = round(r["gsamples_s"] / eq["gsamples_s"], 3)
    info["varlen_over_equal_case_a"] = ratios
    for k, v in ratios.items():
        print(f"varlen / equal-length, case a, {k}: {v:.3f}{'' if v >= 0.85 else '  (below the 0.85 target)'}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
