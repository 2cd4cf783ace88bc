"""Batched WaveletDenoiser (vw_wavelet_denoise) against vw_swt_denoise on the same shape, and against the per-signal
WaveletDenoiser loop.  One JSON line per workload:  python tools/denoise_batch_bench.py [--reps 20] [--out FILE]

Device-resident CUDA tensors, CUDA-event times, median of --reps calls after warm-up; three input sets rotate so that
successive calls do not find their input in L2 (126 MB) where a set is larger than it.  The two engine calls alternate
within one loop so both see the same clocks and neighbours.  The per-signal loop runs the existing single-signal
methods on the first 64 rows (host arrays, one row per call) and reports rows/s."""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import vectorwave_b200 as vw  # noqa: E402
from vectorwave_b200 import _native  # noqa: E402
from vectorwave_b200.denoising import ThresholdMethod as M, ThresholdType as T, WaveletDenoiser  # noqa: E402
from vectorwave_b200.modwt import multilevel_alignment  # noqa: E402

WORKLOADS = [   # (name, wavelet, boundary, batch, n, levels, method)
    ("a_db4_4096x4096_J4_periodic_universal", vw.Daubechies.DB4, vw.BoundaryMode.PERIODIC, 4096, 4096, 4, M.UNIVERSAL),
    ("b_db4_4096x4096_J4_periodic_bayes", vw.Daubechies.DB4, vw.BoundaryMode.PERIODIC, 4096, 4096, 4, M.BAYES),
    ("c_db8_256x2^20_J6_zero_minimax", vw.Daubechies.DB8, vw.BoundaryMode.ZERO_PADDING, 256, 1 << 20, 6, M.MINIMAX),
    ("d_db4_1024x4096_J4_periodic_sure", vw.Daubechies.DB4, vw.BoundaryMode.PERIODIC, 1024, 4096, 4, M.SURE),
]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("denoise_batch_bench needs a CUDA device")
    eng = vw.Engine.get(0)
    gpu = gpu_info()
    lines = []
    for name, wav, mode, b, n, levels, method in WORKLOADS:
        den = WaveletDenoiser(wav, mode)
        ml = vw.MultiLevelMODWTTransform(wav, mode)
        align, order = multilevel_alignment(wav, mode, levels)
        code = getattr(_native, "THR_" + method.value)
        g = torch.Generator(device="cuda").manual_seed(1)
        sets = [torch.randn((b, n), dtype=torch.float64, device="cuda", generator=g) for _ in range(3)]

        def ours(x):
            return eng.wavelet_denoise(x, ml._hs, ml._gs, levels, mode.value, align, order, True, code, 0.0, True)

        def swt(x):
            return eng.denoise(x, ml._hs, ml._gs, levels, mode.value, align, order, -1.0, True)

        for x in sets:
            ours(x)
            swt(x)
        torch.cuda.synchronize()
        t_ours, t_swt = [], []
        for i in range(args.reps):
            for fn, acc in ((ours, t_ours), (swt, t_swt)):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn(sets[i % 3])
                e1.record()
                e1.synchronize()
                acc.append(e0.elapsed_time(e1))
        out, _ = ours(sets[0])
        rows = min(64, b)
        x_host = sets[0][:rows].cpu().numpy()
        den.denoiseMultiLevel(x_host[0], levels, method, T.SOFT)   # warm-up of the per-signal path
        t0 = time.perf_counter()
        per_row = [den.denoiseMultiLevel(x_host[r], levels, method, T.SOFT) for r in range(rows)]
        loop_s = time.perf_counter() - t0
        diff = max(float(np.max(np.abs(out[r].cpu().numpy() - per_row[r]))) for r in range(rows))
        ms, ms_swt = float(np.median(t_ours)), float(np.median(t_swt))
        line = {"workload": name, "gpu_and_power_limit": gpu, "batch": b, "n": n, "levels": levels,
                "method": method.value, "reps": args.reps, "input_set_mb": round(b * n * 8 / 2 ** 20, 1),
                "wavelet_denoise_ms": round(ms, 4), "swt_denoise_ms": round(ms_swt, 4),
                "ratio_to_swt": round(ms / ms_swt, 3), "batch_rows_per_s": round(b / (ms * 1e-3), 1),
                "per_signal_loop_rows_per_s": round(rows / loop_s, 1), "per_signal_rows": rows,
                "max_abs_batch_minus_per_row": diff}
        if name.startswith("a_"):
            # decompose 8(J+2) + median 3 x 8 + reconstruct 8(J+2) bytes per sample (the issue's model)
            model = (8 * (levels + 2) * 2 + 24) * b * n
            line["model_bytes"] = model
            line["model_gb_per_s"] = round(model / (ms * 1e-3) / 1e9, 1)
        print(json.dumps(line), flush=True)
        lines.append(line)
        del sets
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
