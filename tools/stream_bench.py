"""Per-block cost of BatchStreamingMODWT: the device stream state (vw_stream_process, one call per block) against the
chain it replaces (one vw_modwt_stream_level call per level plus the torch copies that assembled [history | block]
rows and cut the new histories).  One JSON line per workload:
    python tools/stream_bench.py [--blocks 200] [--rounds 3] [--out FILE]

Device-resident CUDA tensors; every figure is CUDA-event time over --blocks consecutive blocks of one stream after a
warm-up, divided by the block count, median of --rounds rounds in which the paths alternate.  Host time that keeps the
GPU waiting (Python, ctypes, torch) is part of a block's cost and so part of the figure.  `handle_per_level_us` is the
same state forced onto the generic per-level kernels (VW_FLAG_NO_FUSE: no tile or column kernels either).  `host_blocks_s`
is the end-to-end rate of the Python facade on host (numpy) blocks.  Before timing, both paths run the same seeded
blocks from fresh streams and must agree to 1e-12 * max|x|.  Workload (d) does not fit one CTA per row and takes the
per-level path inside the state."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import vectorwave_b200 as vw  # noqa: E402
from vectorwave_b200 import _native  # noqa: E402
from vectorwave_b200.modwt import SCALE  # noqa: E402

BM = vw.BoundaryMode
WORKLOADS = [   # (name, wavelet, mode, streams, block, levels)
    ("a_db4_256x256_J4_zero", "db4", BM.ZERO_PADDING, 256, 256, 4),
    ("b_sym8_4096x1024_J6_symmetric", "sym8", BM.SYMMETRIC, 4096, 1024, 6),
    ("c_db8_16x8192_J5_zero", "db8", BM.ZERO_PADDING, 16, 8192, 5),
    ("d_coif5_4x65536_J8_symmetric", "coif5", BM.SYMMETRIC, 4, 65536, 8),
]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


class OldChain:
    """the per-level chain of the previous Python facade, restated: per block J + 2 allocations, a copy of the block
    into the level-1 row, per level a history write, one vw_modwt_stream_level call and a clone of the new history"""

    def __init__(self, eng, hs, gs, levels, mode):
        self.eng, self.hs, self.gs, self.levels, self.mode = eng, hs, gs, levels, mode
        self.hl = [(hs.size - 1) << j for j in range(levels)]
        self.hist = None

    def process(self, x):
        import torch
        b, n = x.shape
        w = torch.empty((self.levels, b, n), dtype=torch.float64, device=x.device)
        v_final = torch.empty((b, n), dtype=torch.float64, device=x.device)
        exts = [torch.empty((b, h + n + (h + n) % 2), dtype=torch.float64, device=x.device) for h in self.hl]
        exts[0][:, self.hl[0]:self.hl[0] + n] = x
        if self.hist is None:
            self.hist = [None] * self.levels
        for j in range(self.levels):
            hl = self.hl[j]
            ext = exts[j][:, :hl + n]
            block = ext[:, hl:]
            if self.hist[j] is None:
                if self.mode == BM.ZERO_PADDING:
                    self.hist[j] = torch.zeros((b, hl), dtype=torch.float64, device=x.device)
                else:
                    m = np.mod(np.arange(hl) - hl, 2 * n)
                    self.hist[j] = block[:, torch.as_tensor(np.where(m < n, m, 2 * n - 1 - m), device=x.device)].contiguous()
            ext[:, :hl] = self.hist[j]
            v_out = exts[j + 1][:, self.hl[j + 1]:self.hl[j + 1] + n] if j + 1 < self.levels else v_final
            self.eng.stream_level(ext, hl, self.hs, self.gs, j + 1, w[j], v_out)
            self.hist[j] = ext[:, n:n + hl].clone()
        return w, v_final


def per_block_ms(run, blocks, nblocks):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(nblocks):
        run(blocks[k % len(blocks)])
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / nblocks


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("stream_bench needs a CUDA device")
    eng = vw.Engine.get(0)
    gpu = gpu_info()
    lines = []
    for name, wname, mode, b, n, levels in WORKLOADS:
        wav = vw.get_wavelet(wname)
        hs, gs = wav.lowPassDecomposition() * SCALE, wav.highPassDecomposition() * SCALE
        g = torch.Generator(device="cuda").manual_seed(1)
        blocks = [torch.randn((b, n), dtype=torch.float64, device="cuda", generator=g) for _ in range(4)]
        amax = max(float(torch.max(torch.abs(x))) for x in blocks)

        # same seeded blocks through both paths from fresh streams
        st, old = eng.stream_create(hs, gs, levels, mode.value), OldChain(eng, hs, gs, levels, mode)
        err = 0.0
        for x in blocks:
            wa, va = st.process(x)
            wb, vb = old.process(x)
            err = max(err, float(torch.max(torch.abs(wa - wb))), float(torch.max(torch.abs(va - vb))))
        torch.cuda.synchronize()
        assert err <= 1e-12 * amax, f"{name}: paths differ by {err:.3e}"

        w = torch.empty((levels, b, n), dtype=torch.float64, device="cuda")
        v = torch.empty((b, n), dtype=torch.float64, device="cuda")
        nofuse = eng.stream_create(hs, gs, levels, mode.value)
        runs = {"handle": lambda x: st.process(x, w_out=w, v_out=v),
                "handle_per_level": lambda x: nofuse.process(x, _native.FLAG_NO_FUSE, w_out=w, v_out=v),
                "old_chain": old.process}
        launches = {}
        for key, run in runs.items():
            per_block_ms(run, blocks, 20)           # warm-up
            n0 = eng.launch_count()
            run(blocks[0])
            launches[key] = eng.launch_count() - n0
        times = {k: [] for k in runs}
        for _ in range(args.rounds):
            for key, run in runs.items():
                times[key].append(per_block_ms(run, blocks, args.blocks))

        # host (numpy) blocks end to end through the facade
        hx = [x.cpu().numpy() for x in blocks]
        fac = vw.BatchStreamingMODWT.Builder().wavelet(wav).boundary(mode).levels(levels).build()
        fac.processMultiLevel(hx[0])
        nh = max(10, min(args.blocks, int(2e8 // (b * n * 8 * (levels + 2)))))
        t0 = time.perf_counter()
        for k in range(nh):
            fac.processMultiLevel(hx[k % len(hx)])
        host_rate = nh / (time.perf_counter() - t0)
        fac.close()
        st.close()
        nofuse.close()

        hist = (hs.size - 1) * ((1 << levels) - 1)
        rec = {
            "workload": name, "gpu": gpu, "streams": b, "block": n, "levels": levels, "wavelet": wname, "mode": mode.name,
            "handle_us": round(1e3 * float(np.median(times["handle"])), 2),
            "handle_per_level_us": round(1e3 * float(np.median(times["handle_per_level"])), 2),
            "old_chain_us": round(1e3 * float(np.median(times["old_chain"])), 2),
            "speedup_vs_old": round(float(np.median(times["old_chain"]) / np.median(times["handle"])), 2),
            "handle_launches_per_block": launches["handle"],
            "handle_per_level_launches_per_block": launches["handle_per_level"],
            "old_chain_engine_launches_per_block": launches["old_chain"],
            "old_chain_torch_copies_per_block": 2 * levels + 1,
            "bytes_per_sample_model_handle": round(8 * (levels + 2) + 16 * hist / n, 2),
            "bytes_per_sample_model_old_chain": 24 * levels + 16,
            "host_blocks_s": round(host_rate, 1),
            "max_abs_diff": err, "tolerance": 1e-12 * amax,
            "blocks_timed": args.blocks, "rounds": args.rounds,
        }
        print(json.dumps(rec), flush=True)
        lines.append(json.dumps(rec))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
