#!/usr/bin/env python
"""bench.py -- MODWT forward + inverse throughput (GSamples/s) on B200, per BASELINE.json.

A "step" is one pass of the hot path over one batch of synthetic input: multi-level MODWT decompose
(forward) followed by reconstruct (inverse) of every signal of the workload.  Default workload (N=1):
BASELINE.json configs[1], the extensions batch-facade shape 4096 x 4096 fp64 signals, db4, J=4, PERIODIC.

  value     whole-job GSamples/s (B*N input samples per fwd+inv step), inputs resident in HBM
  e2e       same metric through the public host-buffer API (BatchMODWT.multiLevelAoS + inverseMultiLevelAoS
            -> C ABI with HOST pointers): H2D of the signals, D2H of all coefficients, H2D of the coefficients
            and D2H of the reconstruction are all inside the timed region
  roofline  dominant kernel (the analysis tile kernel) against the measured HBM copy peak: algorithmic bytes
            (24 B/sample/level, SURVEY.md 8d) per launch / its CUDA-event duration; the FP64 roof is measured in the
            same run (vw_probe_fp64)
  cpu_baseline  the oracle's C restatement of the reference's dense loops (kind "port"; the reference is Java and
            no JVM exists on the box) on all host cores, same workload (bounded sample) = the reference's
            structured-concurrency baseline; `variants` adds SURVEY 8(d)'s one-thread core scalar and SoA batch lanes
  extra     measured in the same run, beside the headline (VERDICT r1 item 1): the other BASELINE configs on one GPU
            (c3, c4, c5 in both of its boundary modes, c5_denoise with its own e2e), the span-sharded long signal
            (`span`, strong scaling over the N ranks incl. N=1 self-wrap, halo exchange timed separately), BASELINE
            config #3 as written (`batch_strong_c3`: 1024 signals SPLIT over the N ranks), the small-call latencies
            from a compiled host (`c1_latency_us`), and the decompose -> threshold -> reconstruct pipeline with the
            coefficients resident in HBM (`e2e_resident_result`, 16 B/sample over PCIe instead of 16*(J+2))

Multi-GPU (torchrun, one rank per GPU): the batch shards by signal with no communication (weak scaling: every
rank runs the full per-GPU workload); `--workload span` runs one long coif5 signal span-sharded with NCCL halo
exchange.  `--impl reference` times the CPU restatement only (rank 0; other ranks exit).
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "GSamples/s MODWT fwd+inv fp64 (J levels)"
UNIT = "GSamples/s"
S = 1.0 / math.sqrt(2.0)
MODES = ("PERIODIC", "ZERO_PADDING", "SYMMETRIC")

WORKLOADS = {
    # name: (wavelet, batch, n, levels, boundary mode)
    "batch4096x4096_db4_J4": ("db4", 4096, 4096, 4, 0),
    "batch4096x4096_haar_J4": ("haar", 4096, 4096, 4, 0),
    "batch16x4096_db4_J4": ("db4", 16, 4096, 4, 0),
    "batch1024x65536_sym8_J8": ("sym8", 1024, 65536, 8, 0),
    "single2p28_coif5_J10": ("coif5", 1, 1 << 28, 10, 0),
    "batch256x1M_db8_J6": ("db8", 256, 1 << 20, 6, 0),
}
DEFAULT = "batch4096x4096_db4_J4"


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def n_sets(b, n, levels):
    """rotating input / output sets so no step finds its inputs in L2 (each set is far larger than L2 anyway)"""
    return 1 if (levels + 3) * b * n * 8 * 3 > 60e9 else 3


def config_of(workload):
    """The SAME dict from both arms (the driver compares them)."""
    wname, b, n, levels, mode = WORKLOADS[workload]
    return {"workload": workload, "wavelet": wname, "batch_per_gpu": b, "signal_length": n, "levels": levels,
            "boundary": MODES[mode], "sharding": "by signal, no communication",
            "l2": f"{n_sets(b, n, levels)} rotating input/output sets of {(levels + 3) * b * n * 8 / 2**20:.0f} MiB each "
                  "(> 126 MB L2); inputs larger than L2"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def _cpus_of(spec):
    cpus = set()
    for part in spec.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def bind_near_gpu(props, index):
    """Multi-rank runs: keep this process (and the pinned host buffers it first-touches) on the NUMA node the GPU hangs
    off, so eight ranks do not push their PCIe traffic across the socket link.  sysfs first; containers often hide it
    (numa_node = -1), so the fallback is the CPU-affinity column of `nvidia-smi topo -m`.  Best effort."""
    try:
        bdf = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node >= 0:
            cpus = _cpus_of(open(f"/sys/devices/system/node/node{node}/cpulist").read()) & os.sched_getaffinity(0)
            if cpus:
                os.sched_setaffinity(0, cpus)
                return {"node": node, "cpus": len(cpus), "source": "sysfs"}
    except Exception:
        pass
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        header = None
        for ln in out.splitlines():
            cols = [c.strip() for c in ln.split("\t") if c.strip()]
            if header is None and any(c.startswith("CPU Affinity") for c in cols):
                header = cols
                continue
            if header and cols and cols[0] == f"GPU{index}":
                # the row has one leading name column the header lacks
                k = [i for i, c in enumerate(header) if c.startswith("CPU Affinity")][0] + 1
                cpus = _cpus_of(cols[k]) & os.sched_getaffinity(0)
                numa = cols[k + 1] if k + 1 < len(cols) else None
                if cpus:
                    os.sched_setaffinity(0, cpus)
                    return {"node": numa, "cpus": len(cpus), "source": "nvidia-smi topo -m"}
    except Exception:
        pass
    return None


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def traffic_of(key):
    tr = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(tr)).get(key)
    except Exception:
        return None


def cpu_port(workload, threads, budget_rows=None, inverse=True):
    """Times the CPU restatement of the reference's dense loops on a bounded sample of the workload."""
    import numpy as np
    from oracle import cref
    from oracle.wavelets import filters
    wname, b, n, levels, mode = WORKLOADS[workload]
    h, g, wid = filters(wname)
    macs_per_sample = 2 * sum((len(h) - 1) * (1 << j) + 1 for j in range(levels)) * (2 if inverse else 1)
    # ~1.5e9 dense MAC/s/core: size the sample for roughly 10 s of wall time
    target = 10.0 * 1.2e9 * max(threads, 1)
    n_s = min(n, 1 << 20)
    rows = max(1, min(b, int(target / (macs_per_sample * n_s)))) if budget_rows is None else budget_rows
    rows = max(rows, min(b, threads))
    x = np.random.default_rng(42).standard_normal((rows, n_s))
    cref.lib()
    t0 = time.perf_counter()
    cref.batch_fwd_inv(x, h, g, levels, mode, wid, dense=True, threads=threads, inverse=inverse)
    dt = time.perf_counter() - t0
    return {"value": rows * n_s / dt * 1e-9, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{rows} x {n_s} of the {b} x {n} workload, {wname} J={levels}, dense upsampled taps as the "
                      f"reference (Sum_j 2*L_j MACs/sample/direction), {dt:.2f} s, pthread work queue over signals",
            "seconds": dt}


def cpu_variants(workload):
    """SURVEY 8(d)'s other two CPU baselines on one host thread, ~2 s each: (1) the core scalar path (one signal after
    the other, dense taps, forward + inverse) and (2) the extensions' SoA batch path (lanes = signals, dense taps,
    forward only as in BatchSIMDMODWT.batchMultiLevelMODWTSoA)."""
    import numpy as np
    from oracle import cref
    from oracle.wavelets import filters
    wname, b, n, levels, mode = WORKLOADS[workload]
    h, g, wid = filters(wname)
    macs_fwd = 2 * sum((len(h) - 1) * (1 << j) + 1 for j in range(levels))
    n_s = min(n, 1 << 16)
    out = []
    rows = max(1, min(b, int(2.0 * 0.4e9 / (2 * macs_fwd * n_s))))
    x = np.random.default_rng(42).standard_normal((rows, n_s))
    t0 = time.perf_counter()
    cref.batch_fwd_inv(x, h, g, levels, mode, wid, dense=True, threads=1, inverse=True)
    dt = time.perf_counter() - t0
    out.append({"name": "core_scalar_1_thread", "value": rows * n_s / dt * 1e-9, "unit": UNIT, "cores": 1,
                "sample": f"{rows} x {n_s}, forward + inverse, {dt:.2f} s"})
    if mode == 0:
        lanes = max(1, min(b, int(2.0 * 0.9e9 / (macs_fwd * n_s))))
        xs = np.ascontiguousarray(np.random.default_rng(43).standard_normal((lanes, n_s)).T).reshape(-1)
        t0 = time.perf_counter()
        cref.batch_soa_decompose(xs, lanes, n_s, h, g, levels)
        dt = time.perf_counter() - t0
        out.append({"name": "soa_batch_lanes_1_thread_forward_only", "value": lanes * n_s / dt * 1e-9,
                    "unit": "GSamples/s (forward only)", "cores": 1,
                    "sample": f"{lanes} lanes x {n_s}, batchMultiLevelMODWTSoA restated (gcc -O2 autovectorised), {dt:.2f} s"})
    return out


def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    vals = []
    for _ in range(args.warmup):
        cpu_port(args.workload, threads, budget_rows=max(threads, 8))
    cb = None
    for _ in range(max(1, args.steps)):
        cb = cpu_port(args.workload, threads, budget_rows=args.ref_rows)
        vals.append(cb["value"])
    value = statistics.median(vals)
    cb["value"] = value
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_of(args.workload),
            "cpu_baseline": cb,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "CPU restatement (oracle port) of the reference's scalar loops; the reference is pure Java and "
                    "no JVM exists on the box (probed: gpurun_out/jdk_probe.txt, DESIGN.md)"}
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------------------------------
# extra block
# ---------------------------------------------------------------------------------------------------------------------
class Ctx:
    """what the extra measurements share"""

    def __init__(self, torch, dist, vw, eng, dev, rank, world, peak, fp64_peak):
        self.torch, self.dist, self.vw, self.eng, self.dev = torch, dist, vw, eng, dev
        self.rank, self.world, self.peak, self.fp64_peak = rank, world, peak, fp64_peak

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        if self.world == 1:
            return ms
        t = self.torch.tensor([ms], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, reps, warm=2):
        """CUDA-event time per call of fn over `reps` calls (ms), max over ranks, barrier on both sides"""
        torch = self.torch
        for _ in range(warm):
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1) / reps)

    def free(self):
        import gc
        gc.collect()
        self.torch.cuda.empty_cache()


def roofline_entry(c, key, l, levels, samples, fwd_ms, inv_ms, launches_fwd, launches_inv):
    """whole-direction roofline of a config: 24*J B/sample/direction over the measured HBM copy peak, FP64 beside it"""
    alg = 24.0 * levels * samples
    step_ms = fwd_ms + inv_ms
    return {"bound": "hbm", "achieved": 2.0 * alg / step_ms * 1e-6, "peak": c.peak, "unit": "GB/s",
            "frac": 2.0 * alg / step_ms * 1e-6 / c.peak, "traffic": traffic_of(key),
            "forward_ms": fwd_ms, "inverse_ms": inv_ms, "forward_frac": alg / fwd_ms * 1e-6 / c.peak,
            "inverse_frac": alg / inv_ms * 1e-6 / c.peak, "launches_forward": launches_fwd, "launches_inverse": launches_inv,
            "fp64_tflops_achieved": 2.0 * 4.0 * l * levels * samples / step_ms * 1e-9, "fp64_tflops_peak_measured": c.fp64_peak,
            "frac_of_fp64": (2.0 * 4.0 * l * levels * samples / step_ms * 1e-9) / c.fp64_peak if c.fp64_peak else None,
            "fp64_note": "algorithmic FLOPs of the direct form (4L per sample, level and direction, SURVEY 8d)" +
                         ("; coif5's levels 3-10 run in lattice form and execute L + 2 FP64 instructions per sample and level instead of 2L" if l == 30 else "")}


def extra_batch(c, key, workload, mode, rows=None, reps=8):
    """forward + inverse of `rows` signals of a batch workload in boundary `mode`, device-resident (this rank's share)"""
    from vectorwave_b200.modwt import multilevel_alignment
    torch, vw = c.torch, c.vw
    wname, b, n, levels, _ = WORKLOADS[workload]
    rows = b if rows is None else rows
    wv = vw.get_wavelet(wname)
    hs, gs = wv.lowPassDecomposition() * S, wv.highPassDecomposition() * S
    bm = [vw.BoundaryMode.PERIODIC, vw.BoundaryMode.ZERO_PADDING, vw.BoundaryMode.SYMMETRIC][mode]
    align, order = multilevel_alignment(wv, bm, levels)
    gen = torch.Generator(device=c.dev)
    gen.manual_seed(1234 + c.rank)
    x = torch.randn((rows, n), dtype=torch.float64, device=c.dev, generator=gen)
    w = torch.empty((levels, rows, n), dtype=torch.float64, device=c.dev)
    v = torch.empty((rows, n), dtype=torch.float64, device=c.dev)
    xr = torch.empty((rows, n), dtype=torch.float64, device=c.dev)
    l0 = c.eng.launch_count()
    c.eng.forward(x, hs, gs, levels, mode, 0, w, v)
    lf = c.eng.launch_count() - l0
    c.eng.inverse(w, v, hs, gs, mode, align, order, out=xr)
    li = c.eng.launch_count() - l0 - lf
    fwd_ms = c.timed(lambda: c.eng.forward(x, hs, gs, levels, mode, 0, w, v), reps)
    inv_ms = c.timed(lambda: c.eng.inverse(w, v, hs, gs, mode, align, order, out=xr), reps)
    rt = float((xr - x).abs().max()) if mode == 0 else None
    out = {"workload": workload, "boundary": MODES[mode], "rows_this_rank": rows, "ms_per_step": fwd_ms + inv_ms,
           "round_trip_max_abs_err": rt, "l2": f"working set {(levels + 3) * rows * n * 8 / 2**30:.1f} GiB per rank, far larger than L2",
           "_l": int(hs.size), "_levels": levels, "_n": n, "_lf": lf, "_li": li, "_fwd": fwd_ms, "_inv": inv_ms}
    del x, w, v, xr
    c.free()
    return out


def finish_batch(c, key, d, total_rows):
    """adds value + roofline to an extra_batch record (value over ALL ranks' rows; roofline per GPU)"""
    n, levels = d.pop("_n"), d.pop("_levels")
    l, lf, li, fwd, inv = d.pop("_l"), d.pop("_lf"), d.pop("_li"), d.pop("_fwd"), d.pop("_inv")
    d["value"] = total_rows * n / d["ms_per_step"] * 1e-6
    d["unit"] = UNIT
    d["roofline"] = roofline_entry(c, key, l, levels, d["rows_this_rank"] * n, fwd, inv, lf, li)
    d["roofline_model_gsamples"] = c.peak / (48.0 * levels) * c.world
    d["frac_of_roofline_model"] = d["value"] / d["roofline_model_gsamples"]
    return d


def extra_denoise(c, mode, reps=4):
    """BASELINE config #5 as written: SWT denoise (decompose, universal soft threshold, reconstruct), db8 J=6, 256 x 2^20,
    device-resident and end to end through HOST buffers (8 B/sample each way)."""
    import numpy as np
    from vectorwave_b200.modwt import multilevel_alignment
    torch, vw = c.torch, c.vw
    wname, b, n, levels, _ = WORKLOADS["batch256x1M_db8_J6"]
    wv = vw.get_wavelet(wname)
    hs, gs = wv.lowPassDecomposition() * S, wv.highPassDecomposition() * S
    bm = [vw.BoundaryMode.PERIODIC, vw.BoundaryMode.ZERO_PADDING, vw.BoundaryMode.SYMMETRIC][mode]
    align, order = multilevel_alignment(wv, bm, levels)
    gen = torch.Generator(device=c.dev)
    gen.manual_seed(77)
    x = torch.randn((b, n), dtype=torch.float64, device=c.dev, generator=gen)
    l0 = c.eng.launch_count()
    c.eng.denoise(x, hs, gs, levels, mode, align, order, -1.0, True)
    launches = c.eng.launch_count() - l0
    ms = c.timed(lambda: c.eng.denoise(x, hs, gs, levels, mode, align, order, -1.0, True), reps, warm=1)
    del x
    c.free()
    # end to end: host signal in, host denoised signal out
    eb = 64
    xh = c.eng.pinned_empty((eb, n))
    xh[...] = np.random.default_rng(5).standard_normal((eb, n))
    c.eng.denoise(xh, hs, gs, levels, mode, align, order, -1.0, True)
    t0 = time.perf_counter()
    for _ in range(3):
        c.eng.denoise(xh, hs, gs, levels, mode, align, order, -1.0, True)
    dt = (time.perf_counter() - t0) / 3
    out = {"workload": "batch256x1M_db8_J6 SWT denoise (universal soft threshold)", "boundary": MODES[mode],
           "value": b * n / ms * 1e-6, "unit": UNIT, "ms_per_step": ms, "gpu_launches_per_step": launches,
           "roofline": {"bound": "hbm", "achieved": 48.0 * levels * b * n / ms * 1e-6, "peak": c.peak, "unit": "GB/s",
                        "frac": 48.0 * levels * b * n / ms * 1e-6 / c.peak, "traffic": traffic_of(f"c5_denoise_{MODES[mode]}"),
                        "note": "48*J algorithmic bytes per sample (decompose + reconstruct; the threshold rides on the synthesis "
                                "loads; the universal-threshold selection adds 3 passes over W_1)"},
           "e2e": {"value": eb * n / dt * 1e-9, "unit": UNIT, "h2d_bytes_per_step": eb * n * 8, "d2h_bytes_per_step": eb * n * 8,
                   "batch": eb, "api": "vw_swt_denoise with HOST (pinned) buffers"}}
    del xh
    c.free()
    return out


def extra_span(c, reps=4):
    """BASELINE config #4: one 2^28-sample coif5 J=10 PERIODIC signal span-sharded over the ranks (strong scaling; at one
    rank the ring wraps onto itself through the same code path).  The halo exchange is timed separately."""
    from vectorwave_b200.sharded import SpanShardedMODWT
    torch, vw = c.torch, c.vw
    n_total, levels = 1 << 28, 10
    n_local = n_total // c.world
    sh = SpanShardedMODWT(vw.Coiflet.COIF5, levels, n_local, vw.BoundaryMode.PERIODIC, rank=c.rank, world=c.world, engine=c.eng)
    gen = torch.Generator(device=c.dev)
    gen.manual_seed(42 + c.rank)
    x = torch.randn(n_local, dtype=torch.float64, device=c.dev, generator=gen)
    state = {"res": sh.forward(x)}

    def step():
        state["res"] = sh.forward(x, result=state["res"])
        state["xr"] = sh.inverse(state["res"])
    l0 = c.eng.launch_count()
    step()
    launches = c.eng.launch_count() - l0
    ms = c.timed(step, reps, warm=1)
    rt = float((state["xr"] - x).abs().max())
    ex_ms = c.timed(lambda: sh.exchange_only(state["res"]), 10, warm=2)
    model = c.peak / (48.0 * levels)
    out = {"workload": "single2p28_coif5_J10", "scaling": "strong", "value": n_total / ms * 1e-6, "unit": UNIT,
           "ms_per_step": ms, "halo_exchange_ms_per_step": ex_ms,
           "halo_exchange_note": "both directions' exchanges alone (analysis: lead samples of x; synthesis: pack, send/recv, unpack), "
                                 "CUDA events, max over ranks; NCCL send/recv over NVLink at N>1, a local copy at N=1",
           "halo_bytes_per_rank_per_step": int((sh.plan.lead + sh.plan.inverse_msg) * 8) if sh.plan is not None else None,
           "span_per_rank": n_local, "gpu_launches_per_step": launches, "round_trip_max_abs_err": rt,
           "roofline": {"bound": "hbm", "achieved": 48.0 * levels * n_local / ms * 1e-6, "peak": c.peak, "unit": "GB/s",
                        "frac": 48.0 * levels * n_local / ms * 1e-6 / c.peak, "traffic": traffic_of("single2p28_coif5_J10"),
                        "fp64_tflops_achieved": 8.0 * 30 * levels * n_local / ms * 1e-9, "fp64_tflops_peak_measured": c.fp64_peak,
                        "frac_of_fp64": 8.0 * 30 * levels * n_local / ms * 1e-9 / c.fp64_peak if c.fp64_peak else None,
                        "note": "per GPU, whole step.  fp64_* count the DIRECT form's 4L FLOP per sample, level and direction (the "
                                "algorithmic work of SURVEY 8d); levels 3-10 run in lattice form (L + 2 FP64 instructions instead of 2L, "
                                "two levels per pass at 32 B/sample), so the FP64 pipe executes about 60 % of that figure"},
           "roofline_model_gsamples": model * c.world, "frac_of_roofline_model": n_total / ms * 1e-6 / (model * c.world),
           "l2": "per-rank working set 26 GiB / world, far larger than L2"}
    assert rt < 1e-9, f"span round trip error {rt}"
    del x, state, sh
    c.free()
    return out


def extra_span_one_thread(c, reps=4):
    """The same span-sharded 2^28 coif5 J=10 transform driven the way a JVM would: ONE host thread, every GPU of the job
    through vw_init_multi / vw_modwt_forward_sharded / vw_modwt_inverse_sharded (halos as peer copies over NVLink).  Runs on
    rank 0 while the other ranks wait; host wall clock around synchronous calls (each returns when every device is done)."""
    from vectorwave_b200 import _native
    torch, vw = c.torch, c.vw
    world = c.world
    n_total, levels = 1 << 28, 10
    n_local = n_total // world
    wv = vw.Coiflet.COIF5
    hs, gs = wv.lowPassDecomposition() * S, wv.highPassDecomposition() * S
    plan = _native.span_plan(hs.size, levels, n_local, world)
    lead, lead_w, pad = int(plan.lead), int(plan.lead_w), int(plan.pad)
    row = lead_w + n_local + pad
    devices = list(range(world))
    me = _native.MultiEngine(devices)
    try:
        xext, w, v, xo = [], [], [], []
        for d in devices:
            dev = torch.device("cuda", d)
            gen = torch.Generator(device=dev)
            gen.manual_seed(42 + d)
            e = torch.empty(lead + n_local, dtype=torch.float64, device=dev)
            e[lead:] = torch.randn(n_local, dtype=torch.float64, device=dev, generator=gen)
            xext.append(e)
            w.append(torch.empty((levels, row), dtype=torch.float64, device=dev))
            v.append(torch.empty(n_local + pad, dtype=torch.float64, device=dev))
            xo.append(torch.empty(n_local, dtype=torch.float64, device=dev))
        for d in devices:
            torch.cuda.synchronize(d)
        l0 = me.launch_count()
        ex_f = me.forward(plan, xext, hs, gs, 0, w, v, timed=True)
        ex_i = me.inverse(plan, w, v, hs, gs, 0, 0, xo, timed=True)
        launches = me.launch_count() - l0
        t0 = time.perf_counter()
        for _ in range(reps):
            me.forward(plan, xext, hs, gs, 0, w, v)
            me.inverse(plan, w, v, hs, gs, 0, 0, xo)
        ms = (time.perf_counter() - t0) / reps * 1e3
        rt = max(float((xo[d] - xext[d][lead:]).abs().max()) for d in devices)
    finally:
        me.close()
    assert rt < 1e-9, f"sharded ABI round trip error {rt}"
    model = c.peak / (48.0 * levels) * world
    out = {"workload": "single2p28_coif5_J10", "scaling": "strong", "driver": "one host thread, vw_init_multi over "
           f"{world} device(s), peer-copy halo exchange", "value": n_total / ms * 1e-6, "unit": UNIT, "ms_per_step": ms,
           "halo_exchange_ms": {"analysis": ex_f, "synthesis": ex_i, "note": "device time of the slowest receiving copy, CUDA events"},
           "gpu_launches_per_step": launches, "round_trip_max_abs_err": rt, "timing": "host wall clock around synchronous calls",
           "roofline_model_gsamples": model, "frac_of_roofline_model": n_total / ms * 1e-6 / model}
    del xext, w, v, xo
    c.free()
    return out


def extra_latency(local_rank):
    exe = os.path.join(ROOT, "tools", "_build", "latency")
    if not os.path.exists(exe):
        return {"unavailable": "tools/_build/latency not built (python -c 'import __graft_entry__ as g; g.build()')"}
    try:
        out = subprocess.run([exe, str(local_rank), "2000"], capture_output=True, text=True, timeout=120)
        return json.loads(out.stdout.strip().splitlines()[-1])
    except Exception as ex:
        return {"unavailable": f"latency tool failed: {ex}"}


def extra_resident(c, workload, reps=5):
    """decompose (host signal in) -> universal soft threshold on the resident coefficients -> reconstruct (host signal out):
    the MultiLevelMODWTResult never leaves HBM (vw_modwt_decompose_h / vw_result_* / vw_modwt_reconstruct_h)."""
    import numpy as np
    wname, b, n, levels, mode = WORKLOADS[workload]
    wv = c.vw.get_wavelet(wname)
    hs, gs = wv.lowPassDecomposition() * S, wv.highPassDecomposition() * S
    xh = c.eng.pinned_empty((b, n))
    xh[...] = np.random.default_rng(11).standard_normal((b, n))
    oh = c.eng.pinned_empty((b, n))
    res = c.eng.decompose_resident(xh, hs, gs, levels, mode)

    def step():
        c.eng.decompose_resident(xh, hs, gs, levels, mode, result=res)
        res.universal_threshold(True)
        res.reconstruct(hs, gs, mode, out=oh)
    step()
    t0 = time.perf_counter()
    for _ in range(reps):
        step()
    dt = (time.perf_counter() - t0) / reps
    # the same pipeline with every coefficient crossing PCIe (the double[] API): forward, threshold on the host copy, inverse
    out = {"value": b * n / dt * 1e-9, "unit": UNIT, "h2d_bytes_per_step": b * n * 8, "d2h_bytes_per_step": b * n * 8 + b * 8,
           "pipeline": "decompose -> universal soft threshold -> reconstruct", "workload": workload, "ms_per_step": dt * 1e3,
           "note": f"16 B/sample over PCIe; the all-copies e2e of this line moves {16 * (levels + 2)} B/sample"}
    res.free()
    return out


def pcie_probe(c):
    """achieved pinned-copy rate per direction on this rank (1 GiB, best of 3)"""
    import ctypes as C
    nbytes = 1 << 30
    host = c.eng.pinned_empty((nbytes // 8,))
    devbuf = c.torch.empty(nbytes // 8, dtype=c.torch.float64, device=c.dev)
    lib, ctx = c.eng.lib, c.eng.ctx
    best = {"h2d": 0.0, "d2h": 0.0}
    for _ in range(3):
        t0 = time.perf_counter()
        lib.vw_copy_h2d(ctx, C.c_void_p(devbuf.data_ptr()), C.c_void_p(host.ctypes.data), nbytes)
        best["h2d"] = max(best["h2d"], nbytes / (time.perf_counter() - t0) * 1e-9)
        t0 = time.perf_counter()
        lib.vw_copy_d2h(ctx, C.c_void_p(host.ctypes.data), C.c_void_p(devbuf.data_ptr()), nbytes)
        best["d2h"] = max(best["d2h"], nbytes / (time.perf_counter() - t0) * 1e-9)
    del host, devbuf
    c.free()
    return {"h2d_gbs": best["h2d"], "d2h_gbs": best["d2h"], "bytes": nbytes}


DUMP_BYTES = 48 << 20   # --dump-outputs writes at most this much


def dump_outputs(path, w, v, xr):
    """Writes W [J][B][N], V_J [B][N] and the reconstruction [B][N] of one step as w.npy [J][P], v.npy [P] and xr.npy [P]
    (float64): the values at P (signal, time) positions drawn once from a fixed seed, the same for every array and every
    run of a workload, or at every position when the whole output fits in DUMP_BYTES."""
    import numpy as np
    import torch
    levels, total = w.shape[0], v.numel()
    keep = min(total, DUMP_BYTES // (8 * (levels + 2)))
    idx = np.arange(total) if keep == total else np.sort(np.random.default_rng(1234).choice(total, keep, replace=False))
    idx = torch.as_tensor(idx, device=v.device)
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "w.npy"), w.reshape(levels, total).index_select(1, idx).cpu().numpy())
    np.save(os.path.join(path, "v.npy"), v.reshape(total).index_select(0, idx).cpu().numpy())
    np.save(os.path.join(path, "xr.npy"), xr.reshape(total).index_select(0, idx).cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT, choices=sorted(WORKLOADS) + ["span"])
    ap.add_argument("--ref-rows", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (a seeded sample of W, V_J and the "
                         "reconstruction, float64) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload == "span"):
        ap.error("--dump-outputs applies to the batch workloads of --impl b200")
    if args.impl == "reference":
        if args.workload == "span":
            args.workload = "single2p28_coif5_J10"
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import numpy as np
    import torch
    import torch.distributed as dist

    import vectorwave_b200 as vw

    world = env_int("WORLD_SIZE", 1)
    rank = env_int("RANK", 0)
    local_rank = env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the MODWT engine has no CPU path")
    torch.cuda.set_device(local_rank)
    numa = bind_near_gpu(torch.cuda.get_device_properties(local_rank), local_rank) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    cpu_group = dist.new_group(backend="gloo") if world > 1 else None
    dev = torch.device("cuda", local_rank)
    eng = vw.Engine.get(local_rank)
    peak, peak_src = measured_peaks()
    try:
        fp64_peak, sm_max = eng.probe_fp64()
    except Exception:
        fp64_peak, sm_max = None, None
    c = Ctx(torch, dist, vw, eng, dev, rank, world, peak, fp64_peak)

    if args.workload == "span":
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        d = extra_span(c, reps=args.steps)
        clocks = sampler.stop() if rank == 0 else None
        if rank == 0:
            line = {"metric": METRIC, "value": d["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                    "warmup": 1, "ms_per_step": d["ms_per_step"], "higher_is_better": True, "scaling": "strong",
                    "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                    "config": {"workload": "single2p28_coif5_J10", "wavelet": "coif5", "signal_length": 1 << 28, "levels": 10,
                               "boundary": "PERIODIC", "sharding": f"contiguous spans of {d['span_per_rank']} samples, one halo "
                               "exchange per direction (NCCL send/recv)", "l2": d["l2"]},
                    "roofline": d["roofline"], "cpu_baseline": None, "e2e": None, "gpu_launches": d["gpu_launches_per_step"] * args.steps,
                    "clocks": clocks, "round_trip_max_abs_err": d["round_trip_max_abs_err"],
                    "halo_exchange_ms_per_step": d["halo_exchange_ms_per_step"],
                    "roofline_model_gsamples": d["roofline_model_gsamples"], "frac_of_roofline_model": d["frac_of_roofline_model"]}
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return 0

    wname, b, n, levels, mode = WORKLOADS[args.workload]
    wv = vw.get_wavelet(wname)
    hs, gs = wv.lowPassDecomposition() * S, wv.highPassDecomposition() * S

    # batch sharding by signal: weak scaling, every rank owns a full per-GPU batch; no data-path collective
    nsets = n_sets(b, n, levels)
    gen = torch.Generator(device=dev)
    gen.manual_seed(42 + rank)
    xs = [torch.randn((b, n), dtype=torch.float64, device=dev, generator=gen) for _ in range(nsets)]
    ws = [torch.empty((levels, b, n), dtype=torch.float64, device=dev) for _ in range(nsets)]
    vs = [torch.empty((b, n), dtype=torch.float64, device=dev) for _ in range(nsets)]
    xr = [torch.empty((b, n), dtype=torch.float64, device=dev) for _ in range(nsets)]

    def step(i):
        k = i % nsets
        eng.forward(xs[k], hs, gs, levels, mode, 0, ws[k], vs[k])
        eng.inverse(ws[k], vs[k], hs, gs, mode, None, 0, out=xr[k])

    for i in range(args.warmup):
        step(i)
    c.barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c.barrier()
    e0.record()
    for i in range(args.steps):
        step(i)
    e1.record()
    c.barrier()
    launches = eng.launch_count() - l0
    ms_step = c.max_over_ranks(e0.elapsed_time(e1)) / args.steps
    value = world * b * n / ms_step * 1e-6
    if args.dump_outputs and rank == 0:
        last = (args.steps - 1) % nsets
        dump_outputs(args.dump_outputs, ws[last], vs[last], xr[last])

    # correctness guard inside the bench: the timed path must really invert (PERIODIC round trip)
    rt = float((xr[0] - xs[0]).abs().max())
    assert rt < 1e-9, f"round trip error {rt}: the timed path does not invert"

    # ---- roofline of the dominant kernel: the analysis launch(es), timed alone with CUDA events -------
    reps = max(10, args.steps, int(80.0 / max(ms_step / 2.0, 1e-3)))   # >= 80 ms per direction: stable event timing, clock samples
    reps = min(reps, 2000)
    for _ in range(3):
        eng.forward(xs[0], hs, gs, levels, mode, 0, ws[0], vs[0])
    torch.cuda.synchronize()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    lf0 = eng.launch_count()
    f0.record()
    for i in range(reps):
        k = i % nsets
        eng.forward(xs[k], hs, gs, levels, mode, 0, ws[k], vs[k])
    f1.record()
    torch.cuda.synchronize()
    fwd_ms = f0.elapsed_time(f1) / reps
    fwd_launches = (eng.launch_count() - lf0) // reps
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for i in range(reps):
        k = i % nsets
        eng.inverse(ws[k], vs[k], hs, gs, mode, None, 0, out=xr[k])
    g1.record()
    torch.cuda.synchronize()
    inv_ms = g0.elapsed_time(g1) / reps
    # the sampler ran through the timed steps AND the per-direction loops above (the same kernels under load): a 20-step
    # timed region of this workload lasts ~6 ms, too short for nvidia-smi's sampling period on its own
    clocks = sampler.stop() if rank == 0 else None
    alg_bytes_dir = 24.0 * levels * b * n          # 24 B/sample/level/direction (SURVEY.md 8d)
    achieved = alg_bytes_dir / fwd_ms * 1e-6        # GB/s over the forward direction's launches
    fused_bytes = 8.0 * (levels + 2) * b * n
    roofline = {"bound": "hbm", "kernel": "k_lean_analysis" if fwd_launches == 1 else "analysis launches of one direction",
                "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic_of(args.workload), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes_dir / max(fwd_launches, 1),
                "launches_per_direction": fwd_launches, "avg_launch_ms": fwd_ms / max(fwd_launches, 1),
                "forward_ms": fwd_ms, "inverse_ms": inv_ms,
                "inverse_achieved_gbs": alg_bytes_dir / inv_ms * 1e-6,
                "fused_compulsory_bytes_per_direction": fused_bytes,
                "frac_of_fused_compulsory_bound": (fused_bytes / fwd_ms * 1e-6) / peak,
                "inverse_frac_of_fused_compulsory_bound": (fused_bytes / inv_ms * 1e-6) / peak,
                "fp64_tflops_peak_measured": fp64_peak, "fp64_peak_source": "vw_probe_fp64 in this run (DFMA, uniform-register "
                "operand, 8 chains, 64 warps/SM)", "sm_max_mhz": sm_max,
                "fp64_tflops_achieved": 4.0 * hs.size * levels * b * n / fwd_ms * 1e-9,
                "frac_of_fp64": (4.0 * hs.size * levels * b * n / fwd_ms * 1e-9) / fp64_peak if fp64_peak else None}

    # ---- e2e: host buffers through the public facade, copies inside the timed region (rank-local) ----------
    e2e = None
    if not args.no_e2e:
        eb = b if b * n * 8 * (levels + 2) <= 8e9 else max(1, int(8e9 / (n * 8 * (levels + 2))))
        xh = eng.pinned_empty((eb, n))
        xh[...] = np.random.default_rng(7 + rank).standard_normal((eb, n))
        wh = eng.pinned_empty((levels, eb, n))
        vh = eng.pinned_empty((eb, n))
        oh = eng.pinned_empty((eb, n))

        def e2e_step():
            eng.forward(xh, hs, gs, levels, mode, 0, wh, vh)                 # H2D x, D2H W + V_J
            eng.inverse(wh, vh, hs, gs, mode, None, 0, out=oh)              # H2D W + V_J, D2H x^
        for _ in range(2):
            e2e_step()
        c.barrier()
        esteps = max(3, min(args.steps, 10))
        t0 = time.perf_counter()
        for _ in range(esteps):
            e2e_step()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        assert float(np.max(np.abs(oh - xh))) < 1e-6
        step_bytes = int((levels + 2) * eb * n * 8)
        e2e = {"value": world * eb * n * esteps / dt * 1e-9, "unit": UNIT,
               "h2d_bytes_per_step": step_bytes, "d2h_bytes_per_step": step_bytes,
               "api": "Engine.forward/inverse with HOST (pinned) buffers == vw_modwt_forward / vw_modwt_inverse without "
                      "VW_FLAG_DEVICE_PTRS; coefficients cross PCIe both ways like the Java double[] API",
               "batch": eb, "steps": esteps, "numa_binding": numa,
               "pcie_gbs_per_rank_each_way_in_the_step": step_bytes * esteps / dt * 1e-9}
        del xh, wh, vh, oh

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        try:
            cpu = cpu_port(args.workload, len(os.sched_getaffinity(0)) or 1)
            cpu["variants"] = cpu_variants(args.workload)
        except Exception as ex:  # the checker must never take the bench down
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {ex}"}

    # ---- extra: the other configs, the sharded paths, latencies -- same run, after the headline ----------------
    del xs, ws, vs, xr
    c.free()
    extra = None
    if not args.no_extra:
        extra = {}

        def guarded(key, fn):
            try:
                val = fn()
                if rank == 0:
                    extra[key] = val
            except Exception as ex:   # one failing side measurement must not lose the headline
                if world > 1:
                    raise
                extra[key] = {"failed": f"{type(ex).__name__}: {ex}"[:300]}
                c.free()
        # BASELINE config #3 as written: 1024 x 65536 sym8 J=8 split over the ranks by signal (strong scaling)
        from vectorwave_b200.sharded import shard_batch
        lo, hi = shard_batch(1024, rank, world)
        guarded("batch_strong_c3" if world > 1 else "c3", lambda: finish_batch(
            c, "batch1024x65536_sym8_J8", extra_batch(c, "batch1024x65536_sym8_J8", "batch1024x65536_sym8_J8", 0, rows=hi - lo), 1024))
        if world > 1 and rank == 0 and "batch_strong_c3" in extra:
            extra["batch_strong_c3"]["scaling"] = "strong"
            extra["batch_strong_c3"]["sharding"] = f"1024 signals split by signal over {world} ranks, no communication"
        guarded("span", lambda: extra_span(c))
        # the JVM's way of driving the same transform: rank 0 alone, one host thread over all the job's GPUs.  The other
        # ranks wait on a CPU (gloo) barrier: an NCCL barrier is a kernel spinning on their GPU, which would time-slice
        # against rank 0's kernels there (measured: 34 ms per step instead of 13)
        c.free()
        c.barrier()
        if rank == 0:
            try:
                extra["span_one_host_thread"] = extra_span_one_thread(c)
            except Exception as ex:
                extra["span_one_host_thread"] = {"failed": f"{type(ex).__name__}: {ex}"[:300]}
        if world > 1:
            dist.barrier(group=cpu_group)
        c.barrier()
        if world > 1:
            # what the box's PCIe fabric gives when every rank copies at once (e2e at N > 1 is bound by this, not by the engine)
            c.barrier()
            mine = dict(pcie_probe(c), rank=rank, numa_binding=numa)
            allp = [None] * world
            dist.all_gather_object(allp, mine)
            if rank == 0:
                extra["pcie_all_ranks_concurrently"] = {
                    "h2d_gbs_min": min(p["h2d_gbs"] for p in allp), "h2d_gbs_max": max(p["h2d_gbs"] for p in allp),
                    "d2h_gbs_min": min(p["d2h_gbs"] for p in allp), "d2h_gbs_max": max(p["d2h_gbs"] for p in allp),
                    "h2d_gbs_sum": sum(p["h2d_gbs"] for p in allp), "d2h_gbs_sum": sum(p["d2h_gbs"] for p in allp),
                    "numa_bindings": [p["numa_binding"] for p in allp],
                    "note": "1 GiB pinned copies issued by all ranks at the same time, one direction after the other"}
        if world == 1:
            guarded("pcie", lambda: pcie_probe(c))
            guarded("c4", lambda: finish_batch(c, "single2p28_coif5_J10",
                                               extra_batch(c, "single2p28_coif5_J10", "single2p28_coif5_J10", 0, reps=4), 1))
            for m in (1, 2):
                key = f"c5_{MODES[m]}"
                guarded(key, lambda m=m, key=key: finish_batch(c, key, extra_batch(c, key, "batch256x1M_db8_J6", m, reps=4), 256))
            guarded("c5_PERIODIC", lambda: finish_batch(c, "batch256x1M_db8_J6",
                                                        extra_batch(c, "batch256x1M_db8_J6", "batch256x1M_db8_J6", 0, reps=4), 256))
            for m in (1, 2):
                guarded(f"c5_denoise_{MODES[m]}", lambda m=m: extra_denoise(c, m))
            guarded("c2_haar", lambda: finish_batch(c, "batch4096x4096_haar_J4",
                                                    extra_batch(c, "batch4096x4096_haar_J4", "batch4096x4096_haar_J4", 0, reps=50), 4096))
            guarded("e2e_resident_result", lambda: extra_resident(c, args.workload))
            extra["c1_latency_us"] = extra_latency(local_rank)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config_of(args.workload),
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
                "clocks": clocks, "round_trip_max_abs_err": rt,
                "validation": "input validation (VW_FLAG_CHECK_FINITE, the reference's validateFiniteValues) is NOT in the timed "
                              "region: the device-resident and e2e loops call the engine with flags = 0; the API-compatible "
                              "classes pay one extra read pass + a stream sync for it",
                "roofline_model_gsamples": peak / (48.0 * levels),
                "frac_of_roofline_model": value / world / (peak / (48.0 * levels)),
                "gsample_levels_per_s": value * 2.0 * levels,      # SURVEY 8(d): 2*J*B*N / t
                "extra": extra}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
