"""Generates tests/golden/modwt_golden.npz -- the committed golden vectors of the MODWT / SWT path.

Provenance: the reference (MorphIQ-Labs/VectorWave) is pure Java and no JVM exists in the build image, so its own
code cannot produce these vectors here.  They are the outputs of the CPU oracle (oracle/modwt_oracle.c, a C
restatement of the reference loops compiled -O2 -ffp-contract=off so the JVM's separate multiply / add roundings
hold), which tests/test_oracle_kat.py pins against the reference's literal known answers.  The INPUTS reproduce the
reference's own test fixtures bit for bit: `randomAoS(batch, n, seed)` (java.util.Random nextDouble()*2-1,
ETEST/modwt/BatchMODWTApiTest.java:67-74) and `TestSignals.compositeSin(n, seed, noise)`
(CTEST/testing/TestSignals.java:18-30), via oracle/javarandom.py.

The shapes are the reference's parity-test shapes: B = 3 / 4, N = 128, J = 3 (BatchMODWTMultiLevelParityTest.java:24-46),
N in {128, 129, 256} single level (ModwtPeriodicRoundTripTest.java:25-42), N = 512 with J = min(5, max)
(MultiLevelModwtCorrectnessTest.java:27-72), N in {256, 500} PERIODIC + ZERO_PADDING
(ParallelVsSequentialEquivalenceTest.java:18-49), plus SYMMETRIC and the SWT denoise of config #5's wavelet.

What is stored: the arrays themselves come to 2 MB, so each one (input, W, V, reconstruction, denoised signal) is kept
as the SHA-256 digest of its shape and float64 bytes, which pins every bit, plus a seeded sample of SAMPLE values with
their flat positions, which shows what the values are when a digest stops matching.  The inputs are regenerated from
their seeds by cases(); the SWT thresholds are stored whole.

Run from the repo root:  python tests/golden/make_golden.py
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import cref, javarandom  # noqa: E402
from oracle.wavelets import filters  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "modwt_golden.npz")
SAMPLE = 32


def digest(a):
    """SHA-256 of the shape and the little-endian float64 bytes of `a`, as 32 uint8"""
    a = np.ascontiguousarray(a, dtype="<f8")
    return np.frombuffer(hashlib.sha256(repr(a.shape).encode() + a.tobytes()).digest(), dtype=np.uint8)


def entry(name, a, rng):
    """the stored form of the golden array `name`: {name/sha256, name/idx, name/val}"""
    a = np.ascontiguousarray(a, dtype=np.float64)
    idx = np.sort(rng.choice(a.size, min(a.size, SAMPLE), replace=False)).astype(np.int64)
    return {name + "/sha256": digest(a), name + "/idx": idx, name + "/val": a.ravel()[idx]}


def outputs(key, name, mode, levels, x):
    """the oracle's arrays of one case, {w, v, xr} plus {denoise_soft1, denoise_soft0} for the swt_ cases, and those
    cases' thresholds {thr_soft1, thr_soft0}"""
    h, g, wid = filters(name)
    w = np.empty((levels, x.shape[0], x.shape[1]))
    v = np.empty_like(x)
    xr = np.empty_like(x)
    for i in range(x.shape[0]):
        w[:, i, :], v[i] = cref.decompose(x[i], h, g, levels, mode)
        xr[i] = cref.reconstruct(w[:, i, :], v[i], h, g, mode, wid)
    arrays, thresholds = {"w": w, "v": v, "xr": xr}, {}
    if key.startswith("swt_"):
        for soft in (True, False):
            arrays[f"denoise_soft{int(soft)}"], thresholds[f"thr_soft{int(soft)}"] = \
                cref.swt_denoise(x[0], h, g, levels, mode, wid, -1.0, soft)
    return arrays, thresholds


def cases():
    """(key, wavelet, mode, levels, x[B][N]) -- every case is decomposed, reconstructed and (db8) denoised."""
    out = []
    for name, b, seed in (("haar", 3, 123), ("db4", 4, 456), ("db4", 3, 99)):
        x = javarandom.uniform_pm1(b * 128, seed).reshape(b, 128)          # randomAoS(batch, 128, seed)
        out.append((f"aos_{name}_b{b}_n128_j3_s{seed}", name, 0, 3, x))
    for n in (128, 129, 256):
        x = javarandom.composite_sin(n, 42, 0.05)[None, :]
        for name in ("haar", "db4"):
            out.append((f"sin_{name}_n{n}_j1", name, 0, 1, x))
    x512 = javarandom.composite_sin(512, 7, 0.1)[None, :]
    for name in ("haar", "db2", "db4", "db6", "db8", "sym4", "sym8", "coif2", "coif3", "coif5"):
        lv = min(5, cref.max_levels(512, len(filters(name)[0]), 10))
        for mode in (0, 1, 2):
            out.append((f"ml_{name}_n512_j{lv}_m{mode}", name, mode, lv, x512))
    for n in (256, 500):
        x = javarandom.composite_sin(n, 11, 0.2)[None, :]
        for mode in (0, 1):
            out.append((f"pvs_db4_n{n}_j3_m{mode}", "db4", mode, 3, x))
    x4096 = javarandom.composite_sin(4096, 42, 0.2)[None, :]
    for mode in (0, 1, 2):
        out.append((f"swt_db8_n4096_j5_m{mode}", "db8", mode, 5, x4096))
    return out


def main():
    blobs = {}
    rng = np.random.default_rng(20240607)
    for key, name, mode, levels, x in cases():
        arrays, thresholds = outputs(key, name, mode, levels, x)
        blobs.update(entry(key + "/x", x, rng))
        for k, a in arrays.items():
            blobs.update(entry(f"{key}/{k}", a, rng))
        for k, t in thresholds.items():
            blobs[f"{key}/{k}"] = np.array([t])
    np.savez_compressed(OUT, **blobs)
    print(f"{OUT}: {len(blobs)} arrays, {os.path.getsize(OUT) / 1024:.0f} KiB")


if __name__ == "__main__":
    main()
