#!/usr/bin/env python3
"""Device coverage from aligned reads (coverage_gpu.cuh + rle_encode_kernel) against the HBM roofline,
with numpy's time for the same coverage on the host beside it.  Two cases, seeded reads (synth.reads):
  chr1   one chr1-sized region (249,250,621 bases), 1e7 reads;
  batch  24 hg19 chromosomes x 8 samples in one call, `density` reads per base.
Algorithmic bytes: 4 B per base zeroed + 8 B per base scanned (read + write) + 4 B per base encoded
+ 12 B per row written + 16 B per read (8 B read, two 4 B atomics).
usage: python tools/prof_coverage.py [--density 0.01] [--samples 8] [--out file.jsonl]"""
import argparse, json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import peaksegdisk_b200 as psd
from peaksegdisk_b200 import synth
from peaksegdisk_b200.plan import coverage_rows

ap = argparse.ArgumentParser()
ap.add_argument("--density", type=float, default=0.01)
ap.add_argument("--samples", type=int, default=8)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--out", default=None)
a = ap.parse_args()
peak = 6554.9
try:
    peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
except Exception:
    pass


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:
        q = "nvidia-smi unavailable: %s" % e
    return q


def host_numpy(starts, ends, lo, hi):
    """What a user does without the library: difference array, cumsum, run heads (4-8 B per base)."""
    n = hi - lo
    keep = (ends > lo) & (starts < hi)
    d = np.zeros(n + 1, np.int32)
    np.add.at(d, np.maximum(starts[keep].astype(np.int64) - lo, 0), 1)
    np.add.at(d, np.minimum(ends[keep].astype(np.int64) - lo, n), -1)
    cov = np.cumsum(d[:n], dtype=np.int32)
    heads = np.flatnonzero(np.r_[True, cov[1:] != cov[:-1]])
    return heads, cov[heads]


def measure(name, problems, host_problems, host_scale):
    best, walls = None, []
    for _ in range(a.reps + 1):   # the first call is the warm-up
        t0 = time.time()
        rows, st = coverage_rows(problems, 0)
        walls.append(time.time() - t0)
        if best is None or st["kernel_ms"] < best["kernel_ms"]:
            best = st
    walls = walls[1:]
    alg = 16 * best["bases"] + 12 * best["rows"] + 16 * best["reads"]
    gbps = alg / best["kernel_ms"] / 1e6
    t0 = time.time()
    for p in host_problems:
        host_numpy(*p)
    t_np = (time.time() - t0) * host_scale
    rec = {"case": name, "gpu": gpu_info(), "problems": best["n_problems"], "waves": best["n_waves"], "reads": best["reads"],
           "bases": best["bases"], "rows": best["rows"], "kernel_ms": best["kernel_ms"], "device_ms": best["device_ms"],
           "call_wall_s_min": min(walls), "algorithmic_bytes": alg, "bytes_per_base": alg / best["bases"],
           "achieved_gbps": gbps, "peak_gbps": peak, "frac_of_peak": gbps / peak, "h2d_bytes": best["h2d_bytes"],
           "d2h_bytes": best["d2h_bytes"], "host_numpy_s": t_np,
           "host_numpy_note": "measured" if host_scale == 1 else "measured on sample 0, times %d samples" % host_scale}
    print(json.dumps(rec), flush=True)
    if a.out:
        with open(a.out, "a") as f:
            f.write(json.dumps(rec) + "\n")


n1 = synth.HG19_LEN[0]
s, e = synth.reads(5, 10 ** 7, n1)
measure("chr1", [(s, e, 0, n1)], [(s, e, 0, n1)], 1)
del s, e
batch, sample0 = [], []
for ci, length in enumerate(synth.HG19_LEN):
    for si in range(a.samples):
        s, e = synth.reads(1000 * ci + si, int(a.density * length), length)
        batch.append((s, e, 0, length))
        if si == 0:
            sample0.append((s, e, 0, length))
measure("hg19_24chrom_x%d" % a.samples, batch, sample0, a.samples)
