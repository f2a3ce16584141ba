#!/usr/bin/env python3
"""Device coverage statistics (psd_features, features_gpu.cuh) against the HBM roofline, with the host time
of a numpy weighted-sort computation of the same statistics beside it.  Three cases:
  chr1     one chr1-sized problem (synth.hg19_problem(0, 0, ...), about 8.9 M rows);
  hg19     24 hg19 chromosomes x `samples` samples at row scale `scale` in one call;
  tiny     10,000 problems of 1 to 100 rows.
Algorithmic bytes: 8 B per row per pass (int32 weight and count), four passes.
usage: python tools/prof_features.py [--scale 0.25] [--samples 8] [--out file.jsonl]"""
import argparse, json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
from peaksegdisk_b200 import synth
from peaksegdisk_b200.plan import problem_features

ap = argparse.ArgumentParser()
ap.add_argument("--scale", type=float, default=0.25)
ap.add_argument("--samples", type=int, default=8)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--out", default=None)
a = ap.parse_args()
peak = 6554.9   # GB/s, this project's measured HBM read bandwidth on a B200
PASSES = 4


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, timeout=60)
    if q.returncode != 0:
        raise SystemExit("nvidia-smi failed: no GPU to measure on")
    return q.stdout.strip()


def host_numpy(s, e, c):
    """What a user does without the library: a weighted sort and cumulative weights per problem."""
    w = (e - s).astype(np.int64)
    c = c.astype(np.int64)
    order = np.argsort(c, kind="stable")
    cs, cw = c[order], np.cumsum(w[order])
    B = int(cw[-1])
    q = []
    for p in (0.25, 0.5, 0.75):
        h = (B - 1) * p
        lo = int(np.floor(h))
        x0, x1 = cs[np.searchsorted(cw, [lo, min(lo + 1, B - 1)], "right")]
        q.append(x0 + (h - lo) * (x1 - x0))
    m = float(np.sum(w * c)) / B
    sd = np.sqrt(np.sum(w * (c - m) ** 2) / (B - 1)) if B > 1 else np.nan
    return cs[0], q, cs[-1], m, sd


def measure(name, problems, host_problems, host_scale):
    best, walls = None, []
    for _ in range(a.reps + 1):   # the first call is the warm-up
        t0 = time.time()
        _, st = problem_features(problems, 0, return_stats=True)
        walls.append(time.time() - t0)
        if best is None or st["kernel_ms"] < best["kernel_ms"]:
            best = st
    walls = walls[1:]
    alg = 8 * PASSES * best["rows"]
    gbps = alg / best["kernel_ms"] / 1e6
    t0 = time.time()
    for p in host_problems:
        host_numpy(*p)
    t_np = (time.time() - t0) * host_scale
    rec = {"case": name, "gpu": gpu_info(), "problems": best["n_problems"], "waves": best["n_waves"], "rows": best["rows"],
           "launches": best["n_launches"], "kernel_ms": best["kernel_ms"], "device_ms": best["device_ms"],
           "call_wall_s_min": min(walls), "algorithmic_bytes": alg, "achieved_gbps": gbps, "peak_gbps": peak,
           "frac_of_peak": gbps / peak, "h2d_bytes": best["h2d_bytes"], "d2h_bytes": best["d2h_bytes"],
           "host_numpy_s": t_np,
           "host_numpy_note": "measured" if host_scale == 1 else "measured on sample 0, times %d samples" % host_scale}
    print(json.dumps(rec), flush=True)
    if a.out:
        with open(a.out, "a") as f:
            f.write(json.dumps(rec) + "\n")


gpu_info()
_, bs, be, bc = synth.read_bedgraph(os.path.join(ROOT, "tests", "golden", "Mono27ac_coverage.bedGraph"))
bw = (be - bs).astype(np.int64)
p = synth.hg19_problem(0, 0, bw, bc)[:3]
measure("chr1", [p], [p], 1)
del p
batch, sample0 = [], []
for ci in range(len(synth.HG19_LEN)):
    for si in range(a.samples):
        p = synth.hg19_problem(ci, si, bw, bc, a.scale)[:3]
        batch.append(p)
        if si == 0:
            sample0.append(p)
measure("hg19_24chrom_x%d_scale%g" % (a.samples, a.scale), batch, sample0, a.samples)
del batch, sample0
rng = np.random.default_rng(3)
tiny = []
for k in rng.integers(1, 101, size=10000):
    w = rng.integers(1, 50, size=k)
    end = np.cumsum(w)
    tiny.append(((end - w).astype(np.int32), end.astype(np.int32), rng.poisson(5.0, size=k).astype(np.int32)))
measure("tiny_10000", tiny, tiny, 1)
