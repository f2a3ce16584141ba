#!/usr/bin/env python3
"""Differential fuzz: random problems of varied shapes through the GPU path and the oracle (psd_math
mode, bit-identical to the reference's libm); every summary field and segment must match bit for bit.
usage: tools/fuzz_gpu_vs_oracle.py [n_problems=300] [seed=0]"""
import os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import peaksegdisk_b200 as psd
from peaksegdisk_b200 import synth
import oracle_bind

def problems(n_prob, seed):
    """n_prob draws of the six shapes (k % 6), (chromStart, chromEnd, coverage, penalty) each; draws with
    constant coverage are left out."""
    rng = np.random.default_rng(seed)
    probs = []
    for k in range(n_prob):
        kind = k % 6
        n = int(rng.integers(50, 4000))
        if kind == 0:      # piecewise Poisson with random means
            means = np.repeat(rng.gamma(1.0, 5.0, size=n // 40 + 1), 40)[:n]
            z = rng.poisson(means)
        elif kind == 1:    # mostly zeros with rare bursts
            z = rng.poisson(0.02, size=n) + (rng.random(n) < 0.01) * rng.integers(1, 50, size=n)
        elif kind == 2:    # large counts
            z = rng.poisson(rng.uniform(100, 1e5), size=n)
        elif kind == 3:    # slowly increasing trend (many pieces)
            z = (np.arange(n) // 3) + rng.integers(0, 2, size=n)
        elif kind == 4:    # two-level alternation
            z = np.where((np.arange(n) // rng.integers(2, 30)) % 2 == 0, rng.integers(0, 3), rng.integers(3, 40)) + rng.poisson(0.3, size=n)
        else:              # uniform noise
            z = rng.integers(0, int(rng.integers(2, 1000)), size=n)
        s, e, c = synth.rle_rows(z.astype(np.int64))
        if kind % 2 == 1:  # random bases per row instead of run lengths
            w = rng.integers(1, 5000, size=len(c)); e = np.cumsum(w).astype(np.int32); s = np.concatenate(([0], e[:-1])).astype(np.int32)
        if len(set(c.tolist())) < 2:
            continue
        pen = float(10 ** rng.uniform(-3, 7)) if rng.random() > 0.1 else 0.0
        probs.append((s, e, c, pen))
    return probs


def main():
    n_prob = int(sys.argv[1]) if len(sys.argv) > 1 else 300
    probs = problems(n_prob, int(sys.argv[2]) if len(sys.argv) > 2 else 0)
    plan, ids = psd.solve_batch(probs)
    bad = 0
    for pid, (s, e, c, pen) in zip(ids, probs):
        st, summ, oseg = oracle_bind.solve_rows(s, e, c, pen)
        r = plan.result(pid)
        if r.status != 0 or st != 0:
            print("status", pid, r.status, st); bad += 1; continue
        got = plan.loss_row(pid); seg = plan.segments(pid)
        vals = np.array([got["segments"], got["peaks"], got["mean.pen.cost"], got["total.loss"], got["equality.constraints"], got["mean.intervals"], got["max.intervals"]], dtype=np.float64)
        ref = np.array([summ[1], summ[2], summ[5], summ[6], summ[7], summ[8], summ[9]])
        same = np.array_equal(vals.view(np.uint64), ref.view(np.uint64)) and all(np.array_equal(a, b) for a, b in zip(seg[:3], oseg[:3])) and np.array_equal(seg[3].view(np.uint64), oseg[3].view(np.uint64))
        if not same:
            bad += 1
            print("MISMATCH problem", pid, "rows", len(c), "penalty", pen, vals, ref)
    st = plan.stats()
    print("%d problems, %d rows, %d mismatches; tier-switched %d, max pieces seen %d" % (len(probs), st["rows_solved"], bad, st["n_overflow_tier"], int(max(plan.loss_row(i)["max.intervals"] for i in ids))))
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
