#!/usr/bin/env python3
"""Experiment: config-2 vectors at ONE penalty (function sizes differ a lot between penalties) under
the launch configuration given in the environment (PSD_OCCUPANCY_MODE).
usage: python tools/prof_shares.py <penalty> [n_vectors=1024] [copies=5]"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import peaksegdisk_b200 as psd
from peaksegdisk_b200 import synth
pen = float(sys.argv[1]); nv = int(sys.argv[2]) if len(sys.argv) > 2 else 1024; copies = int(sys.argv[3]) if len(sys.argv) > 3 else 5
plan = psd.Plan(0); rows = 0
for k in range(nv):
    s, e, c = synth.poisson_problem(k)
    for j in range(copies):
        plan.add(s, e, c, pen * (1.0 + 0.01 * j)); rows += len(c)
plan.upload()
for rep in range(2):
    plan.solve(); st = plan.stats()
plan.download()
mi = sum(plan.loss_row(i)["mean.intervals"] for i in range(0, len(plan), 37)) / len(range(0, len(plan), 37))
mx = max(plan.loss_row(i)["max.intervals"] for i in range(len(plan)))
print("penalty=%g occupancy=%s: dp_ms=%.1f rows/s=%.3e warps/sm=%d mean.intervals=%.2f max.intervals=%d overflow_tier_problems=%d" % (
    pen, os.environ.get("PSD_OCCUPANCY_MODE", "0"), st["dp_ms"], rows / st["dp_ms"] * 1e3,
    st["warps_per_sm"], mi, mx, st["n_overflow_tier"]), flush=True)
