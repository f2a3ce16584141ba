#!/usr/bin/env python3
"""Exact model-selection path (psd_model_path, model_path_batch): where the time of a path goes.
Two cases:
  mono27ac  the reference's Mono27ac coverage on [100, Inf): wall time, device time and rounds, beside the
            71 s the parity oracle (oracle/fpop_oracle.cpp) needs for the same path on one host core;
  synth     512 synth.poisson_problem problems on [1e3, Inf), one call: solves, rows x solves per second
            and the share of the wall time spent outside the DP kernel.
The card's name and power limit are read in the same run.
usage: python tools/prof_model_path.py [--problems 512] [--out profiles/model_path.jsonl]"""
import argparse, json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import peaksegdisk_b200 as psd
from peaksegdisk_b200 import synth

ap = argparse.ArgumentParser()
ap.add_argument("--problems", type=int, default=512)
ap.add_argument("--out", default=None)
a = ap.parse_args()


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:
        q = "nvidia-smi unavailable: %s" % e
    return q


def measure(name, problems, pen_min, extra):
    psd.model_path_batch(problems[:1], pen_min=pen_min, pen_max=pen_min * 2)   # module load, plan setup
    t0 = time.perf_counter()
    paths, st = psd.model_path_batch(problems, pen_min=pen_min)
    wall = time.perf_counter() - t0
    rows = sum(len(c) for _, _, c in problems)
    dev_ms = st["dp_ms"] + st["backtrack_ms"] + st["label_ms"]
    rec = {"case": name, "gpu": gpu_info(), "problems": len(problems), "rows": rows, "pen_min": pen_min, "pen_max": "Inf",
           "rounds": st["rounds"], "solves": st["solves"], "models": st["models"], "rows_solved": st["rows_solved"],
           "wall_s": round(wall, 3), "dp_ms": round(st["dp_ms"], 2), "backtrack_ms": round(st["backtrack_ms"], 2),
           "device_ms": round(dev_ms, 2), "rows_x_solves_per_s": round(st["rows_solved"] / wall, 1),
           "share_outside_dp": round(1 - st["dp_ms"] / 1e3 / wall, 4), "h2d_bytes": st["h2d_bytes"], "d2h_bytes": st["d2h_bytes"]}
    rec.update(extra)
    print(json.dumps(rec), flush=True)
    return rec


_, s, e, c = synth.read_bedgraph(os.path.join(ROOT, "tests", "golden", "Mono27ac_coverage.bedGraph"))
recs = [measure("mono27ac", [(s, e, c)], 100.0, {"host_oracle_s": 71, "host_oracle_note": "parity oracle, one host core, Python driver"}),
        measure("synth", [synth.poisson_problem(7000 + k) for k in range(a.problems)], 1e3, {})]
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for r in recs:
            f.write(json.dumps(r) + "\n")
