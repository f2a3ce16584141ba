"""Writes tests/golden/golden_path_mono27ac.json: the exact model path of the reference's Mono27ac
coverage on [100, Inf), computed by the CROPS rules of psd_model_path (tests/path_oracle.py) over the
parity oracle (oracle/fpop_oracle.cpp) on the host.  Takes about a minute and a half on one core."""
import json
import math
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle_bind  # noqa: E402
import path_oracle  # noqa: E402
from peaksegdisk_b200 import synth  # noqa: E402

PEN_MIN = 100.0


def main():
    _, s, e, c = synth.read_bedgraph(os.path.join(ROOT, "tests", "golden", "Mono27ac_coverage.bedGraph"))
    if not oracle_bind.libm_matches_golden():
        sys.exit("this host's libm differs from the one the goldens were made with")
    t0 = time.time()
    models, rounds, solves = path_oracle.crops(path_oracle.oracle_round(s, e, c), PEN_MIN, math.inf)
    secs = time.time() - t0
    out = {"pen_min": PEN_MIN, "pen_max": "Inf", "rounds": rounds, "solves": solves,
           "columns": ["min.lambda", "max.lambda", "penalty", "peaks", "segments", "total.loss"],
           # floats as their repr so that they come back bit for bit
           "models": [[repr(float(m[k])) if isinstance(m[k], float) else m[k] for k in
                       ["min.lambda", "max.lambda", "penalty", "peaks", "segments", "total.loss"]] for m in models]}
    path = os.path.join(ROOT, "tests", "golden", "golden_path_mono27ac.json")
    rows = out.pop("models")
    with open(path, "w") as f:   # one model per line
        f.write(json.dumps(out)[:-1] + ', "models": [\n' + ",\n".join(json.dumps(r) for r in rows) + "\n]}\n")
    print("%d models, %d solves, %d rounds, %.1f s on the host -> %s" % (len(models), solves, rounds, secs, path))


if __name__ == "__main__":
    main()
