#!/usr/bin/env python3
"""Joint single-peak models (psd_joint_models, joint_models_batch) at user sizes: `regions` regions of
`min_kb` to `max_kb` kb, S samples each, at each bin width.  Per case, with CUDA events (the library's stats):
kernel ms, device ms (copies included), the wall time of one call, pair x sample evaluations per second, and
that rate against the fp64 rate tools/microbench/fp64_peak.cu measures in the same run.  The fp64 share is an
upper bound: it charges every evaluation 30 fp64 instructions (the division, psd_log's main path and the loss
arithmetic), which only feasible samples execute.  Beside it, the C oracle (tests/native/joint_oracle.c, libm)
on one host core, timed on the first regions and scaled by evaluations, and a bit-for-bit check of those
regions against it.
usage: python tools/prof_joint.py [--regions 2000] [--samples 8 32 128] [--bins 1 10] [--out file.jsonl]"""
import argparse, ctypes as C, json, os, subprocess, sys, tempfile, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
from peaksegdisk_b200.plan import joint_models_batch

ap = argparse.ArgumentParser()
ap.add_argument("--regions", type=int, default=2000)
ap.add_argument("--samples", type=int, nargs="+", default=[8, 32, 128])
ap.add_argument("--bins", type=int, nargs="+", default=[1, 10])
ap.add_argument("--min-kb", type=float, default=1.0)
ap.add_argument("--max-kb", type=float, default=5.0)
ap.add_argument("--oracle-evals", type=float, default=3e8, help="pair x sample evaluations the host oracle times")
ap.add_argument("--out", default=None)
a = ap.parse_args()
FP64_PER_EVAL = 30
tmp = tempfile.mkdtemp(prefix="prof_joint_")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, timeout=60)
    if q.returncode != 0:
        raise SystemExit("nvidia-smi failed: no GPU to measure on")
    return q.stdout.strip()


def fp64_peak():
    exe = os.path.join(tmp, "fp64_peak")
    subprocess.check_call([os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-o", exe,
                           os.path.join(ROOT, "tools", "microbench", "fp64_peak.cu")])
    return json.loads(subprocess.run([exe], capture_output=True, text=True, check=True).stdout)


def oracle_lib():
    so = os.path.join(tmp, "joint_oracle.so")
    subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-o", so,
                           os.path.join(ROOT, "tests", "native", "joint_oracle.c"), "-lm"])
    lib = C.CDLL(so)
    lib.joint_oracle.restype = C.c_int
    return lib


def region(rng, S, length):
    """S samples over [0, length): Poisson background at a per-sample depth, a peak in about half of them."""
    lo = int(rng.integers(0, length // 2)); hi = lo + int(rng.integers(100, length // 2))
    out = []
    for _ in range(S):
        w = rng.integers(1, 30, size=length // 8 + 2)
        e = np.minimum(np.cumsum(w), length)
        e = e[np.concatenate([[True], e[1:] > e[:-1]])]
        e[-1] = length
        s = np.concatenate([[0], e[:-1]])
        lam = np.full(len(e), float(rng.choice([2, 10, 40])))
        if rng.random() < 0.5:
            lam[(s >= lo) & (e <= hi)] *= 5
        out.append((s.astype(np.int32), e.astype(np.int32), rng.poisson(lam).astype(np.int32)))
    return out


def oracle_check(lib, samples, bin_bases, got):
    """Times the oracle on one region and checks the device's losses and peaks against it."""
    start, end = int(samples[0][0][0]), int(samples[0][1][-1])
    n = -(-(end - start) // bin_bases)
    g = start + np.arange(n + 1, dtype=np.int64) * bin_bases
    g[n] = end
    S = len(samples)
    pref = np.zeros((n + 1, S), np.int64)
    for j, (s, e, c) in enumerate(samples):
        s, e, c = (np.asarray(x, np.int64) for x in (s, e, c))
        cum = np.concatenate([[0], np.cumsum(c * (e - s))])
        r = np.minimum(np.searchsorted(e, g, side="right"), len(c) - 1)
        pref[:, j] = cum[r] + c[r] * (g - s[r])
    loss = np.zeros(S + 1); pa = np.zeros(S + 1, np.int32); pb = np.zeros(S + 1, np.int32)
    f = np.zeros((S + 1, S), np.uint8)
    t0 = time.perf_counter()
    lib.joint_oracle(C.c_int(S), C.c_int(n), C.c_int(bin_bases), C.c_int(end - start), pref.ctypes.data_as(C.POINTER(C.c_int64)),
                     C.c_int(1), C.c_int(n - 1), loss.ctypes.data_as(C.POINTER(C.c_double)), pa.ctypes.data_as(C.POINTER(C.c_int)),
                     pb.ctypes.data_as(C.POINTER(C.c_int)), f.ctypes.data_as(C.POINTER(C.c_uint8)))
    dt = time.perf_counter() - t0
    m = got["models"]
    ks = m["peaks"].to_numpy()
    ok = np.array_equal(np.flatnonzero(np.isfinite(loss)), ks) and \
        np.array_equal(loss[ks].view(np.int64), m["total.loss"].to_numpy().view(np.int64)) and \
        all(k == 0 or (g[pa[k]] == m["peakStart"][i] and g[pb[k]] == m["peakEnd"][i]) for i, k in enumerate(ks))
    return dt, S * (n - 1) * (n - 2) // 2, bool(ok)


info = gpu_info()
peak = fp64_peak()
lib = oracle_lib()
joint_models_batch([region(np.random.default_rng(0), 4, 300)])   # warm-up: module load, first launches
for S in a.samples:
    for b in a.bins:
        rng = np.random.default_rng(1000 * S + b)
        probs = [region(rng, S, int(rng.integers(int(a.min_kb * 1000), int(a.max_kb * 1000) + 1))) for _ in range(a.regions)]
        t0 = time.perf_counter()
        got, st = joint_models_batch(probs, bin_bases=b)
        wall = time.perf_counter() - t0
        rate = st["pair_sample_evals"] / (st["kernel_ms"] * 1e-3)
        o_s, o_ev, ok, n_chk = 0.0, 0, True, 0
        while n_chk < len(probs) and o_ev < a.oracle_evals:
            dt, ev, good = oracle_check(lib, probs[n_chk], b, got[n_chk])
            o_s += dt; o_ev += ev; ok = ok and good; n_chk += 1
        rec = {"case": "regions%d_S%d_bin%d" % (a.regions, S, b), "gpu": info, "regions": a.regions, "samples": S,
               "bin_bases": b, "kb": [a.min_kb, a.max_kb], "pair_sample_evals": st["pair_sample_evals"],
               "kernel_ms": st["kernel_ms"], "device_ms": st["device_ms"], "call_wall_s": wall, "waves": st["n_waves"],
               "launches": st["n_launches"], "h2d_bytes": st["h2d_bytes"], "d2h_bytes": st["d2h_bytes"],
               "evals_per_s": rate, "fp64_dfma_tflops_measured": peak["dfma_tflops"],
               "fp64_share_upper_bound": rate * FP64_PER_EVAL / (peak["dfma_tflops"] * 1e12 / 2),
               "models": int(sum(len(g["models"]) for g in got)),
               "oracle_one_core_s_scaled": o_s * st["pair_sample_evals"] / max(1, o_ev),
               "oracle_note": "libm C oracle timed on %d regions (%d evaluations) and scaled by evaluations" % (n_chk, o_ev),
               "oracle_bit_identical": ok}
        print(json.dumps(rec), flush=True)
        if a.out:
            with open(a.out, "a") as fh:
                fh.write(json.dumps(rec) + "\n")
