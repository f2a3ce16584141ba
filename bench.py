#!/usr/bin/env python3
"""bench.py -- BASELINE.json's metric (FPOP bedGraph rows x penalties per second) on config 2:
1,024 synthetic Poisson count vectors per GPU (N log-uniform 1e4..1e5, RLE'd to bedGraph rows) x
penalties {1e2,1e3,1e4,1e5,1e6} = 5,120 independent problems per GPU.

  python bench.py --gpus N --steps K --warmup W          our arm (CUDA, through the C ABI)
  python bench.py --impl reference ...                   the reference's CPU solver on the host cores
  python bench.py ... --dump-outputs DIR                 also write the value path's results as DIR/*.npy
                                                         (our arm; the reference arm accepts and ignores it)

A "step" is one solve of the whole batch; --steps sets the number of timed steps of the value, e2e and
e2e_plan_api paths (the in-run cpu_baseline sample is one step, the RLE figure the best of four uploads).
  value   K steps of psd_plan_solve (DP + backtrack kernels; the rows are already resident in HBM when the
          timed region starts, as the bench contract asks; no H2D/D2H inside), CUDA events, max over ranks.
  e2e     the DROP-IN path, per step: psd_fpop_disk_batch on the batch's bedGraph FILES (tmpfs) -> text
          parse -> pinned rows -> H2D -> DP -> backtrack -> D2H -> _segments.bed / _loss.tsv written,
          scratch db files created and removed -- exactly what the reference arm pays for.
  e2e_plan_api (secondary)  psd_plan_run on host arrays: H2D -> DP -> backtrack -> D2H, no text.
After the timed steps the result files of 30 problems of the batch are compared with the committed
reference fixture (tests/golden/golden_fullsize.json, section c2): loss line and sha256(segments).
The inputs are generated from fixed seeds, so two builds run with the same arguments solve the same
problems and their --dump-outputs files can be compared array for array.  Nothing is written into the
source tree (no bytecode either): scratch files go to tmpfs or the temporary directory.
Multi-GPU: one process per GPU (torchrun), each rank owns its own 5,120 problems (weak scaling, no
data-path collective); value = all ranks' rows x penalties / max-over-ranks time.
"""
import argparse
import hashlib
import importlib.util
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

sys.dont_write_bytecode = True      # the tree may be read-only and must stay as the build left it
ROOT = os.path.dirname(os.path.abspath(__file__))
METRIC = "fpop_bedgraph_rows_x_penalties_per_sec"
UNIT = "rows*penalties/s"
GOLDEN_SEEDS = (588, 0, 1, 2, 3, 1022)     # the bench vectors pinned in tests/golden/golden_fullsize.json (rank 0)


def _load(name, rel):
    """Import one pure-Python module of the package by path, WITHOUT running peaksegdisk_b200/__init__
    (which loads the CUDA library): the reference arm must not touch our native code."""
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, rel))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


synth = _load("psd_synth", "peaksegdisk_b200/synth.py")
rfmt = _load("psd_rfmt", "peaksegdisk_b200/rfmt.py")
shard = _load("psd_shard", "peaksegdisk_b200/shard.py")
PEN_STRS = [rfmt.r_paste(p) for p in synth.C2_PENALTIES]


def make_config(args):
    """Identical in both arms (the driver compares the two lines' config)."""
    return {"workload": "config2: %d synthetic Poisson count vectors/GPU, N log-uniform 1e4-1e5 (RLE rows), penalties 1e2..1e6 "
                        "=> %d problems/GPU" % (args.vectors, 5 * args.vectors),
            "vectors_per_gpu": args.vectors, "penalties": synth.C2_PENALTIES, "quick": bool(args.quick),
            "l2": "no flush needed: per-step inputs + cost-function store are far larger than the 126 MB L2",
            "sharding": "by problem, no collective"}


def build_vectors(rank, n_vectors, quick):
    return [(seed, synth.poisson_problem(seed, 4000 if quick else None)) for seed in shard.rank_seeds(rank, n_vectors)]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=fd, stderr=subprocess.DEVNULL)
            os.close(fd)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for nm, v in zip(names, f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            os.unlink(self.path)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), samples=len(sm))
        out["reasons"] = sorted(reasons)
        return out


class CpuReference:
    """The unmodified reference solver (oracle/_ref/libref_fpop.so: PeakSegFPOP_disk compiled from the
    reference's own sources) on a bounded sample of the batch: all host threads, one problem per thread
    at a time, longest problems first, bedGraph and db files on tmpfs.  Falls back to our CPU
    restatement (oracle/_build) when the compiled reference is absent."""

    def __init__(self, vectors, target_rows, tmpdir, n_threads):
        import ctypes as C
        self.C = C
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_bind
        self.kind = "reference"
        lib_path = oracle_bind.REF_SO
        if not os.path.exists(lib_path):
            oracle_bind.ensure_built()
        if not os.path.exists(lib_path):
            lib_path, self.kind = oracle_bind.ORACLE_SO, "port"
        self.lib = C.CDLL(lib_path)
        self.n_threads = n_threads if self.kind == "reference" else 1
        # the sample: whole vectors (all five penalties each), evenly spread over the batch's sizes
        total = sum(len(v[1][2]) for v in vectors) * len(PEN_STRS)
        n_pick = max(1, min(len(vectors), int(round(len(vectors) * target_rows / max(1, total)))))
        n_pick = max(n_pick, min(len(vectors), (2 * self.n_threads + len(PEN_STRS) - 1) // len(PEN_STRS)))
        by_size = sorted(range(len(vectors)), key=lambda i: len(vectors[i][1][2]))
        picked = [by_size[int((k + 0.5) * len(by_size) / n_pick)] for k in range(n_pick)]
        jobs = []
        for i in sorted(set(picked)):
            seed, (s, e, c) = vectors[i]
            path = os.path.join(tmpdir, "ref_v%d.bedGraph" % seed)
            synth.write_bedgraph(path, s, e, c)
            for pen in PEN_STRS:
                jobs.append((len(c), path, pen, os.path.join(tmpdir, "ref_v%d_%s.db" % (seed, pen))))
        jobs.sort(key=lambda j: -j[0])          # longest first: a short tail when the threads run dry
        self.jobs = jobs
        self.rows = sum(j[0] for j in jobs)
        self.sample = "%d of %d problems (%d of %d vectors x 5 penalties, %d rows*penalties), %s PeakSegFPOP_disk incl. text parse + file output, files on %s" % (
            len(jobs), len(vectors) * len(PEN_STRS), len(set(picked)), len(vectors), self.rows,
            "the unmodified reference's" if self.kind == "reference" else "the oracle port's", tmpdir)

    def step(self):
        C = self.C
        n = len(self.jobs)
        arr = lambda xs: (C.c_char_p * n)(*[x.encode() for x in xs])
        status = (C.c_int * n)()
        files, pens, dbs = [j[1] for j in self.jobs], [j[2] for j in self.jobs], [j[3] for j in self.jobs]
        if self.kind == "reference":
            self.lib.ref_fpop_batch.restype = C.c_double
            secs = self.lib.ref_fpop_batch(n, arr(files), arr(pens), arr(dbs), self.n_threads, status)
        else:
            self.lib.oracle_fpop_disk.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p]
            t0 = time.time()
            for k, (f, p, d) in enumerate(zip(files, pens, dbs)):
                status[k] = self.lib.oracle_fpop_disk(f.encode(), p.encode(), d.encode())
                if os.path.exists(d):
                    os.unlink(d)
            secs = time.time() - t0
        assert all(s == 0 for s in status), list(status)
        return secs


def check_against_golden(vectors, file_of):
    """Result files of the timed batch vs the committed reference fixture.  Returns (#checked, [mismatches])."""
    try:
        gold = json.load(open(os.path.join(ROOT, "tests", "golden", "golden_fullsize.json")))["c2"]
    except (OSError, KeyError, ValueError):
        return 0, ["golden fixture missing"]
    have = {seed for seed, _ in vectors}
    n, bad = 0, []
    for g in gold:
        seed, npos = g["key"]
        if npos is not None or seed not in have:
            continue
        pre = "%s_penalty=%s" % (file_of[seed], g["penalty"])
        try:
            loss = open(pre + "_loss.tsv").read()
            seg = open(pre + "_segments.bed").read()
        except OSError as exc:
            bad.append("%s: %r" % (pre, exc)); continue
        n += 1
        if loss != g["loss"] or hashlib.sha256(seg.encode()).hexdigest() != g["segments_sha256"]:
            bad.append("seed %d penalty %s differs from the reference" % (seed, g["penalty"]))
    return n, bad


DUMP_BYTES = 64 << 20


def dump_outputs(plan, n_rows, out_dir):
    """What a caller of the timed path (psd_plan_solve, then psd_plan_download) receives, as float64 arrays:
      loss.npy      [n_probs, 10]  the _loss.tsv fields of every problem (plan.LOSS_COLUMNS), problem order
      segments.npy  [n_segs, 5]    problem id, chromStart, chromEnd, is_peak, mean: all segments of the
                                   problems a fixed seeded permutation reaches first while their row counts
                                   (a bound on the segment counts) fit in 64 MB in all, rows sorted by
                                   problem id.  The sample depends on the inputs only, never on the results."""
    import numpy as np
    n_probs = len(n_rows)
    os.makedirs(out_dir, exist_ok=True)
    loss = np.array([list(plan.loss_row(i).values()) for i in range(n_probs)], np.float64)
    budget = DUMP_BYTES - loss.nbytes - 2 * 4096         # .npy headers
    picked, used = [], 0
    for pid in np.random.default_rng(0).permutation(n_probs).tolist():
        nbytes = 5 * 8 * n_rows[pid]
        if used + nbytes > budget:
            break
        picked.append(pid)
        used += nbytes
    parts = [np.column_stack((np.full(len(seg[0]), pid),) + seg).astype(np.float64)
             for pid in sorted(picked) for seg in [plan.segments(pid)]]
    np.save(os.path.join(out_dir, "loss.npy"), loss)
    np.save(os.path.join(out_dir, "segments.npy"), np.concatenate(parts) if parts else np.zeros((0, 5)))
    return {"dir": out_dir, "problems": n_probs, "problems_with_segments": len(picked)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--vectors", type=int, default=1024, help="count vectors per GPU (config 2: 1024)")
    ap.add_argument("--quick", action="store_true", help="small problems (development only; not a bench value)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-seconds", type=float, default=30.0, help="reference arm: CPU work per step, seconds per core")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write the last step's results of the value path as DIR/*.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    config = make_config(args)
    tmp_root = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)

    if args.impl == "reference":
        if rank != 0:
            return
        if args.dump_outputs:
            print("bench.py: --dump-outputs applies to our arm; the reference arm writes no arrays", file=sys.stderr)
        vectors = build_vectors(0, args.vectors, args.quick)
        td = tempfile.mkdtemp(prefix="psd_ref_", dir=tmp_root)
        try:
            ref = CpuReference(vectors, int(cores * 5e4 * args.ref_seconds), td, cores)
            secs = [ref.step() for _ in range(args.warmup + args.steps)][args.warmup:]
        finally:
            shutil.rmtree(td, ignore_errors=True)
        value = ref.rows * len(secs) / sum(secs)
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * sum(secs) / max(1, len(secs)), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": ref.n_threads, "kind": ref.kind, "sample": ref.sample},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "native": "oracle/_ref/libref_fpop.so only (no CUDA library is loaded by this arm)"}
        print(json.dumps(line), flush=True)
        return

    import ctypes as C
    import numpy as np
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- there is no CPU path to benchmark")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    sys.path.insert(0, ROOT)
    import peaksegdisk_b200 as psd
    lib = psd._lib.lib

    vectors = build_vectors(rank, args.vectors, args.quick)
    probs = [(s, e, c, pen) for _, (s, e, c) in vectors for pen in synth.C2_PENALTIES]
    plan = psd.Plan(local_rank)
    for (s, e, c, pen) in probs:
        plan.add(s, e, c, pen)
    stream = torch.cuda.current_stream().cuda_stream
    rows_per_step = sum(len(p[2]) for p in probs)
    dgroup = dist if world > 1 else None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n_warm, n_steps, sample_clocks):
        for _ in range(n_warm):
            fn()
        sampler = ClockSampler(local_rank) if sample_clocks else None
        barrier()
        if sampler:
            sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(n_steps):
            fn()
        ev1.record()
        barrier()
        clocks = sampler.stop() if sampler else None
        mine = ev0.elapsed_time(ev1)
        ms, _ = shard.reduce_time_and_rows(mine, 0, dgroup, "cuda")
        return ms, clocks, mine

    # ---- value: device-resident rows, DP + backtrack only ----------------------------------------------
    plan.upload(stream)
    ms_total, clocks, ms_mine = timed(lambda: plan.solve(stream), args.warmup, args.steps, True)
    st = plan.stats()
    dumped = None
    if args.dump_outputs and rank == 0:
        plan.download(stream)          # outside the timed region: the results of its last step
        dumped = dump_outputs(plan, [len(p[2]) for p in probs], args.dump_outputs)
    ms_per_step = ms_total / args.steps
    _, total_rows = shard.reduce_time_and_rows(0.0, rows_per_step, dgroup, "cuda")
    value = total_rows / (ms_per_step / 1e3)
    per_rank_ms = [ms_mine / args.steps]
    if world > 1:
        t = torch.tensor([ms_mine / args.steps], dtype=torch.float64, device="cuda")
        gathered = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(gathered, t)
        per_rank_ms = [float(g.item()) for g in gathered]
    # ---- secondary: the plan API end to end (host arrays -> H2D -> solve -> D2H) ---------------------------
    ms_plan, _, _ = timed(lambda: plan.run(stream), 1 if args.warmup > 0 else 0, args.steps, False)
    ms_plan /= args.steps
    st_plan = plan.stats()
    bad = [i for i in range(len(probs)) if plan.result(i).status != 0]
    if bad:
        raise SystemExit("bench.py: %d problems failed, first status %d" % (len(bad), plan.result(bad[0]).status))
    plan.close()
    # ---- e2e: the drop-in file path -------------------------------------------------------------------------
    td = tempfile.mkdtemp(prefix="psd_bench_r%d_" % rank, dir=tmp_root)
    try:
        i32p = C.POINTER(C.c_int32)
        file_of = {}
        for seed, (s, e, c) in vectors:
            path = os.path.join(td, "v%d.bedGraph" % seed)
            rc = lib.psd_write_bedgraph(path.encode(), b"chrUnknown", len(c), s.ctypes.data_as(i32p), e.ctypes.data_as(i32p), c.ctypes.data_as(i32p))
            assert rc == 0, rc
            file_of[seed] = path
        files = [file_of[seed] for seed, _ in vectors for _ in PEN_STRS]
        pens = [p for _ in vectors for p in PEN_STRS]
        dbs = ["%s_penalty=%s.db" % (f, p) for f, p in zip(files, pens)]
        n = len(files)
        arr = lambda xs: (C.c_char_p * n)(*[x.encode() for x in xs])
        a_files, a_pens, a_dbs = arr(files), arr(pens), arr(dbs)
        status = (C.c_int * n)()
        text_bytes = sum(os.path.getsize(f) for f in file_of.values())

        def file_step():
            rc = lib.psd_fpop_disk_batch(n, a_files, a_pens, a_dbs, status)
            if rc:
                raise SystemExit("bench.py: psd_fpop_disk_batch failed: " + psd._lib.status_text(rc))
            for d in dbs:              # R/PeakSegFPOP_file.R:74-77 deletes the db after every call
                try:
                    os.unlink(d)
                except OSError:
                    pass

        ms_files, _, _ = timed(file_step, 1 if args.warmup > 0 else 0, args.steps, False)
        bs = psd._lib.last_batch_stats()
        assert all(s == 0 for s in status), "file batch: a problem failed"
        e2e_value = total_rows / (ms_files / args.steps / 1e3)
        n_checked, mismatches = check_against_golden(vectors, file_of) if not args.quick else (0, [])
        if mismatches:
            raise SystemExit("bench.py: results differ from the reference fixture: %s" % mismatches[:3])
        out_bytes = sum(os.path.getsize("%s_penalty=%s_%s" % (f, p, suf)) for f, p in zip(files, pens) for suf in ("segments.bed", "loss.tsv"))
    finally:
        lib.psd_release_cache()
        shutil.rmtree(td, ignore_errors=True)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = peaks.get("hbm_gbs", 6650.0)
    alg_bytes = st["store_bytes_algorithmic"]
    dp_s = st["dp_ms"] / 1e3
    achieved = alg_bytes / dp_s / 1e9 if dp_s > 0 else 0.0
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "dp_kernel_traffic.json"))).get("dram_bytes_per_launch")
    except (OSError, ValueError):
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": "fpop_dp_kernel", "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 (of fallback)",
                "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": st["dp_ms"],
                "backtrack": {"kernel": "fpop_backtrack_kernel", "bytes_read": st["backtrack_bytes_read"], "kernel_ms": st["backtrack_ms"],
                              "achieved": (st["backtrack_bytes_read"] / (st["backtrack_ms"] / 1e3) / 1e9) if st["backtrack_ms"] > 0 else 0.0,
                              "unit": "GB/s", "note": "latency-bound pointer chase: one dependent record read per segment"},
                "note": "the DP is bound by fp64 issue/latency, not HBM (DESIGN.md); kernel_ms is the last timed step's DP kernel, CUDA events on the launching stream"}
    # secondary kernel, measured outside the timed region: the device run-length encoding of the
    # count-vector front end (psd_plan_add_counts) on a sample of the same vectors
    try:
        plan_c = psd.Plan(local_rank)
        for seed in list(shard.rank_seeds(rank, args.vectors))[:256]:
            plan_c.add_counts(synth.poisson_counts(seed, 4000 if args.quick else None).astype("int32"), 1000.0)
        best = None
        for _ in range(4):
            plan_c.upload(stream)
            sc = plan_c.stats()
            if best is None or sc["rle_ms"] < best["rle_ms"]:
                best = sc
        rle_gbs = best["rle_bytes_algorithmic"] / (best["rle_ms"] / 1e3) / 1e9 if best["rle_ms"] > 0 else 0.0
        roofline["rle"] = {"kernel": "rle_encode_kernel", "bound": "hbm", "positions": best["rle_positions"],
                           "algorithmic_bytes_per_launch": best["rle_bytes_algorithmic"], "kernel_ms": best["rle_ms"],
                           "achieved": rle_gbs, "peak": peak, "unit": "GB/s", "frac": rle_gbs / peak,
                           "note": "4 B/position read + 12 B/row written; 256 of the vectors, not part of the timed step"}
        plan_c.close()
    except Exception as exc:   # the headline numbers do not depend on it
        roofline["rle"] = {"error": repr(exc)}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": config,
            "value_region": "psd_plan_solve: DP + backtrack kernels, rows resident in HBM (no H2D/D2H inside the timed region)",
            "run_info": {"problems_per_gpu": len(probs), "rows_x_penalties_per_gpu": rows_per_step, "piece_cap": st["piece_cap"],
                         "warps_per_sm": st["warps_per_sm"], "store_waves": st["n_waves"], "overflow_tier_problems": st["n_overflow_tier"],
                         "per_rank_ms_per_step": per_rank_ms, "host_cores": cores},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": bs["h2d_bytes"], "d2h_bytes_per_step": bs["d2h_bytes"],
                    "ms_per_step": ms_files / args.steps,
                    "path": "psd_fpop_disk_batch: %d bedGraph files (%.0f MB of text, tmpfs) x 5 penalties -> parse -> H2D -> DP -> backtrack -> D2H -> "
                            "%d result files (%.0f MB); db files created and removed" % (len(file_of), text_bytes / 1e6, 2 * n, out_bytes / 1e6),
                    "stages_ms_last_step": {k: round(bs[k], 2) for k in ("parse_ms", "build_ms", "run_ms", "write_ms", "release_ms", "dp_ms", "backtrack_ms")},
                    "results_checked_against_reference_fixture": n_checked},
            "e2e_plan_api": {"value": total_rows / (ms_plan / 1e3), "unit": UNIT, "ms_per_step": ms_plan, "h2d_bytes_per_step": st_plan["h2d_bytes"],
                             "d2h_bytes_per_step": st_plan["d2h_bytes"], "path": "psd_plan_run on host arrays: H2D -> DP -> backtrack -> D2H, no text"},
            "gpu_launches": st["n_launches"] * args.steps + bs["n_launches"] * args.steps, "roofline": roofline}
    if world == 1 and not args.no_cpu_baseline:
        td = tempfile.mkdtemp(prefix="psd_ref_", dir=tmp_root)
        try:
            ref = CpuReference(vectors, int(cores * 5e4 * args.ref_seconds), td, cores)
            secs = ref.step()
        finally:
            shutil.rmtree(td, ignore_errors=True)
        line["cpu_baseline"] = {"value": ref.rows / secs, "unit": UNIT, "cores": ref.n_threads, "kind": ref.kind, "sample": ref.sample, "seconds": secs}
    if dumped:
        line["dump_outputs"] = dumped
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
