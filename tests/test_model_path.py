"""Label errors on the device (psd_plan_set_labels / psd_plan_label_errors, Plan.label_errors) and the exact
model-selection path (psd_model_path, model_path_batch): a numpy label-error oracle against brute force,
the CROPS driver of tests/path_oracle.py against a log grid of oracle solves, and every input error,
without a GPU; on the GPU, device errors against the numpy oracle and paths against the oracle driver
bit for bit."""
import contextlib
import ctypes as C
import json
import math
import os
import numpy as np
import pandas as pd
import pytest
import oracle_bind
import path_oracle
from helpers import GOLD

PSD_ERR_ARG = 111
KIND_NAMES = np.array(list(path_oracle.KINDS))


@pytest.fixture(scope="module")
def psd():
    import peaksegdisk_b200
    return peaksegdisk_b200


@pytest.fixture(scope="module")
def gpu(psd):
    assert psd._lib.lib.psd_device_count() >= 1, "no CUDA device"
    return psd


@contextlib.contextmanager
def option(psd, name, value, default):
    psd._lib.lib.psd_set_option(name.encode(), float(value))
    try:
        yield
    finally:
        psd._lib.lib.psd_set_option(name.encode(), float(default))


@contextlib.contextmanager
def options(psd, opts):
    """option() for each (name, value, default) of opts"""
    with contextlib.ExitStack() as stack:
        for name, value, default in opts:
            stack.enter_context(option(psd, name, value, default))
        yield


TWO_BLOCK = [("latency_mode", 2, 0), ("occupancy_mode", 2, 0)]   # the throughput kernel's two-block build, forced


def label_df(ls, le, kind):
    return pd.DataFrame({"chromStart": np.asarray(ls, np.int64), "chromEnd": np.asarray(le, np.int64),
                         "annotation": KIND_NAMES[np.asarray(kind)]})


def random_labels(rng, lo, hi, bounds, n):
    """n labels inside [lo, hi): ends drawn from the given boundaries (peak boundaries, row ends), their
    neighbours, uniform positions and the first and last base."""
    pts = np.unique(np.clip(np.concatenate([bounds, bounds - 1, bounds + 1, [lo, lo + 1, hi - 1, hi],
                                            rng.integers(lo, hi + 1, size=16)]), lo, hi))
    a = rng.choice(pts, size=n); b = rng.choice(pts, size=n)
    ls, le = np.minimum(a, b), np.maximum(a, b)
    le = np.where(ls == le, np.minimum(ls + 1 + rng.integers(0, 5, size=n), hi), le)
    ls = np.where(ls == le, le - 1, ls)
    return ls, le, rng.integers(0, 4, size=n)


def rows_problem(rng, n, constant=False):
    w = rng.integers(1, 30, size=n)
    end = np.cumsum(w) + int(rng.integers(0, 1000))
    start = end - w
    cov = np.full(n, 3) if constant else rng.poisson(rng.choice([1.0, 8.0], size=n))
    return start.astype(np.int32), end.astype(np.int32), cov.astype(np.int32)


# ---- CPU ---------------------------------------------------------------------------------------------

def test_numpy_label_oracle_matches_brute_force():
    rng = np.random.default_rng(11)
    for case in range(1000):
        lo = int(rng.integers(0, 50)); hi = lo + int(rng.integers(5, 120))
        cuts = np.sort(rng.choice(np.arange(lo + 1, hi), size=2 * int(rng.integers(0, min(6, (hi - lo - 1) // 2) + 1)), replace=False))
        ps, pe = cuts[0::2].astype(np.int64), cuts[1::2].astype(np.int64)
        ls, le, kind = random_labels(rng, lo, hi, cuts, int(rng.integers(1, 12)))
        got = path_oracle.label_errors(ps, pe, ls, le, kind)
        want = path_oracle.label_errors_brute(ps, pe, ls, le, kind)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), case


def test_crops_driver_agrees_with_a_log_grid_of_oracle_solves():
    rng = np.random.default_rng(5)
    grid = np.logspace(-3, 5, 2000)
    for case in range(6):
        s, e, c = rows_problem(rng, int(rng.integers(4, 13)))
        models, rounds, solves = path_oracle.crops(path_oracle.oracle_round(s, e, c), 0.0, math.inf)
        assert solves == 2 * len(models) - 1 or len(models) == 1
        by_peaks = {m["peaks"]: m for m in models}
        seen = set()
        for lam in grid:
            st, summ, _ = oracle_bind.solve_rows(s, e, c, float(lam))
            k = int(summ[2])
            seen.add(k)
            m = by_peaks[k]   # every grid model is on the path
            assert m["min.lambda"] * (1 - 1e-9) <= lam <= m["max.lambda"] * (1 + 1e-9), (case, lam, m)
        for m in models:   # every model whose interval holds a few grid points was seen on the grid
            lo, hi = max(m["min.lambda"], grid[0]), min(m["max.lambda"], grid[-1])
            if hi > lo * (grid[1] / grid[0]) ** 3:
                assert m["peaks"] in seen, (case, m)
        assert models[0]["max.lambda"] == math.inf and models[-1]["min.lambda"] == 0.0


def test_set_labels_input_errors(psd):
    lib = psd._lib.lib
    p32 = C.POINTER(C.c_int32)
    plan = psd.Plan()
    pid = plan.add(np.array([10, 20]), np.array([20, 40]), np.array([1, 5]), 10.0)

    def call(ls, le, kind, id_=pid):
        a, b, k = (np.asarray(x, np.int32) for x in (ls, le, kind))
        return lib.psd_plan_set_labels(plan._h, id_, len(k), a.ctypes.data_as(p32), b.ctypes.data_as(p32), k.ctypes.data_as(p32))
    for args, words in [(([10], [41], [0]), "label 0"), (([9], [20], [0]), "label 0"), (([10, 30], [20, 30], [1, 1]), "label 1"),
                        (([10], [20], [4]), "kind 4"), (([10], [20], [-1]), "kind -1"), (([25, 22], [24, 30], [0, 2]), "label 0")]:
        assert call(*args) == PSD_ERR_ARG
        msg = lib.psd_last_error().decode()
        assert "problem %d" % pid in msg and words in msg, msg
    assert call([10], [20], [0], id_=7) == PSD_ERR_ARG and "problem 7" in lib.psd_last_error().decode()
    assert lib.psd_plan_set_labels(plan._h, pid, 2, None, None, None) == PSD_ERR_ARG
    with pytest.raises(ValueError):
        plan.set_labels(pid, {"chromStart": [10], "chromEnd": [20], "annotation": ["peak"]})
    with pytest.raises(ValueError):   # set but not solved yet
        plan.set_labels(pid, label_df([10], [40], [1]))
        plan.label_errors(pid)


def test_model_path_input_errors(psd):
    s, e, c = np.array([0, 5, 9], np.int32), np.array([5, 9, 20], np.int32), np.array([1, 4, 2], np.int32)
    ok = (s, e, c)
    cases = [
        (dict(pen_min=float("nan")), "pen_min"), (dict(pen_min=-1.0), "pen_min"), (dict(pen_min=5.0, pen_max=4.0), "pen_min > pen_max"),
        (dict(pen_min=math.inf, pen_max=1e9), "infinite"), (dict(pen_max=float("nan")), "pen_max"),
    ]
    for kw, words in cases:
        with pytest.raises(ValueError, match=words):
            psd.model_path_batch([ok], **kw)
    bad_rows = [(s, e + 1, c), (s, e, -c), (s[:0], e[:0], c[:0])]
    for bad in bad_rows:
        with pytest.raises(ValueError, match="problem 1"):
            psd.model_path_batch([ok, bad])
    for lab, words in [(label_df([0], [21], [0]), "label 0"), (label_df([3, 4], [5, 4], [0, 1]), "label 1"),
                       (pd.DataFrame({"chromStart": [1], "chromEnd": [2], "annotation": ["peakStart"]}).assign(chromStart=[-1]), "label 0")]:
        with pytest.raises(ValueError, match="problem 1: " + words):
            psd.model_path_batch([ok, ok], labels=[None, lab])
    lib = psd._lib.lib
    h = C.c_void_p()
    assert lib.psd_model_path(-1, -1, None, 0.0, 1.0, C.byref(h)) == PSD_ERR_ARG
    assert "n_problems" in lib.psd_last_error().decode() and not h.value
    k = (psd._lib.PsdPathProblem * 1)()
    k[0].n_rows = 3; k[0].chromStart = s.ctypes.data_as(C.POINTER(C.c_int32)); k[0].chromEnd = e.ctypes.data_as(C.POINTER(C.c_int32))
    k[0].coverage = c.ctypes.data_as(C.POINTER(C.c_int32)); k[0].n_labels = 1   # null label arrays
    assert lib.psd_model_path(-1, 1, k, 0.0, 1.0, C.byref(h)) == PSD_ERR_ARG
    assert "problem 0" in lib.psd_last_error().decode()


def test_constant_coverage_path_is_solved_on_the_host(psd):
    # one model, no peaks; labels that need a peak are false negatives
    s = np.array([0, 5], np.int32)
    paths, st = psd.model_path_batch([(s, s + 5, np.array([2, 2]))], labels=[label_df([0, 2, 4, 6], [2, 4, 6, 10], [0, 1, 2, 3])])
    m = paths[0]["models"]
    assert len(m) == 1 and m["peaks"][0] == 0 and m["min.lambda"][0] == 0 and math.isinf(m["max.lambda"][0])
    assert list(m[["fp", "fn", "possible.fp", "possible.fn", "errors"]].iloc[0]) == [0, 3, 3, 3, 3]
    assert paths[0]["target"] == (0.0, math.inf, 3)
    assert st["rounds"] == 1 and st["solves"] == 2 and st["rows_solved"] == 0


# ---- GPU ---------------------------------------------------------------------------------------------

def device_errors_case(psd):
    """~200 seeded problems of 1e3..1e5 rows with labels on and between their peak boundaries: penalties 0
    and Inf, a constant-coverage problem and a count-vector problem included."""
    from peaksegdisk_b200 import synth
    rng = np.random.default_rng(2024)
    probs = []
    for k in range(200):
        n = int(round(10 ** rng.uniform(3, 5)))
        if k == 0:
            probs.append(("rows", rows_problem(rng, 1500, constant=True), 1e3))
        elif k == 1:
            probs.append(("counts", synth.poisson_counts(77, 30000), 1e3))
        else:
            pen = [0.0, math.inf][k - 2] if k < 4 else float(10 ** rng.uniform(1, 6))
            if k == 2:
                n = 1000
            probs.append(("rows", synth.poisson_problem(1000 + k, n), pen))
    return probs, rng


def solve_with_labels(psd, probs, rng, labels=None):
    plan = psd.Plan()
    ids = [plan.add_counts(x, pen) if kind == "counts" else plan.add(*x, pen) for kind, x, pen in probs]
    if labels is None:   # label ends on and next to the first solve's peak boundaries
        plan.run()
        labels = []
        for pid, (kind, x, pen) in zip(ids, probs):
            s, e, pk, _ = plan.segments(pid)
            lo, hi = int(s.min()), int(e.max())
            bounds = np.concatenate([s[pk == 1], e[pk == 1], s[:3]]).astype(np.int64)
            labels.append(random_labels(rng, lo, hi, bounds, int(rng.integers(1, 40))))
    for pid, lab in zip(ids, labels):
        plan.set_labels(pid, label_df(*lab))
    plan.run()
    return plan, ids, labels


@pytest.mark.gpu
def test_device_label_errors_equal_the_numpy_oracle(gpu):
    psd = gpu
    probs, rng = device_errors_case(psd)
    plan, ids, labels = solve_with_labels(psd, probs, rng)
    assert plan.stats()["n_launches"] >= 3
    want = []
    for pid, lab in zip(ids, labels):
        s, e, pk, _ = plan.segments(pid)
        ps, pe = path_oracle.peaks_of(s, e, pk)
        fp, fn = path_oracle.label_errors(ps, pe, *lab)
        df, tot = plan.label_errors(pid)
        assert np.array_equal(df["fp"].to_numpy(), fp) and np.array_equal(df["fn"].to_numpy(), fn), pid
        assert tot["errors"] == fp.sum() + fn.sum() and tot["fp"] == fp.sum() and tot["fn"] == fn.sum()
        assert tot["possible.fp"] == int((lab[2] != 1).sum()) and tot["possible.fn"] == int((lab[2] != 0).sum())
        want.append((fp, fn))
    assert plan.result(ids[0]).trivial == 1 and plan.result(ids[3]).trivial == 1
    # the same errors from the latency kernel, from the throughput kernel's two-block build, from several
    # store waves and from the global piece-list tier
    for name, opts in [("latency", [("latency_mode", 1, 0)]), ("two-block", TWO_BLOCK),
                       ("store waves", [("store_gb", 0.1, 0), ("host_spill_gb", 0, -1)]), ("piece_cap", [("piece_cap", 8, 48)])]:
        with options(psd, opts):
            plan2, ids2, _ = solve_with_labels(psd, probs, rng, labels)
        st = plan2.stats()
        if name == "store waves":
            assert st["n_waves"] > 1, st
        for pid, (fp, fn) in zip(ids2, want):
            df, _ = plan2.label_errors(pid)
            assert np.array_equal(df["fp"].to_numpy(), fp) and np.array_equal(df["fn"].to_numpy(), fn), (name, pid)


@pytest.mark.gpu
def test_plan_without_labels_launches_what_it_did(gpu):
    from peaksegdisk_b200 import synth
    plan, ids = gpu.solve_batch([(*synth.poisson_problem(s, 5000), 1e3) for s in range(4)])
    assert plan.stats()["n_launches"] == 2 * plan.stats()["n_waves"]


def assert_table_equal(got, want, what):
    cols = ["min.lambda", "max.lambda", "penalty", "peaks", "segments", "total.loss"]
    assert len(got) == len(want), (what, len(got), len(want))
    for col in cols:
        g = got[col].to_numpy().astype(float)
        w = np.array([float(m[col]) for m in want])
        assert np.array_equal(g, w), (what, col, np.flatnonzero(g != w)[:5])


@pytest.mark.gpu
def test_model_path_equals_the_oracle_driver_bit_for_bit(gpu):
    """With the automatic kernel choice and with the throughput kernel's two-block build forced."""
    from peaksegdisk_b200 import synth
    rng = np.random.default_rng(99)
    small, large = [], []
    for k in range(20):
        n = int(rng.integers(200, 2001))
        (small if n <= 500 else large).append(synth.poisson_problem(500 + k, n))
    for probs, lo, hi in [(small, 0.0, math.inf), (large, 10.0, 1e4)]:
        want = [path_oracle.crops(path_oracle.oracle_round(s, e, c), lo, hi) for s, e, c in probs]
        for build, opts in [("auto", []), ("two-block", TWO_BLOCK)]:
            with options(gpu, opts):
                paths, st = gpu.model_path_batch(probs, pen_min=lo, pen_max=hi)
            for k, (models, rounds, n_solves) in enumerate(want):
                assert_table_equal(paths[k]["models"], models, (build, lo, k))
            assert st["solves"] == sum(w[2] for w in want) and st["models"] == sum(len(p["models"]) for p in paths), build


@pytest.mark.gpu
def test_mono27ac_path_equals_the_golden_table(gpu):
    from peaksegdisk_b200 import synth
    gold = json.load(open(os.path.join(GOLD, "golden_path_mono27ac.json")))
    _, s, e, c = synth.read_bedgraph(os.path.join(GOLD, "Mono27ac_coverage.bedGraph"))
    paths, st = gpu.model_path_batch([(s, e, c)], pen_min=100.0)
    cols = gold["columns"]
    want = [dict(zip(cols, [float(v) if isinstance(v, str) else v for v in row])) for row in gold["models"]]
    assert_table_equal(paths[0]["models"], want, "Mono27ac")
    assert (len(want), gold["solves"], gold["rounds"]) == (380, 759, 14)
    assert (st["models"], st["solves"], st["rounds"]) == (380, 759, 14)
    # the golden solves at penalties >= 100 fall in the interval of a model with their peak count
    m = paths[0]["models"]
    lo, hi, pk = m["min.lambda"].to_numpy(), m["max.lambda"].to_numpy(), m["peaks"].to_numpy()
    g = json.load(open(os.path.join(GOLD, "golden_mono27ac.json")))
    checks = [(float(p), int(v["loss"].split("\t")[2])) for p, v in g["penalties"].items() if p in ("100", "1952.6", "1e6", "1000000", "Inf")]
    checks += [(float(x["penalty_str"]), x["peaks"]) for x in g["search19"] if float(x["penalty_str"]) >= 100]
    assert len(checks) >= 6
    for lam, peaks in checks:
        inside = (lo <= lam) & (lam <= hi)   # on a boundary either neighbour counts
        assert peaks in set(pk[inside]), (lam, peaks)


@pytest.fixture(scope="module")
def synth64(gpu):
    from peaksegdisk_b200 import synth
    probs = [synth.poisson_problem(3000 + k) for k in range(64)]
    rng = np.random.default_rng(64)
    labels = []
    for s, e, c in probs:
        lo, hi = int(s[0]), int(e[-1])
        labels.append(label_df(*random_labels(rng, lo, hi, e[rng.integers(0, len(e), size=20)].astype(np.int64), 12)))
    paths, st = gpu.model_path_batch(probs, labels=labels, pen_min=1e3)
    assert all(p["status"] == 0 for p in paths)
    return probs, labels, paths


@pytest.mark.gpu
def test_synth_paths_midpoints_solve_to_their_models(gpu, synth64):
    probs, _, paths = synth64
    plan = gpu.Plan()
    want = []
    for (s, e, c), p in zip(probs, paths):
        m = p["models"]
        for lo, hi, pk in zip(m["min.lambda"], m["max.lambda"], m["peaks"]):
            if 0 < lo and math.isfinite(hi) and hi > lo * (1 + 1e-9):
                want.append((plan.add(s, e, c, math.sqrt(lo * hi)), int(pk)))
    plan.run()
    assert len(want) > 64
    bad = [(pid, pk, plan.result(pid).n_peaks) for pid, pk in want if plan.result(pid).n_peaks != pk]
    assert not bad, bad[:5]


@pytest.mark.gpu
def test_synth_paths_are_the_same_alone_and_with_store_waves(gpu, synth64):
    probs, labels, paths = synth64
    cols = ["min.lambda", "max.lambda", "penalty", "peaks", "segments", "total.loss", "errors"]
    order = np.argsort([len(c) for _, _, c in probs])
    for k in order[:3]:
        alone, _ = gpu.model_path_batch([probs[k]], labels=[labels[k]], pen_min=1e3)
        pd.testing.assert_frame_equal(alone[0]["models"][cols], paths[k]["models"][cols], check_exact=True)
    with option(gpu, "store_gb", 0.5, 0), option(gpu, "host_spill_gb", 0, -1):   # each round's solve runs in several store waves
        waved, st = gpu.model_path_batch(probs, labels=labels, pen_min=1e3)
    for k in range(len(probs)):
        pd.testing.assert_frame_equal(waved[k]["models"], paths[k]["models"], check_exact=True)


@pytest.mark.gpu
def test_synth_path_errors_and_targets(gpu, synth64):
    probs, labels, paths = synth64
    plan = gpu.Plan()
    jobs = []
    for k, ((s, e, c), p) in enumerate(zip(probs, paths)):
        for row in p["models"].itertuples(index=False):
            jobs.append((k, plan.add(s, e, c, row[4]), row))
    plan.run()
    for k, pid, row in jobs:
        s, e, pk, _ = plan.segments(pid)
        lab = labels[k]
        fp, fn = path_oracle.label_errors(*path_oracle.peaks_of(s, e, pk), lab["chromStart"], lab["chromEnd"],
                                          lab["annotation"].map(path_oracle.KINDS))
        assert plan.result(pid).n_peaks == row[5]
        assert (row[8], row[9], row[12]) == (fp.sum(), fn.sum(), fp.sum() + fn.sum()), (k, row)
    for p in paths:
        m = p["models"]
        want = path_oracle.target_interval(m["min.lambda"].to_numpy(), m["max.lambda"].to_numpy(), m["errors"].to_numpy())
        assert p["target"] == want, (p["target"], want)
