"""GPU parity tests (run with -m gpu on the B200 box).  Everything goes through the C ABI of
libpeaksegdisk_b200.so (ctypes); expected values are the golden vectors generated from the unmodified
reference (tools/make_golden.py) and the oracle on the same seeded inputs.

Bars (BASELINE.json north_star): segment chromStart/chromEnd, peak counts, selected penalty bit-exact;
total Poisson loss within 1e-9 relative.  Because the kernels use the reference's libm bit for bit
(psd_math.h) we in fact require the whole _loss.tsv / _segments.bed text to be byte-identical, which
implies both bars; the 1e-9 comparison is kept for hosts whose libm differs from the goldens'."""
import ctypes as C
import math
import os
import numpy as np
import pytest
import oracle_bind
import oracle_checks
from oracle_checks import check_vs_oracle as _check_vs_oracle, LOSS_RTOL
from helpers import ROOT, GOLD, golden, sha, outputs, synth_rows, rows_text, parse_rows, loss_fields

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def psd():
    import peaksegdisk_b200
    assert peaksegdisk_b200._lib.lib.psd_device_count() >= 1, "no CUDA device"
    return peaksegdisk_b200


BUILDS = {"auto": (0, 0), "throughput-kernel": (2, 1), "two-block": (2, 2)}   # latency_mode, occupancy_mode


@pytest.fixture(autouse=True, params=list(BUILDS))
def kernel_mode(request, psd):
    """Every test runs three times: with the automatic choice (small waves go to the latency kernel: one
    problem per block, one chain per warp), with the throughput kernel's one-block build forced (one
    problem per warp, one block of 14 warps per SM, 48-piece shared-memory tier) and with its two-block
    build forced (two blocks per SM, 24-piece tier), so every kernel build sees every parity case.  The
    environment carries the same choice to the subprocess tools."""
    lat, occ = BUILDS[request.param]
    lib = psd._lib.lib
    lib.psd_set_option(b"latency_mode", float(lat))
    lib.psd_set_option(b"occupancy_mode", float(occ))
    os.environ["PSD_LATENCY_MODE"] = str(lat)
    os.environ["PSD_OCCUPANCY_MODE"] = str(occ)
    yield request.param
    lib.psd_set_option(b"latency_mode", 0.0)
    lib.psd_set_option(b"occupancy_mode", 0.0)
    os.environ.pop("PSD_LATENCY_MODE", None)
    os.environ.pop("PSD_OCCUPANCY_MODE", None)


def _disk(psd, path, pen, db=None):
    return psd._lib.lib.psd_fpop_disk(path.encode(), pen.encode(), (db or path + ".db").encode())


def test_reference_test_vectors_byte_identical(psd, tmp_path):
    """tests/testthat vectors (SURVEY.md Appendix A): every output byte equals the reference's."""
    for k, case in enumerate(golden("golden_small.json")):
        path = str(tmp_path / ("c%d.bedGraph" % k))
        open(path, "w").write(case["input"])
        assert _disk(psd, path, case["penalty"]) == case["status"], case["name"]
        assert outputs(path, case["penalty"]) == (case["segments"], case["loss"]), (case["name"], case["penalty"])
        # db: created on the DP branch only (R reports its size and deletes it)
        assert os.path.isfile(path + ".db") == (case["db_bytes"] is not None), (case["name"], case["penalty"])
        if os.path.isfile(path + ".db"):
            os.unlink(path + ".db")


def test_status_codes_and_created_files(psd, tmp_path):
    dbdir = tmp_path / "dbdir"
    dbdir.mkdir()
    for k, case in enumerate(golden("golden_errors.json")):
        path = str(tmp_path / ("e%d.bedGraph" % k))
        if not case["missing"]:
            open(path, "w").write(case["input"])
        st = _disk(psd, path, case["penalty"], str(dbdir) if case["db"] else None)
        assert st == case["status"], case["name"]
        assert outputs(path, case["penalty"]) == (case["segments"], case["loss"]), case["name"]


def test_mono27ac_config1(psd, tmp_path):
    """BASELINE config 1: Mono27ac chr11 coverage, penalty 10.5 (+ the other probed penalties)."""
    g = golden("golden_mono27ac.json")
    path = str(tmp_path / "coverage.bedGraph")
    open(path, "w").write(open(os.path.join(GOLD, "Mono27ac_coverage.bedGraph")).read())
    pens = list(g["penalties"])
    st = psd.PeakSegFPOP_file_batch([path] * len(pens), pens)
    assert st == [0] * len(pens)
    for pen in pens:
        want = g["penalties"][pen]
        seg, loss = outputs(path, pen)
        assert loss == want["loss"], pen
        assert sha(seg) == want["segments_sha256"], pen
    f = loss_fields(outputs(path, "10.5")[1])
    assert (f["segments"], f["peaks"], f["bases"], f["lines"]) == (2269, 1134, 520000, 6921)
    assert abs(f["total_loss"] - (-127781.95220675057)) <= LOSS_RTOL * 127781.95


def test_seeded_synthetic_vs_reference_golden_one_batch(psd, tmp_path):
    """64 problems (Poisson + worst-case increasing counts, > 1500 pieces per function) in ONE launch;
    the increasing ones overflow the shared-memory tier and are re-run from global-memory lists."""
    cases = golden("golden_synth.json")
    paths, pens = [], []
    files = {}
    for case in cases:
        key = (case["kind"], tuple(case["key"]))
        if key not in files:
            s, e, c = synth_rows(case["kind"], case["key"])
            p = str(tmp_path / ("%s_%s.bedGraph" % (case["kind"], "_".join(map(str, case["key"])))))
            open(p, "w").write(rows_text(s, e, c))
            files[key] = p
        paths.append(files[key]); pens.append(case["penalty"])
    st = psd.PeakSegFPOP_file_batch(paths, pens)
    assert st == [c["status"] for c in cases]
    for case, p, pen in zip(cases, paths, pens):
        seg, loss = outputs(p, pen)
        assert loss == case["loss"], (case["kind"], case["key"], pen)
        assert sha(seg) == case["segments_sha256"], (case["kind"], case["key"], pen)


def test_in_memory_batch_vs_oracle_fresh_seeds(psd):
    from peaksegdisk_b200 import synth
    rng = np.random.default_rng(1234)
    probs = []
    for seed in range(100, 124):
        s, e, c = synth.poisson_problem(seed, int(rng.integers(500, 6000)))
        probs.append((s, e, c, float(10 ** rng.uniform(-1, 6))))
    # ragged / edge shapes
    probs.append((np.array([0, 1], np.int32), np.array([1, 3], np.int32), np.array([5, 3], np.int32), 0.1))
    probs.append((np.array([0, 5, 9], np.int32), np.array([5, 9, 100], np.int32), np.array([0, 7, 0], np.int32), 0.0))
    z = np.zeros(40, np.int32); z[17] = 3
    probs.append((np.arange(40, dtype=np.int32), np.arange(1, 41, dtype=np.int32), z, 2.0))
    plan, ids = psd.solve_batch(probs)
    for pid, (s, e, c, pen) in zip(ids, probs):
        _check_vs_oracle(plan, pid, s, e, c, pen)
    st = plan.stats()
    assert st["n_launches"] >= 2 and st["rows_solved"] == sum(len(p[2]) for p in probs)


def test_trivial_and_mixed_batch(psd):
    """Inf penalty and constant coverage never reach the kernel; mixed with real problems."""
    from peaksegdisk_b200 import synth
    s, e, c = synth.poisson_problem(5, 700)
    five = np.full(3, 5, np.int32)
    plan, ids = psd.solve_batch([(s, e, c, math.inf), (np.array([1, 2, 3], np.int32), np.array([2, 3, 4], np.int32), five, 0.0),
                                 (s, e, c, 30.0)])
    r0, r1 = plan.result(ids[0]), plan.result(ids[1])
    assert r0.trivial == 1 and r0.n_segments == 1 and r1.trivial == 1 and r1.n_peaks == 0
    assert plan.loss_row(ids[1])["total.loss"] == -9.1415686865115048931   # test-CRAN-PeakSegFPOP_dir.R:113-129
    _check_vs_oracle(plan, ids[2], s, e, c, 30.0)


def test_r_api_vectors(psd, tmp_path):
    # test-CRAN-PeakSegFPOP_vec.R
    fit = psd.PeakSegFPOP_vec(np.array([1, 3, 0, 4, 2]), 0)
    assert len(fit["segments"]) == 5 and fit["segments"]["status"].tolist() == ["background", "peak"] * 2 + ["background"]
    assert len(psd.PeakSegFPOP_vec(np.array([1, 3, 0, 4, 2]), float("inf"))["segments"]) == 1
    # test-CRAN-PeakSegFPOP_file.R:30-42
    import pandas as pd
    four = pd.DataFrame({"chrom": "chr1", "chromStart": [0, 10, 20, 30], "chromEnd": [10, 20, 30, 40], "count": [2, 10, 14, 13]})
    d = tmp_path / "prob"
    d.mkdir()
    psd.writeBedGraph(four, str(d / "coverage.bedGraph"))
    fit = psd.PeakSegFPOP_dir(str(d), "10.5")
    assert fit["segments"]["chromStart"].tolist() == [30, 10, 0] and fit["segments"]["chromEnd"].tolist() == [40, 30, 10]
    assert fit["segments"]["status"].tolist() == ["background", "peak", "background"]
    assert np.allclose(fit["segments"]["mean"], [12.3333, 12.3333, 2], atol=1e-3)
    assert int(fit["loss"]["peaks"][0]) == 1 and "megabytes" in fit["loss"] and "seconds" in fit["loss"]
    # cache: second call must not re-run the solver (timing file unchanged)
    t = os.path.getmtime(str(d / "coverage.bedGraph_penalty=10.5_timing.tsv"))
    fit2 = psd.PeakSegFPOP_dir(str(d), "10.5")
    assert os.path.getmtime(str(d / "coverage.bedGraph_penalty=10.5_timing.tsv")) == t
    assert fit2["segments"].equals(fit["segments"])
    # an empty cached loss file is recomputed (test-CRAN-PeakSegFPOP_dir.R:38-43)
    open(str(d / "coverage.bedGraph_penalty=10.5_loss.tsv"), "w").close()
    assert int(psd.PeakSegFPOP_dir(str(d), "10.5")["loss"]["peaks"][0]) == 1
    # unwritable db (test-CRAN-PeakSegFPOP_file.R:64-68)
    with pytest.raises(RuntimeError, match="unable to write to cost function database file"):
        psd.PeakSegFPOP_file(str(d / "coverage.bedGraph"), "10.5", str(tmp_path))
    # (0,0,5) at 0 and 10000 (test-CRAN-PeakSegFPOP_dir.R:139-160)
    zzf = pd.DataFrame({"chrom": "chr1", "chromStart": [1, 2, 3], "chromEnd": [2, 3, 4], "count": [0, 0, 5]})
    fit = psd.PeakSegFPOP_df(zzf, 0, str(tmp_path))
    assert fit["segments"]["mean"].tolist() == [2.5, 2.5, 0] and int(fit["loss"]["peaks"][0]) == 1
    fit = psd.PeakSegFPOP_df(zzf, 10000, str(tmp_path))
    assert len(fit["segments"]) == 1 and abs(fit["segments"]["mean"][0] - 5 / 3) < 1e-5


def test_sequential_search_selected_penalty_bit_exact(psd, tmp_path):
    """config 3 semantics on Mono27ac, target 19 peaks (test-TRAVIS-sequentialSearch.R:25-29): the whole
    penalty chain (15-digit strings) and the selected model equal the reference's."""
    chain = golden("golden_mono27ac.json")["search19"]
    d = tmp_path / "chr11-60000-580000"
    d.mkdir()
    open(str(d / "coverage.bedGraph"), "w").write(open(os.path.join(GOLD, "Mono27ac_coverage.bedGraph")).read())
    fit = psd.sequentialSearch_dir(str(d), 19)
    assert int(fit["loss"]["peaks"][0]) == 19 and len(fit["segments"]) == 39
    others = fit["others"]
    got = sorted((int(r["iteration"]), psd.r_paste(float(r["penalty"])), int(r["peaks"])) for _, r in others.iterrows())
    want = sorted((c["iteration"], c["penalty_str"], c["peaks"]) for c in chain)
    assert got == want
    assert psd.r_paste(float(fit["loss"]["penalty"][0])) == "1715.84956360692"
    for c in chain:   # every loss line of the chain is byte-identical
        assert outputs(str(d / "coverage.bedGraph"), c["penalty_str"])[1] == c["loss"]
    # test-CRAN-sequentialSearch.R: more peaks than possible
    d2 = tmp_path / "supp"
    d2.mkdir()
    open(str(d2 / "coverage.bedGraph"), "w").write("".join("chr1\t%d\t%d\t%d\n" % (i, i + 1, v) for i, v in enumerate([3, 9, 18, 15, 20, 2])))
    with pytest.raises(ValueError, match="peaks.int=5 but max=2 peaks for N=6 data"):
        psd.sequentialSearch_dir(str(d2), 5)
    assert int(psd.sequentialSearch_dir(str(d2), 2)["loss"]["peaks"][0]) == 2


def _poisson_loss(s, e, c, seg):
    """sum_i w_i (m - z_i log m) recomputed from the returned segmentation (independent of the solver)"""
    w = (e - s).astype(np.float64); z = c.astype(np.float64)
    ends = np.concatenate(([0], np.cumsum(w)))
    total = 0.0
    pos = {int(v): k + 1 for k, v in enumerate(e)}
    for st, en, _, m in zip(*seg):
        a = 0 if st == s[0] else pos[int(st)]
        b = pos[int(en)]
        ww, zz = w[a:b], z[a:b]
        total += float(np.sum(ww * m) - (np.sum(ww * zz) * math.log(m) if m > 0 else 0.0))
    return total


def test_full_size_properties_config2_shapes(psd):
    """Problems at BASELINE config-2 sizes (N up to 1e5) are too slow for the scalar oracle in a test,
    so check size-independent properties: contiguous alternating segments, up/down constraint, loss
    identity, loss recomputed from the segmentation, monotonicity in the penalty, and independence of
    batch position."""
    from peaksegdisk_b200 import synth
    rows = [synth.poisson_problem(seed, n) for seed, n in [(900, 100000), (901, 60000), (902, 31000)]]
    pens = [1e2, 1e3, 1e4, 1e5, 1e6]
    probs = [(s, e, c, p) for (s, e, c) in rows for p in pens] + [rows[0] + (1e3,)]
    plan, ids = psd.solve_batch(probs)
    by = {}
    for pid, (s, e, c, pen) in zip(ids, probs):
        r = plan.loss_row(pid)
        seg = plan.segments(pid)
        n = r["segments"]
        assert r["peaks"] == (n - 1) // 2 and n % 2 == 1
        assert seg[1][0] == e[-1] and seg[0][-1] == s[0] and np.array_equal(seg[0][:-1], seg[1][1:])
        assert seg[2].tolist() == [k & 1 for k in range(n)]
        m = seg[3][::-1]            # chromosome order: bg, peak, bg, ...
        up = m[1::2] >= m[0:-1:2]; down = m[2::2] <= m[1::2]
        assert up.all() and down.all()
        assert r["bases"] == int(e[-1] - s[0]) and r["bedGraph.lines"] == len(c)
        assert r["total.loss"] == r["mean.pen.cost"] * r["bases"] - pen * r["peaks"]
        recomputed = _poisson_loss(s, e, c, seg)
        assert abs(recomputed - r["total.loss"]) <= 1e-9 * max(1.0, abs(r["total.loss"])) * 10
        by.setdefault(id(c), []).append((pen, r["peaks"], r["total.loss"]))
    for v in by.values():
        v.sort()
        assert all(a[1] >= b[1] for a, b in zip(v, v[1:])), "peaks must not increase with the penalty"
        assert all(a[2] <= b[2] + 1e-9 * abs(b[2]) for a, b in zip(v, v[1:])), "loss must not decrease with the penalty"
    a, b = plan.loss_row(ids[1]), plan.loss_row(ids[-1])     # same problem at two batch positions
    assert a == b and all(np.array_equal(x, y) for x, y in zip(plan.segments(ids[1]), plan.segments(ids[-1])))


def test_store_waves_and_small_piece_tier_give_identical_results(psd):
    """A store pool too small for the batch forces several waves; a tiny shared-memory tier forces the
    global-memory tier.  Results must not change."""
    from peaksegdisk_b200 import synth
    probs = [synth.poisson_problem(seed, 4000) + (pen,) for seed, pen in [(300, 0.0), (301, 10.0), (302, 1e3), (303, 1e5),
                                                                          (304, 50.0), (305, 2e4)]]
    base, ids = psd.solve_batch(probs)
    want = [(base.loss_row(i), base.segments(i)) for i in ids]
    lib = psd._lib.lib
    try:
        lib.psd_set_option(b"store_gb", 0.004)     # ~4 MB: not enough for all six
        lib.psd_set_option(b"host_spill_gb", 0.0)  # no pinned-host spill: the store must be recycled in waves
        lib.psd_set_option(b"piece_cap", 8.0)
        plan, ids2 = psd.solve_batch(probs)
    finally:
        lib.psd_set_option(b"store_gb", 0.0)
        lib.psd_set_option(b"host_spill_gb", -1.0)
        lib.psd_set_option(b"piece_cap", 48.0)
    st = plan.stats()
    assert st["n_waves"] > 1 and st["n_overflow_tier"] > 0, st
    for i, (loss, seg) in zip(ids2, want):
        assert plan.loss_row(i) == loss
        assert all(np.array_equal(x, y) for x, y in zip(plan.segments(i), seg))


def test_penalty_update_resolves_same_rows(psd):
    from peaksegdisk_b200 import synth
    s, e, c = synth.poisson_problem(77, 3000)
    plan = psd.Plan()
    pid = plan.add(s, e, c, 5.0)
    plan.run()
    first = plan.loss_row(pid)
    plan.set_penalty(pid, 500.0)
    plan.solve(); plan.download()
    _check_vs_oracle(plan, pid, s, e, c, 500.0)
    plan.set_penalty(pid, 5.0)
    plan.solve(); plan.download()
    assert plan.loss_row(pid) == first


def test_config5_worst_case_piece_counts(psd):
    """BASELINE config 5 (vignettes/Worst_case.Rmd): strictly increasing counts make the number of
    pieces per function grow like N/2 (1,575 at N=3000 and penalty 1e6) -- far beyond the shared-memory
    tier and beyond the per-warp spill workspace, so the host re-runs them from large global lists.
    Compared with the oracle on the same rows (golden_synth.json pins N<=3000 against the reference)."""
    from peaksegdisk_b200 import synth
    probs = []
    for n, pen in [(1000, 1e6), (2000, 1e4), (3000, 1e6), (600, 0.0)]:
        probs.append(synth.increasing_problem(n) + (pen,))
    plan, ids = psd.solve_batch(probs)
    for pid, (s, e, c, pen) in zip(ids, probs):
        _check_vs_oracle(plan, pid, s, e, c, pen)
    assert max(plan.loss_row(i)["max.intervals"] for i in ids) > 1000


def test_config3_shape_one_long_problem(psd):
    """BASELINE config 3 shape: one long bedGraph (here 3e5 count positions, about 2.2e5 rows; the
    1e6-row original takes the scalar oracle a minute per penalty) solved at the first penalties a
    sequential search would try; a single warp owns the whole problem."""
    from peaksegdisk_b200 import synth
    s, e, c = synth.poisson_problem(2024, 300000)
    plan = psd.Plan()
    pid0 = plan.add(s, e, c, 0.0)
    pidinf = plan.add(s, e, c, math.inf)
    plan.run()
    over, under = plan.loss_row(pid0), plan.loss_row(pidinf)
    _check_vs_oracle(plan, pid0, s, e, c, 0.0)
    nxt = (over["total.loss"] - under["total.loss"]) / (under["peaks"] - over["peaks"])   # R/sequentialSearch_dir.R:90
    assert nxt > 0
    pen = float(psd.r_paste(nxt))          # the search passes the 15-digit string on
    plan.set_penalty(pid0, pen)
    plan.run()
    _check_vs_oracle(plan, pid0, s, e, c, pen)


def test_file_batch_with_mixed_errors(psd, tmp_path):
    """One launch for a batch in which some entries fail validation: each gets its own status, the
    others are solved."""
    good = str(tmp_path / "good.bedGraph")
    open(good, "w").write("chr1\t0\t10\t2\nchr1\t10\t20\t10\nchr1\t20\t30\t14\nchr1\t30\t40\t13\n")
    gap = str(tmp_path / "gap.bedGraph")
    open(gap, "w").write("chr1 0 1 5\nchr1 2 3 3\n")
    st = psd.PeakSegFPOP_file_batch([good, gap, good, str(tmp_path / "missing"), good],
                                    ["10.5", "1", "-2", "1", "Inf"])
    assert st == [0, 6, 2, 3, 0]
    g = [c for c in golden("golden_small.json") if c["name"] == "four"]
    for pen in ("10.5", "Inf"):
        want = [c for c in g if c["penalty"] == pen][0]
        assert outputs(good, pen) == (want["segments"], want["loss"])


def test_batched_sequential_search_follows_single_chains(psd, tmp_path):
    """sequentialSearch_batch advances many searches in lock step (one launch per iteration); every
    problem must end with exactly the model its own sequentialSearch_dir finds."""
    from peaksegdisk_b200 import synth
    dirs, targets = [], []
    for k, (seed, n, target) in enumerate([(40, 6000, 5), (41, 8000, 12), (42, 5000, 0), (43, 7000, 30)]):
        s, e, c = synth.poisson_problem(seed, n)
        for tag in ("a", "b"):
            d = tmp_path / ("%s%d" % (tag, k))
            d.mkdir()
            synth.write_bedgraph(str(d / "coverage.bedGraph"), s, e, c)
        dirs.append(str(tmp_path / ("a%d" % k))); targets.append(target)
    batch = psd.sequentialSearch_batch(dirs, targets)
    for k, (fit, target) in enumerate(zip(batch, targets)):
        single = psd.sequentialSearch_dir(str(tmp_path / ("b%d" % k)), target)
        assert int(fit["loss"]["peaks"][0]) == int(single["loss"]["peaks"][0]) <= target
        assert psd.r_paste(float(fit["loss"]["penalty"][0])) == psd.r_paste(float(single["loss"]["penalty"][0]))
        assert fit["segments"].equals(single["segments"])
        assert fit["others"]["penalty"].tolist() == single["others"]["penalty"].tolist()


@pytest.mark.parametrize("spill_mode", [0.0, 1.0], ids=["dma-drain", "zero-copy"])
def test_store_spills_to_pinned_host_memory(psd, spill_mode):
    """With an HBM pool far too small for the batch (and fixed, so it cannot grow) the cost-function
    records spill to pinned host memory: by default through an HBM ring that a host thread drains
    with cudaMemcpyAsync on a side stream while the DP kernel runs (spill_mode 0), or by zero-copy
    stores through the mapping (spill_mode 1); the backtrack reads them back through the mapping.
    Results must be identical to the all-HBM run and no extra wave may be needed."""
    from peaksegdisk_b200 import synth
    probs = [synth.poisson_problem(seed, 5000) + (pen,) for seed, pen in [(500, 0.0), (501, 20.0), (502, 1e3), (503, 1e5)]]
    probs += [synth.increasing_problem(1000) + (1e4,)]         # records larger than an 8 KB chunk: written zero-copy in both modes
    base, ids = psd.solve_batch(probs)
    want = [(base.loss_row(i), base.segments(i)) for i in ids]
    lib = psd._lib.lib
    try:
        lib.psd_set_option(b"store_gb", 0.002)       # 2 MB of HBM: a fraction of one problem
        lib.psd_set_option(b"host_spill_gb", 0.25)
        lib.psd_set_option(b"chunk_kb", 8.0)
        lib.psd_set_option(b"spill_mode", spill_mode)
        plan, ids2 = psd.solve_batch(probs)
        st = plan.stats()
        assert (st["store_bytes_drained_dma"] > 0) == (spill_mode == 0.0), st
        # the inspection path reads spilled records from the host region
        hi, bi, bx = plan.store_function(ids2[0], len(probs[0][2]) - 1, 1)
        hi0, bi0, bx0 = base.store_function(ids[0], len(probs[0][2]) - 1, 1)
        assert np.array_equal(hi, hi0) and np.array_equal(bi, bi0) and np.array_equal(bx, bx0)
    finally:
        lib.psd_set_option(b"store_gb", 0.0)
        lib.psd_set_option(b"host_spill_gb", -1.0)
        lib.psd_set_option(b"chunk_kb", 64.0)
        lib.psd_set_option(b"spill_mode", 0.0)
    assert st["store_bytes_spilled_host"] > 0, st
    for i, (loss, seg) in zip(ids2, want):
        assert plan.loss_row(i) == loss
        assert all(np.array_equal(x, y) for x, y in zip(plan.segments(i), seg))


def test_records_larger_than_a_store_chunk(psd):
    """With 1 KB store chunks almost every record spans several chunks (contiguous multi-chunk
    allocation); increasing counts give records of tens of KB."""
    from peaksegdisk_b200 import synth
    probs = [synth.poisson_problem(610, 3000) + (100.0,), synth.increasing_problem(400) + (1e4,)]
    lib = psd._lib.lib
    try:
        lib.psd_set_option(b"chunk_kb", 1.0)
        plan, ids = psd.solve_batch(probs)
    finally:
        lib.psd_set_option(b"chunk_kb", 64.0)
    for pid, (s, e, c, pen) in zip(ids, probs):
        _check_vs_oracle(plan, pid, s, e, c, pen)


def test_extreme_values_match_oracle(psd):
    """Counts up to 2e9, weights up to 1e8 bases per row, long zero runs (log-mean domain starting at
    -inf), penalties from 1e-12 to 1e15: the kernels must follow the oracle through every
    inf/underflow corner of the reference's arithmetic."""
    rng = np.random.default_rng(99)
    s, e, big = oracle_checks.extreme_rows(rng)
    probs = [(s, e, big, pen) for pen in (1e-12, 1.0, 1e9, 1e15)]
    z = np.zeros(300, np.int32); z[100:103] = 7; z[200] = 1
    u = np.arange(300, dtype=np.int32)
    for pen in (0.0, 1e-3, 5.0):
        probs.append((u, u + 1, z, pen))
    tiny = rng.poisson(0.01, size=2000).astype(np.int32)
    tiny[5] = 1
    from peaksegdisk_b200 import synth
    t0, t1, tc = synth.rle_rows(tiny)
    probs.append((t0, t1, tc, 0.5))
    plan, ids = psd.solve_batch(probs)
    for pid, (ps, pe, pc, pen) in zip(ids, probs):
        _check_vs_oracle(plan, pid, ps, pe, pc, pen)


def test_reference_style_caller_runs_the_gpu_solver(psd, tmp_path):
    """The drop-in path end to end: a C++ caller declared like src/interface.cpp's links against the
    library's mangled PeakSegFPOP_disk symbol and gets the reference's files (DP branch)."""
    import subprocess
    exe = str(tmp_path / "dropin")
    libdir = os.path.dirname(psd._lib.LIB_PATH)
    subprocess.check_call(["/usr/bin/g++", "-O1", "-o", exe, os.path.join(ROOT, "tests", "native", "dropin_link.cpp"),
                           "-L" + libdir, "-lpeaksegdisk_b200", "-Wl,-rpath," + libdir])
    case = [c for c in golden("golden_small.json") if c["name"] == "four" and c["penalty"] == "10.5"][0]
    bg = str(tmp_path / "four.bedGraph")
    open(bg, "w").write(case["input"])
    out = subprocess.run([exe, bg, "10.5", bg + ".db"], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert outputs(bg, "10.5") == (case["segments"], case["loss"])
    assert os.path.getsize(bg + ".db") > 0      # R reports its size as `megabytes` and deletes it


def test_reference_interface_cpp_runs_the_gpu_solver(psd, tmp_path):
    """The reference's OWN R glue -- src/interface.cpp compiled UNMODIFIED in the build container
    (oracle/Makefile `interface`: R-header shim + a driver that plays R's .C()) and linked against
    libpeaksegdisk_b200.so -- on the DP branch: R_init_PeakSegDisk registers the routine,
    PeakSegFPOP_interface(char**, char**, char**) calls PeakSegFPOP_disk, the GPU solves, and the
    files equal the reference's; an unwritable db surfaces as interface.cpp's Rf_error text."""
    import subprocess
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_interface_b200")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/ref_interface_b200 not built (make -C oracle interface; needs /root/reference)")
    env = dict(os.environ, PSD_LATENCY_MODE=os.environ.get("PSD_LATENCY_MODE", "0"))
    for case in [c for c in golden("golden_small.json") if c["name"] in ("four", "hap3", "supp") and c["status"] == 0]:
        bg = str(tmp_path / ("%s.bedGraph" % case["name"]))
        open(bg, "w").write(case["input"])
        out = subprocess.run([exe, bg, case["penalty"], bg + ".db"], capture_output=True, text=True, env=env)
        assert out.returncode == 0 and out.stdout.endswith("ok\n"), (case["name"], case["penalty"], out.stderr)
        assert outputs(bg, case["penalty"]) == (case["segments"], case["loss"]), (case["name"], case["penalty"])
    g = golden("golden_mono27ac.json")["penalties"]["10.5"]
    bg = str(tmp_path / "coverage.bedGraph")
    open(bg, "w").write(open(os.path.join(GOLD, "Mono27ac_coverage.bedGraph")).read())
    out = subprocess.run([exe, bg, "10.5", bg + ".db"], capture_output=True, text=True, env=env)
    assert out.returncode == 0, out.stderr
    seg, loss = outputs(bg, "10.5")
    assert loss == g["loss"] and sha(seg) == g["segments_sha256"]
    out = subprocess.run([exe, bg, "10.5", str(tmp_path)], capture_output=True, text=True, env=env)   # db path is a directory
    assert out.returncode == 1 and out.stderr == "Error: unable to write to cost function database file %s\n" % str(tmp_path)


def test_store_contents_equal_the_reference_db(psd, tmp_path, kernel_mode):
    """Row a10 of the scope table: the HBM cost-function store must hold what the reference's
    DiskVector holds.  The reference binary (oracle/_ref/ref_fpop, unmodified sources) solves the
    store problems (oracle_checks.store_problems: Mono27ac at 10.5 and 0, synthetic, extreme-value and
    count-vector problems) and leaves its db; every one of the 2N-1 stored functions -- piece count,
    max_log_mean, data_i, prev_log_mean of every piece, bit for bit -- is read back from the GPU store
    (psd_plan_store_function) and compared."""
    import subprocess
    if not os.path.exists(oracle_bind.REF_BIN):
        pytest.skip("oracle/_ref/ref_fpop not built")
    _store_equals_db(psd, tmp_path, kernel_mode,
                     lambda bg, pen: subprocess.call([oracle_bind.REF_BIN, bg, pen, bg + ".db"], stdout=subprocess.DEVNULL))


def test_store_contents_equal_the_oracle_db(psd, tmp_path, kernel_mode):
    """The same comparison against the db the parity oracle writes (oracle/fpop_oracle.cpp, psd_math
    mode: the reference's DiskVector format, which its size matches in tests/golden), so that the store
    is checked function by function on every machine, also where the compiled reference is absent."""
    _store_equals_db(psd, tmp_path, kernel_mode, lambda bg, pen: oracle_bind.oracle_disk(bg, pen, bg + ".db", 1))


def _store_equals_db(psd, tmp_path, build, write_db):
    probs = oracle_checks.store_problems()
    plan = psd.Plan(0)
    ids = [p.add(plan) for p in probs]
    plan.run()
    for pid, p in zip(ids, probs):
        oracle_checks.assert_store_equals_db(plan, pid, p, p.db(tmp_path, write_db), build)


def test_concurrent_single_problem_calls_from_host_threads(psd, tmp_path):
    """SURVEY 8b "Threading": the replacement must be callable concurrently from several host threads
    (distinct files).  Eight threads call the single-problem entry point repeatedly; every result
    equals the golden file, and the plan parked between calls is reused without cross-talk."""
    import ctypes as C, threading
    g = golden("golden_mono27ac.json")
    pens = list(g["penalties"])
    src = open(os.path.join(GOLD, "Mono27ac_coverage.bedGraph")).read()
    small = [c for c in golden("golden_small.json")][:8]
    errors = []

    def worker(k):
        try:
            path = str(tmp_path / ("t%d.bedGraph" % k))
            open(path, "w").write(src)
            for rep in range(3):
                pen = pens[(k + rep) % len(pens)]
                st = psd._lib.lib.psd_fpop_disk(path.encode(), pen.encode(), (path + ".db").encode())
                assert st == 0, st
                seg, loss = outputs(path, pen)
                assert loss == g["penalties"][pen]["loss"] and sha(seg) == g["penalties"][pen]["segments_sha256"]
                case = small[(k + rep) % len(small)]
                sp = str(tmp_path / ("s%d_%d.bedGraph" % (k, rep)))
                open(sp, "w").write(case["input"])
                st = psd._lib.lib.psd_fpop_disk(sp.encode(), case["penalty"].encode(), (sp + ".db").encode())
                assert st == 0 and outputs(sp, case["penalty"]) == (case["segments"], case["loss"])
        except Exception as e:   # surfaced in the main thread
            errors.append((k, repr(e)))

    threads = [threading.Thread(target=worker, args=(k,)) for k in range(8)]
    [t.start() for t in threads]; [t.join() for t in threads]
    assert not errors, errors
    psd._lib.lib.psd_release_cache()      # drops the parked plan; the next call simply builds a new one
    worker(99)
    assert not errors, errors


def test_batched_file_call_spread_over_two_gpus(psd, tmp_path):
    """SURVEY 8e inside one process: option "devices" deals the problems of one psd_fpop_disk_batch
    call to several GPUs (one plan + host thread each, no exchange).  Same files as on one GPU."""
    if psd._lib.lib.psd_device_count() < 2:
        pytest.skip("needs two GPUs")
    g = golden("golden_mono27ac.json")
    pens = list(g["penalties"])
    path = str(tmp_path / "coverage.bedGraph")
    open(path, "w").write(open(os.path.join(GOLD, "Mono27ac_coverage.bedGraph")).read())
    files, ps, want = [path] * len(pens), list(pens), []
    for k, case in enumerate(c for c in golden("golden_small.json") if c["status"] == 0):
        sp = str(tmp_path / ("s%d.bedGraph" % k))
        open(sp, "w").write(case["input"])
        files.append(sp); ps.append(case["penalty"]); want.append((sp, case))
    try:
        psd._lib.lib.psd_set_option(b"devices", 2.0)
        st = psd.PeakSegFPOP_file_batch(files, ps)
    finally:
        psd._lib.lib.psd_set_option(b"devices", 1.0)
    assert st == [0] * len(files)
    for pen in pens:
        seg, loss = outputs(path, pen)
        assert loss == g["penalties"][pen]["loss"] and sha(seg) == g["penalties"][pen]["segments_sha256"], pen
    for sp, case in want:
        assert outputs(sp, case["penalty"]) == (case["segments"], case["loss"]), case["name"]


def test_count_vectors_are_run_length_encoded_on_the_device(psd):
    """SURVEY 8 row f3: psd_plan_add_counts() takes the raw count vector; the device RLE must give
    exactly the rows R's rle()/cumsum give (R/PeakSegFPOP_vec.R:18-25), so every output equals the
    row-array solve and the oracle.  Shapes: tile-boundary lengths (a tile is 8,192 positions),
    runs that span tiles and warps, single positions, constant vectors, mixed with row problems."""
    from peaksegdisk_b200 import synth
    rng = np.random.default_rng(77)
    vecs = []
    for n in (1, 2, 31, 32, 33, 1023, 1024, 1025, 8191, 8192, 8193, 16384, 20000, 50000):
        vecs.append(synth.poisson_counts(1000 + n, n))
    long_runs = np.repeat(rng.integers(0, 4, size=40), rng.integers(1, 3000, size=40)).astype(np.int64)
    vecs.append(long_runs)                                        # runs crossing several warps / tiles
    vecs.append(np.concatenate([np.zeros(9000, np.int64), [7], np.zeros(9000, np.int64)]))
    vecs.append(np.arange(300) % 2)                               # every position is its own run
    vecs.append(np.repeat([1, 2, 1, 3, 0, 5], [20000, 30000, 1, 50000, 8192, 8191]))   # chains of tiles without any head
    vecs.append(np.full(12345, 3))                                # constant: one-segment model on the host
    vecs.append(np.array([5]))
    pens = [float(10 ** rng.uniform(-1, 5)) for _ in vecs]
    pens[3] = float("inf")
    plan = psd.Plan(0)
    ids = []
    for k, (v, pen) in enumerate(zip(vecs, pens)):
        ids.append(plan.add_counts(v, pen))
        if k % 4 == 0:                                            # interleave a row problem: both kinds share one launch
            s, e, c = synth.poisson_problem(500 + k, 3000)
            ids.append(("rows", plan.add(s, e, c, 50.0), s, e, c))
    plan.run()
    st = plan.stats()
    assert st["n_rle_launches"] == 1 and st["rle_positions"] > 0
    k = 0
    for item in ids:
        if isinstance(item, tuple):
            _, pid, s, e, c = item
            _check_vs_oracle(plan, pid, s, e, c, 50.0)
            continue
        v, pen = vecs[k], pens[k]; k += 1
        s, e, c = synth.rle_rows(v)
        r = plan.result(item)
        assert r.status == 0 and r.n_rows == len(c) and r.bases == len(v)
        if r.trivial:
            seg = plan.segments(item)
            assert (int(seg[0][0]), int(seg[1][0]), int(seg[2][0])) == (0, len(v), 0)
            ref, _ = psd.solve_batch([(s, e, c, pen)])
            assert plan.loss_row(item) == ref.loss_row(0) and seg[3][0] == ref.segments(0)[3][0]
        else:
            _check_vs_oracle(plan, item, s, e, c, pen)
    # the R-named batched front end reports the same tables
    out = psd.PeakSegFPOP_vec_batch([vecs[0], vecs[12]], [pens[0], pens[12]])
    for o, kk in zip(out, (0, 12)):
        s, e, c = synth.rle_rows(vecs[kk])
        stt, summ, oseg = oracle_bind.solve_rows(s, e, c, pens[kk])
        assert int(o["loss"]["peaks"][0]) == int(summ[2]) and float(o["loss"]["total.loss"][0]) == summ[6]
        assert np.array_equal(o["segments"]["chromStart"].to_numpy(), oseg[0])
        assert list(o["segments"]["status"]) == [("peak" if i % 2 else "background") for i in range(len(oseg[0]))]
    with pytest.raises(ValueError):
        plan.add_counts(np.array([1, -2, 3]), 1.0)
    with pytest.raises(ValueError):
        plan.add_counts(np.array([1.5, 2.0]), 1.0)


def test_count_vector_batch_full_size_matches_row_batch(psd):
    """Config-2-sized vectors (1e4..1e5 positions): device-RLE problems and host-RLE row problems
    give bit-identical loss rows and segments; re-upload and penalty updates work on count problems."""
    from peaksegdisk_b200 import synth
    vecs = [synth.poisson_counts(seed) for seed in range(40, 56)]
    a = psd.Plan(0); b = psd.Plan(0)
    for v in vecs:
        for pen in (1e2, 1e4):
            a.add_counts(v, pen)
            b.add(*synth.rle_rows(v), pen)
    a.run(); b.run()
    for pid in range(len(a)):
        assert a.loss_row(pid) == b.loss_row(pid)
        sa, sb = a.segments(pid), b.segments(pid)
        assert all(np.array_equal(x, y) for x, y in zip(sa[:3], sb[:3])) and np.array_equal(sa[3].view(np.uint64), sb[3].view(np.uint64))
    assert a.stats()["rle_positions"] == 2 * sum(len(v) for v in vecs)
    a.set_penalty(0, 1e3); b.set_penalty(0, 1e3)
    a.run(); b.run()
    assert a.loss_row(0) == b.loss_row(0) and a.loss_row(1) == b.loss_row(1)


def test_differential_fuzz_against_oracle():
    """tools/fuzz_gpu_vs_oracle.py: 150 random problems of six shapes (bursty zeros, huge counts,
    trends with hundreds of pieces, random weights, penalties 0 and 1e-3..1e7) in one launch; every
    summary field and every segment bit-identical to the oracle."""
    import subprocess, sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "fuzz_gpu_vs_oracle.py"), "150", "7"],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert " 0 mismatches" in out.stdout
