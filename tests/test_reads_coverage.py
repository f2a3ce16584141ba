"""Coverage from aligned reads (psd_coverage_from_reads, coverage_from_reads, solve_reads_batch): the
device rows against a numpy difference-array oracle, the reference's Mono27ac data rebuilt from reads,
waves, and reads -> segmentation end to end.  Input checks run without a GPU."""
import ctypes as C
import os
import numpy as np
import pandas as pd
import pytest
import oracle_bind
from helpers import GOLD, golden, sha, outputs

PSD_ERR_ARG = 111


@pytest.fixture(scope="module")
def psd():
    import peaksegdisk_b200
    return peaksegdisk_b200


@pytest.fixture(scope="module")
def gpu(psd):
    assert psd._lib.lib.psd_device_count() >= 1, "no CUDA device"
    return psd


def oracle_rows(starts, ends, a, b):
    """numpy oracle: difference array (np.add.at), cumsum, run heads.  Returns int32 (start, end, count)."""
    starts = np.asarray(starts, np.int64); ends = np.asarray(ends, np.int64)
    n = b - a
    keep = (ends > a) & (starts < b)
    d = np.zeros(n + 1, np.int32)
    np.add.at(d, np.maximum(starts[keep] - a, 0), 1)
    np.add.at(d, np.minimum(ends[keep] - a, n), -1)
    cov = np.cumsum(d[:n], dtype=np.int32)
    del d
    heads = np.flatnonzero(np.r_[True, cov[1:] != cov[:-1]])
    return (heads + a).astype(np.int32), (np.r_[heads[1:], n] + a).astype(np.int32), cov[heads]


def brute_rows(starts, ends, a, b):
    cov = [sum(1 for s, e in zip(starts, ends) if s <= x < e) for x in range(a, b)]
    rs, re_, rc = [a], [], [cov[0]]
    for x in range(1, b - a):
        if cov[x] != cov[x - 1]:
            re_.append(a + x); rs.append(a + x); rc.append(cov[x])
    re_.append(b)
    return np.array(rs), np.array(re_), np.array(rc)


def assert_rows_equal(got, want, what=""):
    for g, w, name in zip(got, want, ("chromStart", "chromEnd", "count")):
        assert g.dtype == np.int32 and np.array_equal(g, w), (what, name)


# ---- CPU ---------------------------------------------------------------------------------------------

def test_numpy_oracle_matches_brute_force():
    rng = np.random.default_rng(7)
    for case in range(300):
        a = int(rng.integers(0, 20)); b = a + int(rng.integers(1, 40))
        n = int(rng.integers(0, 12))
        s = rng.integers(0, 70, size=n)
        e = s + rng.integers(1, 15, size=n)
        if case % 5 == 0 and n > 1:
            s[1], e[1] = e[0], e[0] + 3   # abutting reads: their deltas cancel
        got = oracle_rows(s, e, a, b)
        want = brute_rows(s.tolist(), e.tolist(), a, b)
        for g, w in zip(got, want):
            assert np.array_equal(g, w), (case, s, e, a, b)


def _call(psd, problems):
    """psd_coverage_from_reads through ctypes: (status, handle)."""
    arr = (psd._lib.PsdReads * len(problems))()
    keep = []
    for i, (n, s, e, a, b) in enumerate(problems):
        arr[i].n_reads = n; arr[i].region_start = a; arr[i].region_end = b
        if s is not None:
            s = np.ascontiguousarray(s, np.int32); e = np.ascontiguousarray(e, np.int32); keep += [s, e]
            arr[i].read_start = s.ctypes.data_as(C.POINTER(C.c_int32)); arr[i].read_end = e.ctypes.data_as(C.POINTER(C.c_int32))
    h = C.c_void_p()
    rc = psd._lib.lib.psd_coverage_from_reads(-1, len(problems), arr, C.byref(h))
    return rc, h


def test_input_errors_name_problem_and_read_without_gpu(psd):
    ok = (3, [0, 5, 9], [4, 8, 12], 0, 20)
    s = np.array([0, 1, 2, 3, 4]); e = s + 2
    bad = {
        "start < 0": (5, np.where(np.arange(5) == 3, -1, s), e, 0, 20),
        "end <= start": (5, s, np.where(np.arange(5) == 3, 3, e), 0, 20),
        "region_start < 0": (0, None, None, -1, 20),
        "region_end <= region_start": (0, None, None, 20, 20),
        "too long": (0, None, None, 0, 0x3fffffff + 1),
        "null": (4, None, None, 0, 20),
        "2^31 reads": (1 << 31, None, None, 0, 20),
        "negative count": (-1, None, None, 0, 20),
    }
    for what, prob in bad.items():
        rc, h = _call(psd, [ok, ok, prob])
        assert rc == PSD_ERR_ARG and not h.value, what
        msg = psd._lib.lib.psd_last_error().decode()
        assert "problem 2" in msg, (what, msg)
        if what in ("start < 0", "end <= start"):
            assert "read 3" in msg, (what, msg)
    # the longest region allowed is accepted by the checks (no read in it: no device work)
    rc, h = _call(psd, [(0, None, None, 0, 0x3fffffff)])
    assert rc == 0
    assert psd._lib.lib.psd_coverage_n_rows(h, 0) == 1 and psd._lib.lib.psd_coverage_n_rows(h, 1) == -1
    psd._lib.lib.psd_coverage_free(h)


def test_regions_without_reads_give_one_zero_row_without_gpu(psd):
    from peaksegdisk_b200.plan import coverage_rows
    rows, st = coverage_rows([([], [], 3, 7), ([100, 0], [200, 5], 10, 90), (np.zeros(0, np.int32), np.zeros(0, np.int32), 0, 1)])
    assert [tuple(map(list, r)) for r in rows] == [([3], [7], [0]), ([10], [90], [0]), ([0], [1], [0])]
    assert st["n_waves"] == 0 and st["rows"] == 3 and st["n_problems"] == 3


def test_coverage_from_reads_argument_errors(psd):
    df = pd.DataFrame({"chrom": ["chr1", "chr1"], "chromStart": [0, 5], "chromEnd": [10, 9]})
    with pytest.raises(ValueError, match="data.frame"):
        psd.coverage_from_reads({"chrom": []})
    with pytest.raises(ValueError, match="columns"):
        psd.coverage_from_reads(df.drop(columns="chromEnd"))
    with pytest.raises(ValueError, match="integer"):
        psd.coverage_from_reads(df.assign(chromStart=[0.0, 5.5]))
    with pytest.raises(ValueError, match="32-bit"):
        psd.coverage_from_reads(df.assign(chromEnd=[10, 2 ** 31]))
    with pytest.raises(ValueError, match="region"):
        psd.coverage_from_reads(df, region=[("chr1", 0, 10)])
    with pytest.raises(ValueError, match="integer"):
        psd.coverage_from_reads(df, region={"chr1": (0, 10.5)})
    with pytest.raises(ValueError, match="problem 0: read 1: end 4 <= start 5"):
        psd.coverage_from_reads(df.assign(chromEnd=[10, 4]), region={"chr1": (0, 10)})
    with pytest.raises(ValueError, match="same length"):
        psd.plan.coverage_rows([([1, 2], [3], 0, 10)])
    # no read in the region: no device needed
    got = psd.coverage_from_reads(df, region={"chr1": (100, 200), "chr2": (0, 5)})
    assert got.values.tolist() == [["chr1", 100, 200, 0], ["chr2", 0, 5, 0]]
    assert list(got.columns) == psd.col_name_list["coverage"]


# ---- GPU ---------------------------------------------------------------------------------------------

def _mono_reads(seed=11):
    from peaksegdisk_b200 import synth
    chrom, s, e, c = synth.read_bedgraph(os.path.join(GOLD, "Mono27ac_coverage.bedGraph"))
    rs, re_ = np.repeat(s, c), np.repeat(e, c)
    perm = np.random.default_rng(seed).permutation(len(rs))
    return chrom, rs[perm], re_[perm]


@pytest.mark.gpu
def test_mono27ac_from_reads_is_the_reference_fixture(gpu, tmp_path):
    """The reference's Mono27ac coverage expanded into reads (count copies of each row), shuffled,
    and turned back into coverage on the device: the bedGraph text is byte-identical, so every solve
    on it gives the golden outputs."""
    chrom, rs, re_ = _mono_reads()
    assert len(rs) == 50179
    reads = pd.DataFrame({"chrom": chrom, "chromStart": rs, "chromEnd": re_, "name": "r"})
    cov = gpu.coverage_from_reads(reads, region={chrom: (60000, 580000)})
    assert len(cov) == 6921
    d = tmp_path / "chr11-60000-580000"
    d.mkdir()
    path = str(d / "coverage.bedGraph")
    p32 = C.POINTER(C.c_int32)
    cols = [np.ascontiguousarray(cov[k].to_numpy(), np.int32) for k in ("chromStart", "chromEnd", "count")]
    assert gpu._lib.lib.psd_write_bedgraph(path.encode(), chrom.encode(), len(cov), *[a.ctypes.data_as(p32) for a in cols]) == 0
    assert open(path, "rb").read() == open(os.path.join(GOLD, "Mono27ac_coverage.bedGraph"), "rb").read()
    g = golden("golden_mono27ac.json")
    pens = list(g["penalties"])
    assert gpu.PeakSegFPOP_file_batch([path] * len(pens), pens) == [0] * len(pens)
    for pen in pens:
        seg, loss = outputs(path, pen)
        assert loss == g["penalties"][pen]["loss"], pen
        assert sha(seg) == g["penalties"][pen]["segments_sha256"], pen
    fit = gpu.sequentialSearch_dir(str(d), 19)
    assert int(fit["loss"]["peaks"][0]) == 19 and len(fit["segments"]) == 39
    assert gpu.r_paste(float(fit["loss"]["penalty"][0])) == "1715.84956360692"
    for c in g["search19"]:
        assert outputs(path, c["penalty_str"])[1] == c["loss"]


def _edge_problems():
    from peaksegdisk_b200 import synth
    rng = np.random.default_rng(3)
    P = []
    P.append(([], [], 1000, 5000))                                  # no reads
    P.append(([0, 10, 5000], [900, 1000, 7000], 1000, 5000))        # all outside (one ends at region_start, one starts at region_end)
    P.append(([500, 4990, 2000], [1500, 9000, 5000], 1000, 5000))   # straddling either end, one ending at region_end
    P.append(([7, 0, 7, 8], [8, 7, 9, 9], 7, 8))                    # 1-base region
    P.append(([100] * 50, [300] * 50, 0, 1000))                     # identical reads
    P.append(([0, 10, 20, 30, 40], [10, 20, 30, 40, 50], 0, 60))    # abutting: deltas cancel, runs merge
    P.append((list(range(0, 200, 3)), list(range(1, 201, 3)), 0, 200))   # 1-base reads
    P.append(([5, 100], [30000, 8192 * 5 + 3], 0, 8192 * 6))        # single reads across several tiles
    for n in (8191, 8192, 8193, 16384):
        s, e = synth.reads(n, 3000, n)
        P.append((s, e, 0, n))
    s, e = synth.reads(21, 20000, 50000, start=123456)
    P.append((np.sort(s), e[np.argsort(s)], 123456, 123456 + 50000))   # sorted by start
    P.append((s, e, 123456 + 1000, 123456 + 40000))                     # unsorted, a sub-region of the same reads
    s, e = synth.reads(22, 10 ** 6, 3 * 10 ** 7, start=10 ** 6)
    P.append((s, e, 10 ** 6, 10 ** 6 + 3 * 10 ** 7))               # 1e6 reads
    s = rng.integers(0, 10 ** 6, size=1000); P.append((s, s + rng.integers(1, 50000, size=1000), 0, 10 ** 6))   # long reads
    return P


@pytest.mark.gpu
def test_rows_equal_the_oracle_many_problems_one_call(gpu):
    P = _edge_problems()
    rows, st = gpu.plan.coverage_rows(P)
    assert st["n_problems"] == len(P) and st["n_waves"] == 1 and st["kernel_ms"] > 0
    for k, (p, got) in enumerate(zip(P, rows)):
        assert_rows_equal(got, oracle_rows(*p), k)
    assert [len(r[2]) for r in rows[:8]] == [1, 1, 4, 1, 3, 2, 134, 5]
    assert st["rows"] == sum(len(r[2]) for r in rows)


@pytest.mark.gpu
def test_waves_give_the_same_rows(gpu):
    P = _edge_problems()
    one, st1 = gpu.plan.coverage_rows(P)
    gpu._lib.lib.psd_set_option(b"coverage_gb", 0.05)
    try:
        many, st2 = gpu.plan.coverage_rows(P)
    finally:
        gpu._lib.lib.psd_set_option(b"coverage_gb", 0.0)
    assert st1["n_waves"] == 1 and st2["n_waves"] > 1
    for k, (a, b) in enumerate(zip(one, many)):
        assert_rows_equal(a, b, k)


@pytest.mark.gpu
def test_chr1_sized_region_1e7_reads(gpu):
    from peaksegdisk_b200 import synth
    n = 249250621
    s, e = synth.reads(5, 10 ** 7, n)
    (gs, ge, gc), = gpu.plan.coverage_rows([(s, e, 0, n)])[0]
    assert gs[0] == 0 and ge[-1] == n and np.array_equal(gs[1:], ge[:-1]) and np.all(gc[1:] != gc[:-1])
    ws, we, wc = oracle_rows(s, e, 0, n)
    assert len(gc) == len(wc)
    pick = np.random.default_rng(9).choice(len(gc), size=100000, replace=False)
    assert np.array_equal(gs[pick], ws[pick]) and np.array_equal(ge[pick], we[pick]) and np.array_equal(gc[pick], wc[pick])
    assert_rows_equal((gs, ge, gc), (ws, we, wc))


@pytest.mark.gpu
@pytest.mark.parametrize("latency_mode", [0.0, 2.0], ids=["auto", "throughput-kernel"])
def test_solve_reads_batch_end_to_end(gpu, latency_mode):
    from peaksegdisk_b200 import synth
    rng = np.random.default_rng(17)
    probs = []
    for k in range(12):
        length = int(rng.integers(20000, 400000))
        s, e = synth.reads(100 + k, int(length // 40), length, start=int(rng.integers(0, 10 ** 6)))
        probs.append((s, e, int(s.min()) + 500, int(s.min()) + length, float(10 ** rng.uniform(0, 4))))
    gpu._lib.lib.psd_set_option(b"latency_mode", latency_mode)
    try:
        plan, ids = gpu.solve_reads_batch(probs)
        rows = [oracle_rows(*p[:4]) for p in probs]
        ref, rids = gpu.solve_batch([r + (p[4],) for r, p in zip(rows, probs)])
    finally:
        gpu._lib.lib.psd_set_option(b"latency_mode", 0.0)
    for k, (a, b) in enumerate(zip(ids, rids)):
        assert plan.loss_row(a) == ref.loss_row(b), k
        ga, gb = plan.segments(a), ref.segments(b)
        assert all(np.array_equal(x, y) for x, y in zip(ga[:3], gb[:3])), k
        assert np.array_equal(ga[3].view(np.uint64), gb[3].view(np.uint64)), k
    for k in (0, 5, 11):
        st, summ, oseg = oracle_bind.solve_rows(*rows[k], probs[k][4])
        got, seg = plan.loss_row(ids[k]), plan.segments(ids[k])
        assert st == 0 and got["segments"] == int(summ[1]) and got["total.loss"] == summ[6]
        assert all(np.array_equal(x, y) for x, y in zip(seg[:3], oseg[:3]))
        assert np.array_equal(seg[3].view(np.uint64), oseg[3].view(np.uint64))


@pytest.mark.gpu
def test_multi_chromosome_dataframe(gpu, tmp_path):
    from peaksegdisk_b200 import synth
    parts = []
    for k, (ch, length) in enumerate([("chr2", 300000), ("chr1", 200000), ("chrX", 150000)]):
        s, e = synth.reads(50 + k, length // 50, length, start=10000 * (k + 1))
        parts.append(pd.DataFrame({"chrom": ch, "chromStart": s.astype(np.int64), "chromEnd": e.astype(np.int64), "strand": "+"}))
    reads = pd.concat(parts, ignore_index=True).sample(frac=1.0, random_state=4).reset_index(drop=True)
    first = list(pd.unique(reads["chrom"]))
    cov = gpu.coverage_from_reads(reads)
    assert list(cov.columns) == gpu.col_name_list["coverage"] and list(pd.unique(cov["chrom"])) == first
    for ch in first:
        r = reads[reads["chrom"] == ch]
        want = oracle_rows(r["chromStart"], r["chromEnd"], int(r["chromStart"].min()), int(r["chromEnd"].max()))
        c = cov[cov["chrom"] == ch]
        assert_rows_equal(tuple(c[k].to_numpy() for k in ("chromStart", "chromEnd", "count")), want, ch)
    # explicit regions: clipped reads, an extra chromosome without reads at the end
    region = {"chr1": (50000, 120000), "chrY": (0, 1000), "chrX": (30000, 31000)}
    cov2 = gpu.coverage_from_reads(reads, region=region)
    assert list(pd.unique(cov2["chrom"])) == first + ["chrY"]
    for ch in first + ["chrY"]:
        r = reads[reads["chrom"] == ch]
        a, b = region.get(ch, (int(r["chromStart"].min()) if len(r) else 0, int(r["chromEnd"].max()) if len(r) else 0))
        c = cov2[cov2["chrom"] == ch]
        assert_rows_equal(tuple(c[k].to_numpy() for k in ("chromStart", "chromEnd", "count")),
                          oracle_rows(r["chromStart"], r["chromEnd"], a, b), ch)
    # writeBedGraph -> PeakSegFPOP_dir agrees with PeakSegFPOP_df on the same coverage
    one = cov[cov["chrom"] == "chr1"].reset_index(drop=True)
    fit_df = gpu.PeakSegFPOP_df(one, 5000.0, str(tmp_path / "df"))
    d = tmp_path / "dir"
    d.mkdir()
    gpu.writeBedGraph(one, str(d / "coverage.bedGraph"))
    fit_dir = gpu.PeakSegFPOP_dir(str(d), "5000")
    assert fit_df["segments"].equals(fit_dir["segments"])
    L = gpu.col_name_list["loss"]
    assert fit_df["loss"][L].equals(fit_dir["loss"][L])
    assert int(fit_dir["loss"]["bedGraph.lines"][0]) == len(one)
