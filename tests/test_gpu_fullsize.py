"""GPU parity at the STATED sizes of BASELINE.json's configurations, against fixtures produced by the
unmodified reference (tests/golden/golden_fullsize.json, tools/make_golden_fullsize.py): every
_loss.tsv line byte-identical, sha256 of every _segments.bed identical.  Everything goes through the
C ABI's file entry points (psd_fpop_disk_batch), like the reference's own R callers."""
import os
import numpy as np
import pytest
from helpers import ROOT, golden, sha, outputs, synth_rows, c4_lite_problem

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def psd():
    import peaksegdisk_b200
    assert peaksegdisk_b200._lib.lib.psd_device_count() >= 1, "no CUDA device"
    return peaksegdisk_b200


@pytest.fixture(scope="module")
def shm(tmp_path_factory):
    import shutil, tempfile
    d = tempfile.mkdtemp(prefix="psdfull", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    yield d
    shutil.rmtree(d, ignore_errors=True)


def _check(psd, cases, paths, latency_mode=0.0, occupancy_mode=0.0):
    pens = [c["penalty"] for c in cases]
    lib = psd._lib.lib
    try:
        lib.psd_set_option(b"latency_mode", latency_mode)
        lib.psd_set_option(b"occupancy_mode", occupancy_mode)
        st = psd.PeakSegFPOP_file_batch(paths, pens)
    finally:
        lib.psd_set_option(b"latency_mode", 0.0)
        lib.psd_set_option(b"occupancy_mode", 0.0)
    assert st == [0] * len(cases)
    for case, p in zip(cases, paths):
        seg, loss = outputs(p, case["penalty"])
        assert loss == case["loss"], (case.get("key"), case["penalty"])
        assert sha(seg) == case["segments_sha256"], (case.get("key"), case["penalty"])
        assert seg.splitlines()[:2] == case["segments_head"] and seg.splitlines()[-1:] == case["segments_tail"]
        for suf in ("_segments.bed", "_loss.tsv"):
            os.unlink("%s_penalty=%s%s" % (p, case["penalty"], suf))


@pytest.mark.parametrize("mode", [(0.0, 0.0), (2.0, 1.0), (2.0, 2.0)], ids=["auto", "throughput-kernel", "two-block"])
def test_config2_full_size_vs_reference(psd, shm, mode):
    """Config 2 at its stated size: 8 vectors of 1e5 positions and six of the bench's own vectors
    (among them the longest and the shortest of the timed batch) x {1e2..1e6} = 70 problems, one call;
    with the automatic choice, the throughput kernel's one-block build and its two-block build (whose
    24-piece shared-memory tier these 24-34-piece functions outgrow into the global workspace)."""
    from peaksegdisk_b200 import synth
    cases = golden("golden_fullsize.json")["c2"]
    files = {}
    for c in cases:
        key = tuple(c["key"])
        if key not in files:
            files[key] = os.path.join(shm, "c2_%d.bedGraph" % key[0])
            if not os.path.exists(files[key]):
                synth.write_bedgraph(files[key], *synth.poisson_problem(*key))
    _check(psd, cases, [files[tuple(c["key"])] for c in cases], *mode)


def test_config3_million_row_problem_vs_reference(psd, shm):
    """Config 3: the 1,004,608-row problem (seed 2024) at EVERY penalty of the reference's
    sequentialSearch_dir chain to 100 peaks (13 DP solves + Inf), as one batched call: one problem
    per thread block in the latency kernel."""
    from peaksegdisk_b200 import synth
    g = golden("golden_fullsize.json")["c3"]
    path = os.path.join(shm, "c3.bedGraph")
    s, e, c = synth.poisson_problem(g["seed"], g["positions"])
    assert len(c) == g["n_rows"]
    synth.write_bedgraph(path, s, e, c)
    cases = [dict(ch, penalty=ch["penalty_str"]) for ch in g["chain"]]
    _check(psd, cases, [path] * len(cases))
    os.unlink(path)


def test_second_search_chain_selected_penalty_bit_exact(psd, shm):
    """The second pinned sequential search (config 3's generator, 75,892 rows, target 30 peaks):
    sequentialSearch_dir must walk exactly the reference's chain of 15-digit penalty strings."""
    from peaksegdisk_b200 import synth
    g = golden("golden_fullsize.json")["c3s"]
    d = os.path.join(shm, "search30")
    os.makedirs(d)
    synth.write_bedgraph(os.path.join(d, "coverage.bedGraph"), *synth.poisson_problem(g["seed"], g["positions"]))
    fit = psd.sequentialSearch_dir(d, g["target_peaks"])
    chain = g["chain"]
    got = sorted((int(r["iteration"]), psd.r_paste(float(r["penalty"])), int(r["peaks"])) for _, r in fit["others"].iterrows())
    assert got == sorted((c["iteration"], c["penalty_str"], c["peaks"]) for c in chain)
    assert int(fit["loss"]["peaks"][0]) == g["target_peaks"]
    assert psd.r_paste(float(fit["loss"]["penalty"][0])) == chain[-1]["penalty_str"]
    for c in chain:
        seg, loss = outputs(os.path.join(d, "coverage.bedGraph"), c["penalty_str"])
        assert loss == c["loss"] and sha(seg) == c["segments_sha256"], c["penalty_str"]


def test_config5_worst_case_10000_vs_reference(psd, shm):
    """Config 5 at the vignette's size (vignettes/Worst_case.Rmd:19-41): increasing(10000) at 1e2, 1e4
    and 1e6 -- cost functions of up to 4,290 pieces."""
    from peaksegdisk_b200 import synth
    cases = golden("golden_fullsize.json")["c5"]
    path = os.path.join(shm, "c5.bedGraph")
    synth.write_bedgraph(path, *synth.increasing_problem(10000))
    _check(psd, cases, [path] * len(cases))
    assert max(float(c["loss"].split("\t")[9]) for c in cases) == 4290


def test_config4_lite_with_host_spill_vs_reference(psd, shm):
    """Config 4 at 1/20 scale (hg19-shaped problems, Mono27ac-like weights): the largest (463,766
    rows) and the smallest problem of the 48 plus four others, with the HBM pool capped so that most
    of the cost-function store goes through the pinned-host spill path."""
    from peaksegdisk_b200 import synth
    cases = golden("golden_fullsize.json")["c4"]
    paths, pens, want = [], [], []
    for k in (2, 42, 7, 19, 30, 45):
        s, e, c, pen = c4_lite_problem(k, 2, 0.05)
        p = os.path.join(shm, "c4_%d.bedGraph" % k)
        synth.write_bedgraph(p, s, e, c)
        paths.append(p); pens.append(psd.r_paste(pen))
        g = [x for x in cases if x["key"][2] == k]
        want.append(g[0] if g else None)
        if g:
            assert g[0]["n_rows"] == len(c) and g[0]["penalty"] == pens[-1]
    lib = psd._lib.lib
    try:
        lib.psd_set_option(b"store_gb", 0.25)
        lib.psd_set_option(b"host_spill_gb", 2.0)
        st = psd.PeakSegFPOP_file_batch(paths, pens)
    finally:
        lib.psd_set_option(b"store_gb", 0.0)
        lib.psd_set_option(b"host_spill_gb", -1.0)
    assert st == [0] * len(paths)
    for p, pen, g in zip(paths, pens, want):
        if g is None:
            continue
        seg, loss = outputs(p, pen)
        assert loss == g["loss"] and sha(seg) == g["segments_sha256"], g["key"]
