"""Joint single-peak models of many samples (psd_joint_models, joint_models_batch).  Without a GPU: the C oracle
(tests/native/joint_oracle.c, libm's log) against a brute force over every peak and every subset of samples,
model selection against a dense penalty grid, the label errors and targets of the reference against
path_oracle, problems with no possible peak through the library, and every input error.  On the GPU: every
output bit for bit against the oracle on about 300 problems, in one call and in forced waves, a large problem,
a planted signal, coverage from reads, and labels."""
import ctypes as C
import itertools
import math
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor
import numpy as np
import pandas as pd
import pytest
import path_oracle
from helpers import ROOT

PSD_ERR_ARG = 111
KIND_NAMES = ["noPeaks", "peaks", "peakStart", "peakEnd"]


@pytest.fixture(scope="module")
def psd():
    import peaksegdisk_b200
    return peaksegdisk_b200


@pytest.fixture(scope="module")
def gpu(psd):
    assert psd._lib.lib.psd_device_count() >= 1, "no CUDA device"
    return psd


@pytest.fixture(scope="module")
def oracle(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("joint") / "joint_oracle.so")
    subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-o", so,
                           os.path.join(ROOT, "tests", "native", "joint_oracle.c"), "-lm"])
    lib = C.CDLL(so)
    lib.joint_oracle.restype = C.c_int
    lib.joint_oracle.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int64), C.c_int, C.c_int,
                                 C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_uint8)]
    return lib


# ---- the reference: prefix sums, the C oracle, selection, labels ------------------------------------------

def grid_of(start, end, bin_bases):
    n = -(-(end - start) // bin_bases)
    g = start + np.arange(n + 1, dtype=np.int64) * bin_bases
    g[n] = end
    return g


def prefix(samples, bin_bases):
    """C_s(0, i) at every grid point, [grid index][sample], exact int64."""
    start, end = int(samples[0][0][0]), int(samples[0][1][-1])
    g = grid_of(start, end, bin_bases)
    out = np.zeros((len(g), len(samples)), np.int64)
    for j, (s, e, c) in enumerate(samples):
        s, e, c = (np.asarray(a, np.int64) for a in (s, e, c))
        cum = np.concatenate([[0], np.cumsum(c * (e - s))])
        r = np.minimum(np.searchsorted(e, g, side="right"), len(c) - 1)
        out[:, j] = cum[r] + c[r] * (g - s[r])
    return start, end, g, out


def oracle_models(oracle, pref, bin_bases, length, pieces=1):
    """(loss[k], a[k], b[k], in_peak[k, s]) for k = 0..S; with pieces > 1 the rows of a are scored in
    parallel (ctypes releases the GIL) and merged with the tie rule."""
    N, S = pref.shape[0] - 1, pref.shape[1]
    pref = np.ascontiguousarray(pref)
    pp = pref.ctypes.data_as(C.POINTER(C.c_int64))

    def run(lo_hi):
        lo, hi = lo_hi
        loss = np.zeros(S + 1); a = np.zeros(S + 1, np.int32); b = np.zeros(S + 1, np.int32)
        f = np.zeros((S + 1, S), np.uint8)
        oracle.joint_oracle(S, N, bin_bases, length, pp, lo, hi, loss.ctypes.data_as(C.POINTER(C.c_double)),
                            a.ctypes.data_as(C.POINTER(C.c_int)), b.ctypes.data_as(C.POINTER(C.c_int)),
                            f.ctypes.data_as(C.POINTER(C.c_uint8)))
        return loss, a, b, f
    if pieces <= 1 or N < 8:
        return run((1, N - 1))
    # row a holds N - 1 - a pairs: cut the rows into pieces of about equal pairs
    w = np.array([N - 1 - a for a in range(1, N - 1)], np.float64)
    cuts = np.searchsorted(np.cumsum(w) / w.sum(), np.linspace(0, 1, pieces + 1)[1:-1]) + 1
    bounds = [1] + sorted(set(int(x) for x in cuts)) + [N - 1]
    with ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        parts = list(ex.map(run, zip(bounds[:-1], bounds[1:])))
    loss, a, b, f = (x.copy() for x in parts[0])
    for pl, pa, pb, pf in parts[1:]:   # later pieces hold larger a: they win only with a strictly smaller loss
        for k in range(1, S + 1):
            if pl[k] < loss[k]:
                loss[k], a[k], b[k], f[k] = pl[k], pa[k], pb[k], pf[k]
    return loss, a, b, f


def select(ks, loss):
    """Selectable models (indices) and their [min_lambda, max_lambda]: the rule of psd_joint_models."""
    def lam(i, j):
        return (loss[i] - loss[j]) / float(ks[j] - ks[i])
    hull = [0]
    for j in range(1, len(ks)):
        while len(hull) >= 2 and not lam(hull[-2], hull[-1]) > lam(hull[-1], j):
            hull.pop()
        hull.append(j)
    while len(hull) >= 2 and not lam(hull[-2], hull[-1]) > 0:
        hull.pop()
    lo = np.full(len(ks), np.nan); hi = np.full(len(ks), np.nan)
    for h, m in enumerate(hull):
        hi[m] = math.inf if h == 0 else lam(hull[h - 1], m)
        lo[m] = 0.0 if h + 1 == len(hull) else lam(m, hull[h + 1])
    return hull, lo, hi


def label_totals(in_peak, ps, pe, labels, brute=False):
    """fp, fn, possible.fp, possible.fn, errors of one model summed over the samples' labels."""
    tot = np.zeros(5, np.int64)
    fun = path_oracle.label_errors_brute if brute else path_oracle.label_errors
    for s, lab in enumerate(labels):
        if lab is None:
            continue
        ls = np.asarray(lab["chromStart"], np.int64); le = np.asarray(lab["chromEnd"], np.int64)
        kind = np.array([path_oracle.KINDS[x] for x in lab["annotation"]], np.int64)
        peaks = (np.array([ps], np.int64), np.array([pe], np.int64)) if in_peak[s] else (np.zeros(0, np.int64), np.zeros(0, np.int64))
        fp, fn = fun(peaks[0], peaks[1], ls, le, kind)
        tot += [int(np.sum(fp)), int(np.sum(fn)), int(np.sum(kind != 1)), int(np.sum(kind != 0)), int(np.sum(fp) + np.sum(fn))]
    return tot


def reference(oracle, samples, bin_bases, labels=None, pieces=1, brute_labels=False):
    """What joint_models_batch returns for one problem, from the C oracle and the host rules."""
    start, end, g, pref = prefix(samples, bin_bases)
    loss, a, b, f = oracle_models(oracle, pref, bin_bases, end - start, pieces)
    ks = [k for k in range(len(loss)) if math.isfinite(loss[k])]
    L = [float(loss[k]) for k in ks]
    hull, lo, hi = select(ks, L)
    cols = {"peaks": np.array(ks, np.int64), "total.loss": np.array(L),
            "peakStart": np.array([-1 if k == 0 else int(g[a[k]]) for k in ks], np.int64),
            "peakEnd": np.array([-1 if k == 0 else int(g[b[k]]) for k in ks], np.int64),
            "selectable": np.isin(np.arange(len(ks)), hull), "min.lambda": lo, "max.lambda": hi}
    target = None
    if labels is not None and any(x is not None for x in labels):
        err = np.array([label_totals(f[k].astype(bool), cols["peakStart"][i], cols["peakEnd"][i], labels, brute_labels)
                        for i, k in enumerate(ks)])
        for j, col in enumerate(["fp", "fn", "possible.fp", "possible.fn", "errors"]):
            cols[col] = err[:, j]
        target = path_oracle.target_interval(lo[hull], hi[hull], err[hull, 4])
    return {"models": pd.DataFrame(cols), "in_peak": f[ks].astype(bool), "target": target}


def same_bits(x, y):
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    return x.shape == y.shape and bool(np.all((x.view(np.int64) == y.view(np.int64)) | (np.isnan(x) & np.isnan(y))))


def assert_same(got, want, what):
    gm, wm = got["models"], want["models"]
    assert list(gm["peaks"]) == list(wm["peaks"]), (what, list(gm["peaks"]), list(wm["peaks"]))
    for col in wm.columns:
        if wm[col].dtype == np.float64:
            assert same_bits(gm[col], wm[col]), (what, col, gm[col].tolist(), wm[col].tolist())
        else:
            assert np.array_equal(np.asarray(gm[col]), np.asarray(wm[col])), (what, col, gm[col].tolist(), wm[col].tolist())
    assert np.array_equal(got["in_peak"], want["in_peak"]), what
    if want["target"] is None:
        assert got["target"] is None, what
    else:
        assert got["target"] is not None and same_bits(got["target"][:2], want["target"][:2]) and got["target"][2] == want["target"][2], \
            (what, got["target"], want["target"])


# ---- problem generators ------------------------------------------------------------------------------------

def tile(rng, start, end, counts_fn, max_w=20):
    """Rows tiling [start, end) with random widths; counts_fn(n) gives the counts."""
    w = []
    left = end - start
    while left > 0:
        x = int(min(left, rng.integers(1, max_w + 1)))
        w.append(x); left -= x
    e = start + np.cumsum(w)
    return (e - np.array(w)).astype(np.int32), e.astype(np.int32), np.asarray(counts_fn(len(w))).astype(np.int32)


def sample_set(rng, S, start, end, kind, max_w=20):
    big = 2 ** 31 - 1
    if kind == "zero":
        return [tile(rng, start, end, lambda n: np.zeros(n), max_w) for _ in range(S)]
    if kind == "constant":
        return [tile(rng, start, end, lambda n, v=int(rng.integers(0, 50)): np.full(n, v), max_w) for _ in range(S)]
    if kind == "huge":
        return [tile(rng, start, end, lambda n: rng.choice([big, big - 1, 2 ** 30, 0, 7], size=n), max_w) for _ in range(S)]
    if kind == "duplicate":
        base = [tile(rng, start, end, lambda n: rng.poisson(8, size=n), max_w) for _ in range(max(1, S // 3))]
        return [base[i % len(base)] for i in range(S)]
    if kind == "mirror":   # the coverage of every sample is symmetric around the region's middle
        out = []
        for _ in range(S):
            half = (end - start) // 2
            s, e, c = tile(rng, 0, half, lambda n: rng.poisson(6, size=n), max_w)
            mid = end - start - 2 * half
            ws = list(e - s)
            cs = list(c)
            widths = ws + ([mid] if mid else []) + ws[::-1]
            cnts = cs + ([int(rng.integers(0, 20))] if mid else []) + cs[::-1]
            ee = start + np.cumsum(widths)
            out.append(((ee - np.array(widths)).astype(np.int32), ee.astype(np.int32), np.array(cnts, np.int32)))
        return out
    # noise with a bump in some samples
    lo, hi = sorted(int(x) for x in rng.integers(start, end, size=2))
    out = []
    for _ in range(S):
        depth = float(rng.choice([0.5, 3, 20]))
        bump = rng.random() < 0.5

        def counts(n, depth=depth):
            return rng.poisson(depth, size=n)
        s, e, c = tile(rng, start, end, counts, max_w)
        if bump:
            c = np.where((s >= lo) & (e <= hi), c * 4 + 3, c).astype(np.int32)
        out.append((s, e, c))
    return out


def labels_for(rng, samples):
    out = []
    for s, e, _ in samples:
        if rng.random() < 0.3:
            out.append(None)
            continue
        a0, a1 = int(s[0]), int(e[-1])
        n = int(rng.integers(1, 5))
        ls, le = [], []
        for _ in range(n):
            x, y = sorted(int(v) for v in rng.integers(a0, a1 + 1, size=2))
            if x == y:
                y = min(a1, x + 1); x = y - 1
            ls.append(x); le.append(y)
        out.append(pd.DataFrame({"chromStart": ls, "chromEnd": le, "annotation": list(rng.choice(KIND_NAMES, size=n))}))
    return out


# ---- CPU: oracle against brute force, selection, labels ------------------------------------------------------

def brute(samples, bin_bases):
    """Every peak and every subset of samples, each sample with its own feasibility test (Python ints, libm log).
    Returns {k: (loss, a, b, frozenset)}; ties: the smaller loss, then a, then b, then the subset whose samples
    in (r desc, s asc) order come first."""
    start, end, g, pref = prefix(samples, bin_bases)
    N, S = len(g) - 1, len(samples)
    P = [[int(x) for x in row] for row in pref]

    def L(c, w):
        return 0.0 if c == 0 else float(c) - float(c) * math.log(float(c) / float(w))
    W = [int(x - g[0]) for x in g]
    l1 = [L(P[N][s], W[N]) for s in range(S)]
    flat = 0.0
    for x in l1:
        flat += x
    best = {0: (flat, -1, -1, frozenset())}
    for a in range(1, N - 1):
        for b in range(a + 1, N):
            r = {}
            for s in range(S):
                c0a, cab, cbn = P[a][s], P[b][s] - P[a][s], P[N][s] - P[b][s]
                w0a, wab, wbn = W[a], W[b] - W[a], W[N] - W[b]
                if cab * w0a > c0a * wab and cab * wbn > cbn * wab:
                    r[s] = l1[s] - ((L(c0a, w0a) + L(cab, wab)) + L(cbn, wbn))
            for k in range(1, S + 1):
                for sub in itertools.combinations(range(S), k):
                    if any(s not in r for s in sub):
                        continue
                    order = sorted(sub, key=lambda s: (-r[s], s))
                    R = 0.0
                    for s in order:
                        R += r[s]
                    key = (flat - R, a, b, [(-r[s], s) for s in order])
                    if k not in best or key < best[k][4]:
                        best[k] = (flat - R, a, b, frozenset(sub), key)
    return {k: v[:4] for k, v in best.items()}


def test_oracle_matches_brute_force(oracle):
    rng = np.random.default_rng(7)
    kinds = ["noise", "noise", "zero", "constant", "huge", "duplicate", "mirror"]
    for case in range(500):
        S = int(rng.integers(1, 6))
        bin_bases = int(rng.choice([1, 2, 3, 7]))
        N = int(rng.integers(1, 13))
        length = N * bin_bases - int(rng.integers(0, bin_bases))
        start = int(rng.integers(0, 1000))
        samples = sample_set(rng, S, start, start + length, kinds[case % len(kinds)], max_w=4)
        want = brute(samples, bin_bases)
        _, end, g, pref = prefix(samples, bin_bases)
        loss, a, b, f = oracle_models(oracle, pref, bin_bases, end - start)
        for k in range(S + 1):
            if k not in want:
                assert math.isinf(loss[k]) and a[k] == -1, (case, k)
                continue
            wl, wa, wb, wset = want[k]
            assert same_bits(loss[k], wl) and a[k] == wa and b[k] == wb, (case, k, loss[k], wl, a[k], wa, b[k], wb)
            assert set(np.flatnonzero(f[k])) == set(wset), (case, k)


def test_selection_matches_penalty_grid(oracle):
    """The selectable models and their intervals are the argmin of loss_k + lambda k over a dense lambda grid."""
    rng = np.random.default_rng(11)
    lams = np.concatenate([[0.0], np.logspace(-4, 7, 4000)])
    n_sel = 0
    for case in range(60):
        S = int(rng.integers(1, 12))
        samples = sample_set(rng, S, 0, int(rng.integers(5, 60)), ["noise", "duplicate", "mirror"][case % 3], max_w=3)
        ref = reference(oracle, samples, 1)["models"]
        k, loss = ref["peaks"].to_numpy(), ref["total.loss"].to_numpy()
        sel = ref["selectable"].to_numpy()
        assert sel[0] and ref["max.lambda"][0] == math.inf
        n_sel += int(sel.sum())
        for lam in lams:
            cost = loss + lam * k
            m = int(np.argmin(cost))
            if np.sum(cost == cost[m]) > 1:
                continue   # a breakpoint of the grid
            assert sel[m], (case, lam, m)
            assert ref["min.lambda"][m] <= lam <= ref["max.lambda"][m], (case, lam, m)
        # every selectable model is the argmin at the middle of its interval (duplicated samples make points
        # collinear up to rounding: the breakpoints then decide, and an interval of a few ulps is not probed)
        for m in np.flatnonzero(sel):
            lo, hi = ref["min.lambda"][m], ref["max.lambda"][m]
            if hi - lo <= 1e-9 * hi:
                continue
            mid = lo * 2 + 1 if math.isinf(hi) else (lo + hi) / 2
            assert int(np.argmin(loss + mid * k)) == m, (case, m)
        assert not np.any(np.isfinite(ref["min.lambda"][~sel]))
    assert n_sel > 60


def test_reference_labels_match_path_oracle(oracle):
    """Label errors summed over samples equal path_oracle's brute force, and the target equals
    path_oracle.target_interval over the selectable models."""
    rng = np.random.default_rng(5)
    n_target = 0
    for case in range(80):
        S = int(rng.integers(1, 7))
        samples = sample_set(rng, S, 100, 100 + int(rng.integers(3, 40)), "noise", max_w=3)
        labels = labels_for(rng, samples)
        if all(x is None for x in labels):
            labels[0] = pd.DataFrame({"chromStart": [100], "chromEnd": [101], "annotation": ["noPeaks"]})
        got = reference(oracle, samples, 1, labels)
        want = reference(oracle, samples, 1, labels, brute_labels=True)
        assert_same(got, want, case)
        m = got["models"]
        sel = m["selectable"].to_numpy()
        t = path_oracle.target_interval(m["min.lambda"][sel].to_numpy(), m["max.lambda"][sel].to_numpy(), m["errors"][sel].to_numpy())
        assert t == got["target"]
        n_target += 1
    assert n_target == 80


def test_no_peak_problems_on_the_host(psd, oracle):
    """Regions of one or two bins have only the flat model; they never reach the device, so the library
    answers them without a GPU, with labels."""
    rng = np.random.default_rng(3)
    probs, labs, bins = [], [], []
    for case in range(40):
        S = int(rng.integers(1, 9))
        b = int(rng.choice([1, 5, 50]))
        length = int(rng.integers(1, 2 * b + 1))
        samples = sample_set(rng, S, 1000, 1000 + length, ["noise", "huge", "zero"][case % 3], max_w=7)
        probs.append(samples); labs.append(labels_for(rng, samples)); bins.append(b)
    for b in sorted(set(bins)):
        idx = [i for i in range(len(probs)) if bins[i] == b]
        got, st = psd.joint_models_batch([probs[i] for i in idx], bin_bases=b, labels=[labs[i] for i in idx])
        assert st["n_waves"] == 0 and st["pair_sample_evals"] == 0
        for r, i in zip(got, idx):
            assert len(r["models"]) == 1
            assert_same(r, reference(oracle, probs[i], b, labs[i]), i)


def _joint_struct(psd, problems):
    """ctypes problems; each problem (region, bin, samples) with samples (s, e, c, labels or None) and None
    standing for a null array."""
    arr = (psd._lib.PsdJointProblem * max(1, len(problems)))()
    keep = []
    p32 = C.POINTER(C.c_int32)

    def ptr(a):
        if a is None:
            return None
        a = np.ascontiguousarray(a, np.int32)
        keep.append(a)
        return a.ctypes.data_as(p32)
    for i, (region, bin_bases, samples, n_samples) in enumerate(problems):
        sa = (psd._lib.PsdJointSample * max(1, len(samples or [])))()
        keep.append(sa)
        for j, (s, e, c, lab) in enumerate(samples or []):
            sa[j].n_rows = len(c) if c is not None else 3
            sa[j].chromStart, sa[j].chromEnd, sa[j].coverage = ptr(s), ptr(e), ptr(c)
            if lab is not None:
                ls, le, lk = lab
                sa[j].n_labels = len(lk) if lk is not None else 2
                sa[j].label_start, sa[j].label_end, sa[j].label_kind = ptr(ls), ptr(le), ptr(lk)
        arr[i].region_start, arr[i].region_end = region
        arr[i].bin_bases = bin_bases
        arr[i].n_samples = n_samples
        arr[i].samples = sa if samples is not None else None
    return arr, keep


def test_joint_input_errors(psd):
    """Every bad input is refused on the host with PSD_ERR_ARG, naming the problem and the sample, before any
    device work (these run without a GPU)."""
    lib = psd._lib.lib
    s, e, c = np.array([0, 5]), np.array([5, 9]), np.array([1, 2])
    good_sample = (s, e, c, None)
    good = ((0, 9), 1, [good_sample, good_sample], 2)
    lab_ok = (np.array([1]), np.array([4]), np.array([1]))
    cases = [
        (((0, 9), 1, [good_sample], 0), "n_samples 0"),
        (((0, 9), 1, [good_sample] * 257, 257), "n_samples 257"),
        (((0, 9), 1, None, 2), "samples is null"),
        (((0, 9), 0, [good_sample] * 2, 2), "bin_bases 0"),
        (((0, 9), -3, [good_sample] * 2, 2), "bin_bases -3"),
        (((0, 40000), 1, [(np.array([0]), np.array([40000]), np.array([1]), None)] * 2, 2), "PSD_JOINT_MAX_BINS"),
        (((0, 9), 1, [good_sample, (np.array([0, 6]), np.array([5, 9]), c, None)], 2), "sample 1: row 1"),     # gap
        (((0, 9), 1, [good_sample, (np.array([0, 5]), np.array([5, 9]), np.array([1, -1]), None)], 2), "sample 1: row 1"),
        (((0, 9), 1, [good_sample, (np.array([0, 5]), np.array([5, 10]), c, None)], 2), "sample 1: rows cover [0, 10)"),
        (((0, 9), 1, [good_sample, (np.array([1, 5]), np.array([5, 9]), c, None)], 2), "sample 1: rows cover [1, 9)"),
        (((0, 10), 1, [good_sample, good_sample], 2), "sample 0: rows cover [0, 9)"),   # the region differs from the rows
        (((0, 9), 1, [good_sample, (None, e, c, None)], 2), "sample 1: a row array is null"),
        (((0, 9), 1, [good_sample, (s, e, None, None)], 2), "sample 1: a row array is null"),
        (((0, 9), 1, [good_sample, (s, e, c, (np.array([1]), np.array([4]), np.array([4])))], 2), "sample 1: label 0: kind 4"),
        (((0, 9), 1, [good_sample, (s, e, c, (np.array([4]), np.array([4]), np.array([1])))], 2), "sample 1: label 0: chromStart 4 >= chromEnd 4"),
        (((0, 9), 1, [good_sample, (s, e, c, (np.array([5]), np.array([10]), np.array([0])))], 2), "sample 1: label 0: [5, 10) is not inside"),
        (((0, 9), 1, [good_sample, (s, e, c, (None, np.array([4]), np.array([1])))], 2), "sample 1: a label array is null"),
    ]
    h = C.c_void_p()
    for bad, text in cases:
        arr, keep = _joint_struct(psd, [good, bad, good])
        h.value = None
        assert lib.psd_joint_models(-1, 3, arr, C.byref(h)) == PSD_ERR_ARG, text
        msg = lib.psd_last_error().decode()
        assert "problem 1" in msg and text in msg, (text, msg)
        assert not h.value
    arr, keep = _joint_struct(psd, [good])
    assert lib.psd_joint_models(-1, -1, arr, C.byref(h)) == PSD_ERR_ARG
    assert lib.psd_joint_models(-1, 1, None, C.byref(h)) == PSD_ERR_ARG
    assert lib.psd_joint_models(-1, 1, arr, None) == PSD_ERR_ARG
    # zero problems: no device needed
    assert lib.psd_joint_models(-1, 0, None, C.byref(h)) == 0 and h.value
    st = psd._lib.PsdJointStats()
    assert lib.psd_joint_get_stats(h, C.byref(st)) == 0 and st.n_problems == 0 and st.n_waves == 0
    assert lib.psd_joint_n_models(h, 0) == -1
    lib.psd_joint_free(h)
    # the Python entry
    with pytest.raises(ValueError, match="problem 0: sample 1: rows cover"):
        psd.joint_models_batch([[(s, e, c), (np.array([0, 5]), np.array([5, 10]), c)]])
    with pytest.raises(ValueError, match="problem 0: n_samples 0"):
        psd.joint_models_batch([[]])
    with pytest.raises(ValueError, match="bin_bases 0"):
        psd.joint_models_batch([[(s, e, c)]], bin_bases=0)
    with pytest.raises(ValueError, match="label 0"):
        psd.joint_models_batch([[(s, e, c)]], labels=[[pd.DataFrame({"chromStart": [3], "chromEnd": [20], "annotation": ["peaks"]})]])
    with pytest.raises(ValueError, match="one entry"):
        psd.joint_models_batch([[(s, e, c)]], labels=[[None, None]])
    assert psd.joint_models_batch([])[0] == []
    for name in ("psd_joint_models", "psd_joint_model_table", "psd_joint_samples", "psd_joint_target"):
        assert name in psd._lib.C_ABI_SYMBOLS


# ---- GPU: bit for bit against the oracle -------------------------------------------------------------------

def gpu_problem_set(seed=2026):
    """About 300 problems: S in {1, 2, 7, 32, 33, 100, 256}, N from 1 to about 1,000, bins of 1 and more with a
    short last bin, zero, constant, huge-count, duplicated and mirrored samples."""
    rng = np.random.default_rng(seed)
    Ss = [1, 2, 7, 32, 33, 100, 256]
    kinds = ["noise", "noise", "zero", "constant", "huge", "duplicate", "mirror"]
    out = []   # (samples, bin)
    for i in range(294):
        S = Ss[i % 7]
        kind = kinds[(i // 7) % 7]
        n_max = int(min(1000, math.sqrt(2 * 3e6 / S)))
        N = [1, 2, 3][i % 3] if i < 21 else int(round(n_max ** rng.uniform(0.3, 1.0)))
        bin_bases = int(rng.choice([1, 1, 4, 10])) if kind != "huge" else int(rng.choice([1, 1000, 1000000]))
        N = min(N, 1000 if bin_bases < 1000000 else 1000)
        length = N * bin_bases - int(rng.integers(0, bin_bases))
        start = int(rng.integers(0, 10 ** 6))
        out.append((sample_set(rng, S, start, start + length, kind, max_w=max(1, min(3 * bin_bases, 10 ** 7))), bin_bases))
    for S, N in ((1, 1000), (2, 997), (7, 640)):   # the longest grids
        out.append((sample_set(rng, S, 0, N, "noise", max_w=3), 1))
    return out


def run_joint(psd, problems, labels=None):
    """joint_models_batch on (samples, bin) problems of mixed bins: one call per bin width."""
    got = [None] * len(problems)
    stats = []
    for b in sorted(set(p[1] for p in problems)):
        idx = [i for i, p in enumerate(problems) if p[1] == b]
        res, st = psd.joint_models_batch([problems[i][0] for i in idx], bin_bases=b,
                                         labels=None if labels is None else [labels[i] for i in idx])
        stats.append(st)
        for i, r in zip(idx, res):
            got[i] = r
    return got, stats


@pytest.fixture(scope="module")
def gpu_set(oracle):
    probs = gpu_problem_set()
    with ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        want = list(ex.map(lambda p: reference(oracle, p[0], p[1]), probs))
    return probs, want


@pytest.mark.gpu
def test_gpu_bit_identical_to_oracle(gpu, gpu_set):
    probs, want = gpu_set
    got, stats = run_joint(gpu, probs)
    for i, (g, w) in enumerate(zip(got, want)):
        assert_same(g, w, "problem %d (S %d, bin %d)" % (i, len(probs[i][0]), probs[i][1]))
    assert sum(st["pair_sample_evals"] for st in stats) == sum(
        len(s) * max(0, (len(grid_of(int(s[0][0][0]), int(s[0][1][-1]), b)) - 2) * (len(grid_of(int(s[0][0][0]), int(s[0][1][-1]), b)) - 3) // 2)
        for s, b in probs)
    # something happened: models with peaks, selectable ones, exact ties from duplicated samples
    assert sum(len(g["models"]) for g in got) > 2 * len(got)


@pytest.mark.gpu
def test_gpu_forced_waves(gpu, gpu_set):
    probs, want = gpu_set
    lib = gpu._lib.lib
    lib.psd_set_option(b"coverage_gb", 1e-6)   # about 1 KB: every problem runs in a wave of its own
    try:
        got, stats = run_joint(gpu, probs)
    finally:
        lib.psd_set_option(b"coverage_gb", 0.0)
    n_dev = sum(1 for s, b in probs if -(-(int(s[0][1][-1]) - int(s[0][0][0])) // b) >= 3)
    assert sum(st["n_waves"] for st in stats) == n_dev
    for i, (g, w) in enumerate(zip(got, want)):
        assert_same(g, w, "problem %d in waves" % i)


@pytest.mark.gpu
def test_gpu_large_problem(gpu, oracle):
    """N = 4,096 bins and S = 64 samples: 8.4 M peaks, 5.4e8 pair x sample evaluations."""
    rng = np.random.default_rng(99)
    samples = sample_set(rng, 64, 5000, 5000 + 4096, "noise", max_w=6)
    want = reference(oracle, samples, 1, pieces=256)
    got, st = gpu.joint_models_batch([samples])
    assert_same(got[0], want, "N 4096, S 64")
    assert st["pair_sample_evals"] == 64 * 4095 * 4094 // 2


@pytest.mark.gpu
def test_gpu_planted_peak(gpu, oracle):
    """20 samples at high depth, 12 of them with one peak on bins [80, 120) of 10 bases: the 12-sample model is
    selectable, with exactly those samples and those boundaries."""
    rng = np.random.default_rng(12)
    start, bin_bases, n_bins = 30000, 10, 200
    carriers = sorted(int(x) for x in rng.choice(20, size=12, replace=False))
    samples = []
    for s in range(20):
        w = np.full(n_bins * bin_bases // 5, 5)
        e = start + np.cumsum(w)
        st = e - w
        lam = np.full(len(w), 60.0)
        if s in carriers:
            lam[(st >= start + 80 * bin_bases) & (e <= start + 120 * bin_bases)] = 600.0
        samples.append((st.astype(np.int32), e.astype(np.int32), rng.poisson(lam).astype(np.int32)))
    got, _ = gpu.joint_models_batch([samples], bin_bases=bin_bases)
    assert_same(got[0], reference(oracle, samples, bin_bases), "planted")
    m = got[0]["models"]
    r = int(np.flatnonzero(m["peaks"].to_numpy() == 12)[0])
    assert bool(m["selectable"][r])
    assert (m["peakStart"][r], m["peakEnd"][r]) == (start + 800, start + 1200)
    assert list(np.flatnonzero(got[0]["in_peak"][r])) == carriers


@pytest.mark.gpu
def test_gpu_from_reads(gpu, oracle):
    """Aligned reads of several samples over one region -> coverage_rows on the device -> joint models."""
    from peaksegdisk_b200.plan import coverage_rows
    rng = np.random.default_rng(21)
    start, end = 100000, 101500
    problems = []
    for s in range(9):
        n = int(rng.integers(200, 800))
        st = rng.integers(start - 100, end, size=n)
        if s % 3:   # a peak in two of three samples
            st = np.concatenate([st, rng.integers(start + 600, start + 800, size=400)])
        problems.append((st, st + rng.integers(30, 120, size=len(st)), start, end))
    rows, _ = coverage_rows(problems, device=0)
    for b in (1, 10):
        got, st = gpu.joint_models_batch([rows], bin_bases=b)
        assert_same(got[0], reference(oracle, rows, b), "reads, bin %d" % b)
        assert len(got[0]["models"]) > 1 and st["n_waves"] == 1


@pytest.mark.gpu
def test_gpu_labels(gpu, oracle):
    rng = np.random.default_rng(31)
    probs, labs = [], []
    for case in range(40):
        S = int(rng.choice([1, 3, 8, 40]))
        b = int(rng.choice([1, 5]))
        start = int(rng.integers(0, 10 ** 5))
        samples = sample_set(rng, S, start, start + int(rng.integers(3, 120)) * b, "noise", max_w=4)
        probs.append((samples, b)); labs.append(labels_for(rng, samples))
    labs[0] = [None] * len(probs[0][0])   # a problem without labels in a call with labels
    got, _ = run_joint(gpu, probs, labs)
    n_target = 0
    for i, (g, (samples, b)) in enumerate(zip(got, probs)):
        want = reference(oracle, samples, b, labs[i])
        assert_same(g, want, "labelled problem %d" % i)
        n_target += want["target"] is not None
    assert n_target >= 30
