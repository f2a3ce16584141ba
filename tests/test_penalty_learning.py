"""Penalty learning: coverage statistics on the device (psd_features, problem_features) and interval
regression (IntervalRegressionCV).  Without a GPU: an exact statistics oracle against brute force, every
psd_features input error, and the fit's optimality conditions, objective, lambda_max, determinism and choice
of lambda.  On the GPU: psd_features against the oracle bit for bit, in one call and in forced waves, and
the whole workflow -- labelled paths, features, fit, predicted penalties, labelled solves -- end to end."""
import ctypes as C
import math
import os
import time
import numpy as np
import pandas as pd
import pytest
from helpers import GOLD

PSD_ERR_ARG = 111
PSD_ERR_INCONSISTENT = 6
NINE = ["quartile.0%", "quartile.25%", "quartile.50%", "quartile.75%", "quartile.100%", "mean", "sd", "bases", "data"]


@pytest.fixture(scope="module")
def psd():
    import peaksegdisk_b200
    return peaksegdisk_b200


@pytest.fixture(scope="module")
def gpu(psd):
    assert psd._lib.lib.psd_device_count() >= 1, "no CUDA device"
    return psd


# ---- the statistics oracle ------------------------------------------------------------------------------

def _type7(x_at, B, p):
    h = float(B - 1) * p
    lo = math.floor(h)
    g = h - lo
    x0 = x_at(lo)
    if g == 0:
        return float(x0)
    x1 = x_at(lo + 1)
    return float(x0) if x1 == x0 else (1 - g) * x0 + g * x1


def _finish(B, S1, S2, n_rows, x_at, lo_c, hi_c):
    q = [float(lo_c)] + [_type7(x_at, B, p) for p in (0.25, 0.5, 0.75)] + [float(hi_c)]
    sd = math.nan if B == 1 else math.sqrt(float(B * S2 - S1 * S1) / (float(B) * float(B - 1)))
    return q + [float(S1) / float(B), sd, float(B), float(n_rows)]


def features_oracle(s, e, c):
    """The nine statistics of one problem in exact integer arithmetic (S2 from 16-bit limbs of c^2 so that
    numpy sums never overflow) and R's type-7 formula on a weighted sort, as the library defines them."""
    w = (np.asarray(e, np.int64) - np.asarray(s, np.int64))
    c = np.asarray(c, np.int64)
    B = int(w.sum())
    S1 = int(np.sum(w * c))   # < 2^63 for B < 2^32 and int32 counts
    c2 = (c * c).astype(np.uint64)
    S2 = 0
    for li in range(4):
        limb = ((c2 >> np.uint64(16 * li)) & np.uint64(0xffff)).astype(np.int64)
        for k in range(0, len(c), 1 << 16):   # w * limb < 2^47, 2^16 of them < 2^63
            S2 += int(np.sum(w[k:k + (1 << 16)] * limb[k:k + (1 << 16)])) << (16 * li)
    order = np.argsort(c, kind="stable")
    cs, cw = c[order], np.cumsum(w[order])
    return _finish(B, S1, S2, len(c), lambda k: int(cs[np.searchsorted(cw, k, "right")]), int(c.min()), int(c.max()))


def features_brute(s, e, c):
    """The same from the expanded, sorted per-base vector and Python-int sums."""
    x = np.sort(np.repeat(np.asarray(c, np.int64), np.asarray(e, np.int64) - np.asarray(s, np.int64)))
    xs = [int(v) for v in x]
    B = len(xs)
    return _finish(B, sum(xs), sum(v * v for v in xs), len(c), lambda k: xs[k], xs[0], xs[-1])


def oracle_frame(problems):
    rows = []
    for s, e, c in problems:
        base = np.array(features_oracle(s, e, c))
        with np.errstate(divide="ignore", invalid="ignore"):
            rows.append(np.concatenate([base, np.log(base + 1), np.log(base), np.log(np.log(base))]))
    return np.array(rows)


def random_rows(rng, n, start=None, max_w=20, counts=None):
    w = rng.integers(1, max_w + 1, size=n)
    s0 = int(rng.integers(0, 1000)) if start is None else start
    end = s0 + np.cumsum(w)
    c = rng.integers(0, 50, size=n) if counts is None else counts
    return (end - w).astype(np.int32), end.astype(np.int32), np.asarray(c).astype(np.int32)


def assert_bits_equal(got, want, what):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    same = (got.view(np.int64) == want.view(np.int64)) | (np.isnan(got) & np.isnan(want))
    if not same.all():
        i, j = np.argwhere(~same)[0]
        raise AssertionError("%s: row %d column %d: %r != %r" % (what, i, j, got[i, j], want[i, j]))


# ---- CPU: oracle, input errors -------------------------------------------------------------------------

def test_statistics_oracle_matches_brute_force():
    rng = np.random.default_rng(2024)
    for case in range(1000):
        n = int(rng.integers(1, 40))
        kind = case % 4
        if kind == 0:
            counts = rng.integers(0, 10, size=n)
        elif kind == 1:
            counts = rng.integers(0, 2 ** 31, size=n)   # wide values: 128-bit S2, every digit
        elif kind == 2:
            counts = np.full(n, int(rng.integers(0, 2 ** 31)))
        else:
            counts = rng.choice([0, 1, 2 ** 31 - 1, 2 ** 24, 2 ** 16 + 3], size=n)
        s, e, c = random_rows(rng, n, max_w=int(rng.choice([1, 3, 30])), counts=counts)
        got, want = features_oracle(s, e, c), features_brute(s, e, c)
        assert_bits_equal(np.array([got]), np.array([want]), "case %d" % case)


def _rows_struct(psd, problems):
    arr = (psd._lib.PsdRows * max(1, len(problems)))()
    keep = []
    p32 = C.POINTER(C.c_int32)
    for i, (s, e, c) in enumerate(problems):
        s, e, c = (None if a is None else np.ascontiguousarray(a, np.int32) for a in (s, e, c))
        keep += [s, e, c]
        arr[i].n_rows = len(c) if c is not None else 3
        arr[i].chromStart = s.ctypes.data_as(p32) if s is not None else None
        arr[i].chromEnd = e.ctypes.data_as(p32) if e is not None else None
        arr[i].coverage = c.ctypes.data_as(p32) if c is not None else None
    return arr, keep


def test_features_input_errors(psd):
    """Every bad input is refused on the host, naming the problem, before any device work (these run
    without a GPU: a check that came after the device work would return PSD_ERR_CUDA here)."""
    lib = psd._lib.lib
    good = (np.array([0, 5]), np.array([5, 9]), np.array([1, 2]))
    out = (psd._lib.PsdProblemFeatures * 4)()
    st = psd._lib.PsdFeaturesStats()
    cases = [
        ((np.array([0, 5]), np.array([5, 9]), np.array([1, -2])), PSD_ERR_ARG, "row 1"),     # negative count
        ((np.array([0, 5]), np.array([5, 5]), np.array([1, 2])), PSD_ERR_ARG, "row 1"),      # empty row
        ((np.array([0, 6]), np.array([5, 9]), np.array([1, 2])), PSD_ERR_INCONSISTENT, "row 1"),   # gap
        ((np.array([0, 4]), np.array([5, 9]), np.array([1, 2])), PSD_ERR_INCONSISTENT, "row 1"),   # overlap
        ((None, np.array([5, 9, 12]), np.array([1, 2, 3])), PSD_ERR_ARG, "null"),
        ((np.array([0, 5, 9]), np.array([5, 9, 12]), None), PSD_ERR_ARG, "null"),
        ((np.zeros(0), np.zeros(0), np.zeros(0)), PSD_ERR_ARG, "n_rows 0"),
    ]
    for bad, code, text in cases:
        arr, keep = _rows_struct(psd, [good, bad, good])
        assert lib.psd_features(-1, 3, arr, out, C.byref(st)) == code, text
        msg = lib.psd_last_error().decode()
        assert "problem 1" in msg and text in msg, msg
        if all(a is not None for a in bad):   # null arrays cannot come from Python
            with pytest.raises(ValueError, match="problem 1"):
                psd.problem_features([good, bad, good])
    arr, keep = _rows_struct(psd, [good])
    assert lib.psd_features(-1, -1, arr, out, None) == PSD_ERR_ARG
    assert lib.psd_features(-1, 1, None, out, None) == PSD_ERR_ARG
    assert lib.psd_features(-1, 1, arr, None, None) == PSD_ERR_ARG
    # zero problems: 0, no device needed, stats zeroed
    st.n_waves = 7
    assert lib.psd_features(-1, 0, None, None, C.byref(st)) == 0 and st.n_waves == 0 and st.n_launches == 0
    df = psd.problem_features([])
    assert list(df.columns) == psd.plan.FEATURE_COLUMNS and len(df) == 0 and len(df.columns) == 36
    with pytest.raises(ValueError, match="same length"):
        psd.problem_features([(np.array([0]), np.array([5, 6]), np.array([1]))])
    assert "psd_features" in psd._lib.C_ABI_SYMBOLS


# ---- CPU: interval regression --------------------------------------------------------------------------

def regression_data(seed, n=80, p=10, inf_share=0.3, width=(0.5, 3.0)):
    """Features with a few informative columns, a constant and a non-finite column, and target intervals
    around a linear function with noise; some limits infinite."""
    rng = np.random.default_rng(seed)
    X = rng.normal(size=(n, p)) * rng.uniform(0.5, 20, size=p) + rng.uniform(-5, 5, size=p)
    X[:, 3] = 7.0                       # constant: dropped
    X[rng.integers(0, n), 5] = -np.inf  # non-finite on one row: dropped
    f = 2.0 + 0.3 * X[:, 0] - 0.1 * X[:, 1] + 0.05 * X[:, 2] + rng.normal(0, 0.3, size=n)
    half = rng.uniform(*width, size=n) / 2
    lo, hi = f - half, f + half
    u = rng.uniform(size=n)
    lo[u < inf_share / 2] = -np.inf
    hi[(u >= inf_share / 2) & (u < inf_share)] = np.inf
    return pd.DataFrame(X, columns=["x%d" % j for j in range(p)]), np.column_stack([lo, hi])


def scaled(model, X):
    return (np.asarray(X[model.columns], np.float64) - model.centre) / model.scale


def objective(Xs, lo, hi, lam, b, w, margin=1.0):
    f = b + Xs @ w
    return float(np.mean(np.maximum(0, lo + margin - f) ** 2 + np.maximum(0, f - hi + margin) ** 2) + lam * np.abs(w).sum())


def kkt(Xs, lo, hi, lam, b, w, margin=1.0):
    f = b + Xs @ w
    g = 2 * (np.maximum(0, f - hi + margin) - np.maximum(0, lo + margin - f)) / len(f)
    gw = Xs.T @ g
    v = np.where(w != 0, np.abs(gw + lam * np.sign(w)), np.maximum(np.abs(gw) - lam, 0))
    return max(abs(g.sum()), v.max())


def test_regression_optimality_conditions_along_the_path(psd):
    X, T = regression_data(1)
    m = psd.IntervalRegressionCV(X, T, tol=1e-6)
    assert "x3" not in m.columns and "x5" not in m.columns and len(m.columns) == 8
    Xs = scaled(m, X)
    assert np.allclose(Xs.mean(axis=0), 0) and np.allclose(Xs.std(axis=0, ddof=1), 1)
    assert np.isinf(T).any()
    for i, lam in enumerate(m.path["lambda"]):
        assert kkt(Xs, T[:, 0], T[:, 1], lam, m.path_intercepts[i], m.path_weights[i]) <= 1e-6, i
    lam = m.path["lambda"].to_numpy()
    assert lam[0] == m.lambda_max and np.isclose(lam[-1], m.lambda_max * 1e-3) and np.all(np.diff(lam) < 0)


def test_regression_objective_matches_scipy():
    from scipy.optimize import minimize
    from peaksegdisk_b200 import learn
    X, T = regression_data(2, n=60, p=6)
    Xa = np.asarray(X, np.float64)[:, [0, 1, 2, 4]]
    Xs = (Xa - Xa.mean(axis=0)) / Xa.std(axis=0, ddof=1)
    lo, hi = T[:, 0], T[:, 1]
    lmax = learn.lambda_max(Xs, lo, hi)
    lams = lmax * np.array([0.5, 0.05, 0.002])
    b, W = learn.interval_regression_path(Xs, lo, hi, lams, tol=1e-11)
    p = Xs.shape[1]
    for i, lam in enumerate(lams):
        def fun(z):
            bb, w = z[0], z[1:1 + p] - z[1 + p:]
            f = bb + Xs @ w
            a, c = np.maximum(0, lo + 1 - f), np.maximum(0, f - hi + 1)
            g = 2 * (c - a) / len(f)
            gw = Xs.T @ g
            return (np.mean(a ** 2 + c ** 2) + lam * z[1:].sum(), np.concatenate([[g.sum()], gw + lam, -gw + lam]))
        r = minimize(fun, np.zeros(1 + 2 * p), jac=True, method="L-BFGS-B", bounds=[(None, None)] + [(0, None)] * (2 * p),
                     options={"ftol": 1e-16, "gtol": 1e-12, "maxiter": 100000, "maxcor": 50})
        ours = objective(Xs, lo, hi, lam, b[i], W[i])
        assert abs(ours - r.fun) <= 1e-7 * abs(r.fun), (lam, ours, r.fun)


def test_regression_lambda_max_is_the_first_nonzero_point(psd):
    from peaksegdisk_b200 import learn
    X, T = regression_data(3)
    m = psd.IntervalRegressionCV(X, T)
    assert np.all(m.path_weights[0] == 0) and m.path["nonzero"].iloc[0] == 0
    Xs = scaled(m, X)
    b, W = learn.interval_regression_path(Xs, T[:, 0], T[:, 1], [m.lambda_max * (1 - 1e-3)])
    assert np.count_nonzero(W[0]) >= 1
    b, W = learn.interval_regression_path(Xs, T[:, 0], T[:, 1], [m.lambda_max])
    assert np.all(W[0] == 0)
    # the intercept at lambda_max is the exact 1-D minimiser: a fine grid finds nothing lower
    grid = b[0] + np.linspace(-1e-3, 1e-3, 2001)
    obj = [objective(Xs, T[:, 0], T[:, 1], 0.0, g, np.zeros(Xs.shape[1])) for g in grid]
    assert objective(Xs, T[:, 0], T[:, 1], 0.0, b[0], np.zeros(Xs.shape[1])) <= min(obj) + 1e-15


def test_regression_separable_set_has_no_training_errors(psd):
    X, T = regression_data(4, n=60, inf_share=0.2, width=(3.0, 5.0))
    rng = np.random.default_rng(4)
    f = 1.0 + 0.4 * X["x0"].to_numpy() - 0.2 * X["x1"].to_numpy()
    half = rng.uniform(1.5, 2.5, size=len(f))   # no noise, room for the margin
    T = np.column_stack([f - half, f + half])
    m = psd.IntervalRegressionCV(X, T)
    assert m.path["train.errors"].iloc[-1] == 0
    assert m.path["train.errors"].iloc[0] > 0


def test_regression_is_deterministic_and_chooses_the_documented_lambda(psd):
    X, T = regression_data(5)
    a = psd.IntervalRegressionCV(X, T, seed=7)
    b = psd.IntervalRegressionCV(X, T, seed=7)
    pd.testing.assert_frame_equal(a.path, b.path)
    assert np.array_equal(a.folds, b.folds) and np.array_equal(a.weights, b.weights)
    v = a.path["validation.errors"].to_numpy()
    best = np.flatnonzero(v == v.min())
    assert a.lambda_ == a.path["lambda"].iloc[best[0]] == a.path["lambda"].iloc[best].max()
    i = best[0]
    assert np.array_equal(a.weights, a.path_weights[i]) and a.intercept == a.path_intercepts[i]
    assert np.bincount(a.folds).min() >= len(T) // 5
    pred = a.predict(X)
    assert np.allclose(pred, a.intercept + scaled(a, X) @ a.weights)
    assert np.allclose(a.predict(np.asarray(X)), pred)


def test_regression_bad_input_raises(psd):
    X, T = regression_data(6, n=20)
    for row, (lo, hi) in [(3, (-np.inf, np.inf)), (4, (2.0, 2.0)), (5, (3.0, 1.0)), (6, (np.nan, 1.0))]:
        bad = T.copy()
        bad[row] = (lo, hi)
        with pytest.raises(ValueError, match="target row %d" % row):
            psd.IntervalRegressionCV(X, bad)
    with pytest.raises(ValueError):
        psd.IntervalRegressionCV(X, T[:, :1])
    m = psd.IntervalRegressionCV(X, T)
    Y = X.copy()
    Y.loc[2, m.columns[0]] = np.nan
    with pytest.raises(ValueError, match="feature row 2"):
        m.predict(Y)
    Y = X.copy()
    Y.loc[1, "x5"] = np.inf   # a dropped column may be anything
    m.predict(Y)


# ---- GPU: psd_features against the oracle ---------------------------------------------------------------

def feature_problems():
    from peaksegdisk_b200 import synth
    from peaksegdisk_b200.plan import coverage_rows
    rng = np.random.default_rng(77)
    probs = {}
    _, s, e, c = synth.read_bedgraph(os.path.join(GOLD, "Mono27ac_coverage.bedGraph"))
    probs["Mono27ac"] = [(s, e, c)]
    probs["one row"] = [(np.array([100], np.int32), np.array([137], np.int32), np.array([9], np.int32))]
    probs["one base"] = [(np.array([5], np.int32), np.array([6], np.int32), np.array([3], np.int32))]
    probs["constant"] = [random_rows(rng, 5000, counts=np.full(5000, 17))]
    n = 64   # counts of 2^31 - 1 and weights near 2^31 / n: S2 near 2^93, B near 2^31
    w = (2 ** 31 // n) - rng.integers(0, 1000, size=n)
    end = np.cumsum(w) - 2 ** 30
    probs["wide"] = [((end - w).astype(np.int32), end.astype(np.int32),
                      rng.choice([2 ** 31 - 1, 2 ** 31 - 2, 2 ** 30, 1, 0, 0x01020304], size=n).astype(np.int32))]
    # quartile ranks lo and lo + 1 in different rows: B = 9 -> h = 2, 4, 6 exactly; B = 10 -> h = 2.25, 4.5, 6.75
    probs["rank split"] = [(np.arange(k, dtype=np.int32), np.arange(1, k + 1, dtype=np.int32),
                            rng.permutation(np.arange(k) * 1000 + 7).astype(np.int32)) for k in (9, 10, 11, 12, 2, 3)]
    probs["1e7 rows"] = [random_rows(rng, 10 ** 7, start=0, max_w=60, counts=rng.poisson(rng.choice([0.2, 3.0, 40.0], size=10 ** 7)))]
    probs["10000 tiny"] = [random_rows(rng, int(k), max_w=int(rng.integers(1, 100))) for k in rng.integers(1, 101, size=10000)]
    reads = [synth.reads(31 + i, 20000, 500000, start=1000 * i) for i in range(4)]
    rows, _ = coverage_rows([(rs, re_, 1000 * i, 1000 * i + 500000) for i, (rs, re_) in enumerate(reads)], 0)
    probs["coverage_rows"] = rows
    return probs


@pytest.fixture(scope="module")
def feature_cases(gpu):
    probs = feature_problems()
    names, flat = [], []
    for k, v in probs.items():
        names += ["%s[%d]" % (k, i) for i in range(len(v))]
        flat += v
    return names, flat, oracle_frame(flat)


@pytest.mark.gpu
def test_features_equal_the_oracle_bit_for_bit(gpu, feature_cases):
    names, flat, want = feature_cases
    t0 = time.time()
    df, st = gpu.problem_features(flat, device=0, return_stats=True)
    wall = time.time() - t0
    assert list(df.columns) == gpu.plan.FEATURE_COLUMNS
    got = df.to_numpy()
    for i in np.flatnonzero(~np.all((got.view(np.int64) == want.view(np.int64)) | (np.isnan(got) & np.isnan(want)), axis=1))[:1]:
        raise AssertionError("%s: got %s want %s" % (names[i], got[i, :9], want[i, :9]))
    assert np.isnan(df["sd"].iloc[names.index("one base[0]")]) and df["bases"].iloc[names.index("one base[0]")] == 1
    assert np.isneginf(df["log.quartile.0%"]).any()   # log 0 is -inf, not an error
    assert st["n_problems"] == len(flat) and st["n_waves"] == 1 and st["n_launches"] == 8
    assert st["rows"] == sum(len(p[2]) for p in flat)
    print("psd_features: %d problems, %d rows, kernels %.2f ms, device %.2f ms, call %.2f s"
          % (len(flat), st["rows"], st["kernel_ms"], st["device_ms"], wall))


@pytest.mark.gpu
def test_features_in_forced_waves_are_identical(gpu, feature_cases):
    names, flat, want = feature_cases
    lib = gpu._lib.lib
    lib.psd_set_option(b"coverage_gb", 0.002)
    try:
        df, st = gpu.problem_features(flat, device=0, return_stats=True)
    finally:
        lib.psd_set_option(b"coverage_gb", 0.0)
    assert st["n_waves"] > 1 and st["n_launches"] == 8 * st["n_waves"]
    assert_bits_equal(df.to_numpy(), want, "waves")


# ---- GPU: end to end ------------------------------------------------------------------------------------

def labelled_problem(seed, depth):
    """A count vector of 2e4 to 5e4 positions with known peaks (background mean 0.1 x depth, peaks 1 x depth,
    300 to 900 bases) and, in the middle of every gap between peaks, a 1,000-base bump of twice the
    background that is not a peak.  Labels: peaks on the peak centres, peakStart / peakEnd at the edges,
    noPeaks on the gaps (bumps included).  A bump's likelihood gain grows with depth (about 39 x depth) and a
    peak's too (420 to 1,260 x depth): at depth 1 the bumps never show at penalties >= 1e2 and the peaks vanish
    above about 1e3, at depth 100 the bumps need penalties above about 4e3, so no constant penalty suits both."""
    from peaksegdisk_b200 import synth
    rng = np.random.default_rng(seed)
    n = int(rng.integers(20000, 50001))
    mu = np.full(n, 0.1 * depth)
    peaks = []
    pos = int(rng.integers(1000, 3000))
    while pos + 1500 < n:
        width = int(rng.integers(300, 900))
        peaks.append((pos, pos + width))
        mu[pos:pos + width] = depth
        pos += width + int(rng.integers(2500, 6000))
    for (_, b), (a, _) in zip(peaks[:-1], peaks[1:]):
        mid = (a + b) // 2
        mu[mid - 500:mid + 500] = 0.2 * depth
    counts = rng.poisson(mu)
    s, e, c = synth.rle_rows(counts)
    ls, le, ann = [], [], []
    prev_end = 0
    for a, b in peaks:
        mid = (a + b) // 2
        ls += [a - 150, mid - 50, b - 150]; le += [a + 150, mid + 50, b + 150]; ann += ["peakStart", "peaks", "peakEnd"]
        if a - 400 > prev_end + 400:
            ls.append(prev_end + 400); le.append(a - 400); ann.append("noPeaks")
        prev_end = b
    if n - 100 > prev_end + 400:
        ls.append(prev_end + 400); le.append(n - 100); ann.append("noPeaks")
    return (s, e, c), pd.DataFrame({"chromStart": ls, "chromEnd": le, "annotation": ann})


def errors_at(models, pen):
    """Label errors of the path model whose [min.lambda, max.lambda] contains pen."""
    m = models[(models["min.lambda"] <= pen) & (pen <= models["max.lambda"])]
    assert len(m) >= 1, pen
    return int(m["errors"].iloc[0])


@pytest.mark.gpu
def test_learned_penalties_beat_the_best_constant_end_to_end(gpu):
    t0 = time.time()
    pen_min = 1e2
    data = [labelled_problem(9000 + i, 1 if i % 4 < 2 else 100) for i in range(96)]   # depths 1, 1, 100, 100, ...
    rows = [d[0] for d in data]
    labels = [d[1] for d in data]
    paths, pst = gpu.model_path_batch(rows, labels, pen_min=pen_min, device=0)
    assert all(p["status"] == 0 and p["target"] is not None for p in paths)
    train, test = np.arange(0, 96, 2), np.arange(1, 96, 2)
    feats = gpu.problem_features(rows, device=0)
    targets = np.log([paths[i]["target"][:2] for i in train])
    model = gpu.IntervalRegressionCV(feats.iloc[train].reset_index(drop=True), targets)
    # the paths cover [pen_min, inf): a prediction below it is raised to it
    pen = np.maximum(np.exp(model.predict(feats.iloc[test].reset_index(drop=True))), pen_min)
    plan = gpu.Plan(0)
    ids = []
    for i, p in zip(test, pen):
        ids.append(plan.add(*rows[i], float(p)))
        plan.set_labels(ids[-1], labels[i])
    plan.run()
    learned = 0
    for pid, i, p in zip(ids, test, pen):
        dev = plan.label_errors(pid)[1]["errors"]
        assert dev == errors_at(paths[i]["models"], p), (i, p)
        learned += dev
    # the best constant penalty on the training paths: the geometric midpoints of all their breakpoints
    bp = np.unique(np.concatenate([paths[i]["models"]["min.lambda"].to_numpy() for i in train]))
    bp = bp[np.isfinite(bp) & (bp >= pen_min)]
    cand = np.concatenate([np.sqrt(bp[:-1] * bp[1:]), [bp[-1] * 2]])
    train_err = np.array([sum(errors_at(paths[i]["models"], p) for i in train) for p in cand])
    const = cand[int(np.argmin(train_err))]
    const_test = sum(errors_at(paths[i]["models"], const) for i in test)
    wall = time.time() - t0
    print("end to end: %d path solves in %d rounds; lambda %.3g of %d; test errors: learned %d, best constant "
          "penalty %.4g %d (train %d); %.1f s" % (pst["solves"], pst["rounds"], model.lambda_, len(model.path), learned,
                                                 const, const_test, train_err.min(), wall))
    assert learned < const_test
