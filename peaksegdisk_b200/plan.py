"""Batched in-memory solves: many (rows, penalty) problems in one launch, one warp per problem."""
import ctypes as C
import math
import numpy as np
from . import _lib

LOSS_COLUMNS = ["penalty", "segments", "peaks", "bases", "bedGraph.lines", "mean.pen.cost", "total.loss",
                "equality.constraints", "mean.intervals", "max.intervals"]   # R/col.name.list.R:12-15
SEGMENT_COLUMNS = ["chrom", "chromStart", "chromEnd", "status", "mean"]     # R/col.name.list.R:16
LABEL_KINDS = {"noPeaks": 0, "peaks": 1, "peakStart": 2, "peakEnd": 3}      # PeakError's annotations
PATH_ERROR_COLUMNS = ["fp", "fn", "possible.fp", "possible.fn", "errors"]


def _i32(a):
    a = np.asarray(a)
    if a.dtype != np.int32 and a.size and np.issubdtype(a.dtype, np.integer):
        if int(a.max()) > 2147483647 or int(a.min()) < -2147483648:   # R integers are 32-bit; do not wrap silently
            raise ValueError("values do not fit a 32-bit integer")
    a = np.ascontiguousarray(a, dtype=np.int32)
    return a, a.ctypes.data_as(C.POINTER(C.c_int32))


def _coords(a, what):
    """int32 view of a coordinate array; non-integer or out-of-int32 values raise ValueError."""
    a = np.asarray(a)
    if a.size and not np.issubdtype(a.dtype, np.integer):
        raise ValueError("%s must be integer" % what)
    return _i32(a)


def _coord(x, what):
    if isinstance(x, bool) or not isinstance(x, (int, np.integer)):
        raise ValueError("%s must be an integer" % what)
    if not -2147483648 <= int(x) <= 2147483647:
        raise ValueError("%s does not fit a 32-bit integer" % what)
    return int(x)


class Plan:
    """A batch of independent problems.  add() copies rows to the host side of the plan;
    upload()/solve()/download() are the three timed phases; run() does all three."""

    def __init__(self, device=-1):
        self._h = _lib.lib.psd_plan_create(int(device))
        if not self._h:
            raise RuntimeError("peaksegdisk_b200: cannot create a plan: " + _lib.lib.psd_last_error().decode())

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib.psd_plan_destroy(self._h)
            self._h = None

    __del__ = close

    def __len__(self):
        return _lib.lib.psd_plan_size(self._h)

    def add(self, chrom_start, chrom_end, coverage, penalty):
        s, sp = _i32(chrom_start)
        e, ep = _i32(chrom_end)
        c, cp = _i32(coverage)
        if not (len(s) == len(e) == len(c)):
            raise ValueError("chromStart, chromEnd and coverage must have the same length")
        is_inf = 1 if (isinstance(penalty, float) and math.isinf(penalty) and penalty > 0) else 0
        pid = _lib.lib.psd_plan_add(self._h, len(c), sp, ep, cp, 0.0 if is_inf else float(penalty), is_inf)
        if pid < 0:
            raise ValueError(_lib.status_text(-pid, penalty=str(penalty)))
        return pid

    def add_counts(self, counts, penalty):
        """One problem from a count vector (counts[i] = coverage of base [i, i+1)); the run-length
        encoding into rows happens on the device at upload (R/PeakSegFPOP_vec.R:18-25 does it in R)."""
        v = np.asarray(counts)
        if not np.issubdtype(v.dtype, np.integer):
            raise ValueError("count.vec must be integer")
        c, cp = _i32(v)
        is_inf = 1 if (isinstance(penalty, float) and math.isinf(penalty) and penalty > 0) else 0
        pid = _lib.lib.psd_plan_add_counts(self._h, len(c), cp, 0.0 if is_inf else float(penalty), is_inf)
        if pid < 0:
            raise ValueError(_lib.status_text(-pid, penalty=str(penalty)))
        return pid

    def set_penalty(self, pid, penalty):
        is_inf = 1 if (math.isinf(penalty) and penalty > 0) else 0
        rc = _lib.lib.psd_plan_set_penalty(self._h, pid, 0.0 if is_inf else float(penalty), is_inf)
        if rc:
            raise ValueError(_lib.status_text(rc, penalty=str(penalty)))

    def set_labels(self, pid, labels):
        """Labels of problem pid: a DataFrame (or dict) with columns chromStart, chromEnd and annotation
        (noPeaks / peaks / peakStart / peakEnd), 0-based half-open.  They are scored on the device by
        every later solve (label_errors)."""
        s, e, k = label_arrays(labels)
        p32 = C.POINTER(C.c_int32)
        rc = _lib.lib.psd_plan_set_labels(self._h, pid, len(k), s.ctypes.data_as(p32), e.ctypes.data_as(p32), k.ctypes.data_as(p32))
        if rc:
            raise ValueError("peaksegdisk_b200: " + _lib.status_text(rc))
        if not hasattr(self, "_labels"):
            self._labels = {}
        self._labels[pid] = (s, e, k)

    def label_errors(self, pid):
        """Label errors of problem pid's last solve: (DataFrame with one row per label -- chromStart,
        chromEnd, annotation, fp, fn, possible.fp, possible.fn -- and a dict of the totals fp, fn,
        possible.fp, possible.fn, errors)."""
        import pandas as pd
        if pid not in getattr(self, "_labels", {}):
            raise ValueError("peaksegdisk_b200: problem %d has no labels" % pid)
        s, e, k = self._labels[pid]
        fp = np.zeros(len(k), np.int32); fn = np.zeros(len(k), np.int32)
        tot = _lib.PsdLabelErrors()
        p32 = C.POINTER(C.c_int32)
        rc = _lib.lib.psd_plan_label_errors(self._h, pid, C.byref(tot), fp.ctypes.data_as(p32), fn.ctypes.data_as(p32))
        if rc:
            raise (ValueError if rc == 111 else RuntimeError)("peaksegdisk_b200: " + _lib.status_text(rc))
        names = np.array(list(LABEL_KINDS))
        df = pd.DataFrame({"chromStart": s, "chromEnd": e, "annotation": names[k], "fp": fp, "fn": fn,
                           "possible.fp": (k != 1).astype(np.int32), "possible.fn": (k != 0).astype(np.int32)})
        return df, {"fp": tot.fp, "fn": tot.fn, "possible.fp": tot.possible_fp, "possible.fn": tot.possible_fn,
                    "errors": tot.errors}

    def _call(self, fn, stream):
        rc = fn(self._h, C.c_void_p(int(stream) if stream else 0))
        if rc:
            raise RuntimeError("peaksegdisk_b200: " + _lib.status_text(rc))

    def upload(self, stream=0):
        self._call(_lib.lib.psd_plan_upload, stream)

    def solve(self, stream=0):
        self._call(_lib.lib.psd_plan_solve, stream)

    def download(self, stream=0):
        self._call(_lib.lib.psd_plan_download, stream)

    def run(self, stream=0):
        self._call(_lib.lib.psd_plan_run, stream)

    def result(self, pid):
        r = _lib.PsdResult()
        rc = _lib.lib.psd_plan_result(self._h, pid, C.byref(r))
        if rc:
            raise RuntimeError(_lib.status_text(rc))
        return r

    def loss_row(self, pid):
        """The 10 fields of _loss.tsv as a dict (R/col.name.list.R:12-15)."""
        r = self.result(pid)
        if r.status:
            raise RuntimeError("peaksegdisk_b200: " + _lib.status_text(r.status))
        vals = [r.penalty, r.n_segments, r.n_peaks, int(r.bases), r.n_rows, r.mean_pen_cost, r.total_loss,
                r.n_equality, r.mean_intervals, r.max_intervals]
        return dict(zip(LOSS_COLUMNS, vals))

    def segments(self, pid):
        """(chromStart, chromEnd, is_peak, mean) arrays, last segment first as in _segments.bed."""
        r = self.result(pid)
        if r.status:
            raise RuntimeError("peaksegdisk_b200: " + _lib.status_text(r.status))
        n = r.n_segments
        s = np.zeros(n, np.int32); e = np.zeros(n, np.int32); k = np.zeros(n, np.int32); m = np.zeros(n)
        rc = _lib.lib.psd_plan_segments(self._h, pid, s.ctypes.data_as(C.POINTER(C.c_int32)),
                                        e.ctypes.data_as(C.POINTER(C.c_int32)), k.ctypes.data_as(C.POINTER(C.c_int32)),
                                        m.ctypes.data_as(C.POINTER(C.c_double)))
        if rc:
            raise RuntimeError(_lib.status_text(rc))
        return s, e, k, m

    def store_function(self, pid, row, which, cap=65536):
        """The stored cost function `which` (0 up, 1 down) of row `row`: (max_log_mean, data_i,
        prev_log_mean) arrays, the fields of the reference's db record (src/PeakSegFPOPLog.cpp:18-34)."""
        n = C.c_int32(0)
        hi = np.zeros(cap); bi = np.zeros(cap, np.int32); bx = np.zeros(cap)
        rc = _lib.lib.psd_plan_store_function(self._h, pid, row, which, cap, C.byref(n), hi.ctypes.data_as(C.POINTER(C.c_double)),
                                              bi.ctypes.data_as(C.POINTER(C.c_int32)), bx.ctypes.data_as(C.POINTER(C.c_double)))
        if rc:
            raise RuntimeError(_lib.status_text(rc))
        return hi[:n.value].copy(), bi[:n.value].copy(), bx[:n.value].copy()

    def stats(self):
        st = _lib.PsdStats()
        _lib.lib.psd_plan_get_stats(self._h, C.byref(st))
        return {name: getattr(st, name) for name, _ in st._fields_}


def solve_batch(problems, device=-1, stream=0):
    """problems: iterable of (chromStart, chromEnd, coverage, penalty).  Returns (plan, ids)."""
    plan = Plan(device)
    ids = [plan.add(s, e, c, pen) for (s, e, c, pen) in problems]
    plan.run(stream)
    return plan, ids


def solve_counts_batch(problems, device=-1, stream=0):
    """problems: iterable of (count_vector, penalty): the in-memory form of PeakSegFPOP_vec for many
    vectors at once; the vectors are run-length encoded on the device.  Returns (plan, ids)."""
    plan = Plan(device)
    ids = [plan.add_counts(v, pen) for (v, pen) in problems]
    plan.run(stream)
    return plan, ids


def coverage_rows(problems, device=-1):
    """problems: iterable of (read_start, read_end, region_start, region_end), reads half-open and in any
    order.  The per-base coverage of each region and its run-length encoding into rows, computed on the
    device in ONE psd_coverage_from_reads call (coverage_gpu.cuh).  Returns (rows, stats): rows[i] is
    problem i's (chromStart, chromEnd, count) int32 arrays, which tile [region_start, region_end);
    stats is the call's psd_coverage_stats as a dict."""
    problems = list(problems)
    arr = (_lib.PsdReads * max(1, len(problems)))()
    keep = []   # the int32 copies must outlive the call
    for i, (rs, re_, a, b) in enumerate(problems):
        s, sp = _coords(rs, "read_start")
        e, ep = _coords(re_, "read_end")
        if len(s) != len(e):
            raise ValueError("read_start and read_end must have the same length")
        keep += [s, e]
        arr[i].n_reads = len(s); arr[i].read_start = sp; arr[i].read_end = ep
        arr[i].region_start = _coord(a, "region_start"); arr[i].region_end = _coord(b, "region_end")
    h = C.c_void_p()
    rc = _lib.lib.psd_coverage_from_reads(int(device), len(problems), arr, C.byref(h))
    if rc:
        raise (ValueError if rc == 111 else RuntimeError)("peaksegdisk_b200: " + _lib.status_text(rc))
    try:
        rows = []
        for i in range(len(problems)):
            n = _lib.lib.psd_coverage_n_rows(h, i)
            s = np.empty(n, np.int32); e = np.empty(n, np.int32); c = np.empty(n, np.int32)
            p32 = C.POINTER(C.c_int32)
            _lib.lib.psd_coverage_rows(h, i, s.ctypes.data_as(p32), e.ctypes.data_as(p32), c.ctypes.data_as(p32))
            rows.append((s, e, c))
        st = _lib.PsdCoverageStats()
        _lib.lib.psd_coverage_get_stats(h, C.byref(st))
        return rows, {name: getattr(st, name) for name, _ in st._fields_}
    finally:
        _lib.lib.psd_coverage_free(h)


def solve_reads_batch(problems, device=-1, stream=0):
    """problems: iterable of (read_start, read_end, region_start, region_end, penalty): aligned reads in,
    segmentations out.  One coverage call for all problems (coverage_rows), then Plan.add on each
    problem's rows and one run.  Returns (plan, ids)."""
    problems = list(problems)
    rows, _ = coverage_rows([p[:4] for p in problems], device)
    plan = Plan(device)
    ids = [plan.add(s, e, c, p[4]) for (s, e, c), p in zip(rows, problems)]
    plan.run(stream)
    return plan, ids


FEATURE_NAMES = ["quartile.0%", "quartile.25%", "quartile.50%", "quartile.75%", "quartile.100%", "mean", "sd",
                 "bases", "data"]   # PeakSegPipeline's problem.features
FEATURE_COLUMNS = FEATURE_NAMES + [pre + f for pre in ("log+1.", "log.", "log.log.") for f in FEATURE_NAMES]


def problem_features(problems, device=-1, return_stats=False):
    """problems: iterable of (chromStart, chromEnd, coverage) rows.  The coverage statistics of each
    problem's per-base vector (each row repeated chromEnd - chromStart times), computed on the device in
    ONE psd_features call without expanding the rows (features_gpu.cuh).  Returns a DataFrame with one
    row per problem and 36 columns: quartile.0% .. quartile.100% (R's type 7), mean, sd (NaN for one
    base), bases and data (rows), then the same nine with the prefixes log+1., log. and log.log. (-inf for
    the log of 0, NaN for the log of a negative).  With return_stats, also the call's psd_features_stats
    as a dict."""
    import pandas as pd
    problems = list(problems)
    arr = (_lib.PsdRows * max(1, len(problems)))()
    keep = []   # the int32 copies must outlive the call
    for i, (s, e, c) in enumerate(problems):
        s, sp = _i32(s)
        e, ep = _i32(e)
        c, cp = _i32(c)
        if not (len(s) == len(e) == len(c)):
            raise ValueError("chromStart, chromEnd and coverage must have the same length")
        keep += [s, e, c]
        arr[i].n_rows = len(c); arr[i].chromStart = sp; arr[i].chromEnd = ep; arr[i].coverage = cp
    out = (_lib.PsdProblemFeatures * max(1, len(problems)))()
    st = _lib.PsdFeaturesStats()
    rc = _lib.lib.psd_features(int(device), len(problems), arr, out, C.byref(st))
    if rc in (111, 6):   # PSD_ERR_ARG, PSD_ERR_INCONSISTENT_CHROMSTART_CHROMEND: the message names the problem
        raise ValueError("peaksegdisk_b200: " + _lib.lib.psd_last_error().decode())
    if rc:
        raise RuntimeError("peaksegdisk_b200: " + _lib.status_text(rc))
    a = np.ctypeslib.as_array(out)[:len(problems)]
    base = np.column_stack([a["quartile"].reshape(-1, 5), a["mean"], a["sd"], a["bases"].astype(np.float64),
                            a["rows"].astype(np.float64)]) if len(problems) else np.zeros((0, 9))
    with np.errstate(divide="ignore", invalid="ignore"):
        x = np.hstack([base, np.log(base + 1), np.log(base), np.log(np.log(base))])
    df = pd.DataFrame(x, columns=FEATURE_COLUMNS)
    if return_stats:
        return df, {name: getattr(st, name) for name, _ in st._fields_}
    return df


def label_arrays(labels):
    """(chromStart, chromEnd, kind) int32 arrays of a label table with columns chromStart, chromEnd and
    annotation (noPeaks / peaks / peakStart / peakEnd; kind 0..3 in that order)."""
    try:
        ann = list(labels["annotation"])
        s, _ = _coords(labels["chromStart"], "chromStart")
        e, _ = _coords(labels["chromEnd"], "chromEnd")
    except KeyError as err:
        raise ValueError("labels need the columns chromStart, chromEnd and annotation") from err
    bad = [a for a in ann if a not in LABEL_KINDS]
    if bad:
        raise ValueError("label annotation %r is not one of %s" % (bad[0], ", ".join(LABEL_KINDS)))
    if not len(s) == len(e) == len(ann):
        raise ValueError("chromStart, chromEnd and annotation must have the same length")
    return s, e, np.array([LABEL_KINDS[a] for a in ann], np.int32)


def model_path_batch(problems, labels=None, pen_min=0.0, pen_max=math.inf, device=-1):
    """Every model that is optimal for some penalty in [pen_min, pen_max], for each problem
    (chromStart, chromEnd, coverage), in one psd_model_path call: the pending crossing penalties of all
    problems are solved together, one batched solve per round (CROPS).  labels: None, or one label
    DataFrame (or None) per problem; label errors are counted on the device.

    Returns (paths, stats).  paths[i] is {"models": DataFrame, "target": (min.lambda, max.lambda, errors)
    or None}; the models are sorted by peaks, with penaltyLearning::modelSelection's columns (min.lambda,
    max.lambda, min.log.lambda, max.log.lambda, penalty, peaks, segments, total.loss) and, for a problem
    with labels, fp, fn, possible.fp, possible.fn and errors.  A problem whose solve failed has
    {"status": code, "models": None, "target": None}.  stats is the call's psd_path_stats as a dict."""
    import pandas as pd
    problems = list(problems)
    if labels is None:
        labels = [None] * len(problems)
    labels = list(labels)
    if len(labels) != len(problems):
        raise ValueError("labels needs one entry (a DataFrame or None) per problem")
    arr = (_lib.PsdPathProblem * max(1, len(problems)))()
    keep = []   # the int32 copies must outlive the call
    p32 = C.POINTER(C.c_int32)
    for i, ((s, e, c), lab) in enumerate(zip(problems, labels)):
        s, sp = _i32(s)
        e, ep = _i32(e)
        c, cp = _i32(c)
        if not (len(s) == len(e) == len(c)):
            raise ValueError("chromStart, chromEnd and coverage must have the same length")
        keep += [s, e, c]
        arr[i].n_rows = len(c); arr[i].chromStart = sp; arr[i].chromEnd = ep; arr[i].coverage = cp
        if lab is not None:
            ls, le, lk = label_arrays(lab)
            keep += [ls, le, lk]
            arr[i].n_labels = len(lk)
            arr[i].label_start = ls.ctypes.data_as(p32); arr[i].label_end = le.ctypes.data_as(p32)
            arr[i].label_kind = lk.ctypes.data_as(p32)
    h = C.c_void_p()
    rc = _lib.lib.psd_model_path(int(device), len(problems), arr, float(pen_min), float(pen_max), C.byref(h))
    if rc:
        raise (ValueError if rc == 111 else RuntimeError)("peaksegdisk_b200: " + _lib.status_text(rc))
    try:
        paths = []
        for i in range(len(problems)):
            st = _lib.lib.psd_path_status(h, i)
            if st:
                paths.append({"status": st, "models": None, "target": None})
                continue
            n = _lib.lib.psd_path_n_models(h, i)
            m = (_lib.PsdPathModel * n)()
            _lib.lib.psd_path_models(h, i, m)
            a = np.ctypeslib.as_array(m)
            lo, hi = a["min_lambda"].copy(), a["max_lambda"].copy()
            with np.errstate(divide="ignore"):
                cols = {"min.lambda": lo, "max.lambda": hi, "min.log.lambda": np.log(lo), "max.log.lambda": np.log(hi),
                        "penalty": a["penalty"].copy(), "peaks": a["peaks"].astype(np.int64),
                        "segments": a["segments"].astype(np.int64), "total.loss": a["total_loss"].copy()}
            target = None
            if labels[i] is not None:
                for col, f in zip(PATH_ERROR_COLUMNS, ["fp", "fn", "possible_fp", "possible_fn", "errors"]):
                    cols[col] = a[f].astype(np.int64)
                tlo, thi, terr = C.c_double(), C.c_double(), C.c_int32()
                _lib.lib.psd_path_target(h, i, C.byref(tlo), C.byref(thi), C.byref(terr))
                if terr.value >= 0:
                    target = (tlo.value, thi.value, terr.value)
            paths.append({"status": 0, "models": pd.DataFrame(cols), "target": target})
        st = _lib.PsdPathStats()
        _lib.lib.psd_path_get_stats(h, C.byref(st))
        return paths, {name: getattr(st, name) for name, _ in st._fields_}
    finally:
        _lib.lib.psd_path_free(h)


JOINT_COLUMNS = ["peaks", "total.loss", "peakStart", "peakEnd", "selectable", "min.lambda", "max.lambda",
                 "min.log.lambda", "max.log.lambda"]


def joint_models_batch(problems, bin_bases=1, labels=None, device=-1):
    """Exact joint single-peak models (the model of PeakSegJoint: one peak shared by position, per-sample
    means, the number of peaked samples as the complexity) of many regions in ONE psd_joint_models call.
    problems: per region, a list with one (chromStart, chromEnd, coverage) per sample; the region is sample 0's
    [first chromStart, last chromEnd), and every sample's rows must tile it.  bin_bases: the grid's bin width
    (peak ends are on bin boundaries).  labels: None or, per problem, a list with one label DataFrame (or None)
    per sample; label errors are summed over samples.

    Returns (results, stats).  results[i] is {"models": DataFrame, "in_peak": bool array (models x samples),
    "target": (min.lambda, max.lambda, errors) or None}; the models, one per k that has one (k ascending), have
    the columns peaks (k), total.loss, peakStart, peakEnd (-1 for k = 0), selectable, min.lambda, max.lambda,
    min.log.lambda, max.log.lambda (NaN when not selectable) and, with labels, fp, fn, possible.fp, possible.fn
    and errors.  stats is the call's psd_joint_stats as a dict."""
    import pandas as pd
    problems = [list(p) for p in problems]
    if labels is None:
        labels = [None] * len(problems)
    labels = list(labels)
    if len(labels) != len(problems):
        raise ValueError("labels needs one entry (a list per sample, or None) per problem")
    arr = (_lib.PsdJointProblem * max(1, len(problems)))()
    keep = []   # the int32 copies and sample arrays must outlive the call
    p32 = C.POINTER(C.c_int32)
    has_labels = []
    for i, (samples, lab) in enumerate(zip(problems, labels)):
        if lab is not None:
            lab = list(lab)
            if len(lab) != len(samples):
                raise ValueError("problem %d: labels needs one entry (a DataFrame or None) per sample" % i)
        sa = (_lib.PsdJointSample * max(1, len(samples)))()
        keep.append(sa)
        for j, (s, e, c) in enumerate(samples):
            s, sp = _i32(s)
            e, ep = _i32(e)
            c, cp = _i32(c)
            if not (len(s) == len(e) == len(c)):
                raise ValueError("problem %d sample %d: chromStart, chromEnd and coverage must have the same length" % (i, j))
            keep += [s, e, c]
            sa[j].n_rows = len(c); sa[j].chromStart = sp; sa[j].chromEnd = ep; sa[j].coverage = cp
            if lab is not None and lab[j] is not None:
                ls, le, lk = label_arrays(lab[j])
                keep += [ls, le, lk]
                sa[j].n_labels = len(lk)
                sa[j].label_start = ls.ctypes.data_as(p32); sa[j].label_end = le.ctypes.data_as(p32)
                sa[j].label_kind = lk.ctypes.data_as(p32)
        s0 = samples[0] if samples else None
        if s0 is not None and len(s0[0]):
            arr[i].region_start = int(s0[0][0]); arr[i].region_end = int(s0[1][-1])
        arr[i].bin_bases = int(bin_bases); arr[i].n_samples = len(samples); arr[i].samples = sa
        has_labels.append(lab is not None and any(x is not None for x in lab))
    h = C.c_void_p()
    rc = _lib.lib.psd_joint_models(int(device), len(problems), arr, C.byref(h))
    if rc == 111:
        raise ValueError("peaksegdisk_b200: " + _lib.lib.psd_last_error().decode())
    if rc:
        raise RuntimeError("peaksegdisk_b200: " + _lib.status_text(rc))
    try:
        out = []
        for i in range(len(problems)):
            n = _lib.lib.psd_joint_n_models(h, i)
            m = (_lib.PsdJointModel * n)()
            _lib.lib.psd_joint_model_table(h, i, m)
            a = np.ctypeslib.as_array(m)
            lo, hi = a["min_lambda"].copy(), a["max_lambda"].copy()
            with np.errstate(divide="ignore"):
                cols = {"peaks": a["peaks"].astype(np.int64), "total.loss": a["total_loss"].copy(),
                        "peakStart": a["peak_start"].astype(np.int64), "peakEnd": a["peak_end"].astype(np.int64),
                        "selectable": a["selectable"] != 0, "min.lambda": lo, "max.lambda": hi,
                        "min.log.lambda": np.log(lo), "max.log.lambda": np.log(hi)}
            S = len(problems[i])
            flags = np.zeros((n, S), np.uint8)
            for r in range(n):
                _lib.lib.psd_joint_samples(h, i, int(a["peaks"][r]), flags[r].ctypes.data_as(C.POINTER(C.c_uint8)))
            target = None
            if has_labels[i]:
                for col, f in zip(PATH_ERROR_COLUMNS, ["fp", "fn", "possible_fp", "possible_fn", "errors"]):
                    cols[col] = a[f].astype(np.int64)
                tlo, thi, terr = C.c_double(), C.c_double(), C.c_int32()
                _lib.lib.psd_joint_target(h, i, C.byref(tlo), C.byref(thi), C.byref(terr))
                if terr.value >= 0:
                    target = (tlo.value, thi.value, terr.value)
            out.append({"models": pd.DataFrame(cols), "in_peak": flags.astype(bool), "target": target})
        st = _lib.PsdJointStats()
        _lib.lib.psd_joint_get_stats(h, C.byref(st))
        return out, {name: getattr(st, name) for name, _ in st._fields_}
    finally:
        _lib.lib.psd_joint_free(h)
