"""Host-side mirror of the reference's R API for the PeakSegFPOP path, on top of the C ABI.

Same names, argument meaning and error behaviour as the R functions (R is not available in the
build image, so this Python layer stands where the R layer stands in the reference):

    PeakSegFPOP_file      R/PeakSegFPOP_file.R:1-86
    PeakSegFPOP_dir       R/PeakSegFPOP_dir.R:1-117     (result cache: _timing.tsv / _loss.tsv / _segments.bed)
    PeakSegFPOP_df        R/PeakSegFPOP_df.R:1-36
    PeakSegFPOP_vec       R/PeakSegFPOP_vec.R:1-26
    sequentialSearch_dir  R/sequentialSearch_dir.R:1-103
    writeBedGraph         R/writeBedGraph.R:1-37
    col_name_list         R/col.name.list.R:10-18

Every solve goes through libpeaksegdisk_b200.so (CUDA); nothing here computes a segmentation.
"""
import ctypes as C
import math
import os
import shutil
import tempfile
import time

import numpy as np
import pandas as pd

from . import _lib

col_name_list = {
    "loss": ["penalty", "segments", "peaks", "bases", "bedGraph.lines", "mean.pen.cost", "total.loss",
             "equality.constraints", "mean.intervals", "max.intervals"],
    "segments": ["chrom", "chromStart", "chromEnd", "status", "mean"],
    "coverage": ["chrom", "chromStart", "chromEnd", "count"],
}


from .rfmt import r_paste  # noqa: E402,F401  (kept importable as api.r_paste)


def writeBedGraph(count_df, coverage_bedGraph):
    """R/writeBedGraph.R:13-37."""
    if not isinstance(count_df, pd.DataFrame):
        raise ValueError("count.df must be data.frame")
    exp_names = ["chrom", "chromStart", "chromEnd", "count"]
    if list(count_df.columns) != exp_names:
        raise ValueError("count.df must have names " + ", ".join(exp_names))
    if not pd.api.types.is_integer_dtype(count_df["chromStart"]):
        raise ValueError("count.df$chromStart must be integer")
    if not pd.api.types.is_integer_dtype(count_df["chromEnd"]):
        raise ValueError("count.df$chromEnd must be integer")
    if not pd.api.types.is_numeric_dtype(count_df["count"]):
        raise ValueError("count.df$count must be numeric")
    if (count_df["chromStart"] < 0).any():
        raise ValueError("count.df$chromStart must always be non-negative")
    if not (count_df["chromStart"] < count_df["chromEnd"]).all():
        raise ValueError("chromStart must be less than chromEnd for all rows of count.df")
    with open(coverage_bedGraph, "w") as f:
        cnt = count_df["count"].to_numpy()
        as_int = pd.api.types.is_integer_dtype(count_df["count"])
        for ch, s, e, c in zip(count_df["chrom"].tolist(), count_df["chromStart"].tolist(),
                               count_df["chromEnd"].tolist(), cnt.tolist()):
            f.write("%s\t%d\t%d\t%s\n" % (ch, s, e, ("%d" % c) if as_int else r_paste(c)))


def _as_numeric(s):
    """R's as.numeric() on a character scalar (NA on failure)."""
    t = s.strip()
    try:
        if t in ("Inf", "inf", "+Inf"):
            return math.inf
        if t == "-Inf":
            return -math.inf
        if t in ("NA", "NaN", ""):
            return math.nan
        return float(t) if not t.lower().startswith("0x") else float(int(t, 16))
    except ValueError:
        return math.nan


def PeakSegFPOP_file(bedGraph_file, pen_str, db_file=None):
    """Run the solver on a bedGraph file and write <file>_penalty=<pen>_segments.bed / _loss.tsv.
    Returns dict(bedGraph.file, penalty, db.file, megabytes) like the R function."""
    if not (isinstance(bedGraph_file, str) and os.path.exists(bedGraph_file)):
        raise ValueError("bedGraph.file=%s must be the name of a data file to segment" % (bedGraph_file,))
    if not isinstance(pen_str, str):
        raise ValueError("pen.str must be a character string that can be converted to a non-negative numeric scalar")
    penalty = _as_numeric(pen_str)
    if not (0 <= penalty <= math.inf):
        raise ValueError("as.numeric(pen.str)=%s but it must be a non-negative numeric scalar"
                         % ("NA" if math.isnan(penalty) else r_paste(penalty)))
    norm_file = os.path.realpath(bedGraph_file)
    if db_file is None:
        db_file = "%s_penalty=%s.db" % (norm_file, pen_str)
    if not isinstance(db_file, str):
        raise ValueError("db.file=%s must be a temporary file name where cost function db can be written" % (db_file,))
    if os.path.isfile(db_file):
        os.unlink(db_file)
    status = _lib.lib.psd_fpop_disk(norm_file.encode(), pen_str.encode(), db_file.encode())
    if status != 0:
        raise RuntimeError(_lib.status_text(status, norm_file, pen_str, db_file))
    megabytes = os.path.getsize(db_file) / 1024 / 1024 if os.path.isfile(db_file) else 0
    if os.path.isfile(db_file):
        os.unlink(db_file)
    loss_tsv = "%s_penalty=%s_loss.tsv" % (bedGraph_file, pen_str)
    if os.path.getsize(loss_tsv) == 0:
        raise RuntimeError("unable to write to loss output file %s (disk is probably full)" % loss_tsv)
    return {"bedGraph.file": norm_file, "penalty": pen_str, "db.file": db_file, "megabytes": megabytes}


def PeakSegFPOP_file_batch(bedGraph_files, pen_strs, db_files=None):
    """Batch form of PeakSegFPOP_file: all problems go to the GPU in one launch (one warp each).
    Returns the list of status codes (0 = ok); raises nothing for per-problem input errors."""
    n = len(bedGraph_files)
    norm = [os.path.realpath(f) for f in bedGraph_files]
    if db_files is None:
        db_files = ["%s_penalty=%s.db" % (f, p) for f, p in zip(norm, pen_strs)]
    arr = lambda xs: (C.c_char_p * n)(*[x.encode() for x in xs])
    status = (C.c_int * n)()
    rc = _lib.lib.psd_fpop_disk_batch(n, arr(norm), arr(pen_strs), arr(db_files), status)
    for d in db_files:
        if os.path.isfile(d):
            os.unlink(d)
    if rc:
        raise RuntimeError("peaksegdisk_b200: " + _lib.status_text(rc))
    return list(status)


def _read_loss(path):
    """One _loss.tsv line.  The %.20g doubles are parsed with Python's float() (correctly rounded;
    pandas' default parser is not): the sequential search derives its next 15-digit penalty string
    from total.loss differences, where one ulp can change the string."""
    with open(path) as f:
        lines = [ln for ln in f.read().split("\n") if ln != ""]
    names = col_name_list["loss"]
    int_cols = {"segments", "peaks", "bases", "bedGraph.lines", "equality.constraints"}
    cols = {n: [] for n in names}
    for ln in lines:
        fields = ln.split("\t")
        if len(fields) != len(names):
            raise ValueError("%s: expected %d tab-separated fields, found %d" % (path, len(names), len(fields)))
        for n, v in zip(names, fields):
            cols[n].append(int(v) if n in int_cols else _as_numeric(v))
    return pd.DataFrame(cols, columns=names)


def _read_segments(path):
    return pd.read_csv(path, sep="\t", header=None, names=col_name_list["segments"])


def _first_last_line(path):
    with open(path, "rb") as f:
        first = f.readline()
        f.seek(0, os.SEEK_END)
        size = f.tell()
        back = min(size, 4096)
        f.seek(size - back)
        tail = f.read().splitlines()
        last = tail[-1] if tail else b""
    return first.decode().rstrip("\n").split("\t"), last.decode().split("\t")


def _already_computed(cov, seg_bed, loss_tsv, timing_tsv):
    """The cache test of R/PeakSegFPOP_dir.R:70-93."""
    try:
        timing = pd.read_csv(timing_tsv, sep="\t", header=None, names=["penalty", "megabytes", "seconds"],
                             float_precision="round_trip")
        loss = _read_loss(loss_tsv)
        fs, ls = _first_last_line(seg_bed)
        fc, lc = _first_last_line(cov)
        if len(timing) != 1 or len(loss) != 1 or len(fs) != 5 or len(ls) != 5:
            return None
        fc = fc if len(fc) == 4 else " ".join(fc).split()
        lc = lc if len(lc) == 4 else " ".join(lc).split()
        consistent = int(fs[2]) - int(ls[1]) == int(loss["bases"][0])
        start_ok = int(fc[1]) == int(ls[1])
        end_ok = int(lc[2]) == int(fs[2])
        if consistent and start_ok and end_ok:
            return timing, loss
    except Exception:
        return None
    return None


def PeakSegFPOP_dir(problem_dir, penalty_param, db_file=None):
    """Solve problem_dir/coverage.bedGraph at one penalty, with the reference's result cache.
    Returns {"segments": DataFrame, "loss": DataFrame(one row, + megabytes, seconds)}."""
    if not (isinstance(problem_dir, str) and os.path.isdir(problem_dir)):
        raise ValueError("problem.dir=%s must be the name of a directory containing a file named coverage.bedGraph"
                         % (problem_dir,))
    ok_type = isinstance(penalty_param, (str, int, float, np.integer, np.floating)) and not isinstance(penalty_param, bool)
    if not ok_type or (not isinstance(penalty_param, str) and math.isnan(float(penalty_param))):
        raise ValueError("penalty.param must be numeric or character, length 1, not missing")
    penalty_str = r_paste(penalty_param)
    cov = os.path.join(problem_dir, "coverage.bedGraph")
    pre = "%s_penalty=%s" % (cov, penalty_str)
    seg_bed, loss_tsv, timing_tsv = pre + "_segments.bed", pre + "_loss.tsv", pre + "_timing.tsv"
    cached = _already_computed(cov, seg_bed, loss_tsv, timing_tsv)
    if cached is None:
        t0 = time.time()
        result = PeakSegFPOP_file(cov, penalty_str, db_file)
        seconds = time.time() - t0
        timing = pd.DataFrame({"penalty": [_as_numeric(penalty_str)], "megabytes": [result["megabytes"]], "seconds": [seconds]})
        with open(timing_tsv, "w") as f:
            f.write("%s\t%s\t%s\n" % (r_paste(timing["penalty"][0]), r_paste(result["megabytes"]), r_paste(seconds)))
        loss = _read_loss(loss_tsv)
    else:
        timing, loss = cached
    segs = _read_segments(seg_bed)
    loss = loss.copy()
    loss["megabytes"] = timing["megabytes"].to_numpy()
    loss["seconds"] = timing["seconds"].to_numpy()
    return {"segments": segs, "loss": loss}


def PeakSegFPOP_df(count_df, pen_num, base_dir=None):
    """R/PeakSegFPOP_df.R: write the data.frame under base_dir/<chrom>-<start>-<end>/ and solve."""
    if not (isinstance(pen_num, (int, float, np.integer, np.floating)) and not isinstance(pen_num, bool)
            and not math.isnan(float(pen_num)) and 0 <= pen_num):
        raise ValueError("pen.num must be non-negative numeric scalar")
    if base_dir is None:
        base_dir = tempfile.gettempdir()
    data_dir = os.path.join(base_dir, "%s-%d-%d" % (count_df["chrom"].iloc[0], int(count_df["chromStart"].min()),
                                                      int(count_df["chromEnd"].max())))
    shutil.rmtree(data_dir, ignore_errors=True)
    os.makedirs(data_dir, exist_ok=True)
    writeBedGraph(count_df, os.path.join(data_dir, "coverage.bedGraph"))
    L = PeakSegFPOP_dir(data_dir, r_paste(pen_num))
    L["data"] = count_df
    return L


def PeakSegFPOP_vec(count_vec, pen_num):
    """R/PeakSegFPOP_vec.R: run-length encode an integer vector and solve."""
    if not (isinstance(pen_num, (int, float, np.integer, np.floating)) and not isinstance(pen_num, bool)
            and not math.isnan(float(pen_num)) and 0 <= pen_num):
        raise ValueError("pen.num must be non-negative numeric scalar")
    v = np.asarray(count_vec)
    if not np.issubdtype(v.dtype, np.integer):
        raise ValueError("count.vec must be integer")
    from .synth import rle_rows
    s, e, c = rle_rows(v)
    df = pd.DataFrame({"chrom": "chrUnknown", "chromStart": s.astype(np.int64), "chromEnd": e.astype(np.int64),
                       "count": c.astype(np.int64)})
    return PeakSegFPOP_df(df, pen_num)


def PeakSegFPOP_vec_batch(count_vecs, pen_nums):
    """Many PeakSegFPOP_vec calls as ONE in-memory batch: no bedGraph files, the count vectors go to
    the device as they are and are run-length encoded there (rle_gpu.cuh).  Returns one dict per
    problem with the `loss` row and `segments` table PeakSegFPOP_vec reports (chrom "chrUnknown")."""
    from .plan import solve_counts_batch
    pens = list(pen_nums)
    for pen_num in pens:
        if not (isinstance(pen_num, (int, float, np.integer, np.floating)) and not isinstance(pen_num, bool)
                and not math.isnan(float(pen_num)) and 0 <= pen_num):
            raise ValueError("pen.num must be non-negative numeric scalar")
    plan, ids = solve_counts_batch(zip(count_vecs, [float(p) for p in pens]))
    out = []
    for pid in ids:
        st, en, pk, mean = plan.segments(pid)
        seg = pd.DataFrame({"chrom": "chrUnknown", "chromStart": st, "chromEnd": en,
                            "status": np.where(pk == 1, "peak", "background"), "mean": mean})
        out.append({"loss": pd.DataFrame([plan.loss_row(pid)]), "segments": seg})
    return out


def coverage_from_reads(reads, region=None, device=-1):
    """Coverage of aligned reads as a bedGraph data.frame, computed on the device (not an R function of
    the reference: its Spatial_correlation vignette builds coverage from reads in R before solving).

    reads: data.frame with columns chrom, chromStart, chromEnd (half-open read intervals, any order;
    other columns are ignored).  region: None (each chromosome's [min chromStart, max chromEnd)) or a
    dict chrom -> (start, end); reads are clipped to their region and reads outside it are ignored, and
    a dict chromosome without reads gives one zero row.  All chromosomes go to the device in one call.
    Returns a data.frame with col_name_list["coverage"] columns, chromosomes in order of first appearance
    (then the dict's other chromosomes), whose rows tile each region: input for writeBedGraph /
    PeakSegFPOP_df / sequentialSearch_dir."""
    from .plan import coverage_rows
    if not isinstance(reads, pd.DataFrame):
        raise ValueError("reads must be data.frame")
    if not all(c in reads.columns for c in ("chrom", "chromStart", "chromEnd")):
        raise ValueError("reads must have columns chrom, chromStart, chromEnd")
    for col in ("chromStart", "chromEnd"):
        if len(reads) and not pd.api.types.is_integer_dtype(reads[col]):
            raise ValueError("reads$%s must be integer" % col)
    if region is not None and not isinstance(region, dict):
        raise ValueError("region must be None or a dict chrom -> (start, end)")
    region = region or {}
    chroms = list(pd.unique(reads["chrom"]))
    seen = set(chroms)
    chroms += [c for c in region if c not in seen]
    groups = reads.groupby("chrom", sort=False).indices if len(reads) else {}
    starts, ends = reads["chromStart"].to_numpy(), reads["chromEnd"].to_numpy()
    problems = []
    for ch in chroms:
        idx = groups.get(ch, np.zeros(0, np.int64))
        s, e = starts[idx], ends[idx]
        if ch in region:
            if len(region[ch]) != 2:
                raise ValueError("region[%r] must be (start, end)" % (ch,))
            a, b = region[ch]
        else:
            a, b = s.min(), e.max()
        problems.append((s, e, a, b))
    rows, _ = coverage_rows(problems, device)
    n = [len(r[2]) for r in rows]
    if not rows:
        return pd.DataFrame({k: pd.Series(dtype=object if k == "chrom" else np.int32) for k in col_name_list["coverage"]})
    return pd.DataFrame({"chrom": np.repeat(np.array(chroms, dtype=object), n),
                         "chromStart": np.concatenate([r[0] for r in rows]),
                         "chromEnd": np.concatenate([r[1] for r in rows]),
                         "count": np.concatenate([r[2] for r in rows])})


def _solve_many(requests):
    """requests: list of (problem_dir, penalty_str).  Everything that is not already cached goes to
    the GPU in ONE batched launch; returns the PeakSegFPOP_dir result of every request."""
    todo = []
    for d, s in requests:
        cov = os.path.join(d, "coverage.bedGraph")
        pre = "%s_penalty=%s" % (cov, s)
        if os.path.exists(cov) and _already_computed(cov, pre + "_segments.bed", pre + "_loss.tsv", pre + "_timing.tsv") is None:
            todo.append((cov, s))
    if len(todo) > 1:
        t0 = time.time()
        st = PeakSegFPOP_file_batch([c for c, _ in todo], [s for _, s in todo])
        seconds = time.time() - t0
        for (cov, s), code in zip(todo, st):
            if code == 0:
                with open("%s_penalty=%s_timing.tsv" % (cov, s), "w") as f:
                    f.write("%s\t0\t%s\n" % (r_paste(_as_numeric(s)), r_paste(seconds)))
    return [PeakSegFPOP_dir(d, s) for d, s in requests]


class _Search:
    """The state machine of R/sequentialSearch_dir.R:31-98 for one problem."""

    def __init__(self, problem_dir, peaks_int):
        self.dir, self.target = problem_dir, peaks_int
        self.models = {}
        self.next_pen = [0.0, math.inf]
        self.iteration = 0
        self.under = self.over = None
        self.candidate = None

    def requests(self):
        return [(self.dir, r_paste(p)) for p in self.next_pen]

    def update(self, fits):
        self.iteration += 1
        next_str = [r_paste(p) for p in self.next_pen]
        for s, L in zip(next_str, fits):
            L["loss"]["iteration"] = self.iteration
            L["loss"]["under"] = np.nan if self.under is None else self.under["peaks"]
            L["loss"]["over"] = np.nan if self.over is None else self.over["peaks"]
            self.models[s] = L
        if self.iteration == 1:
            self.under = self.models["Inf"]["loss"].iloc[0]
            self.over = self.models["0"]["loss"].iloc[0]
            max_peaks = math.floor((self.over["bases"] - 1) / 2)
            if max_peaks < self.target:
                raise ValueError("peaks.int=%d but max=%d peaks for N=%d data" % (self.target, max_peaks, int(self.over["bases"])))
        else:
            m_new = self.models[next_str[0]]["loss"].iloc[0]
            if m_new["peaks"] in (self.under["peaks"], self.over["peaks"]):   # not a new model
                self.candidate = self.under
                self.next_pen = []
            elif m_new["peaks"] < self.target:
                self.under = m_new
            else:
                self.over = m_new
        if self.target == self.under["peaks"]:
            self.candidate = self.under
            self.next_pen = []
        if self.target == self.over["peaks"]:
            self.candidate = self.over
            self.next_pen = []
        if self.next_pen:
            p = (self.over["total.loss"] - self.under["total.loss"]) / (self.under["peaks"] - self.over["peaks"])
            if p < 0:
                self.candidate = self.under
                self.next_pen = []
            else:
                self.next_pen = [float(p)]

    def result(self):
        out = dict(self.models[r_paste(float(self.candidate["penalty"]))])
        others = pd.concat([m["loss"] for m in self.models.values()], ignore_index=True)
        out["others"] = others.sort_values("iteration", kind="stable").reset_index(drop=True)
        return out


def _check_search_args(problem_dir, peaks_int):
    if not (isinstance(peaks_int, (int, np.integer)) and not isinstance(peaks_int, bool) and 0 <= peaks_int):
        raise ValueError("is.integer(peaks.int) && length(peaks.int) == 1 && 0 <= peaks.int is not TRUE")
    if not isinstance(problem_dir, str):
        raise ValueError("is.character(problem.dir) is not TRUE")


def sequentialSearch_dir(problem_dir, peaks_int, verbose=0):
    """R/sequentialSearch_dir.R:22-103: find the model with peaks_int peaks (or the next simpler one)
    by a sequence of penalized solves.  The first two penalties (0, Inf) are solved as one batch
    (the reference runs them through future_lapply)."""
    _check_search_args(problem_dir, peaks_int)
    st = _Search(problem_dir, peaks_int)
    while st.next_pen:
        if verbose:
            print("Next =", ", ".join(r_paste(p) for p in st.next_pen))
        st.update(_solve_many(st.requests()))
    return st.result()


def sequentialSearch_batch(problem_dirs, peaks_int, verbose=0):
    """Many sequential searches advanced in lock step: iteration k of every unfinished problem is one
    batched GPU launch (one warp per (problem, penalty)).  peaks_int: one target or one per problem.
    Returns the list of sequentialSearch_dir results; each problem follows exactly the chain the
    single-problem search would."""
    targets = [peaks_int] * len(problem_dirs) if isinstance(peaks_int, (int, np.integer)) else list(peaks_int)
    for d, t in zip(problem_dirs, targets):
        _check_search_args(d, t)
    states = [_Search(d, t) for d, t in zip(problem_dirs, targets)]
    while True:
        active = [s for s in states if s.next_pen]
        if not active:
            break
        reqs, spans = [], []
        for s in active:
            r = s.requests()
            spans.append((len(reqs), len(reqs) + len(r)))
            reqs.extend(r)
        if verbose:
            print("iteration with %d solves for %d problems" % (len(reqs), len(active)))
        fits = _solve_many(reqs)
        for s, (a, b) in zip(active, spans):
            s.update(fits[a:b])
    return [s.result() for s in states]
