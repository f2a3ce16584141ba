"""Host restatements of the model-path feature, the references its tests compare against:
label errors (PeakError semantics, 0-based half-open) in numpy and by brute force, and the CROPS driver
of psd_model_path over any solver (the parity oracle in the tests and in tools/make_golden_path.py)."""
import math

import numpy as np

KINDS = {"noPeaks": 0, "peaks": 1, "peakStart": 2, "peakEnd": 3}


def peaks_of(start, end, is_peak):
    """(peak starts, peak ends), ascending, of segments given in any order."""
    start, end, is_peak = (np.asarray(a) for a in (start, end, is_peak))
    k = np.flatnonzero(is_peak != 0)
    o = np.argsort(start[k], kind="stable")
    return start[k][o].astype(np.int64), end[k][o].astype(np.int64)


def label_errors(ps, pe, ls, le, kind):
    """Per-label (fp, fn) int arrays for peaks [ps, pe) (ascending, disjoint) and labels [ls, le) of kind 0..3."""
    ls, le, kind = (np.asarray(a, np.int64) for a in (ls, le, kind))
    # o: ps < le and pe > ls; a: ls <= ps < le; b: ls < pe <= le
    o = np.searchsorted(ps, le, "left") - np.searchsorted(pe, ls, "right")
    o = np.maximum(o, 0)
    a = np.searchsorted(ps, le, "left") - np.searchsorted(ps, ls, "left")
    b = np.searchsorted(pe, le, "right") - np.searchsorted(pe, ls, "right")
    c = np.where(kind == 2, a, b)
    fp = np.where(kind == 0, o > 0, np.where(kind == 1, False, c > 1))
    fn = np.where(kind == 0, False, np.where(kind == 1, o == 0, c == 0))
    return fp.astype(np.int32), fn.astype(np.int32)


def label_errors_brute(ps, pe, ls, le, kind):
    """The same, label by label and peak by peak."""
    fp, fn = [], []
    for s, e, k in zip(ls, le, kind):
        o = sum(1 for a, b in zip(ps, pe) if a < e and s < b)
        na = sum(1 for a in ps if s <= a < e)
        nb = sum(1 for b in pe if s < b <= e)
        if k == 0:
            fp.append(int(o > 0)); fn.append(0)
        elif k == 1:
            fp.append(0); fn.append(int(o == 0))
        else:
            c = na if k == 2 else nb
            fp.append(int(c > 1)); fn.append(int(c == 0))
    return np.array(fp, np.int32), np.array(fn, np.int32)


def crops(solve_round, pen_min, pen_max):
    """psd_model_path's rules (model_path.cpp) over solve_round(penalties) -> [(peaks, total_loss,
    segments), ...], called once per round.  Returns (models sorted by peaks ascending, each a dict with
    min.lambda, max.lambda, penalty, peaks, segments, total.loss; rounds; solves)."""
    rounds, solves = 0, 0
    found, closed, pending = [], [], []

    def model(pen, r):
        return {"penalty": pen, "peaks": r[0], "total.loss": r[1], "segments": r[2]}

    def add_pair(i, j):
        mi, mj = found[i], found[j]
        lam = (mj["total.loss"] - mi["total.loss"]) / float(mi["peaks"] - mj["peaks"])
        if not math.isfinite(lam) or lam < pen_min or lam > pen_max:
            closed.append((i, j, min(max(lam, pen_min), pen_max)))
        else:
            pending.append((i, j, lam))

    pens = [pen_min] if pen_min == pen_max else [pen_min, pen_max]
    res = solve_round(pens)
    rounds, solves = 1, len(pens)
    a = model(pen_min, res[0])
    found.append(a)
    if len(pens) == 2 and res[1][0] != a["peaks"]:
        found.append(model(pen_max, res[1]))
        if a["peaks"] > found[1]["peaks"]:
            add_pair(0, 1)
        else:
            add_pair(1, 0)
    while pending:
        todo, pending = pending, []
        res = solve_round([lam for _, _, lam in todo])
        rounds += 1
        solves += len(todo)
        for (i, j, lam), r in zip(todo, res):
            k = model(lam, r)
            mi, mj = found[i], found[j]
            if mj["peaks"] < k["peaks"] < mi["peaks"] and k["total.loss"] + lam * k["peaks"] < mi["total.loss"] + lam * mi["peaks"]:
                found.append(k)
                add_pair(i, len(found) - 1)
                add_pair(len(found) - 1, j)
            else:
                closed.append((i, j, lam))
    for i, j, lam in closed:
        found[i]["max.lambda"] = lam
        found[j]["min.lambda"] = lam
    max(found, key=lambda m: m["peaks"])["min.lambda"] = pen_min
    min(found, key=lambda m: m["peaks"])["max.lambda"] = pen_max
    return sorted(found, key=lambda m: m["peaks"]), rounds, solves


def target_interval(min_lambda, max_lambda, errors):
    """(min.lambda, max.lambda, errors) of the widest run, in log penalty, of consecutive models (sorted
    by peaks ascending) with the fewest errors; runs reaching 0 or infinity are infinitely wide; ties go
    to the smaller min.lambda."""
    errors = np.asarray(errors)
    best = errors.min()
    out, best_w = None, -1.0
    a = 0
    while a < len(errors):
        if errors[a] != best:
            a += 1
            continue
        b = a
        while b + 1 < len(errors) and errors[b + 1] == best:
            b += 1
        hi, lo = float(max_lambda[a]), float(min_lambda[b])
        w = math.inf if (lo == 0 or math.isinf(hi)) else math.log(hi) - math.log(lo)
        if out is None or w > best_w or (w == best_w and lo < out[0]):
            out, best_w = (lo, hi, int(best)), w
        a = b + 1
    return out


def oracle_round(s, e, c):
    """solve_round for crops() over the parity oracle on rows (s, e, c)."""
    import oracle_bind

    def solve_round(pens):
        out = []
        for p in pens:
            st, summ, _ = oracle_bind.solve_rows(s, e, c, p)
            assert st == 0, st
            out.append((int(summ[2]), float(summ[6]), int(summ[1])))
        return out
    return solve_round
