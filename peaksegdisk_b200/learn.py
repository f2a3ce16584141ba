"""Penalty learning: penaltyLearning's IntervalRegressionCV in numpy.

A problem's target interval (model_path_batch) is the range of log penalties whose model makes the
fewest label errors.  IntervalRegressionCV learns a linear function of problem features
(plan.problem_features) whose value falls inside those intervals, so that unlabelled problems get a
predicted penalty exp(predict(features)).  The fit is a small host problem (n problems x at most 36
features): L1-regularised squared-hinge interval regression, solved by FISTA down a path of lambda values,
with lambda chosen by cross-validation.
"""
import math
import numpy as np


def _targets(targets, n):
    t = np.asarray(targets, dtype=np.float64)
    if t.shape != (n, 2):
        raise ValueError("targets must be an n x 2 array of (lower, upper) log penalties, one row per feature row")
    lo, hi = t[:, 0].copy(), t[:, 1].copy()
    for i in range(n):
        if np.isnan(lo[i]) or np.isnan(hi[i]):
            raise ValueError("target row %d is NaN" % i)
        if not (np.isfinite(lo[i]) or np.isfinite(hi[i])):
            raise ValueError("target row %d has no finite limit" % i)
        if lo[i] >= hi[i]:
            raise ValueError("target row %d: lower limit %r is not below the upper limit %r" % (i, lo[i], hi[i]))
    return lo, hi


def _matrix(features):
    """(float64 matrix, column names) of a DataFrame or a 2-D array (names are then column indices)."""
    names = list(features.columns) if hasattr(features, "columns") else None
    X = np.asarray(features, dtype=np.float64)
    if X.ndim != 2:
        raise ValueError("features must be a 2-D table")
    return X, (names if names is not None else list(range(X.shape[1])))


def _slopes(f, lo, hi, margin):
    """Per-row derivative of max(0, lo + margin - f)^2 + max(0, f - hi + margin)^2 (infinite limits give 0)."""
    return 2.0 * (np.maximum(0.0, f - hi + margin) - np.maximum(0.0, lo + margin - f))


def best_intercept(lo, hi, margin=1.0):
    """The exact minimiser over a constant b of sum max(0, lo + margin - b)^2 + max(0, b - hi + margin)^2.
    Its derivative is piecewise linear and non-decreasing, with breakpoints at lo + margin and hi - margin;
    between the two breakpoints where it changes sign the active terms are fixed and the root is the mean
    of their breakpoints."""
    cl = np.sort((lo + margin)[np.isfinite(lo)])   # (c - b)^2 is active for b < c
    ch = np.sort((hi - margin)[np.isfinite(hi)])   # (b - c)^2 is active for b > c
    sum_l = np.concatenate([[0.0], np.cumsum(cl)])
    sum_h = np.concatenate([[0.0], np.cumsum(ch)])

    def active(b):
        i = np.searchsorted(cl, b, "right")
        j = np.searchsorted(ch, b, "left")
        return len(cl) - i + j, sum_l[-1] - sum_l[i] + sum_h[j]

    t = np.unique(np.concatenate([cl, ch]))
    cnt, tot = active(t)
    d = cnt * t - tot   # the derivative at each breakpoint, up to the factor 2 / n; d[0] <= 0 <= d[-1]
    k = int(np.searchsorted(d, 0.0, "left"))
    if k == 0 or d[k] == 0:
        return float(t[k])
    cnt, tot = active(0.5 * (t[k - 1] + t[k]))
    return float(min(max(tot / cnt, t[k - 1]), t[k]))


def lambda_max(Xs, lo, hi, margin=1.0):
    """The smallest lambda at which all weights 0 are optimal for the scaled matrix Xs: the largest
    |gradient| of the loss with respect to a weight, at the best intercept."""
    if Xs.shape[1] == 0:
        return 0.0
    g = _slopes(np.full(len(lo), best_intercept(lo, hi, margin)), lo, hi, margin) / len(lo)
    return float(np.max(np.abs(Xs.T @ g)))


def interval_regression_path(Xs, lo, hi, lambdas, margin=1.0, tol=1e-6, max_iter=200000):
    """Solutions of min (1/n) sum [max(0, lo + margin - f)^2 + max(0, f - hi + margin)^2] + lam ||w||_1
    with f = b + Xs w (b not penalised), for each lam of a decreasing sequence, by FISTA with adaptive
    restart, each warm-started from the one before and the first from w = 0 and the best intercept.  Each
    stops when the largest violation of the optimality conditions (|d/db|; |d/dw_j + lam sign(w_j)| for
    w_j != 0; |d/dw_j| - lam for w_j = 0) is <= tol, and raises RuntimeError if that does not happen
    within max_iter iterations.  Returns (intercepts [k], weights [k, p])."""
    n, p = Xs.shape
    A = np.hstack([np.ones((n, 1)), Xs])
    L = 4.0 / n * float(np.linalg.norm(A, 2)) ** 2   # the loss's Hessian is (2/n) A' D A with D <= 2
    x = np.zeros(p + 1)
    x[0] = best_intercept(lo, hi, margin)
    out = np.zeros((len(lambdas), p + 1))
    for li, lam in enumerate(lambdas):
        thr = lam / L

        def grad(th):
            return A.T @ (_slopes(A @ th, lo, hi, margin) / n)

        def viol(th, g):
            w, gw = th[1:], g[1:]
            nz = w != 0
            v = abs(g[0])
            if nz.any():
                v = max(v, float(np.max(np.abs(gw[nz] + lam * np.sign(w[nz])))))
            if (~nz).any():
                v = max(v, float(np.max(np.abs(gw[~nz]) - lam)))
            return v

        y, t = x.copy(), 1.0
        it = 0
        while viol(x, grad(x)) > tol:
            it += 1
            if it > max_iter:
                raise RuntimeError("interval regression did not reach tol %g at lambda %g in %d iterations" % (tol, lam, max_iter))
            z = y - grad(y) / L
            xn = z.copy()
            xn[1:] = np.sign(z[1:]) * np.maximum(np.abs(z[1:]) - thr, 0.0)
            if np.dot(y - xn, xn - x) > 0:   # the momentum points uphill: restart it
                y, t = xn.copy(), 1.0
            else:
                tn = 0.5 * (1.0 + math.sqrt(1.0 + 4.0 * t * t))
                y = xn + ((t - 1.0) / tn) * (xn - x)
                t = tn
            x = xn
        out[li] = x
    return out[:, 0].copy(), out[:, 1:].copy()


def _errors(f, lo, hi):
    """Predictions outside their closed target interval (non-finite predictions count as errors)."""
    return int(np.sum(~((f >= lo) & (f <= hi))))


class _Scaling:
    """Columns finite on every given row and not constant, centred and scaled by their sample sd."""

    def __init__(self, X):
        finite = np.all(np.isfinite(X), axis=0)
        keep = finite.copy()
        keep[finite] = np.ptp(X[:, finite], axis=0) > 0
        self.keep = np.flatnonzero(keep)
        Xk = X[:, self.keep]
        self.centre = Xk.mean(axis=0)
        self.scale = Xk.std(axis=0, ddof=1)

    def apply(self, X):
        return (X[:, self.keep] - self.centre) / self.scale


class IntervalRegressionCV:
    """L1-regularised interval regression with lambda chosen by cross-validation (penaltyLearning's
    IntervalRegressionCV).

    features: n x p DataFrame (e.g. plan.problem_features) or array.  targets: n x 2 (lower, upper) log
    penalties with lower < upper; either may be infinite, not both (from model_path_batch:
    np.log([p["target"][:2] for p in paths])).

    A column is used only if it is finite on every training row and not constant; it is centred and scaled
    by its sample sd.  The model f = intercept + x~' weights minimises
        (1/n) sum [max(0, lo + margin - f)^2 + max(0, f - hi + margin)^2] + lambda ||weights||_1
    for n_lambda log-spaced lambdas from lambda_max (the smallest lambda at which all weights 0 are optimal)
    down to lambda_max * lambda_ratio, each solved until the optimality conditions hold within tol.  The n
    rows are dealt into n_folds folds by a seeded permutation; each fold chooses its columns and scaling from
    its own training rows and fits the same lambdas; lambda_ is the one with the fewest validation predictions
    outside their interval, summed over folds (ties go to the larger lambda), and the model is the fit on
    all rows at lambda_.

    Attributes: columns (the kept feature names), centre, scale, weights (on the scaled columns),
    intercept, lambda_, lambda_max, folds, path (DataFrame: lambda, validation.errors, train.errors,
    nonzero), path_intercepts and path_weights (the fit on all rows at each lambda)."""

    def __init__(self, features, targets, n_folds=5, seed=0, margin=1.0, n_lambda=50, lambda_ratio=1e-3, tol=1e-6):
        import pandas as pd
        X, names = _matrix(features)
        n = X.shape[0]
        lo, hi = _targets(targets, n)
        if not 2 <= n_folds <= n:
            raise ValueError("n_folds must be in [2, n rows]")
        if not (n_lambda >= 1 and 0 < lambda_ratio <= 1 and margin >= 0 and tol > 0):
            raise ValueError("n_lambda >= 1, 0 < lambda_ratio <= 1, margin >= 0 and tol > 0 are required")
        self.margin, self.tol = float(margin), float(tol)
        sc = _Scaling(X)
        Xs = sc.apply(X)
        self.lambda_max = lambda_max(Xs, lo, hi, margin)
        lambdas = (self.lambda_max * np.logspace(0.0, math.log10(lambda_ratio), n_lambda) if self.lambda_max > 0
                   else np.zeros(1))
        self.folds = np.random.default_rng(seed).permutation(np.arange(n) % n_folds)
        val_err = np.zeros(len(lambdas), np.int64)
        for k in range(n_folds):
            tr, va = self.folds != k, self.folds == k
            fsc = _Scaling(X[tr])
            b, W = interval_regression_path(fsc.apply(X[tr]), lo[tr], hi[tr], lambdas, margin, tol)
            with np.errstate(invalid="ignore", over="ignore"):
                F = b[:, None] + W @ fsc.apply(X[va]).T
            val_err += [_errors(f, lo[va], hi[va]) for f in F]
        b, W = interval_regression_path(Xs, lo, hi, lambdas, margin, tol)
        train_err = [_errors(b[i] + Xs @ W[i], lo, hi) for i in range(len(lambdas))]
        best = int(np.argmin(val_err))   # the first minimum: lambdas decrease, so ties go to the larger
        self.path = pd.DataFrame({"lambda": lambdas, "validation.errors": val_err, "train.errors": train_err,
                                  "nonzero": np.count_nonzero(W, axis=1)})
        self.path_intercepts, self.path_weights = b, W
        self.lambda_ = float(lambdas[best])
        self.columns = [names[j] for j in sc.keep]
        self._index = sc.keep
        self._names = names
        self.centre, self.scale = sc.centre, sc.scale
        self.weights, self.intercept = W[best].copy(), float(b[best])

    def predict(self, features):
        """Log penalties of the rows of features (a DataFrame with the training columns, or an array with
        the training column order).  A row with a non-finite value in a kept column raises ValueError."""
        if hasattr(features, "columns"):
            missing = [c for c in self.columns if c not in features.columns]
            if missing:
                raise ValueError("features lack the columns %s" % missing)
            Xk = np.asarray(features[self.columns], dtype=np.float64)
        else:
            X, _ = _matrix(features)
            if X.shape[1] != len(self._names):
                raise ValueError("features need %d columns, got %d" % (len(self._names), X.shape[1]))
            Xk = X[:, self._index]
        bad = np.flatnonzero(~np.all(np.isfinite(Xk), axis=1))
        if len(bad):
            raise ValueError("feature row %d has a non-finite value in a column the model uses" % bad[0])
        return self.intercept + ((Xk - self.centre) / self.scale) @ self.weights
