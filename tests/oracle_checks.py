"""Device results against the parity oracle, shared by the GPU test modules: every output of a solved
problem (check_vs_oracle) and the cost-function store row by row against a DiskVector db
(assert_store_equals_db), with the problems the store comparison runs on (store_problems)."""
import os
import numpy as np
import oracle_bind
from helpers import GOLD, parse_reference_db

LOSS_RTOL = 1e-9   # north_star tolerance for the fp64 total loss


def check_vs_oracle(plan, pid, s, e, c, pen, want=None, what=None):
    """Summary fields and segments of problem pid bit for bit against the oracle's solve of the same
    rows (want: a cached oracle_bind.solve_rows result of them)."""
    st, summ, oseg = want if want is not None else oracle_bind.solve_rows(s, e, c, pen)
    assert st == 0, what
    r = plan.result(pid)
    assert r.status == 0, (what, r.status)
    got = plan.loss_row(pid)
    seg = plan.segments(pid)
    # bit-exact integer outputs
    assert (got["segments"], got["peaks"], got["equality.constraints"]) == (int(summ[1]), int(summ[2]), int(summ[7])), what
    assert np.array_equal(seg[0], oseg[0]) and np.array_equal(seg[1], oseg[1]) and np.array_equal(seg[2], oseg[2]), what
    # fp64 outputs: north_star bar 1e-9; we additionally expect bit equality with the psd_math oracle
    assert abs(got["total.loss"] - summ[6]) <= LOSS_RTOL * max(1.0, abs(summ[6])), what
    assert got["total.loss"] == summ[6] and got["mean.pen.cost"] == summ[5], what
    assert got["mean.intervals"] == summ[8] and got["max.intervals"] == summ[9], what
    assert np.array_equal(seg[3].view(np.uint64), oseg[3].view(np.uint64)), what


class StoreProblem:
    """One problem of the store comparison: rows (s, e, c) with a penalty string, added to a plan as
    rows or, when counts is given, as the count vector whose run-length encoding the rows are."""

    def __init__(self, name, rows, pen, counts=None):
        self.name, self.pen, self.counts = name, pen, counts
        self.s, self.e, self.c = rows

    def add(self, plan):
        if self.counts is not None:
            return plan.add_counts(self.counts, float(self.pen))
        return plan.add(self.s, self.e, self.c, float(self.pen))

    def db(self, tmpdir, write_db):
        """write_db(bedgraph, penalty_str) solves the problem's file and leaves bedgraph + '.db'; returns
        the parsed db ({(row, which): (chromEnd, max_log_mean, data_i, prev_log_mean)})."""
        from peaksegdisk_b200 import synth
        bg = os.path.join(str(tmpdir), self.name + ".bedGraph")
        synth.write_bedgraph(bg, self.s, self.e, self.c)
        assert write_db(bg, self.pen) == 0, self.name
        ref = parse_reference_db(bg + ".db", len(self.c))
        os.unlink(bg + ".db")
        assert len(ref) == 2 * len(self.c) - 1 and (0, 0) not in ref, self.name   # up_0 does not exist
        return ref


def extreme_rows(rng=None):
    """The zero-run / 2e9-count / wide-row rows of test_extreme_values_match_oracle: 400 rows of up to
    1.5e6 bases, counts up to 2e9, 30 % zeros (zero runs start the log-mean domain at -inf)."""
    if rng is None:
        rng = np.random.default_rng(99)
    n = 400
    w = rng.integers(1, 100000000, size=n).astype(np.int64)
    e = np.cumsum(w) // 64 + np.arange(1, n + 1)          # strictly increasing, below 2^31
    s = np.concatenate(([0], e[:-1]))
    big = rng.integers(0, 2000000000, size=n)
    big[rng.random(n) < 0.3] = 0
    return s.astype(np.int32), e.astype(np.int32), big.astype(np.int32)


def rising_rows():
    """Poisson counts whose mean rises from 1 to 400 over 1,500 positions: at penalty 1000 its largest
    cost function has 34 pieces, more than the two-block build's 24-piece shared-memory tier holds
    and fewer than the one-block build's 48."""
    from peaksegdisk_b200 import synth
    return synth.rle_rows(np.random.default_rng(0).poisson(np.linspace(1, 400, 1500)))


def store_problems():
    from peaksegdisk_b200 import synth
    _, ms, me, mc = synth.read_bedgraph(os.path.join(GOLD, "Mono27ac_coverage.bedGraph"))
    counts = synth.poisson_counts(78, 8000)
    return [StoreProblem("mono27ac_10.5", (ms, me, mc), "10.5"),
            StoreProblem("mono27ac_0", (ms, me, mc), "0"),
            StoreProblem("poisson_11", synth.poisson_problem(11, 3000), "250"),
            StoreProblem("increasing_150", synth.increasing_problem(150), "1000"),
            StoreProblem("extreme_1e-12", extreme_rows(), "1e-12"),
            StoreProblem("extreme_1e15", extreme_rows(), "1e15"),
            StoreProblem("rising_1000", rising_rows(), "1000"),
            StoreProblem("counts_78", synth.rle_rows(counts), "1000", counts=counts)]


def assert_store_equals_db(plan, pid, prob, ref, build):
    """Every stored function of problem pid (piece count, max_log_mean, data_i, prev_log_mean of every
    piece, bit for bit) equals the db's; a mismatch names the build, the problem, the row, the function
    and the first differing piece."""
    n_pieces = 0
    for (row, which), (chrom_end, hi, bi, bx) in sorted(ref.items()):
        where = "%s build, problem %s, row %d, %s function" % (build, prob.name, row, ("up", "down")[which])
        assert chrom_end == prob.e[row], where
        ghi, gbi, gbx = plan.store_function(pid, row, which, cap=4096)
        assert len(ghi) == len(hi), "%s: %d pieces, the oracle has %d" % (where, len(ghi), len(hi))
        diff = (ghi.view(np.uint64) != hi.view(np.uint64)) | (gbi != bi) | (gbx.view(np.uint64) != bx.view(np.uint64))
        if diff.any():
            k = int(np.flatnonzero(diff)[0])
            raise AssertionError("%s: piece %d of %d differs: (max_log_mean, data_i, prev_log_mean) = (%r, %d, %r), "
                                 "the oracle has (%r, %d, %r)" % (where, k, len(hi), ghi[k], gbi[k], gbx[k], hi[k], bi[k], bx[k]))
        n_pieces += len(hi)
    assert n_pieces == round(plan.loss_row(pid)["mean.intervals"] * 2 * len(prob.c)), (build, prob.name)
    hi0, _, _ = plan.store_function(pid, 0, 0)
    assert len(hi0) == 0, (build, prob.name)
