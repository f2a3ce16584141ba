"""Synthetic bedGraph problems of the shapes BASELINE.json names (SURVEY.md 8d "Synthetic inputs").

Pure numpy; used by bench.py and the tests to build seeded inputs.  Nothing here touches the GPU.
"""
import numpy as np

HG19_LEN = [249250621, 243199373, 198022430, 191154276, 180915260, 171115067, 159138663, 146364022,
            141213431, 135534747, 135006516, 133851895, 115169878, 107349540, 102531392, 90354753,
            81195210, 78077248, 59128983, 63025520, 48129895, 51304566, 155270560, 59373566]
HG19_NAMES = ["chr%d" % i for i in range(1, 23)] + ["chrX", "chrY"]


def rle_rows(counts, start=0):
    """Run-length encode a count vector into (chromStart, chromEnd, coverage) int32 arrays,
    as R/PeakSegFPOP_vec.R:18-25 does with rle()."""
    counts = np.asarray(counts, dtype=np.int64)
    n = counts.size
    if n == 0:
        z = np.zeros(0, np.int32)
        return z, z.copy(), z.copy()
    change = np.flatnonzero(counts[1:] != counts[:-1]) + 1
    first = np.concatenate(([0], change))
    last = np.concatenate((change, [n]))
    return ((first + start).astype(np.int32), (last + start).astype(np.int32), counts[first].astype(np.int32))


def poisson_counts(seed, n=None):
    """One config-2 count vector: alternating background/peak segments, Poisson draws.
    n log-uniform in [1e4, 1e5] unless given."""
    rng = np.random.default_rng(seed)
    if n is None:
        n = int(round(10 ** rng.uniform(4.0, 5.0)))
    means = np.empty(n)
    pos, peak = 0, False
    while pos < n:
        if peak:
            ln, mu = int(rng.integers(50, 201)), float(rng.choice([5.0, 10.0, 30.0]))
        else:
            ln, mu = int(rng.integers(100, 401)), float(rng.choice([0.5, 1.0, 2.0]))
        means[pos:pos + ln] = mu
        pos += ln
        peak = not peak
    return rng.poisson(means[:n]).astype(np.int64)


def poisson_problem(seed, n=None):
    """(chromStart, chromEnd, coverage) rows of one config-2 problem."""
    return rle_rows(poisson_counts(seed, n))


C2_PENALTIES = [1e2, 1e3, 1e4, 1e5, 1e6]


def increasing_problem(n):
    """Config 5 (vignettes/Worst_case.Rmd:19-41): count = 1..n, unit weights."""
    s = np.arange(n, dtype=np.int32)
    return s, s + 1, np.arange(1, n + 1, dtype=np.int32)


def write_bedgraph(path, chrom_start, chrom_end, coverage, chrom="chrUnknown"):
    """Tab-separated, no header: the text R/writeBedGraph.R:35-37 produces."""
    with open(path, "w") as f:
        f.write("".join("%s\t%d\t%d\t%d\n" % (chrom, s, e, c)
                        for s, e, c in zip(chrom_start.tolist(), chrom_end.tolist(), coverage.tolist())))


def read_bedgraph(path):
    a = np.loadtxt(path, dtype=str, ndmin=2)
    return a[0, 0], a[:, 1].astype(np.int32), a[:, 2].astype(np.int32), a[:, 3].astype(np.int32)


def reads(seed, n_reads, length, start=0, n_peaks=None, read_len=(36, 300)):
    """Seeded aligned reads for [start, start + length): half uniform background, half around n_peaks
    centres (default one per 20 kb), lengths uniform in read_len.  Returns unsorted half-open int32
    (read_start, read_end); a read may run past the region's end."""
    rng = np.random.default_rng(seed)
    if n_peaks is None:
        n_peaks = max(1, length // 20000)
    centres = rng.integers(0, length, size=n_peaks)
    n_bg = n_reads // 2
    pos = np.concatenate([rng.integers(0, length, size=n_bg),
                          centres[rng.integers(0, n_peaks, size=n_reads - n_bg)] + rng.normal(0, 300, size=n_reads - n_bg).astype(np.int64)])
    pos = np.clip(pos, 0, length - 1) + start
    rng.shuffle(pos)
    rl = rng.integers(read_len[0], read_len[1] + 1, size=n_reads)
    return pos.astype(np.int32), (pos + rl).astype(np.int32)


def hg19_problem(chrom_index, sample_index, base_weight, base_count, scale_rows=1.0):
    """One config-4 problem: tile the Mono27ac (weight, count) rows up to the chromosome's row
    target, redraw counts, RLE, re-accumulate coordinates (SURVEY.md 8d, C4)."""
    rng = np.random.default_rng(64 * chrom_index + sample_index)
    target = int(round(1e7 * scale_rows * HG19_LEN[chrom_index] / HG19_LEN[0]))
    nb = base_weight.size
    tiles = -(-target // nb)
    scale_s = float(np.exp(rng.uniform(np.log(0.5), np.log(4.0))))
    u = rng.uniform(0.5, 1.5, size=tiles)
    lam = (base_count[None, :] * (scale_s * u[:, None])).reshape(-1)[:target]
    w = np.tile(base_weight, tiles)[:target].astype(np.int64)
    z = rng.poisson(lam).astype(np.int64)
    change = np.flatnonzero(z[1:] != z[:-1]) + 1
    first = np.concatenate(([0], change))
    wsum = np.add.reduceat(w, first)
    end = np.cumsum(wsum)
    start = end - wsum
    penalty = float(np.exp(rng.uniform(np.log(1e2), np.log(1e5))))
    return start.astype(np.int32), end.astype(np.int32), z[first].astype(np.int32), penalty
