"""Every compiled DP kernel build and launch shape, each forced on its own, against the parity oracle:
the stored cost functions row by row and every output bit for bit, plus the check that each forced
build is the one that ran and that the automatic choice of the two-block build on a large batch of
short problems gives what the one-block build gives.

Builds (csrc/fpop_gpu.cu): the throughput kernel's one-block build (fpop_dp_kernel<16, 1>: one block
of 14 warps per SM, 48-piece shared-memory tier) and two-block build (fpop_dp_kernel<14, 2>: two
blocks per SM, 24-piece tier, about 1.3 KB of spills per thread); the latency kernel (fpop_lat.cu,
one problem per block) with helper warps (waves of at most one problem per SM) and without; and the
re-run of problems that outgrew every tier (status 101) from global-memory piece lists only, in the
throughput and in the latency kernel."""
import contextlib
import importlib.util
import math
import os
import numpy as np
import pytest
import oracle_bind
import oracle_checks
from helpers import ROOT

pytestmark = pytest.mark.gpu

# piece_cap / spill_cap of the global-list builds: an 8-piece shared tier and no per-warp global
# workspace, so every problem with more than 8 pieces per function returns 101 and is re-run
GLOBAL_CAPS = {"piece_cap": 8, "spill_cap": 0}
BUILDS = {   # options (their defaults are restored after each solve), and whether the wave exceeds n_SM
    "one-block": ({"latency_mode": 2, "occupancy_mode": 1}, False),
    "two-block": ({"latency_mode": 2, "occupancy_mode": 2}, False),
    "latency-helpers": ({"latency_mode": 1}, False),
    "latency-no-helpers": ({"latency_mode": 1}, True),
    "global-throughput": (dict(GLOBAL_CAPS, latency_mode=2, occupancy_mode=1), False),
    # a wave of more than n_SM problems: the latency kernel's global workspace is then spill_cap (with one
    # problem per SM it is sized for the worst case and nothing would return 101)
    "global-latency": (dict(GLOBAL_CAPS, latency_mode=1), True),
}
DEFAULTS = {"latency_mode": 0, "occupancy_mode": 0, "piece_cap": 48, "spill_cap": 512}


@contextlib.contextmanager
def options(psd, opts):
    """Sets process-wide options for the plans created inside; restores the defaults on the way out.
    A PSD_* environment variable would override them, so none may be set."""
    assert not [k for k in os.environ if k in ("PSD_" + n.upper() for n in DEFAULTS)]
    lib = psd._lib.lib
    try:
        for name, value in opts.items():
            assert lib.psd_set_option(name.encode(), float(value)) == 0
        yield
    finally:
        for name in opts:
            lib.psd_set_option(name.encode(), float(DEFAULTS[name]))


def solve(psd, opts, add):
    """A fresh plan under the options, add(plan) -> ids, run; returns (plan, ids)."""
    with options(psd, opts):
        plan = psd.Plan(0)
        ids = add(plan)
        plan.run()
    return plan, ids


@pytest.fixture(scope="module")
def psd():
    import peaksegdisk_b200
    assert peaksegdisk_b200._lib.lib.psd_device_count() >= 1, "no CUDA device"
    return peaksegdisk_b200


@pytest.fixture(scope="module")
def one_block(psd):
    """stats() of a one-block solve: n_sm, and the one-block build's warps_per_sm and piece_cap."""
    from peaksegdisk_b200 import synth
    plan, _ = solve(psd, BUILDS["one-block"][0], lambda p: [p.add(*synth.poisson_problem(1, 500), 10.0)])
    return plan.stats()


def fuzz_problems(n, seed):
    spec = importlib.util.spec_from_file_location("fuzz_gpu_vs_oracle", os.path.join(ROOT, "tools", "fuzz_gpu_vs_oracle.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.problems(n, seed)


@pytest.fixture(scope="module")
def batch(psd, one_block, tmp_path_factory):
    """The store problems (with their oracle dbs, computed once) and the six fuzz shapes at three seeds;
    `pad` are further fuzz problems that take a wave past n_SM.  Oracle results are cached by index."""
    store = oracle_checks.store_problems()
    d = tmp_path_factory.mktemp("store_db")
    dbs = [p.db(d, lambda bg, pen: oracle_bind.oracle_disk(bg, pen, bg + ".db", 1)) for p in store]
    rising = [p for p in store if p.name == "rising_1000"][0]
    pieces = max(len(v[1]) for v in dbs[store.index(rising)].values())
    two_block_cap = one_block["piece_cap"] // 2
    assert two_block_cap < pieces <= one_block["piece_cap"], pieces   # leaves the two-block build's shared tier only
    fuzz = [x for seed in (1, 2, 3) for x in fuzz_problems(12, seed)]
    rows = [(p.s, p.e, p.c, float(p.pen)) for p in store] + fuzz
    pad = fuzz_problems(2 * one_block["n_sm"], 4)[:one_block["n_sm"] + 8 - len(rows)]
    assert len(rows) <= one_block["n_sm"] < len(rows) + len(pad)
    return {"store": store, "dbs": dbs, "rows": rows, "pad": pad, "oracle": {}}


def oracle(batch, k):
    if k not in batch["oracle"]:
        s, e, c, pen = (batch["rows"] + batch["pad"])[k]
        batch["oracle"][k] = oracle_bind.solve_rows(s, e, c, pen)
    return batch["oracle"][k]


@pytest.fixture(scope="module")
def solved(psd, batch):
    """One solve of the batch per build, shared by the tests below."""
    cache = {}

    def get(build):
        if build not in cache:
            opts, padded = BUILDS[build]
            store = batch["store"]
            extra = batch["rows"][len(store):] + (batch["pad"] if padded else [])

            def add(plan):
                return [p.add(plan) for p in store] + [plan.add(*x) for x in extra]
            cache[build] = solve(psd, opts, add)
        return cache[build]
    return get


@pytest.mark.parametrize("build", list(BUILDS))
def test_forced_build_is_the_one_that_ran(psd, one_block, batch, solved, build):
    """Without this the parametrization could pass vacuously: a build that cannot be configured falls
    back to another one without an error.  stats() holds the last wave's launch shape."""
    plan, ids = solved(build)
    st = plan.stats()
    n_sm = st["n_sm"]
    n_gpu = len(ids)
    assert n_gpu == len(batch["rows"]) + (len(batch["pad"]) if BUILDS[build][1] else 0)
    assert (n_gpu > n_sm) == BUILDS[build][1]                    # helpers run with at most one problem per SM
    if build in ("one-block", "two-block", "global-throughput"):
        assert st["n_latency_waves"] == 0, st
    else:
        assert st["n_latency_waves"] == st["n_waves"], st
    if build == "one-block":
        assert (st["warps_per_sm"], st["piece_cap"], st["n_waves"]) == (one_block["warps_per_sm"], one_block["piece_cap"], 1), st
    elif build == "two-block":
        # two blocks per SM of one_block's warps, and half its shared-memory tier (24 / 28 against 48 / 14 on B200)
        assert (st["warps_per_sm"], st["piece_cap"], st["n_waves"]) == (2 * one_block["warps_per_sm"], one_block["piece_cap"] // 2, 1), st
    elif build.startswith("latency"):
        assert st["n_waves"] == 1, st
    else:   # the first wave, then the re-run of every problem that returned 101 from global lists
        assert st["n_waves"] > 1, st


def last_wave(plan, pid, n_rows):
    """True when problem pid was solved in the plan's last store wave (only its records can be read)."""
    try:
        plan.store_function(pid, n_rows - 1, 1, cap=4096)
        return True
    except RuntimeError:
        return False


@pytest.mark.parametrize("build", list(BUILDS))
def test_store_rows_equal_the_oracle_db(psd, batch, solved, build):
    """Every stored function of every store problem, row by row, against the parity oracle's db.  In
    the global-list builds the inspected problems are the re-run ones: every problem with more than 8
    pieces in some function must be among them."""
    plan, ids = solved(build)
    inspected = 0
    for pid, p, db in zip(ids, batch["store"], batch["dbs"]):
        if build.startswith("global"):
            pieces = max(len(v[1]) for v in db.values())
            rerun = last_wave(plan, pid, len(p.c))
            assert rerun or pieces <= GLOBAL_CAPS["piece_cap"], (build, p.name, pieces)
            if not rerun:
                continue
        oracle_checks.assert_store_equals_db(plan, pid, p, db, build)
        inspected += 1
    assert inspected == len(batch["store"]) or (build.startswith("global") and inspected > 0), inspected


@pytest.mark.parametrize("build", list(BUILDS))
def test_outputs_equal_the_oracle(psd, batch, solved, build):
    """Store problems and fuzz shapes (and the padding): every summary field and the segment bits."""
    plan, ids = solved(build)
    probs = batch["rows"] + batch["pad"]
    for k, pid in enumerate(ids):
        s, e, c, pen = probs[k]
        oracle_checks.check_vs_oracle(plan, pid, s, e, c, pen, oracle(batch, k), (build, k, len(c), pen))


def test_automatic_choice_runs_the_two_block_build_on_many_short_problems(psd, one_block):
    """A wave of many short count vectors is what the automatic choice gives the two-block build, and it
    is the only test in which the two-block build runs with every slot busy, its warps taking further
    problems from the queue.  choose_config picks it when its simulated queue makespan beats the
    one-block build's by 5 %: with every problem on its own warp (2,072 problems on B200) the one-block
    build wins, so the batch holds three problems per one-block slot; and more than 16 problems per SM,
    so that the latency kernel is not considered.  If choose_config is retuned, adjust the batch rather
    than drop the assertion.  Results must be bit-identical to a forced one-block solve, and a seeded
    tenth of the problems equal the oracle."""
    from peaksegdisk_b200 import synth
    rng = np.random.default_rng(2300)
    n_gpu = 3 * one_block["n_sm"] * one_block["warps_per_sm"]
    assert n_gpu > 16 * one_block["n_sm"]
    probs = []
    for k in range(n_gpu):
        probs.append((synth.poisson_counts(7000 + k, int(rng.integers(1000, 3001))), float(10 ** rng.uniform(0, 5))))
        if k % 40 == 39:   # trivial problems mixed in (constant counts, penalty Inf): solved on the host, not in the wave
            probs.append((np.full(int(rng.integers(1, 3000)), 4), 3.0) if k % 80 == 39 else (synth.poisson_counts(k, 1000), math.inf))

    def add(plan):
        return [plan.add_counts(v, pen) for v, pen in probs]
    auto, ids = solve(psd, {}, add)
    st = auto.stats()
    assert st["n_latency_waves"] == 0 and st["n_waves"] == 1, st
    assert (st["warps_per_sm"], st["piece_cap"]) == (2 * one_block["warps_per_sm"], one_block["piece_cap"] // 2), \
        "the automatic choice did not run the two-block build: %s" % st
    ref, ids1 = solve(psd, BUILDS["one-block"][0], add)
    assert ref.stats()["warps_per_sm"] == one_block["warps_per_sm"]
    trivial = 0
    for a, b in zip(ids, ids1):
        trivial += auto.result(a).trivial
        assert auto.loss_row(a) == ref.loss_row(b), a
        sa, sb = auto.segments(a), ref.segments(b)
        assert all(np.array_equal(x, y) for x, y in zip(sa[:3], sb[:3])) and np.array_equal(sa[3].view(np.uint64), sb[3].view(np.uint64)), a
    assert trivial == len(probs) - n_gpu, trivial
    for k in np.random.default_rng(7).choice(len(probs), size=len(probs) // 10, replace=False):
        v, pen = probs[k]
        if not auto.result(ids[k]).trivial:
            oracle_checks.check_vs_oracle(auto, ids[k], *synth.rle_rows(v), pen, what=("auto", int(k)))
