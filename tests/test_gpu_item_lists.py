"""
The repeat of a count whose work-item lists overflowed, against the host oracle.  `count_impl` sizes the planner's
lists before it knows how many items there are: 4 per (pair, tile) combination of a patch with itself plus 1024 for
the heavy list, 2 per other combination plus 1024 for the light list, both CCAP / CCAP_SMALL = 7 times that for a
small job.  A planner that runs past a list sets a flag (`counters[6]`); the host then clears the outputs and the
counters and runs the planner and the count kernel again with lists sized from the exact item counts.

Many items per (pair, tile) make the lists overflow: every patch here is a strip (3.2e-6 x 0.2 rad), so the sky-cell
grid of a first catalog has about 150 cell rows in one column, and a second catalog with fewer than YAWB_TILE rows per
patch makes one tile per patch whose box spans the whole strip.  Each such tile walks every cell row of every z-bin:
about 7 items per z-bin in a small job (CCAP_SMALL = 24 runs per item) and one in a large job (CCAP = 160), against a
list of 28 or 4 per combination.  The search radius stays below 1.3e-3 rad, so the oracle's candidate pairs stay few.

- heavy list: every patch on its own strip, 0.01 rad apart, all pairs listed: the box test drops every combination of
  two patches, so only the heavy list has items;
- light list: all patches on one strip, only pairs of two different patches listed: only the light list has items.

Each case runs in a small and in a large job (40 and 300 patches), checks that the count ran twice (launch count),
compares with the oracle, repeats the same call, and runs a control of the same catalogs whose z-bins are all empty but
one, which fits the first lists.
"""

import numpy as np
import pytest
from numpy.testing import assert_array_equal

import oracle
from test_gpu_paths_vs_oracle import (SMALL_JOB_ITEMS, STREAM_CTAS, STREAM_WARPS, TILE, Rows, all_pairs, compare,
                                      expect, kernel_path, sky, thresholds)

pytestmark = pytest.mark.gpu

STRIP_RA, STRIP_DEC = (0.0, 3.2e-6), (-0.1, 0.1)
SPACING = 0.01  # RA between the strips of the heavy-list layout: far beyond the search radius
REGIMES = {"small": (40, 64), "large": (300, 16)}  # (patches, z-bins)

# (id, count, regime, list): every path meets both regimes and both lists
CASES = [
    ("single-small-heavy", "single", "small", "heavy"),
    ("single-large-light", "single", "large", "light"),
    ("union-small-light", "union", "small", "light"),
    ("union-large-heavy", "union", "large", "heavy"),
    ("cumul-small-light", "cumul", "small", "light"),
    ("cumul-large-heavy", "cumul", "large", "heavy"),
    ("singlew-small-heavy", "weighted", "small", "heavy"),
    ("singlew-large-light", "weighted", "large", "light"),
]
N_EDGES = {"single": 2, "union": 2, "cumul": 4, "weighted": 2}
PATHS = {"single": "Single", "union": "SingleUnion", "cumul": "Cumulative", "weighted": "SingleWeighted"}


@pytest.fixture(scope="module")
def engine():
    from yet_another_wizz_b200 import Engine

    eng = Engine(0)
    yield eng
    eng.close()


def _strips(rng, n_patch, per_patch, separate, n_bins=None, w=False):
    """`per_patch` rows in each of `n_patch` patches, each on the strip, shifted by SPACING per patch if `separate`"""
    n = n_patch * per_patch
    _, ra, dec = sky(rng, n, STRIP_RA, STRIP_DEC)
    patch = np.repeat(np.arange(n_patch), per_patch)
    if separate:
        ra = ra + SPACING * patch
    return Rows(oracle.radec_to_xyz(ra, dec), patch, n_patch, None if n_bins is None else rng.integers(0, n_bins, n),
                rng.uniform(0.5, 1.5, n) if w else None)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_overflowed_lists_are_repeated(engine, case):
    name, count, regime, which = case
    rng = np.random.default_rng(4000 + CASES.index(case))
    n_patch, n_bins = REGIMES[regime]
    n_edges = N_EDGES[count]
    separate = which == "heavy"
    n_first = 2 if count == "union" else 1
    firsts = [_strips(rng, n_patch, 2 * n_bins, separate, n_bins) for _ in range(n_first)]
    per2 = (100, 60) if count == "union" else (150,)  # fewer than TILE rows of the (union) index per patch
    seconds = [_strips(rng, n_patch, n, separate, w=count == "weighted") for n in per2]
    pi, pj = all_pairs(n_patch)
    if which == "light":
        pi, pj = pi[pi != pj], pj[pi != pj]
    assert kernel_path(count == "weighted", n_edges, n_bins, n_first, n_second=len(seconds)) == (PATHS[count], False)

    # the regime: (pair, tile) combinations of the index the tiles come from (no straggler cuts below 8 tiles a patch)
    rows2 = sum(np.diff(s.off) for s in seconds)
    n_flat = int(((rows2 + TILE - 1) // TILE)[pj].sum())
    threshold = SMALL_JOB_ITEMS * engine.num_sms * STREAM_CTAS * STREAM_WARPS
    assert (n_flat < threshold) == (regime == "small"), (n_flat, threshold)

    edges = thresholds(rng, n_bins, n_edges, 2e-4, 1e-3)
    control = edges.copy()  # every z-bin but the first empty: no query walks their cell rows
    control[1:] = control[1:, -1:]
    devs = [r.upload(engine, n_bins) for r in firsts] + [s.upload(engine) for s in seconds]
    weighted = count == "weighted"

    def run(r2):
        """the count of every (first, second) combination, and the stats"""
        if count == "union":
            out, st = engine.count4(*devs, pi, pj, r2)
            return out, st, [(f, s) for s in seconds for f in firsts]
        ci, cf, st = engine.count(devs[0], devs[1], pi, pj, r2)
        return [(ci, cf)], st, [(firsts[0], seconds[0])]

    # launches of the fast path: one planner launch per tile index (one here: a catalog's own, or the union) and the
    # count kernel; index builds are not counted
    n_plan = 1
    for r2, launches, what in ((edges, 2 * (n_plan + 1), "overflow"), (control, n_plan + 1, "control")):
        out, st, combos = run(r2)
        assert st["launches"] == launches, f"{name} ({what}): {st['launches']} launches"
        for k, ((gi, gf), (c1, c2)) in enumerate(zip(out, combos)):
            wi, wf = expect(c1, c2, pi, pj, r2, binned2=False)
            compare(gi, gf, wi, wf, weighted, f"{name} ({what}): output {k}")
        if what == "overflow":  # nothing of the discarded attempt or of the last call may stay behind
            again, st2, _ = run(r2)
            assert st2["launches"] == launches
            for (gi, gf), (ai, af) in zip(out, again):
                assert_array_equal(ai, gi, err_msg=f"{name}: repeated call")
                if not weighted:  # FP64 atomic sums may differ in the last bits from run to run
                    assert_array_equal(af, gf, err_msg=f"{name}: repeated call")
    for d in devs:
        d.free()
