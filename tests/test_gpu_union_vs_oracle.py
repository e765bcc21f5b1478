"""
`count4` on union tiles (`CountPath::SingleUnion`) against the host oracle.  An unweighted `count4` with one sub-bin and
no labels cuts its register tiles from one second-role index over BOTH second catalogs (`yawb_rindex_get_union`): the
union has its own segment offsets (the sum of both catalogs'), takes the patch frames of the first of the two second
catalogs, sizes its Hilbert keys from both row counts, takes the straggler guard's density from the union, and the test
loop splits every count by the catalog bit of each register row into the accumulators [catalog][first catalog][z-bin].

Each case compares all four outputs with `oracle.binned_pair_counts` on the rows that output should see, never with
another device count: z-bin counts around the 32 lanes of a warp, lower edges of 0 and empty z-bins, binned and
unbinned second catalogs (also the autocorrelation shape, where a first catalog is a second one too), very unequal
sizes, an empty second catalog, a patch empty in one second catalog only (on either side: the frames come from the
first), a patch where one second catalog has a single row or all rows at one point (degenerate frames), every geometry
of the oracle file, union segments that cross a tile boundary only together, a large job with row-split items, the
edge-adversarial golden case output by output, and the union cache across second-role masks and catalog order.

Bar: integer pair counts bit-exact (the sums of an unweighted count are the counts as doubles).
"""

import numpy as np
import pytest
from numpy.testing import assert_array_equal

import golden_io
import oracle
from test_gpu_paths_vs_oracle import (GEOMETRIES, SMALL_JOB_ITEMS, STREAM_CTAS, STREAM_WARPS, TILE, Rows, _geometry,
                                      all_pairs, compare, expect, kernel_path, sky, thresholds)

pytestmark = pytest.mark.gpu

# output t of count4 pairs first catalog t % 2 with second catalog t // 2
OUTPUTS = ((0, 0), (1, 0), (0, 1), (1, 1))


@pytest.fixture(scope="module")
def engine():
    from yet_another_wizz_b200 import Engine

    eng = Engine(0)
    yield eng
    eng.close()


def subset(rows: Rows, keep) -> Rows:
    """the rows of `rows` selected by `keep` (a mask or indices), as a catalog of their own"""
    return Rows(rows.xyz[keep], rows.patch[keep], rows.n_patch, None if rows.zbin is None else rows.zbin[keep])


def check_union(engine, firsts, seconds, pi, pj, edges, *, binned2, what, devs=None, prune=True):
    """`count4` of two first and two second catalogs on union tiles: every output against the oracle on the rows of
    its own catalogs.  `devs`: the uploaded catalogs (first a, first b, second a, second b) when the caller keeps
    them; uploaded and freed here otherwise.  Returns the stats."""
    n_bins, n_edges = edges.shape
    assert kernel_path(False, n_edges, n_bins, 2, n_second=2) == ("SingleUnion", False)
    own = devs is None
    if own:
        devs = [r.upload(engine, n_bins) for r in firsts] + [r.upload(engine, n_bins if binned2 else None) for r in seconds]
    out, st = engine.count4(*devs, pi, pj, edges)
    assert st["launches"] == 2, f"{what}: one planner launch over the union tiles and one count kernel"
    for t, ((gi, gf), (c1, c2)) in enumerate(zip(out, OUTPUTS)):
        wi, wf = expect(firsts[c1], seconds[c2], pi, pj, edges, binned2=binned2)
        if len(seconds[c2].xyz) == 0:  # nothing to pair with: the other catalog's counts must not land here
            assert gi.shape == wi.shape and not gi.any() and not gf.any(), f"{what}: output {t} of an empty catalog"
            continue
        compare(gi, gf, wi, wf, False, f"{what}: output {t}")
    if prune:
        assert 0 < st["pair_tests"] < st["pair_tests_naive"], what
    if own:
        for d in devs:
            d.free()
    return st


# --------------------------------------------------------------------------------------------------------------------
# 1. z-bins, thresholds, binned and unbinned second catalogs, sizes, empty and degenerate patches
# --------------------------------------------------------------------------------------------------------------------
# (id, n_bins, binned second catalogs, layout); every case counts unweighted with one sub-bin and no labels
UNION_CASES = [
    ("B1", 1, False, "plain"),
    ("B31-binned", 31, True, "plain"),
    ("B32", 32, False, "plain"),
    ("B33-binned", 33, True, "plain"),
    ("B64", 64, False, "plain"),
    ("auto-B5", 5, True, "auto"),
    ("10-to-1", 4, False, "10:1"),
    ("1-to-10", 4, True, "1:10"),
    ("a-empty", 3, False, "a-empty"),
    ("b-empty", 3, True, "b-empty"),
    ("a-hole", 3, False, "a-hole"),
    ("b-hole", 3, True, "b-hole"),
    ("a-point", 3, False, "a-point"),
    ("b-point", 3, True, "b-point"),
]


def union_case_path(case):
    """the launch of a case of UNION_CASES"""
    return kernel_path(False, 2, case[1], 2, n_second=2)


def _union_catalogs(rng, n_bins, binned2, layout):
    """(first a, first b, second a, second b) on six patches of 0.01 rad; a first catalog drops 1 / (n_bins + 1) of its
    rows, a binned second catalog too"""
    n_patch = 6

    def cat(n):
        xyz, r, _ = sky(rng, n, (0.0, 0.06), (-0.03, 0.03))
        patch = np.minimum((r / 0.01).astype(int), n_patch - 1)
        return Rows(xyz, patch, n_patch, rng.integers(-1, n_bins, n))

    n2a, n2b = {"10:1": (30000, 3000), "1:10": (3000, 30000)}.get(layout, (11000, 14000))
    r1a, r1b, r2a, r2b = cat(5000), cat(8000), cat(n2a), cat(n2b)
    if layout == "auto":  # count4(data, rand, data, rand): each first catalog is also a second catalog
        return r1a, r1b, r1a, r1b
    seconds = [r2a, r2b]
    side = 0 if layout.startswith("a-") else 1
    if layout.endswith("-empty"):
        seconds[side] = subset(seconds[side], np.zeros(len(seconds[side].xyz), dtype=bool))
    elif layout.endswith("-hole"):  # patch 2 has rows in the other second catalog only
        seconds[side] = subset(seconds[side], seconds[side].patch != 2)
    elif layout.endswith("-point"):  # patch 2: one row; patch 4: every row at one point; the other catalog spread
        s = seconds[side]
        keep = (s.patch != 2) | (np.arange(len(s.xyz)) == s.off[2])
        s.xyz[s.off[4]:s.off[5]] = s.xyz[s.off[4]]
        seconds[side] = subset(s, keep)
    if not binned2:
        for s in seconds:
            s.zbin = None
    return r1a, r1b, *seconds


@pytest.mark.parametrize("case", UNION_CASES, ids=[c[0] for c in UNION_CASES])
def test_union_against_oracle(engine, case):
    name, n_bins, binned2, layout = case
    rng = np.random.default_rng(3000 + UNION_CASES.index(case))
    r1a, r1b, r2a, r2b = _union_catalogs(rng, n_bins, binned2, layout)
    edges = thresholds(rng, n_bins, 2, 2e-4, 3e-3)  # lower edges of 0, every eighth z-bin empty, per z-bin scales
    pi, pj = all_pairs(6)
    if layout == "auto":  # the same device catalogs in both roles
        d1a, d1b = r1a.upload(engine, n_bins), r1b.upload(engine, n_bins)
        check_union(engine, [r1a, r1b], [r2a, r2b], pi, pj, edges, binned2=binned2, what=name, devs=[d1a, d1b, d1a, d1b])
        d1a.free(); d1b.free()
        return
    check_union(engine, [r1a, r1b], [r2a, r2b], pi, pj, edges, binned2=binned2, what=name)


# --------------------------------------------------------------------------------------------------------------------
# 2. geometry: every case of the oracle file with its second catalog split in two, and union segments that cross a
# tile boundary only together
# --------------------------------------------------------------------------------------------------------------------
def _split(rng, rows: Rows, how: str):
    if how == "alternate":
        pick = np.arange(len(rows.xyz)) % 2 == 0
    else:
        pick = rng.random(len(rows.xyz)) < 0.4
    return subset(rows, pick), subset(rows, ~pick)


@pytest.mark.parametrize("name", GEOMETRIES + ["tiles-union"])
def test_union_geometry_against_oracle(engine, name):
    """`irregular` cuts tiles with the straggler guard, whose density comes from both catalogs; `strip` (5000 patches)
    sizes the Hilbert keys from both row counts"""
    rng = np.random.default_rng(3500 + (GEOMETRIES + ["tiles-union"]).index(name))
    n_bins = 3
    if name == "tiles-union":  # union segments of 255 + 1, 1 + 255, 256 + 1, 0 + 513 and 128 + 129 rows
        sa, sb, s1 = [255, 1, 256, 0, 128], [1, 255, 1, 513, 129], [300, 1, 256, 257, 255]
        n_patch, lo, hi = 5, 5e-4, 6e-3

        def rows(sizes):
            return Rows(sky(rng, sum(sizes), (0.0, 0.02), (-0.01, 0.01))[0], np.repeat(np.arange(n_patch), sizes), n_patch)

        r1, r2a, r2b = rows(s1), rows(sa), rows(sb)
    else:
        r1, r2, n_patch, (lo, hi) = _geometry(rng, name)
        r2a, r2b = _split(rng, r2, "alternate" if GEOMETRIES.index(name) % 2 == 0 else "random")
    r1.zbin = rng.integers(0, n_bins, len(r1.xyz))
    r1b = subset(r1, np.arange(len(r1.xyz)) % 3 == 1)
    live = np.flatnonzero(np.diff(r1.off) * (np.diff(r2a.off) + np.diff(r2b.off)))
    pi, pj = (live[k].astype(np.int32) for k in all_pairs(len(live)))
    edges = np.array([oracle.chord_sq_edges(np.geomspace(lo * s, hi, 2)) for s in rng.uniform(0.7, 1.0, n_bins)])
    check_union(engine, [r1, r1b], [r2a, r2b], pi, pj, edges, binned2=False, what=name,
                prune=not name.startswith("wide"))  # a search radius of 100 degrees and more reaches every row


# --------------------------------------------------------------------------------------------------------------------
# 3. a large job on union tiles: items of CCAP runs and single z-bins split into row ranges
# --------------------------------------------------------------------------------------------------------------------
def test_union_large_job_with_row_split(engine):
    """the row-split case of the oracle file's large job (56 patches on one strip, all 3136 pairs linked, 64 z-bins,
    every query spanning more than CCAP cell rows) with the second catalog split at random into the two catalogs of
    the union"""
    rng = np.random.default_rng(2026)
    n_patch, n_bins = 56, 64
    strip_ra, strip_dec = (0.0, 3.2e-6), (-0.1, 0.1)

    def cat(per_seg):
        n = n_patch * n_bins * per_seg
        xyz, _, _ = sky(rng, n, strip_ra, strip_dec)
        return Rows(xyz, rng.integers(0, n_patch, n), n_patch, rng.integers(0, n_bins, n))

    r1, r2 = cat(5), cat(4)
    r1b = subset(r1, np.arange(len(r1.xyz)) % 2 == 0)
    r2a, r2b = _split(rng, r2, "random")
    pi, pj = all_pairs(n_patch)
    seg2 = np.zeros((n_patch, n_bins), dtype=np.int64)  # union segments: the rows of both catalogs
    np.add.at(seg2, (r2.patch, r2.zbin), 1)
    n_flat = int(((seg2 + TILE - 1) // TILE).sum(axis=1)[pj].sum())
    assert n_flat > 2 * SMALL_JOB_ITEMS * engine.num_sms * STREAM_CTAS * STREAM_WARPS
    edges = np.array([oracle.chord_sq_edges(np.geomspace(1e-3, 0.205 * s, 2)) for s in rng.uniform(1.0, 1.3, n_bins)])
    # a search radius longer than the strip reaches every row: nothing to prune
    st = check_union(engine, [r1, r1b], [r2a, r2b], pi, pj, edges, binned2=True, what="large job", prune=False)
    assert st["work_items"] >= 2 * n_flat * 0.9  # nearly every (pair, union tile) became two items


# --------------------------------------------------------------------------------------------------------------------
# 4. pairs within a few ulp of the edges: a lane flagged for the FP64 recheck holds rows of both catalogs
# --------------------------------------------------------------------------------------------------------------------
def test_union_edge_adversarial_every_output(engine):
    g = golden_io.load("edge_adversarial")
    a, b = g["a_xyz"], g["b_xyz"]
    lim = oracle.parse_ang_limits(g["upper_ang_min"], g["upper_ang_max"])
    r2 = oracle.chord_sq_edges(oracle.get_ang_bins(lim, None, 50))
    assert len(r2) == 2
    one = Rows(a, np.zeros(len(a), dtype=int), 1, np.zeros(len(a), dtype=int))
    second = Rows(b, np.zeros(len(b), dtype=int), 1)
    firsts = [one, subset(one, np.arange(len(a)) % 3 == 0)]
    seconds = [subset(second, np.arange(len(b)) % 2 == 0), subset(second, np.arange(len(b)) % 2 == 1)]
    pi = pj = np.zeros(1, dtype=np.int32)
    st = check_union(engine, firsts, seconds, pi, pj, r2[None, :], binned2=False, what="edge_adversarial", prune=False)
    assert st["rechecks"] > 0


# --------------------------------------------------------------------------------------------------------------------
# 5. the union cache: second-role masks set, changed and cleared between counts, and the other catalog order
# --------------------------------------------------------------------------------------------------------------------
def test_union_cache_follows_masks_and_order(engine):
    rng = np.random.default_rng(3900)
    n_bins = 4
    r1a, r1b, r2a, r2b = _union_catalogs(rng, n_bins, False, "plain")
    edges = thresholds(rng, n_bins, 2, 2e-4, 3e-3)
    pi, pj = all_pairs(6)
    devs = [r1a.upload(engine, n_bins), r1b.upload(engine, n_bins), r2a.upload(engine), r2b.upload(engine)]
    ma = (rng.random(len(r2a.xyz)) < 0.6).astype(np.uint8)
    mb = (rng.random(len(r2b.xyz)) < 0.3).astype(np.uint8)

    def check(sa, sb, what, order=(2, 3)):
        check_union(engine, [r1a, r1b], [sa, sb], pi, pj, edges, binned2=False, what=what,
                    devs=devs[:2] + [devs[k] for k in order])

    devs[2].set_second_rows(ma)
    devs[3].set_second_rows(mb)
    check(subset(r2a, ma != 0), subset(r2b, mb != 0), "both masked")
    ma2 = (rng.random(len(r2a.xyz)) < 0.5).astype(np.uint8)  # a new mask on one catalog of the cached union
    devs[2].set_second_rows(ma2)
    check(subset(r2a, ma2 != 0), subset(r2b, mb != 0), "mask of the first second catalog changed")
    devs[3].set_second_rows(None)
    check(subset(r2a, ma2 != 0), r2b, "mask of the second second catalog cleared")
    devs[2].set_second_rows(None)
    check(r2a, r2b, "both masks cleared")
    # (b, a) is another union, with b's frames; (a, b) stays cached next to it
    check(r2b, r2a, "second catalogs swapped", order=(3, 2))
    out, st = engine.count4(*devs, pi, pj, edges)
    assert st["index_ms"] == 0.0  # both unions were cached
    for (gi, _), (c1, c2) in zip(out, OUTPUTS):
        assert_array_equal(gi, expect((r1a, r1b)[c1], (r2a, r2b)[c2], pi, pj, edges, binned2=False)[0])
    for d in devs:
        d.free()
