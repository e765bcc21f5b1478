"""
The pair-count kernels against the host oracle, at every place where `yawb_launch_count_fast` or the streaming kernel
switches to other code or other constants: the kernel paths and where their accumulators live (the union-tile path
of `count4`, `SingleUnion`, has its cases in `test_gpu_union_vs_oracle.py`; the repeat of a count whose work-item
lists overflowed is in `test_gpu_item_lists.py`), the group size of
the cumulative path, sub-bin counts up to `YAWB_MAX_EDGES`, z-bin counts around the 32 lanes of a warp, small and
large jobs (items of `CCAP_SMALL` or `CCAP` cell-row runs) with the row-range split of the planner, weights on either
side, per-bin thresholds with lower edges of 0, equal edges and empty z-bins, extreme geometry, short tiles and tiles cut
by the straggler guard, the three kinds of z-bin upload, both kinds of labels, and the two rejections.

Every result is compared with `oracle.binned_pair_counts` (the reference expression in float64 on k-d-tree candidates),
never with another device kernel: the exact kernel `k_count_exact` reads the same index data as the streaming one, so
an index that dropped a row or attached a weight to the wrong row would pass a device-against-device comparison.  The
exact kernel is held to the same oracle on the same cases.

Bar: integer pair counts bit-exact; weighted sums within 1e-12 relative.
"""

import math

import numpy as np
import pytest
from numpy.testing import assert_allclose, assert_array_equal

import oracle

pytestmark = pytest.mark.gpu

RTOL_WEIGHTED = 1e-12

# constants of csrc/yawb_count.cu and yawb_count_stream.cuh that select the code of a count
CUM_MAX_EDGES = 8
SMALL_JOB_ITEMS, STREAM_CTAS, STREAM_WARPS = 30, 4, 4
CCAP = 160
TILE = 256  # YAWB_TILE: rows of a register tile of the second catalog
# constants of csrc/yawb_index.cu that size the sky-cell grid of a first-role index
TARGET_PER_CELL, MAX_GRID_SPAN_CELLS = 5.5, 2048


def kernel_path(weighted: bool, n_edges: int, n_bins: int, n_types: int, n_second: int = 1, labels: bool = False,
                exact: bool = False) -> tuple[str, bool]:
    """the choice of `count_impl` and `yawb_launch_count_fast`: (CountPath, acc_global), or ("Exact", False) for the
    exact kernel.  Two second catalogs (`count4`) share tiles cut from their union only on the single-bin path without
    weights and labels; every other joint launch keeps per-catalog tiles and the path of one second catalog."""
    if exact:
        return "Exact", False
    if n_second == 2 and not weighted and n_edges == 2 and not labels:
        return "SingleUnion", False
    multi = n_edges > 2
    cumul = multi and not weighted and n_edges <= CUM_MAX_EDGES
    acc_bytes = n_types * n_bins * (n_edges - 1) * (16 if weighted else 8)
    acc_global = multi and not cumul and acc_bytes > 2048
    if weighted:
        return ("HistogramWeighted" if multi else "SingleWeighted"), acc_global
    if cumul:
        return "Cumulative", False
    return ("Histogram" if multi else "Single"), acc_global


def cumul_group(n_edges: int) -> int:
    """group size of `phase2_cumul`"""
    return 3 if n_edges <= 3 else 6 if n_edges in (5, 6) else 4


@pytest.fixture(scope="module")
def engine():
    from yet_another_wizz_b200 import Engine

    eng = Engine(0)
    yield eng
    eng.close()


# --------------------------------------------------------------------------------------------------------------------
# catalogs, thresholds, comparison
# --------------------------------------------------------------------------------------------------------------------
class Rows:
    """a catalog on the host, its rows sorted by patch: unit vectors, patch ids, z-bin ids (< 0: dropped; None:
    unbinned), weights (or None)"""

    def __init__(self, xyz, patch, n_patch, zbin=None, w=None, redshift=None):
        order = np.argsort(patch, kind="stable")
        self.redshift = None if redshift is None else np.asarray(redshift)[order]
        self.xyz = np.ascontiguousarray(xyz[order])
        self.patch = np.asarray(patch)[order]
        self.zbin = None if zbin is None else np.asarray(zbin, dtype=np.int64)[order]
        self.w = None if w is None else np.asarray(w, dtype=np.float64)[order]
        self.n_patch = n_patch
        self.off = np.concatenate([[0], np.cumsum(np.bincount(self.patch, minlength=n_patch))]).astype(np.int64)

    def upload(self, engine, n_bins=None):
        if self.zbin is None or n_bins is None:
            return engine.upload_catalog(self.xyz, self.off, weights=self.w)
        return engine.upload_catalog(self.xyz, self.off, weights=self.w, zbin=self.zbin.astype(np.int32), n_bins=n_bins)


def sky(rng, n, ra, dec):
    """`n` unit vectors uniform on the sky in an RA range and a Dec range (radian)"""
    r = rng.uniform(ra[0], ra[1], n)
    d = np.arcsin(rng.uniform(np.sin(dec[0]), np.sin(dec[1]), n))
    return oracle.radec_to_xyz(r % (2.0 * np.pi), d), r, d


def thresholds(rng, n_bins, n_edges, theta_lo, theta_hi, variety=True):
    """squared chord edges per z-bin, different in every z-bin (as angles from a fixed physical scale are).  With
    `variety`: a lower edge of 0 in every fourth z-bin (and in a single one), two equal neighbouring edges in every
    fourth, and every eighth z-bin empty (all edges equal: hi <= lo)"""
    rows = []
    for b in range(n_bins):
        s = rng.uniform(0.7, 1.3)
        r2 = oracle.chord_sq_edges(np.geomspace(theta_lo * s, theta_hi * s, n_edges))
        if variety:
            if b % 4 == 1 or n_bins == 1:
                r2[0] = 0.0
            elif b % 4 == 2 and n_edges > 2:
                r2[1] = r2[2]
            elif b % 8 == 3:
                r2[:] = r2[-1]
        rows.append(r2)
    return np.array(rows)


def expect(r1: Rows, r2: Rows, pi, pj, edges, *, binned2: bool):
    """the oracle's `(counts, sums)` of `count(r1, r2)`, `(n_pairs, n_bins, n_edges - 1)`"""
    wi, wf = oracle.binned_pair_counts(r1.xyz, r1.patch, r1.zbin, r2.xyz, r2.patch, pi, pj, edges, w1=r1.w, w2=r2.w,
                                       zbin2=r2.zbin if binned2 else None)
    return wi[0], wf[0]


def compare(got_i, got_f, want_i, want_f, weighted: bool, what=""):
    assert got_i.shape == want_i.shape, what
    assert want_i.sum() > 0, f"{what}: nothing to compare"
    if not np.array_equal(got_i, want_i):
        bad = np.argwhere(got_i != want_i)
        pytest.fail(f"{what}: {len(bad)} counts differ from the oracle, first at {tuple(bad[0])}: "
                    f"{got_i[tuple(bad[0])]} != {want_i[tuple(bad[0])]}; totals {got_i.sum()} != {want_i.sum()}")
    if weighted:
        assert want_f.sum() > 0, what
        assert_allclose(got_f, want_f, rtol=RTOL_WEIGHTED, atol=0, err_msg=what)
    else:
        assert_array_equal(got_f, want_i.astype(np.float64), err_msg=what)


def all_pairs(n_patch):
    pi, pj = np.meshgrid(np.arange(n_patch), np.arange(n_patch), indexing="ij")
    return pi.ravel().astype(np.int32), pj.ravel().astype(np.int32)


# --------------------------------------------------------------------------------------------------------------------
# 1. kernel paths: CountPath x acc_global, cumulative group sizes, n_edges, z-bins, weights, thresholds
# --------------------------------------------------------------------------------------------------------------------
# (id, n_edges, n_bins, weights, n_types, binned second catalog)
PATH_CASES = [
    ("single-B1", 2, 1, "none", 1, False),
    ("single-B33-binned", 2, 33, "none", 1, True),
    ("singlew-first-B31", 2, 31, "first", 1, False),
    ("singlew-second-B32", 2, 32, "second", 1, False),
    ("singlew-both-B33", 2, 33, "both", 1, True),
    ("singlew-second-count2", 2, 5, "second", 2, False),
    ("cumul-e3-B33", 3, 33, "none", 1, False),
    ("cumul-e4-B1", 4, 1, "none", 1, False),
    ("cumul-e5-B32", 5, 32, "none", 1, True),
    ("cumul-e6-B31", 6, 31, "none", 1, False),
    ("cumul-e6-count2", 6, 4, "none", 2, False),
    ("cumul-e7-B64", 7, 64, "none", 1, False),
    ("cumul-e8-count2-B33", 8, 33, "none", 2, False),
    ("hist-e9-B32-shared", 9, 32, "none", 1, False),
    ("hist-e10-B32-global", 10, 32, "none", 1, True),
    ("hist-e9-count2-B16-shared", 9, 16, "none", 2, False),
    ("hist-e10-count2-B16-global", 10, 16, "none", 2, False),
    ("hist-e33-B1", 33, 1, "none", 1, False),
    ("hist-e256-B1-shared", 256, 1, "none", 1, False),
    ("hist-e12-B256-fallback", 12, 256, "none", 1, True),
    ("histw-e9-first-B16-shared", 9, 16, "first", 1, False),
    ("histw-e10-second-B16-global", 10, 16, "second", 1, False),
    ("histw-e5-both-count2-B16-shared", 5, 16, "both", 2, False),
    ("histw-e6-both-count2-B16-global", 6, 16, "both", 2, True),
    ("histw-e34-both-B1", 34, 1, "both", 1, False),
    ("histw-e256-second-B2", 256, 2, "second", 1, False),
    ("singlew-first-count2-binned", 2, 5, "first", 2, True),
]


def _case_path(case):
    _, n_edges, n_bins, weights, n_types, _ = case
    return kernel_path(weights != "none", n_edges, n_bins, n_types)


def test_path_cases_cover_every_launch():
    """the cases below and the union cases of `test_gpu_union_vs_oracle` reach every (CountPath, acc_global)
    combination that can be launched, every cumulative group size (7 and 8 edges in two passes), the listed edge and
    z-bin counts, and both sides of the 2048-byte accumulator limit for one and two first catalogs, weighted and
    unweighted"""
    from test_gpu_union_vs_oracle import UNION_CASES, union_case_path

    union = {union_case_path(c) for c in UNION_CASES}
    assert union == {("SingleUnion", False)}
    assert {1, 31, 32, 33, 64} <= {c[1] for c in UNION_CASES} and {c[2] for c in UNION_CASES} == {False, True}
    combos = {_case_path(c) for c in PATH_CASES} | union
    assert combos == {("Single", False), ("SingleWeighted", False), ("Cumulative", False), ("Histogram", False),
                      ("Histogram", True), ("HistogramWeighted", False), ("HistogramWeighted", True),
                      ("SingleUnion", False)}
    # count4 keeps per-catalog tiles with a weighted catalog, sub-bins or labels (test_four_counts_against_oracle,
    # test_second_labels_against_oracle), and the exact kernel counts one pair of catalogs at a time
    assert kernel_path(True, 2, 5, 2, n_second=2) == ("SingleWeighted", False)
    assert kernel_path(False, 5, 5, 2, n_second=2) == ("Cumulative", False)
    assert kernel_path(False, 2, 5, 2, n_second=2, labels=True) == ("Single", False)
    assert kernel_path(False, 2, 5, 1, exact=True) == ("Exact", False)
    cum = [c[1] for c in PATH_CASES if _case_path(c)[0] == "Cumulative"]
    assert {cumul_group(e) for e in cum} == {3, 4, 6} and {7, 8} <= set(cum)
    assert {2, 3, 4, 5, 6, 7, 8, 9, 33, 34, 256} <= {c[1] for c in PATH_CASES}
    assert {1, 31, 32, 33, 64} <= {c[2] for c in PATH_CASES}
    for n_types in (1, 2):
        for weighted in (False, True):
            sides = set()
            for c in PATH_CASES:
                path, glob = _case_path(c)
                if c[4] == n_types and (c[3] != "none") == weighted and path.startswith("Histogram"):
                    acc = n_types * c[2] * (c[1] - 1) * (16 if weighted else 8)
                    sides.add(glob)
                    assert glob == (acc > 2048)
            assert sides == {False, True}, (n_types, weighted)
    # the last per-warp table of a sub-bin path, `cum`, alone takes 64 bytes per z-bin and warp: 256 z-bins need
    # more than a quarter of the 227 KB of an SM, so the kernel runs with fewer than STREAM_CTAS CTAs per SM
    assert STREAM_WARPS * 256 * 16 * 4 + 1024 > 227 * 1024 // STREAM_CTAS


def _path_catalogs(rng, n_bins, weights, n_types, binned2):
    n_patch = 6
    ra, dec = (0.0, 0.06), (-0.03, 0.03)

    def cat(n, w):
        xyz, r, _ = sky(rng, n, ra, dec)
        patch = np.minimum((r / 0.01).astype(int), n_patch - 1)
        z = rng.integers(0, n_bins, n)
        z[rng.random(n) < 0.05] = -1
        if w:  # 400 rows at one position in one z-bin: one sort key, whose rows the index stores in any order
            xyz[1000:1400], patch[1000:1400], z[1000:1400] = xyz[1000].copy(), patch[1000], 0
        return xyz, patch, z, rng.uniform(0.5, 1.5, n) if w else None

    firsts = []
    for k, n in enumerate((12000, 7000)[:n_types]):  # "first": the first of two first catalogs only
        xyz, patch, z, w = cat(n, weights == "both" or (weights == "first" and k == 0))
        firsts.append(Rows(xyz, patch, n_patch, z, w))
    xyz, patch, z, w = cat(16000, weights in ("second", "both"))
    xyz[:600], patch[:600] = firsts[0].xyz[:600], firsts[0].patch[:600]  # duplicated rows: d2 = 0
    second = Rows(xyz, patch, n_patch, z if binned2 else None, w)
    return firsts, second


@pytest.mark.parametrize("case", PATH_CASES, ids=[c[0] for c in PATH_CASES])
def test_paths_against_oracle(engine, case):
    name, n_edges, n_bins, weights, n_types, binned2 = case
    rng = np.random.default_rng(1000 + PATH_CASES.index(case))
    firsts, second = _path_catalogs(rng, n_bins, weights, n_types, binned2)
    edges = thresholds(rng, n_bins, n_edges, 2e-4, 3e-3)
    pi, pj = all_pairs(6)
    d1 = [r.upload(engine, n_bins) for r in firsts]
    d2 = second.upload(engine, n_bins if binned2 else None)
    weighted = weights != "none"
    wants = [expect(r, second, pi, pj, edges, binned2=binned2) for r in firsts]
    if n_types == 1:
        ci, cf, st = engine.count(d1[0], d2, pi, pj, edges)
        got = [(ci, cf)]
    else:
        a, b, st = engine.count2(d1[0], d1[1], d2, pi, pj, edges)
        got = [a, b]
    for k, ((gi, gf), (wi, wf)) in enumerate(zip(got, wants)):
        compare(gi, gf, wi, wf, weighted, f"{name}: first catalog {k}")
    assert 0 < st["pair_tests"] < st["pair_tests_naive"]  # the planner and the query boxes pruned
    for k, (d, (wi, wf)) in enumerate(zip(d1, wants)):  # the exact kernel, one first catalog at a time
        ei, ef, es = engine.count(d, d2, pi, pj, edges, exact=True)
        compare(ei, ef, wi, wf, weighted, f"{name}: exact kernel, first catalog {k}")
        assert es["pair_tests"] == es["pair_tests_naive"]
    for d in (*d1, d2):
        d.free()


def test_four_counts_against_oracle(engine):
    """`count4` (two first x two second catalogs in one launch): every output against the oracle, weights on one
    second catalog only, single-bin, cumulative and histogram paths"""
    rng = np.random.default_rng(77)
    n_patch, n_bins = 6, 5
    for n_edges, w2a, w2b in ((2, False, True), (5, False, False), (12, True, False)):
        def cat(n, binned, w):
            xyz, r, _ = sky(rng, n, (0.0, 0.06), (-0.03, 0.03))
            patch = np.minimum((r / 0.01).astype(int), n_patch - 1)
            return Rows(xyz, patch, n_patch, rng.integers(-1, n_bins, n) if binned else None,
                        rng.uniform(0.5, 1.5, n) if w else None)

        r1a, r1b = cat(5000, True, False), cat(9000, True, False)
        r2a, r2b = cat(11000, False, w2a), cat(14000, False, w2b)
        edges = thresholds(rng, n_bins, n_edges, 2e-4, 3e-3)
        pi, pj = all_pairs(n_patch)
        devs = [r1a.upload(engine, n_bins), r1b.upload(engine, n_bins), r2a.upload(engine), r2b.upload(engine)]
        out, st = engine.count4(*devs, pi, pj, edges)
        for (gi, gf), (c1, c2) in zip(out, ((r1a, r2a), (r1b, r2a), (r1a, r2b), (r1b, r2b))):
            wi, wf = expect(c1, c2, pi, pj, edges, binned2=False)
            compare(gi, gf, wi, wf, c2.w is not None, f"count4, {n_edges} edges")
        assert 0 < st["pair_tests"] < st["pair_tests_naive"]
        for d in devs:
            d.free()


# --------------------------------------------------------------------------------------------------------------------
# 2. a large job: items of CCAP runs, and single z-bins of more than CCAP cell rows split into row ranges
# --------------------------------------------------------------------------------------------------------------------
def _grid_rows(rows: Rows, n_bins: int) -> np.ndarray:
    """cell rows (gv) of the sky-cell grid of every patch of a first-role index (`findex_build`)"""
    gv = np.zeros(rows.n_patch, dtype=np.int64)
    for p in range(rows.n_patch):
        x = rows.xyz[rows.off[p]:rows.off[p + 1]]
        c = x.sum(axis=0)
        c /= np.linalg.norm(c)
        a = np.array([1.0, 0.0, 0.0]) if abs(c[2]) > 0.9 else np.array([0.0, 0.0, 1.0])
        e1 = np.cross(a, c)
        e1 /= np.linalg.norm(e1)
        e2 = np.cross(c, e1)
        u, v = (x - c) @ e1, (x - c) @ e2
        du, dv = u.max() - u.min(), v.max() - v.min()
        cell = math.sqrt(TARGET_PER_CELL * max(du * dv, 1e-30) / max(len(x) / n_bins, 1.0))
        cell = max(cell, max(du, dv) / MAX_GRID_SPAN_CELLS)
        gv[p] = int(math.floor(dv / cell)) + 1
    return gv


LARGE_PATHS = [(2, "none"), (6, "none"), (12, "none"), (2, "second"), (5, "both")]


@pytest.mark.parametrize("n_edges,weights", LARGE_PATHS, ids=[f"e{e}-{w}" for e, w in LARGE_PATHS])
def test_large_job_with_row_split(engine, n_edges, weights):
    """56 patches of random rows on one narrow strip (3e-6 x 0.2 rad, running north-south): every patch overlaps
    every other, so all 3136 patch pairs are linked, and a second catalog with a few rows in each of 64 z-bins of
    each patch makes more than twice the (pair, tile) combinations of the small-job limit.  The first catalog's
    grids have 180-300 cell rows (one column), and a search radius longer than the strip makes every query span all
    of them: every item is a single z-bin with more than CCAP cell rows, which the planner must cut into row ranges."""
    rng = np.random.default_rng(2024 + n_edges)
    n_patch, n_bins = 56, 64
    strip_ra, strip_dec = (0.0, 3.2e-6), (-0.1, 0.1)

    def cat(per_seg, w):
        n = n_patch * n_bins * per_seg
        xyz, _, _ = sky(rng, n, strip_ra, strip_dec)
        return Rows(xyz, rng.integers(0, n_patch, n), n_patch, rng.integers(0, n_bins, n),
                    rng.uniform(0.5, 1.5, n) if w else None)

    r1 = cat(5, weights in ("first", "both"))
    r2 = cat(4, weights in ("second", "both"))
    pi, pj = all_pairs(n_patch)
    # the job is large: (pair, tile) combinations; the straggler guard of the tile table can only add tiles
    seg2 = np.zeros((n_patch, n_bins), dtype=np.int64)
    np.add.at(seg2, (r2.patch, r2.zbin), 1)
    n_flat = int(((seg2 + TILE - 1) // TILE).sum(axis=1)[pj].sum())
    threshold = SMALL_JOB_ITEMS * engine.num_sms * STREAM_CTAS * STREAM_WARPS
    print(f"large job: {n_flat} (pair, tile) combinations, small-job threshold {threshold} ({engine.num_sms} SMs)")
    assert n_flat > 2 * threshold
    # every query of every item spans all cell rows of its grid, and those are more than CCAP (at most 2 CCAP)
    gv = _grid_rows(r1, n_bins)
    assert gv.min() > CCAP + 20 and gv.max() <= 2 * CCAP - 20, (gv.min(), gv.max())
    edges = np.array([oracle.chord_sq_edges(np.geomspace(1e-3, 0.205 * s, n_edges))
                      for s in rng.uniform(1.0, 1.3, n_bins)])
    assert np.sqrt(edges[:, -1]).min() > 0.2  # longer than the strip
    d1, d2 = r1.upload(engine, n_bins), r2.upload(engine, n_bins)
    wi, wf = expect(r1, r2, pi, pj, edges, binned2=True)
    weighted = weights != "none"
    ci, cf, st = engine.count(d1, d2, pi, pj, edges)
    compare(ci, cf, wi, wf, weighted, "large job")
    assert st["work_items"] >= 2 * n_flat * 0.9  # nearly every (pair, tile) became two items
    ei, ef, _ = engine.count(d1, d2, pi, pj, edges, exact=True)
    compare(ei, ef, wi, wf, weighted, "large job, exact kernel")
    d1.free(); d2.free()


# --------------------------------------------------------------------------------------------------------------------
# 3. geometry: pole, RA = 0, a patch of more than 90 degrees, very large and very small angles, short tiles, hollow
# patches, and a strip among thousands of patches
# --------------------------------------------------------------------------------------------------------------------
def _geometry(rng, name):
    """(first catalog, second catalog, n_patch, (theta_lo, theta_hi) in radian)"""
    if name == "pole":  # a cap around the north pole, four patches of RA quadrants meeting at the pole
        def cat(n):
            xyz, r, _ = sky(rng, n, (0.0, 2.0 * np.pi), (np.deg2rad(86.0), np.pi / 2))
            return xyz, (r // (np.pi / 2)).astype(int) % 4
        (x1, p1), (x2, p2) = cat(8000), cat(10000)
        return Rows(x1, p1, 4), Rows(x2, p2, 4), 4, (2e-4, 1.5e-2)
    if name == "ra0":  # four patches meeting at RA = 0 on the equator
        def cat(n):
            xyz, r, d = sky(rng, n, (-0.04, 0.04), (-0.04, 0.04))
            return xyz, (r >= 0).astype(int) + 2 * (d >= 0).astype(int)
        (x1, p1), (x2, p2) = cat(9000), cat(11000)
        return Rows(x1, p1, 4), Rows(x2, p2, 4), 4, (2e-4, 8e-3)
    if name.startswith("wide"):  # the sky above Dec = -40 deg is one patch (radius > 90 deg), the rest another
        theta = np.deg2rad(float(name[4:]))
        def cat(n):
            xyz, _, d = sky(rng, n, (0.0, 2.0 * np.pi), (-np.pi / 2, np.pi / 2))
            return xyz, (d < np.deg2rad(-40.0)).astype(int)
        (x1, p1), (x2, p2) = cat(2500), cat(3000)
        return Rows(x1, p1, 2), Rows(x2, p2, 2), 2, (theta / 3, theta)
    if name == "tiny":  # sparse rows, each first row with a second row within 1.5e-6 rad
        n = 3000
        x1, r, d = sky(rng, n, (0.0, 0.5), (-0.25, 0.25))
        x2 = oracle.radec_to_xyz(r + rng.uniform(-1e-6, 1e-6, n) / np.cos(d), d + rng.uniform(-1e-6, 1e-6, n))
        xr, rr, _ = sky(rng, n, (0.0, 0.5), (-0.25, 0.25))
        p1 = np.minimum((r / 0.125).astype(int), 3)
        p2 = np.concatenate([p1, np.minimum((rr / 0.125).astype(int), 3)])
        return Rows(x1, p1, 4), Rows(np.concatenate([x2, xr]), p2, 4), 4, (1e-7, 1.5e-6)
    if name == "tiles":  # patches of 1, 255, 256, 257 and 513 rows: one tile of 1 row, full, full + 1 row, ...
        sizes2, sizes1 = [1, 255, 256, 257, 513], [300, 1, 256, 257, 255]
        x2, _, _ = sky(rng, sum(sizes2), (0.0, 0.02), (-0.01, 0.01))
        x1, _, _ = sky(rng, sum(sizes1), (0.0, 0.02), (-0.01, 0.01))
        p2 = np.repeat(np.arange(5), sizes2)
        p1 = np.repeat(np.arange(5), sizes1)
        return Rows(x1, p1, 5), Rows(x2, p2, 5), 5, (5e-4, 6e-3)
    if name == "irregular":  # a ring and an L: the Hilbert curve of a patch box crosses empty parts of the patch
        def cat(n):
            r, phi = np.sqrt(rng.uniform(0.012**2, 0.02**2, n)), rng.uniform(0.0, 2.0 * np.pi, n)
            u, v = rng.uniform(0.0, 0.04, 4 * n), rng.uniform(0.0, 0.04, 4 * n)
            keep = (u < 0.008) | (v < 0.008)
            ra = np.concatenate([0.05 + r * np.cos(phi), 0.08 + u[keep][:n]])
            dec = np.concatenate([r * np.sin(phi), -0.02 + v[keep][:n]])
            return oracle.radec_to_xyz(ra, dec), np.repeat([0, 1], n)
        (x1, p1), (x2, p2) = cat(6000), cat(10000)
        return Rows(x1, p1, 2), Rows(x2, p2, 2), 2, (2e-4, 1e-3)
    if name == "strip":  # 5000 patches, all but two empty: 5000 x 16 > 2^16 Hilbert cells leave one level of the curve
        # (two key bits) below each (patch, z-bin), and patch 0 is a 6 : 1 strip, wide enough for more than 4 squares
        def cat(n_strip, n_box):
            xs = sky(rng, n_strip, (0.0, 0.06), (-0.005, 0.005))[0]
            xb = sky(rng, n_box, (0.1, 0.11), (-0.005, 0.005))[0]
            return np.concatenate([xs, xb]), np.repeat([0, 1], [n_strip, n_box])
        (x1, p1), (x2, p2) = cat(3000, 500), cat(4000, 600)
        return Rows(x1, p1, 5000), Rows(x2, p2, 5000), 5000, (2e-4, 3e-3)
    if name == "off-sphere":  # rows 1e-6 off the unit sphere: the FP32 test widens its undecided band by that much
        def cat(n, dev):
            xyz, r, _ = sky(rng, n, (0.0, 0.02), (-0.01, 0.01))
            return xyz * (1.0 + dev * rng.uniform(-1.0, 1.0, n))[:, None], np.minimum((r / 0.01).astype(int), 1)
        (x1, p1), (x2, p2) = cat(8000, 1e-6), cat(10000, 1e-6)
        return Rows(x1, p1, 2), Rows(x2, p2, 2), 2, (2e-4, 2e-3)
    raise ValueError(name)


GEOMETRIES = ["pole", "ra0", "wide100", "wide150", "wide179", "tiny", "tiles", "off-sphere", "irregular", "strip"]


def second_role_index_bytes(engine, rows: Rows) -> int:
    """device bytes that the second-role index of the unbinned catalog `rows` adds to it"""
    dev = rows.upload(engine)
    before = dev.info()[1]
    dev.build_index(2)  # YAWB_ROLE_SECOND
    extra = dev.info()[1] - before
    dev.free()
    return extra


@pytest.mark.parametrize("name", GEOMETRIES)
def test_geometry_against_oracle(engine, name):
    rng = np.random.default_rng(GEOMETRIES.index(name) + 500)
    r1, r2, n_patch, (lo, hi) = _geometry(rng, name)
    n_bins = 3
    r1.zbin = rng.integers(0, n_bins, len(r1.xyz))
    r2.w = rng.uniform(0.5, 1.5, len(r2.xyz))
    if name == "irregular":  # the straggler guard cut tiles: more tiles than for as many rows per patch in compact patches
        compact = Rows(sky(rng, len(r2.xyz), (0.0, 0.04), (-0.02, 0.02))[0], r2.patch, n_patch, w=r2.w)
        assert second_role_index_bytes(engine, r2) > second_role_index_bytes(engine, compact)
    live = np.flatnonzero(np.diff(r1.off) * np.diff(r2.off))  # patches with rows in both catalogs
    pi, pj = (live[k].astype(np.int32) for k in all_pairs(len(live)))
    d1 = r1.upload(engine, n_bins)
    plain, weighted = Rows(r2.xyz, r2.patch, n_patch), r2
    for n_edges, second in ((2, plain), (5, plain), (12, plain), (2, weighted), (9, weighted)):
        # lower edges that differ per z-bin, the largest angle exactly
        edges = np.array([oracle.chord_sq_edges(np.geomspace(lo * s, hi, n_edges)) for s in rng.uniform(0.7, 1.0, n_bins)])
        d2 = second.upload(engine)
        wi, wf = expect(r1, second, pi, pj, edges, binned2=False)
        w = second.w is not None
        ci, cf, st = engine.count(d1, d2, pi, pj, edges)
        compare(ci, cf, wi, wf, w, f"{name}, {n_edges} edges")
        if not name.startswith("wide"):  # a search radius of 100 degrees and more reaches every row of the sky
            assert 0 < st["pair_tests"] < st["pair_tests_naive"]
        ei, ef, _ = engine.count(d1, d2, pi, pj, edges, exact=True)
        compare(ei, ef, wi, wf, w, f"{name}, {n_edges} edges, exact kernel")
        d2.free()
    d1.free()


# --------------------------------------------------------------------------------------------------------------------
# 4. uploads: int32 and uint8 z-bin ids, z-bins assigned on the device
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["int32", "uint8", "digitize-right", "digitize-left"])
def test_zbin_uploads_against_oracle(engine, mode):
    rng = np.random.default_rng(["int32", "uint8", "digitize-right", "digitize-left"].index(mode) + 40)
    n_patch, n_bins = 4, 7
    zedges = np.linspace(0.1, 1.0, n_bins + 1)
    closed = "left" if mode == "digitize-left" else "right"

    def cat(n, w):
        xyz, r, _ = sky(rng, n, (0.0, 0.04), (-0.02, 0.02))
        z = rng.uniform(0.0, 1.1, n)
        z[:300] = rng.choice(zedges, 300)  # on an edge
        z[300:310] = np.nan
        ids = np.digitize(z, zedges, right=closed == "right") - 1
        ids[(ids < 0) | (ids >= n_bins)] = -1
        return Rows(xyz, np.minimum((r / 0.01).astype(int), n_patch - 1), n_patch, ids,
                    rng.uniform(0.5, 1.5, n) if w else None, redshift=z)

    def up(rows):
        if mode.startswith("digitize"):
            return engine.upload_catalog(rows.xyz, rows.off, weights=rows.w, redshifts=rows.redshift, edges=zedges,
                                         closed=closed)
        if mode == "uint8":  # 255: dropped row
            ids = np.where(rows.zbin < 0, 255, rows.zbin).astype(np.uint8)
            return engine.upload_catalog(rows.xyz, rows.off, weights=rows.w, zbin=ids, n_bins=n_bins)
        return rows.upload(engine, n_bins)

    pi, pj = all_pairs(n_patch)
    for weighted_second, n_edges in ((False, 2), (True, 6), (False, 13)):
        r1, r2 = cat(10000, False), cat(14000, weighted_second)
        d1, d2 = up(r1), up(r2)
        assert d1.info()[0] == int((r1.zbin >= 0).sum())
        edges = thresholds(rng, n_bins, n_edges, 2e-4, 3e-3)
        wi, wf = expect(r1, r2, pi, pj, edges, binned2=True)
        ci, cf, st = engine.count(d1, d2, pi, pj, edges)
        compare(ci, cf, wi, wf, weighted_second, f"{mode}, {n_edges} edges")
        assert 0 < st["pair_tests"] < st["pair_tests_naive"]
        ei, ef, _ = engine.count(d1, d2, pi, pj, edges, exact=True)
        compare(ei, ef, wi, wf, weighted_second, f"{mode}, {n_edges} edges, exact kernel")
        d1.free(); d2.free()


# --------------------------------------------------------------------------------------------------------------------
# 5. labels: `labels=True` (the second catalog's ids are sample labels) and binned labels (`n_labels=`)
# --------------------------------------------------------------------------------------------------------------------
def _labelled_rows(rng, n, n_patch, n_ids, w):
    xyz, r, _ = sky(rng, n, (0.0, 0.04), (-0.02, 0.02))
    ids = rng.integers(0, n_ids, n)
    ids[rng.random(n) < 0.05] = -1
    return Rows(xyz, np.minimum((r / 0.01).astype(int), n_patch - 1), n_patch, ids,
                rng.uniform(0.5, 1.5, n) if w else None)


def test_second_labels_against_oracle(engine):
    """`labels=True`: every row of label l of the second catalog meets every z-bin of the first catalog, results
    in block l; `count`, `count2` and `count4` (a labelled and an unbinned second catalog in one launch)"""
    rng = np.random.default_rng(61)
    n_patch, n_bins, n_lab = 4, 5, 3
    pi, pj = all_pairs(n_patch)
    for n_edges, w in ((2, False), (6, False), (12, True), (2, True)):
        r1a = _labelled_rows(rng, 8000, n_patch, n_bins, False)
        r1b = _labelled_rows(rng, 5000, n_patch, n_bins, False)
        lab = _labelled_rows(rng, 12000, n_patch, n_lab, w)
        rand = Rows(sky(rng, 9000, (0.0, 0.04), (-0.02, 0.02))[0], rng.integers(0, n_patch, 9000), n_patch)
        edges = thresholds(rng, n_bins, n_edges, 2e-4, 3e-3)
        d1a, d1b, dl, dr = r1a.upload(engine, n_bins), r1b.upload(engine, n_bins), lab.upload(engine, n_lab), rand.upload(engine)

        def want(r1, r2, labelled):
            if not labelled:
                return expect(r1, r2, pi, pj, edges, binned2=False)
            return oracle.binned_pair_counts(r1.xyz, r1.patch, r1.zbin, r2.xyz, r2.patch, pi, pj, edges, w1=r1.w,
                                             w2=r2.w, label2=r2.zbin, n_labels=n_lab)

        wa, wb = want(r1a, lab, True), want(r1b, lab, True)
        ci, cf, st = engine.count(d1a, dl, pi, pj, edges, labels=True)
        compare(ci, cf, *wa, w, f"labels=True, {n_edges} edges")
        assert 0 < st["pair_tests"] < st["pair_tests_naive"]
        (ia, fa), (ib, fb), _ = engine.count2(d1a, d1b, dl, pi, pj, edges, labels=True)
        compare(ia, fa, *wa, w, f"count2 labels=True, {n_edges} edges")
        compare(ib, fb, *wb, w, f"count2 labels=True, {n_edges} edges")
        out, _ = engine.count4(d1a, d1b, dl, dr, pi, pj, edges, labels=True)
        for (gi, gf), (r1, r2, labelled) in zip(out, ((r1a, lab, True), (r1b, lab, True), (r1a, rand, False),
                                                      (r1b, rand, False))):
            wi, wf = want(r1, r2, labelled)
            if not labelled:
                assert gi.shape == (1, *wi.shape)  # an unbinned catalog is one label
                gi, gf = gi[0], gf[0]
            compare(gi, gf, wi, wf, r2.w is not None, f"count4 labels=True, {n_edges} edges")
        for d in (d1a, d1b, dl, dr):
            d.free()


@pytest.mark.parametrize("rule", ["same-labels", "unlabelled-first"])
def test_binned_labels_against_oracle(engine, rule):
    """binned labels (ids = label * B + z-bin): row (l, z) of the second catalog meets row (l, z) of a first
    catalog with the same labels, or row z of a binned first catalog without labels; results in block l"""
    rng = np.random.default_rng(71 + (rule == "same-labels"))
    n_patch, n_bins, n_lab = 4, 6, 4
    pi, pj = all_pairs(n_patch)
    for n_edges, w1, w2 in ((2, False, False), (5, False, False), (9, True, False), (2, False, True), (14, True, True)):
        lab = _labelled_rows(rng, 14000, n_patch, n_lab * n_bins, w2)
        dl = engine.upload_catalog(lab.xyz, lab.off, weights=lab.w,
                                   zbin=np.where(lab.zbin < 0, 255, lab.zbin).astype(np.uint8),
                                   n_bins=n_lab * n_bins, n_labels=n_lab)
        if rule == "same-labels":
            r1 = _labelled_rows(rng, 9000, n_patch, n_lab * n_bins, w1)
            d1 = engine.upload_catalog(r1.xyz, r1.off, weights=r1.w, zbin=r1.zbin.astype(np.int32),
                                       n_bins=n_lab * n_bins, n_labels=n_lab)
            z1 = np.where(r1.zbin < 0, -1, r1.zbin % n_bins)
            l1 = np.where(r1.zbin < 0, -1, r1.zbin // n_bins)
        else:
            r1 = _labelled_rows(rng, 9000, n_patch, n_bins, w1)
            d1 = r1.upload(engine, n_bins)
            z1, l1 = r1.zbin, None
        edges = thresholds(rng, n_bins, n_edges, 2e-4, 3e-3)
        wi, wf = oracle.binned_pair_counts(r1.xyz, r1.patch, z1, lab.xyz, lab.patch, pi, pj, edges, w1=r1.w, w2=lab.w,
                                           zbin2=np.where(lab.zbin < 0, -1, lab.zbin % n_bins),
                                           label1=l1, label2=np.where(lab.zbin < 0, -1, lab.zbin // n_bins),
                                           n_labels=n_lab)
        ci, cf, st = engine.count(d1, dl, pi, pj, edges)
        compare(ci, cf, wi, wf, w1 or w2, f"binned labels ({rule}), {n_edges} edges")
        assert 0 < st["pair_tests"] < st["pair_tests_naive"]
        d1.free(); dl.free()


# --------------------------------------------------------------------------------------------------------------------
# 6. rejections
# --------------------------------------------------------------------------------------------------------------------
def test_rejections_leave_the_engine_usable(engine):
    """a count whose per-warp tables exceed 227 KB of shared memory (700 z-bins x 255 sub-bins, weighted) and a count
    with 257 edges are refused with their messages; the same engine then still counts what the oracle counts"""
    from yet_another_wizz_b200._lib import YawbError

    rng = np.random.default_rng(91)
    n_patch, n_bins = 2, 700
    xyz, r, _ = sky(rng, 20000, (0.0, 0.02), (-0.01, 0.01))
    big = Rows(xyz, (r > 0.01).astype(int), n_patch, rng.integers(0, n_bins, 20000), rng.uniform(0.5, 1.5, 20000))
    other = Rows(sky(rng, 5000, (0.0, 0.02), (-0.01, 0.01))[0], rng.integers(0, n_patch, 5000), n_patch)
    d1, d2 = big.upload(engine, n_bins), other.upload(engine)
    pi, pj = all_pairs(n_patch)
    edges = thresholds(rng, n_bins, 256, 1e-4, 2e-3, variety=False)
    with pytest.raises(YawbError, match="too many z-bins x sub-bins for the shared-memory accumulators"):
        engine.count(d1, d2, pi, pj, edges)
    with pytest.raises(YawbError, match=r"n_edges must be in 2\.\.256 \(got 257\)"):
        engine.count(d1, d2, pi, pj, thresholds(rng, n_bins, 257, 1e-4, 2e-3, variety=False))
    # 700 weighted z-bins need 236 288 B even with one sub-bin; the same rows in 7 z-bins, on the same engine:
    few = Rows(big.xyz, big.patch, n_patch, big.zbin % 7, big.w)
    d7 = few.upload(engine, 7)
    for n_edges in (2, 40):
        edges = thresholds(rng, 7, n_edges, 1e-4, 2e-3)
        wi, wf = expect(few, other, pi, pj, edges, binned2=False)
        ci, cf, _ = engine.count(d7, d2, pi, pj, edges)
        compare(ci, cf, wi, wf, True, f"after the rejections, {n_edges} edges")
    for d in (d1, d2, d7):
        d.free()
