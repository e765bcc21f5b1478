"""
`count4` on its single-bin path cuts the register tiles from ONE second-role index over the union of both second
catalogs: a tile holds rows of both, and every count is split by the catalog of the row.  Each case compares the four
outputs with four separate `count` calls (per-catalog tiles) and with the FP64 exact kernel, both of which see one
second catalog at a time.

Cases: equal and very unequal second-catalog sizes, a second catalog without rows in some patches, rows within a few
ulp of a bin edge (the FP64 recheck has to split one lane's count between the two catalogs), rows off the unit sphere,
and a recount after `drop_index()` of one catalog.
"""

import numpy as np
import pytest
from numpy.testing import assert_array_equal

import golden_io
import oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from yet_another_wizz_b200 import Engine

    eng = Engine(0)
    yield eng
    eng.close()


def sky(rng, n, ra, dec):
    r = rng.uniform(ra[0], ra[1], n)
    d = np.arcsin(rng.uniform(np.sin(dec[0]), np.sin(dec[1]), n))
    return oracle.radec_to_xyz(r, d), r


def upload(engine, xyz, patch, n_patch, zbin=None, n_bins=None):
    order = np.argsort(patch, kind="stable")
    off = np.concatenate([[0], np.cumsum(np.bincount(patch, minlength=n_patch))]).astype(np.int64)
    if zbin is None:
        return engine.upload_catalog(np.ascontiguousarray(xyz[order]), off)
    return engine.upload_catalog(np.ascontiguousarray(xyz[order]), off, zbin=zbin[order].astype(np.int32), n_bins=n_bins)


def check_four(engine, firsts, seconds, pi, pj, edges, what):
    """count4 against count and against the exact kernel, output by output; returns count4's stats and the summed
    pair tests of the four separate counts"""
    out, st = engine.count4(*firsts, *seconds, pi, pj, edges)
    separate_tests = 0
    for (gi, gf), (c1, c2) in zip(out, ((0, 0), (1, 0), (0, 1), (1, 1))):
        wi, _, s = engine.count(firsts[c1], seconds[c2], pi, pj, edges)
        ei, _, _ = engine.count(firsts[c1], seconds[c2], pi, pj, edges, exact=True)
        assert_array_equal(ei, wi, err_msg=f"{what}: count vs exact kernel ({c1}, {c2})")
        assert_array_equal(gi, wi, err_msg=f"{what}: count4 vs count ({c1}, {c2})")
        assert_array_equal(gf, wi.astype(np.float64), err_msg=what)
        separate_tests += s["pair_tests"]
    assert sum(o[0].sum() for o in out) > 0, what
    return st, separate_tests


@pytest.mark.parametrize("sizes", [(20000, 20000), (40000, 4000), (3000, 30000)])
def test_union_tiles_sizes(engine, sizes):
    rng = np.random.default_rng(sum(sizes))
    n_patch, n_bins = 6, 4

    def pos(n):
        xyz, r = sky(rng, n, (0.0, 0.06), (-0.03, 0.03))
        return xyz, np.minimum((r / 0.01).astype(int), n_patch - 1)

    firsts = [upload(engine, *pos(n), n_patch, rng.integers(-1, n_bins, n), n_bins) for n in (6000, 12000)]
    seconds = [upload(engine, *pos(n), n_patch) for n in sizes]
    edges = np.array([oracle.chord_sq_edges(np.array([1e-4, 2e-3]) * s) for s in rng.uniform(0.7, 1.3, n_bins)])
    pi, pj = (a.ravel().astype(np.int32) for a in np.meshgrid(np.arange(n_patch), np.arange(n_patch), indexing="ij"))
    st, separate = check_four(engine, firsts, seconds, pi, pj, edges, f"sizes {sizes}")
    if sizes[0] == sizes[1]:  # tiles over both catalogs cover half the sky: fewer tests than per-catalog tiles
        assert st["pair_tests"] < 0.9 * separate
    for d in firsts + seconds:
        d.free()


def test_union_tiles_empty_patches(engine):
    """one second catalog has no rows in two patches, the other none in a third"""
    rng = np.random.default_rng(5)
    n_patch, n_bins = 5, 3

    def pos(n, skip=()):
        xyz, r = sky(rng, n, (0.0, 0.05), (-0.02, 0.02))
        patch = np.minimum((r / 0.01).astype(int), n_patch - 1)
        keep = ~np.isin(patch, skip)
        return xyz[keep], patch[keep]

    firsts = []
    for n in (5000, 8000):
        xyz, patch = pos(n)
        firsts.append(upload(engine, xyz, patch, n_patch, rng.integers(0, n_bins, len(patch)), n_bins))
    seconds = [upload(engine, *pos(15000, (1, 3)), n_patch), upload(engine, *pos(9000, (2,)), n_patch)]
    edges = np.array([oracle.chord_sq_edges(np.array([0.0, 1.5e-3]) * s) for s in rng.uniform(0.7, 1.3, n_bins)])
    pi, pj = (a.ravel().astype(np.int32) for a in np.meshgrid(np.arange(n_patch), np.arange(n_patch), indexing="ij"))
    check_four(engine, firsts, seconds, pi, pj, edges, "empty patches")
    for d in firsts + seconds:
        d.free()


def test_union_tiles_edge_adversarial(engine):
    """pairs within a few ulp of the edges: the second catalogs take alternate rows of the golden catalog, so that a
    lane flagged for the FP64 recheck holds rows of both"""
    g = golden_io.load("edge_adversarial")
    a, b = g["a_xyz"], g["b_xyz"]
    lim = oracle.parse_ang_limits(g["upper_ang_min"], g["upper_ang_max"])
    r2 = oracle.chord_sq_edges(oracle.get_ang_bins(lim, None, 50))
    assert len(r2) == 2
    one = np.zeros(len(a), dtype=int)
    firsts = [upload(engine, a, one, 1, np.zeros(len(a)), 1), upload(engine, a[::3], one[::3], 1, np.zeros(len(a[::3])), 1)]
    seconds = [upload(engine, b[0::2], np.zeros(len(b[0::2]), dtype=int), 1),
               upload(engine, b[1::2], np.zeros(len(b[1::2]), dtype=int), 1)]
    pi = pj = np.zeros(1, dtype=np.int32)
    st, _ = check_four(engine, firsts, seconds, pi, pj, r2[None, :], "edge_adversarial")
    assert st["rechecks"] > 0
    out, _ = engine.count4(*firsts, *seconds, pi, pj, r2[None, :])
    whole = oracle.pair_histogram(a, b, None, None, r2)  # both second catalogs together are the golden b
    assert_array_equal(out[0][0][0, 0] + out[2][0][0, 0], whole)
    for d in firsts + seconds:
        d.free()


def test_union_tiles_off_sphere(engine):
    """rows 1e-6 off the unit sphere in both second catalogs"""
    rng = np.random.default_rng(11)
    n_patch, n_bins = 2, 3

    def pos(n, dev=0.0):
        xyz, r = sky(rng, n, (0.0, 0.02), (-0.01, 0.01))
        return xyz * (1.0 + dev * rng.uniform(-1.0, 1.0, n))[:, None], np.minimum((r / 0.01).astype(int), n_patch - 1)

    firsts = [upload(engine, *pos(n, 1e-6), n_patch, rng.integers(0, n_bins, n), n_bins) for n in (6000, 9000)]
    seconds = [upload(engine, *pos(n, 1e-6), n_patch) for n in (10000, 7000)]
    edges = np.array([oracle.chord_sq_edges(np.array([2e-4, 2e-3]) * s) for s in rng.uniform(0.7, 1.0, n_bins)])
    pi, pj = (a.ravel().astype(np.int32) for a in np.meshgrid(np.arange(n_patch), np.arange(n_patch), indexing="ij"))
    check_four(engine, firsts, seconds, pi, pj, edges, "off-sphere")
    for d in firsts + seconds:
        d.free()


def test_union_tiles_drop_index(engine):
    """the union index is cached with both catalogs and rebuilt after `drop_index()` of either"""
    rng = np.random.default_rng(23)
    n_patch, n_bins = 4, 3

    def pos(n):
        xyz, r = sky(rng, n, (0.0, 0.04), (-0.02, 0.02))
        return xyz, np.minimum((r / 0.01).astype(int), n_patch - 1)

    firsts = [upload(engine, *pos(n), n_patch, rng.integers(0, n_bins, n), n_bins) for n in (5000, 7000)]
    seconds = [upload(engine, *pos(n), n_patch) for n in (12000, 9000)]
    edges = np.array([oracle.chord_sq_edges(np.array([1e-4, 2e-3]) * s) for s in rng.uniform(0.7, 1.3, n_bins)])
    pi, pj = (a.ravel().astype(np.int32) for a in np.meshgrid(np.arange(n_patch), np.arange(n_patch), indexing="ij"))
    first, _ = engine.count4(*firsts, *seconds, pi, pj, edges)
    again, st = engine.count4(*firsts, *seconds, pi, pj, edges)
    assert st["index_ms"] == 0.0  # every index was cached
    for dropped in (seconds[1], seconds[0]):
        dropped.drop_index()
        out, st = engine.count4(*firsts, *seconds, pi, pj, edges)
        assert st["index_ms"] > 0.0
        for (gi, _), (wi, _), (ai, _) in zip(out, first, again):
            assert_array_equal(gi, wi)
            assert_array_equal(ai, wi)
    # ... and a freed catalog takes the union with it: a new catalog in its place is counted from its own rows
    seconds[1].free()
    seconds[1] = upload(engine, *pos(9000), n_patch)
    check_four(engine, firsts, seconds, pi, pj, edges, "after free")
    for d in firsts + seconds:
        d.free()
