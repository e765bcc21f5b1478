"""
GPU parity tests at the C-ABI level (`yawb_count` vs the oracle), the
equivalent of the reference's `tests/catalog/test_trees.py::TestAngularTree`.

Bar: integer pair counts bit-exact; weighted sums within 1e-12 relative.
"""

from itertools import product

import numpy as np
import pytest
from numpy.testing import assert_allclose, assert_array_equal

import golden_io
import oracle

pytestmark = pytest.mark.gpu

RTOL_WEIGHTED = 1e-12
DELTA = 1e-9


@pytest.fixture(scope="module")
def engine():
    from yet_another_wizz_b200 import Engine

    eng = Engine(0)
    yield eng
    eng.close()


def great_circle_points():
    points = np.array([[0.0, 0.0], [90.0, 0.0], [180.0, 0.0], [270.0, 0.0], [0.0, 90.0], [0.0, -90.0]])
    base = np.arange(1.0, 90.0, 1.0)
    for offset in (0.0, 90.0, 180.0, 270.0):
        points = np.concatenate([points, np.column_stack([base + offset, np.zeros_like(base)])])
    for sign, ra in product([-1.0, 1.0], [0.0, 180.0]):
        points = np.concatenate([points, np.column_stack([np.full_like(base, ra), sign * base])])
    for sign, ra in product([-1.0, 1.0], [90.0, 270.0]):
        points = np.concatenate([points, np.column_stack([np.full_like(base, ra), sign * base])])
    radec = np.deg2rad(points)
    return oracle.radec_to_xyz(radec[:, 0], radec[:, 1])


def single_patch_hist(engine, xyz1, w1, xyz2, w2, r2, exact):
    c1 = engine.upload_catalog(xyz1, np.array([0, len(xyz1)]), weights=w1)
    c2 = engine.upload_catalog(xyz2, np.array([0, len(xyz2)]), weights=w2)
    ci, cf, stats = engine.count(c1, c2, [0], [0], r2, exact=exact)
    c1.free(); c2.free()
    return ci[0, 0], cf[0, 0], stats


@pytest.mark.parametrize("exact", [True, False])
class TestGreatCircleKAT:
    """reference tests/catalog/test_trees.py:181-247 through the C ABI"""

    @pytest.mark.parametrize("ang_max", [1.0, 2.0, 10.0, 89.0])
    def test_count_single(self, engine, ang_max, exact):
        pts = great_circle_points()
        single = oracle.radec_to_xyz(np.array([0.0]), np.array([0.0]))
        amax = ang_max + DELTA
        r2 = oracle.chord_sq_edges(np.deg2rad([amax - 1.0, amax]))
        ci, cf, _ = single_patch_hist(engine, pts, np.full(len(pts), 2.0), single, np.array([2.0]), r2, exact)
        assert ci[0] == 4
        assert cf[0] == 4 * 2.0**2

    @pytest.mark.parametrize("ang_max", [2.0, 10.0, 89.0])
    def test_count_bins(self, engine, ang_max, exact):
        pts = great_circle_points()
        single = oracle.radec_to_xyz(np.array([0.0]), np.array([0.0]))
        edges = np.deg2rad(np.concatenate([[0.0], np.arange(1.0, ang_max)]) + DELTA)
        r2 = oracle.chord_sq_edges(edges)
        ci, cf, _ = single_patch_hist(engine, pts, None, single, None, r2, exact)
        assert_array_equal(ci, np.full(len(edges) - 1, 4))
        assert_array_equal(cf, np.full(len(edges) - 1, 4.0))

    def test_count_dualtree(self, engine, exact):
        pts = great_circle_points()
        r2 = oracle.chord_sq_edges(np.deg2rad([0.0, 1.0]) + DELTA)
        ci, _, _ = single_patch_hist(engine, pts, None, pts, None, r2, exact)
        assert ci[0] == 4 * 6 + 2 * (len(pts) - 6)

    def test_count_empty(self, engine, exact):
        empty = np.empty((0, 3))
        r2 = oracle.chord_sq_edges(np.array([0.1, 0.5, 1.0]))
        ci, cf, _ = single_patch_hist(engine, empty, None, empty, None, r2, exact)
        assert_array_equal(ci, [0, 0])
        pts = great_circle_points()
        ci, cf, _ = single_patch_hist(engine, pts, None, empty, None, r2, exact)
        assert_array_equal(ci, [0, 0])


def engine_inputs(cat: dict, zedges, closed, binned: bool):
    xyz = oracle.radec_to_xyz(cat["ra"], cat["dec"])
    n_patch = len(cat["radii"])
    order = np.argsort(cat["patch"], kind="stable")
    patch_off = np.concatenate([[0], np.cumsum(np.bincount(cat["patch"], minlength=n_patch))])
    zbin = None
    if binned:
        zbin = (np.digitize(cat["z"], zedges, right=(closed == "right")) - 1)[order].astype(np.int32)
    w = None if cat["w"] is None else cat["w"][order]
    return xyz[order], patch_off, w, zbin


def oracle_hists(cat1, cat2, pairs, zedges, closed, r2, binned2):
    """brute-force sub-bin histograms per (pair, z-bin) with the oracle"""
    n_bins = len(zedges) - 1
    xyz1 = oracle.radec_to_xyz(cat1["ra"], cat1["dec"])
    xyz2 = oracle.radec_to_xyz(cat2["ra"], cat2["dec"])
    b1 = np.digitize(cat1["z"], zedges, right=(closed == "right")) - 1
    b2 = np.digitize(cat2["z"], zedges, right=(closed == "right")) - 1 if binned2 else None
    weighted = cat1["w"] is not None or cat2["w"] is not None
    out = np.zeros((len(pairs), n_bins, r2.shape[1] - 1), dtype=np.float64 if weighted else np.int64)
    for k, (i, j) in enumerate(pairs):
        for b in range(n_bins):
            m1 = (cat1["patch"] == i) & (b1 == b)
            m2 = (cat2["patch"] == j) & ((b2 == b) if binned2 else True)
            w1 = None if cat1["w"] is None else cat1["w"][m1]
            w2 = None if cat2["w"] is None else cat2["w"][m2]
            out[k, b] = oracle.pair_histogram(xyz1[m1], xyz2[m2], w1, w2, r2[b])
    return out


def r2_table(cfg):
    rows = []
    for b in range(len(cfg["zedges"]) - 1):
        lim = oracle.parse_ang_limits(cfg["ang_min"][b], cfg["ang_max"][b])
        rows.append(oracle.chord_sq_edges(oracle.get_ang_bins(lim, cfg["rweight"], cfg["resolution"])))
    return np.array(rows)


@pytest.mark.parametrize("exact", [True, False])
@pytest.mark.parametrize("name", ["cross_unweighted", "cross_weighted_multiscale"])
def test_cross_histograms_match_oracle(engine, name, exact):
    g = golden_io.load(name)
    cfg = golden_io.config_of(g)
    r2 = r2_table(cfg)
    pairs = [tuple(p) for p in g["links"]]
    pi = np.array([p[0] for p in pairs]); pj = np.array([p[1] for p in pairs])
    n_bins = len(cfg["zedges"]) - 1
    for a, b in (("ref", "unk"), ("ref", "unk_rand"), ("ref_rand", "unk"), ("ref_rand", "unk_rand")):
        ca, cb = golden_io.catalog_arrays(g, a), golden_io.catalog_arrays(g, b)
        xyz1, off1, w1, z1 = engine_inputs(ca, cfg["zedges"], cfg["closed"], True)
        xyz2, off2, w2, _ = engine_inputs(cb, cfg["zedges"], cfg["closed"], False)
        d1 = engine.upload_catalog(xyz1, off1, weights=w1, zbin=z1, n_bins=n_bins)
        d2 = engine.upload_catalog(xyz2, off2, weights=w2)
        ci, cf, stats = engine.count(d1, d2, pi, pj, r2, exact=exact)
        want = oracle_hists(ca, cb, pairs, cfg["zedges"], cfg["closed"], r2, False)
        if want.dtype == np.int64:
            assert_array_equal(ci, want)
            assert_array_equal(cf, want.astype(np.float64))
        else:
            assert_allclose(cf, want, rtol=RTOL_WEIGHTED, atol=0)
        assert want.sum() > 0
        # sum of weights, trees.py:225-234
        sw = d1.sum_weights()
        for b in range(n_bins):
            for p in range(len(ca["radii"])):
                m = (ca["patch"] == p) & (np.digitize(ca["z"], cfg["zedges"], right=cfg["closed"] == "right") - 1 == b)
                exp = m.sum() if ca["w"] is None else ca["w"][m].sum()
                assert_allclose(sw[b, p], exp, rtol=1e-13)
        d1.free(); d2.free()


@pytest.mark.parametrize("exact", [True, False])
@pytest.mark.parametrize("name", ["auto_unweighted", "auto_rweight_polewrap"])
def test_auto_histograms_match_oracle(engine, name, exact):
    g = golden_io.load(name)
    cfg = golden_io.config_of(g)
    r2 = r2_table(cfg)
    pairs = [tuple(p) for p in g["links"]]
    pi = np.array([p[0] for p in pairs]); pj = np.array([p[1] for p in pairs])
    n_bins = len(cfg["zedges"]) - 1
    data, rand = golden_io.catalog_arrays(g, "data"), golden_io.catalog_arrays(g, "rand")
    for ca, cb in ((data, data), (data, rand), (rand, rand)):
        xyz1, off1, w1, z1 = engine_inputs(ca, cfg["zedges"], cfg["closed"], True)
        xyz2, off2, w2, z2 = engine_inputs(cb, cfg["zedges"], cfg["closed"], True)
        d1 = engine.upload_catalog(xyz1, off1, weights=w1, zbin=z1, n_bins=n_bins)
        d2 = engine.upload_catalog(xyz2, off2, weights=w2, zbin=z2, n_bins=n_bins)
        ci, cf, stats = engine.count(d1, d2, pi, pj, r2, exact=exact)
        want = oracle_hists(ca, cb, pairs, cfg["zedges"], cfg["closed"], r2, True)
        if want.dtype == np.int64:
            assert_array_equal(ci, want)
        else:
            assert_allclose(cf, want, rtol=RTOL_WEIGHTED, atol=0)
        d1.free(); d2.free()


@pytest.mark.parametrize("exact", [True, False])
def test_edge_adversarial(engine, exact):
    """pairs within a few ulp of a bin edge: only the reference's FP64 evaluation
    order reproduces scipy (SURVEY.md section 7.2); golden counts from the reference"""
    g = golden_io.load("edge_adversarial")
    a, b = g["a_xyz"], g["b_xyz"]  # exact doubles of the reference trees
    # edges exactly as the reference forms them: limits -> log10 -> unique -> 10** (trees.py:107-117)
    for key in ("upper", "lower", "multi"):
        lim = oracle.parse_ang_limits(g[f"{key}_ang_min"], g[f"{key}_ang_max"])
        ang_bins = oracle.get_ang_bins(lim, None, 50)
        r2 = oracle.chord_sq_edges(ang_bins)
        ci, _, stats = single_patch_hist(engine, a, None, b, None, r2, exact)
        got = oracle.get_counts_for_limits(ci.astype(np.float64), ang_bins, lim)
        assert_array_equal(got, g[f"{key}_counts"])
    if not exact:
        assert stats["rechecks"] > 0  # the FP64 recheck path was exercised


def test_random_dense_fast_vs_exact(engine):
    """property test: pruned FP32+recheck kernel == unpruned FP64 kernel, several patches, bins, edges"""
    rng = np.random.default_rng(42)
    n_patch, n_bins = 5, 3
    n1, n2 = 20000, 30000
    def cat(n, binned, weighted):
        ra = rng.uniform(0.0, 0.05, n); dec = np.arcsin(rng.uniform(-0.02, 0.02, n))
        patch = np.minimum((ra / 0.05 * n_patch).astype(int), n_patch - 1)
        order = np.argsort(patch, kind="stable")
        xyz = oracle.radec_to_xyz(ra, dec)[order]
        off = np.concatenate([[0], np.cumsum(np.bincount(patch, minlength=n_patch))])
        zbin = rng.integers(-1, n_bins + 1, n).astype(np.int32) if binned else None
        w = rng.uniform(0.5, 1.5, n) if weighted else None
        return xyz, off, w, zbin
    pi, pj = np.meshgrid(np.arange(n_patch), np.arange(n_patch), indexing="ij")
    pi, pj = pi.ravel(), pj.ravel()
    for weighted in (False, True):
        for n_edges in (2, 7):
            r2 = np.sort(rng.uniform(1e-8, 4e-6, (n_bins, n_edges)), axis=1)
            x1, o1, w1, z1 = cat(n1, True, weighted)
            x2, o2, w2, _ = cat(n2, False, False)
            d1 = engine.upload_catalog(x1, o1, weights=w1, zbin=z1, n_bins=n_bins)
            d2 = engine.upload_catalog(x2, o2, weights=w2)
            fi, ff, fs = engine.count(d1, d2, pi, pj, r2)
            ei, ef, es = engine.count(d1, d2, pi, pj, r2, exact=True)
            assert_array_equal(fi, ei)
            assert_allclose(ff, ef, rtol=RTOL_WEIGHTED, atol=0)
            assert ei.sum() > 1000
            assert fs["pair_tests"] < es["pair_tests"]  # pruning happened
            assert es["pair_tests"] == es["pair_tests_naive"]
            d1.free(); d2.free()


def test_fused_count_equals_two_counts(engine):
    """`yawb_count2` (two first catalogs in one pass over a fused sky-cell index) must return exactly what two
    `yawb_count` calls return: different sizes, weights on one side only, dropped z-bins, several edge counts,
    and a patch that is empty in the larger catalog"""
    rng = np.random.default_rng(11)
    n_patch, n_bins = 6, 4

    def cat(n, binned, weighted, empty_patch=None):
        ra = rng.uniform(0.0, 0.06, n); dec = np.arcsin(rng.uniform(-0.02, 0.02, n))
        patch = np.minimum((ra / 0.06 * n_patch).astype(int), n_patch - 1)
        if empty_patch is not None:
            keep = patch != empty_patch
            ra, dec, patch = ra[keep], dec[keep], patch[keep]
        order = np.argsort(patch, kind="stable")
        xyz = oracle.radec_to_xyz(ra, dec)[order]
        off = np.concatenate([[0], np.cumsum(np.bincount(patch, minlength=n_patch))])
        zbin = rng.integers(-1, n_bins + 1, len(ra)).astype(np.int32) if binned else None
        w = rng.uniform(0.5, 1.5, len(ra)) if weighted else None
        return xyz, off, w, zbin

    pi, pj = np.meshgrid(np.arange(n_patch), np.arange(n_patch), indexing="ij")
    pi, pj = pi.ravel(), pj.ravel()
    for wa, wb, w2, n_edges in ((False, False, False, 2), (True, False, False, 2), (False, False, True, 5), (True, True, False, 12)):
        r2 = np.sort(rng.uniform(1e-8, 4e-6, (n_bins, n_edges)), axis=1)
        xa, oa, wwa, za = cat(3000, True, wa)
        xb, ob, wwb, zb = cat(40000, True, wb, empty_patch=2)
        x2, o2, ww2, _ = cat(30000, False, w2)
        da = engine.upload_catalog(xa, oa, weights=wwa, zbin=za, n_bins=n_bins)
        db = engine.upload_catalog(xb, ob, weights=wwb, zbin=zb, n_bins=n_bins)
        d2 = engine.upload_catalog(x2, o2, weights=ww2)
        (ia, fa), (ib, fb), st = engine.count2(da, db, d2, pi, pj, r2)
        sa_i, sa_f, _ = engine.count(da, d2, pi, pj, r2)
        sb_i, sb_f, _ = engine.count(db, d2, pi, pj, r2)
        assert_array_equal(ia, sa_i)
        assert_array_equal(ib, sb_i)
        assert_allclose(fa, sa_f, rtol=RTOL_WEIGHTED, atol=0)
        assert_allclose(fb, sb_f, rtol=RTOL_WEIGHTED, atol=0)
        assert sa_i.sum() > 100 and sb_i.sum() > 1000 and st["pair_tests"] > 0
        # the other order of the two catalogs (the smaller one supplies the frames where the larger is empty)
        (ib2, _), (ia2, _), _ = engine.count2(db, da, d2, pi, pj, r2)
        assert_array_equal(ia2, sa_i)
        assert_array_equal(ib2, sb_i)
        for d in (da, db, d2):
            d.free()


def test_four_counts_in_one_launch_equal_four_counts(engine):
    """`yawb_count4` (two first catalogs x two second catalogs in one launch) must return exactly what four
    `yawb_count` calls return: second catalogs of different sizes, weights on one of them only, dropped z-bins,
    several edge counts (single bin, cumulative and general sub-bin kernels), results kept on the host"""
    rng = np.random.default_rng(17)
    n_patch, n_bins = 5, 3

    def cat(n, binned, weighted):
        ra = rng.uniform(0.0, 0.05, n); dec = np.arcsin(rng.uniform(-0.02, 0.02, n))
        patch = np.minimum((ra / 0.05 * n_patch).astype(int), n_patch - 1)
        order = np.argsort(patch, kind="stable")
        xyz = oracle.radec_to_xyz(ra, dec)[order]
        off = np.concatenate([[0], np.cumsum(np.bincount(patch, minlength=n_patch))])
        zbin = rng.integers(-1, n_bins + 1, len(ra)).astype(np.int32) if binned else None
        w = rng.uniform(0.5, 1.5, len(ra)) if weighted else None
        return xyz, off, w, zbin

    pi, pj = np.meshgrid(np.arange(n_patch), np.arange(n_patch), indexing="ij")
    pi, pj = pi.ravel(), pj.ravel()
    for w1, w2a, w2b, n_edges in ((False, False, False, 2), (False, False, False, 5), (False, True, False, 2), (True, False, True, 12)):
        r2 = np.sort(rng.uniform(1e-8, 4e-6, (n_bins, n_edges)), axis=1)
        xa, oa, wwa, za = cat(2500, True, w1)
        xb, ob, wwb, zb = cat(30000, True, w1)
        x2a, o2a, ww2a, _ = cat(20000, False, w2a)
        x2b, o2b, ww2b, _ = cat(45000, False, w2b)
        da = engine.upload_catalog(xa, oa, weights=wwa, zbin=za, n_bins=n_bins)
        db = engine.upload_catalog(xb, ob, weights=wwb, zbin=zb, n_bins=n_bins)
        d2a = engine.upload_catalog(x2a, o2a, weights=ww2a)
        d2b = engine.upload_catalog(x2b, o2b, weights=ww2b)
        out4, st = engine.count4(da, db, d2a, d2b, pi, pj, r2)
        total = 0
        for (ci, cf), (c1, c2) in zip(out4, ((da, d2a), (db, d2a), (da, d2b), (db, d2b))):
            si, sf, _ = engine.count(c1, c2, pi, pj, r2)
            assert_array_equal(ci, si)
            assert_allclose(cf, sf, rtol=RTOL_WEIGHTED, atol=0)
            total += int(si.sum())
        assert total > 1000 and st["pair_tests"] > 0
        for d in (da, db, d2a, d2b):
            d.free()


def test_pair_test_variants_exact(engine):
    """the saturating-ramp FP32 pair test of the unweighted single-bin kernel must reproduce the reference's
    counts on the adversarial on-edge set and on dense random data"""
    g = golden_io.load("edge_adversarial")
    a, b = g["a_xyz"], g["b_xyz"]
    for key in ("upper", "lower"):
        lim = oracle.parse_ang_limits(g[f"{key}_ang_min"], g[f"{key}_ang_max"])
        ang_bins = oracle.get_ang_bins(lim, None, 50)
        ci, _, stats = single_patch_hist(engine, a, None, b, None, oracle.chord_sq_edges(ang_bins), False)
        assert ci[0] == int(g[f"{key}_counts"][0])
        assert stats["rechecks"] > 0
    # dense small-angle data: thousands of pairs per edge band
    rng = np.random.default_rng(3)
    n = 40000
    ra = rng.uniform(0.0, 0.02, n); dec = np.arcsin(rng.uniform(-0.01, 0.01, n))
    xyz = oracle.radec_to_xyz(ra, dec)
    r2 = oracle.chord_sq_edges(np.array([3e-4, 2e-3]))
    fi, _, fs = single_patch_hist(engine, xyz[: n // 2], None, xyz[n // 2 :], None, r2, False)
    ei, _, _ = single_patch_hist(engine, xyz[: n // 2], None, xyz[n // 2 :], None, r2, True)
    assert_array_equal(fi, ei)
    assert ei[0] > 1e6 and fs["rechecks"] > 0


@pytest.mark.parametrize("dev", [1e-13, 1e-9, 1e-4])
def test_rows_off_the_unit_sphere_stay_exact(engine, dev):
    """The pair test takes |r|^2 of a tile row from the identity for unit vectors; rows that are NOT unit vectors
    (the C ABI takes any doubles) only widen the band of tests that go through the FP64 recheck: the counts still
    equal the plain double-precision evaluation of the reference's expression."""
    rng = np.random.default_rng(11)
    n = 6000
    ra = rng.uniform(0.0, 0.01, n); dec = np.arcsin(rng.uniform(-0.005, 0.005, n))
    xyz = oracle.radec_to_xyz(ra, dec) * (1.0 + dev * rng.uniform(-1.0, 1.0, n))[:, None]
    a, b = xyz[: n // 2], xyz[n // 2 :]
    r2 = oracle.chord_sq_edges(np.array([2e-4, 1.5e-3]))
    want = oracle.pair_histogram(a, b, None, None, r2)
    ci, _, stats = single_patch_hist(engine, a, None, b, None, r2, False)
    assert_array_equal(ci, want.astype(np.int64))
    assert ci[0] > 1e5
    r2m = oracle.chord_sq_edges(np.array([2e-4, 5e-4, 1.0e-3, 1.5e-3]))
    want = oracle.pair_histogram(a, b, None, None, r2m)
    ci, _, _ = single_patch_hist(engine, a, None, b, None, r2m, False)
    assert_array_equal(ci, want.astype(np.int64))


@pytest.mark.parametrize("closed", ["right", "left"])
def test_device_digitize_matches_numpy(engine, closed):
    """yawb_upload_catalog_z: z-bins assigned on the device == np.digitize on the host (reference
    src/yaw/catalog/trees.py:408-414), values on the edges, outside the binning and NaN included: the per-(bin, patch)
    row counts and every pair count agree with an upload of host-assigned ids"""
    rng = np.random.default_rng(21)
    n = 40000
    ra = rng.uniform(0.0, 0.03, n); dec = np.arcsin(rng.uniform(-0.015, 0.015, n))
    xyz = oracle.radec_to_xyz(ra, dec)
    edges = np.linspace(0.1, 1.0, 8)
    z = rng.uniform(0.0, 1.1, n)
    z[:200] = rng.choice(edges, 200)  # exactly on an edge
    z[200:210] = np.nan
    order = np.argsort(ra > 0.015, kind="stable")
    xyz, z = xyz[order], z[order]
    off = np.array([0, int((ra <= 0.015).sum()), n], dtype=np.int64)
    ids = np.digitize(z, edges, right=(closed == "right")).astype(np.int32) - 1
    a = engine.upload_catalog(xyz, off, zbin=ids, n_bins=len(edges) - 1)
    b = engine.upload_catalog(xyz, off, redshifts=z, edges=edges, closed=closed)
    assert_array_equal(a.sum_weights(), b.sum_weights())
    assert a.info()[0] == b.info()[0] < n
    unk = engine.upload_catalog(xyz, off)
    pi = np.array([0, 0, 1, 1], dtype=np.int32); pj = np.array([0, 1, 0, 1], dtype=np.int32)
    r2 = oracle.chord_sq_edges(np.array([2e-4, 2e-3]))
    ca, _, _ = engine.count(a, unk, pi, pj, r2)
    cb, _, _ = engine.count(b, unk, pi, pj, r2)
    assert_array_equal(ca, cb)
    assert ca.sum() > 1e5
    for c in (a, b, unk):
        c.free()


def test_device_patch_metadata(engine):
    """yawb_patch_metadata == the reference's Metadata.compute (src/yaw/catalog/patch.py:104-147): centre = normalised
    mean direction, radius = largest angular distance from it, rows per patch"""
    rng = np.random.default_rng(22)
    sizes = [5000, 0, 12000, 1]
    ras, decs = [], []
    for k, m in enumerate(sizes):
        ras.append(rng.uniform(0.1 * k, 0.1 * k + 0.08, m)); decs.append(rng.uniform(-0.3, -0.25 + 0.02 * k, m))
    ra, dec = np.concatenate(ras), np.concatenate(decs)
    xyz = oracle.radec_to_xyz(ra, dec)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    cat = engine.upload_catalog(xyz, off)
    center, radius, num = cat.patch_metadata()
    assert_array_equal(num, sizes)
    for p, m in enumerate(sizes):
        if m == 0:
            continue
        rows = xyz[off[p]:off[p + 1]]
        c = rows.mean(axis=0)
        c /= np.linalg.norm(c)
        np.testing.assert_allclose(center[p], c, rtol=0, atol=1e-14)
        want = 2.0 * np.arcsin(np.sqrt(((rows - c) ** 2).sum(axis=1).max()) / 2.0)
        np.testing.assert_allclose(radius[p], want, rtol=1e-9, atol=1e-13)
    cat.free()


def test_device_jackknife_matches_einsum(engine):
    """yawb_jackknife == SampledPatchSum of the reference (src/yaw/correlation/paircounts.py:113-141: total - row -
    column + diagonal), exactly for integer counts, to rounding for weighted sums"""
    from yet_another_wizz_b200.binning import Binning
    from yet_another_wizz_b200.paircounts import PatchedCounts, _sample_patch_sum

    rng = np.random.default_rng(31)
    n_patch, n_bins = 24, 7
    binning = Binning(np.linspace(0.1, 1.0, n_bins + 1))
    dense = np.zeros((n_bins, n_patch, n_patch))
    link = rng.random((n_patch, n_patch)) < 0.25
    np.fill_diagonal(link, True)
    dense[:, link] = rng.integers(0, 10**9, size=(n_bins, int(link.sum())))
    counts = PatchedCounts(binning, dense, auto=False)
    want = _sample_patch_sum(binning, dense)
    got = counts.sample_patch_sum(engine)
    assert_array_equal(got.data, want.data)
    assert_array_equal(got.samples, want.samples)
    dense_w = dense * rng.uniform(0.5, 1.5, size=dense.shape)
    want = _sample_patch_sum(binning, dense_w)
    got = PatchedCounts(binning, dense_w, auto=False).sample_patch_sum(engine)
    np.testing.assert_allclose(got.data, want.data, rtol=1e-13)
    np.testing.assert_allclose(got.samples, want.samples, rtol=1e-12)
    # no linked pairs at all
    total, samples = engine.sample_patch_sum(np.zeros((0, n_bins)), np.zeros(0, np.int32), np.zeros(0, np.int32), n_patch)
    assert not total.any() and samples.shape == (n_patch, n_bins) and not samples.any()


def test_device_memory_is_recycled(engine):
    """upload / count / free cycles of varying size: the context's caching allocator reuses its blocks, the
    footprint on the device stops growing after the first cycles"""
    import torch

    rng = np.random.default_rng(5)
    r2 = np.array([[1e-8, 4e-6]])

    def cycle(n):
        a = oracle.radec_to_xyz(rng.uniform(0.0, 0.05, n), rng.uniform(-0.02, 0.02, n))
        off = np.array([0, n // 2, n], dtype=np.int64)
        cat = engine.upload_catalog(a, off)
        ci, _, _ = engine.count(cat, cat, np.array([0, 1], dtype=np.int32), np.array([0, 1], dtype=np.int32), r2)
        cat.free()
        return int(ci.sum())

    sizes = [200_000, 50_000, 120_000, 200_000, 80_000]
    first = [cycle(n) for n in sizes]
    engine.sync()
    free0, _ = torch.cuda.mem_get_info(0)
    for _ in range(4):
        for n in sizes:
            cycle(n)
    engine.sync()
    free1, _ = torch.cuda.mem_get_info(0)
    assert free0 - free1 < 32 << 20, f"device footprint grew by {(free0 - free1) >> 20} MiB"
    assert all(c > 0 for c in first)


def test_assign_patches_matches_scipy_vq(engine):
    """`yawb_assign_patches` against `scipy.cluster.vq.vq` (what the reference's `assign_patch_centers` calls,
    catalog.py:229-249): random rows, many centres (several shared-memory blocks), exact ties (first
    centre wins), and the catalog constructor that uses it"""
    from scipy.cluster import vq

    import yet_another_wizz_b200 as yb

    rng = np.random.default_rng(17)
    for n, p in ((200_000, 64), (50_000, 2500), (1000, 1)):
        xyz = oracle.radec_to_xyz(rng.uniform(0, 0.7, n), rng.uniform(-0.2, 0.2, n))
        cen = oracle.radec_to_xyz(rng.uniform(0, 0.7, p), rng.uniform(-0.2, 0.2, p))
        want, _ = vq.vq(xyz, cen)
        assert_array_equal(engine.assign_patches(xyz, cen), want.astype(np.int32))
    # exact ties: rows on the mirror plane of two centres, duplicated centres
    cen = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [1.0, 0.0, 0.0], [0.0, 0.0, 1.0]])
    rows = np.array([[0.5, 0.5, 0.0], [0.25, 0.25, 0.1], [1.0, 0.0, 0.0], [0.0, 0.5, 0.5], [0.3, 0.3, 0.3]])
    want, _ = vq.vq(rows, cen)
    assert_array_equal(engine.assign_patches(rows, cen), want.astype(np.int32))
    # through the catalog constructor
    ra, dec = rng.uniform(0, 40, 30_000), rng.uniform(-12, 12, 30_000)
    centers = yb.AngularCoordinates(np.deg2rad([[5.0, -6.0], [15.0, 6.0], [25.0, -6.0], [35.0, 6.0]]))
    a = yb.Catalog.from_arrays(ra, dec, patch_centers=centers)
    b = yb.Catalog.from_arrays(ra, dec, patch_centers=centers, engine=engine)
    assert a.get_num_records() == b.get_num_records()
    for pid in a.keys():
        assert_array_equal(a[pid].load_data()["ra"], b[pid].load_data()["ra"])


def test_more_than_65535_patch_pairs(engine):
    """a densely linked catalog of 300 patches: 90 000 patch pairs in one call (the planner runs on a flat grid, so
    the number of pairs is not limited by a grid dimension)"""
    rng = np.random.default_rng(5)
    n_patch, n = 300, 6000
    ra = rng.uniform(0.0, 0.003, n); dec = np.arcsin(rng.uniform(-0.0015, 0.0015, n))
    patch = rng.integers(0, n_patch, n)
    order = np.argsort(patch, kind="stable")
    xyz = oracle.radec_to_xyz(ra, dec)[order]
    off = np.concatenate([[0], np.cumsum(np.bincount(patch, minlength=n_patch))])
    zbin = rng.integers(0, 2, n).astype(np.int32)[order]
    pi, pj = np.meshgrid(np.arange(n_patch), np.arange(n_patch), indexing="ij")
    pi, pj = pi.ravel(), pj.ravel()
    assert len(pi) > 65535
    r2 = np.tile(oracle.chord_sq_edges(np.array([1e-4, 8e-4])), (2, 1))
    d1 = engine.upload_catalog(xyz, off, zbin=zbin, n_bins=2)
    d2 = engine.upload_catalog(xyz, off)
    fi, _, _ = engine.count(d1, d2, pi, pj, r2)
    ei, _, _ = engine.count(d1, d2, pi, pj, r2, exact=True)
    assert_array_equal(fi, ei)
    # the total over all patch pairs is the single-patch count of the same rows
    whole1 = engine.upload_catalog(xyz, np.array([0, n]), zbin=zbin, n_bins=2)
    whole2 = engine.upload_catalog(xyz, np.array([0, n]))
    wi, _, _ = engine.count(whole1, whole2, [0], [0], r2)
    assert_array_equal(fi.sum(axis=0), wi[0])
    assert wi.sum() > 10000
    for d in (d1, d2, whole1, whole2):
        d.free()
