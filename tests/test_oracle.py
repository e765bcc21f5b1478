"""
CPU tests that PIN the oracle (`oracle/oracle.py`, `oracle/paircount_ref.c`):

  * the reference's own known-answer tests for the pair-count primitive,
    restated from `/root/reference/tests/catalog/test_trees.py:134-254`;
  * golden vectors produced by the unmodified reference
    (`tests/golden/make_golden.py`).

Tolerances: unweighted (integer) counts bit-exact; weighted sums 1e-12 relative
(the reference's own tree sums differ from a brute-force sum by ~1e-14).
"""

from itertools import product

import numpy as np
import pytest
from numpy.testing import assert_allclose, assert_array_equal

import golden_cases
import golden_io
import oracle

DELTA = 1e-9  # test_trees.py:162
RTOL_WEIGHTED = 1e-12


def great_circle_points():
    """restates fixture_test_points, test_trees.py:134-159"""
    points = np.array(
        [[0.0, 0.0], [90.0, 0.0], [180.0, 0.0], [270.0, 0.0], [0.0, 90.0], [0.0, -90.0]]
    )
    base = np.arange(1.0, 90.0, 1.0)
    for offset in (0.0, 90.0, 180.0, 270.0):
        points = np.concatenate([points, np.column_stack([base + offset, np.zeros_like(base)])])
    for sign, ra in product([-1.0, 1.0], [0.0, 180.0]):
        points = np.concatenate([points, np.column_stack([np.full_like(base, ra), sign * base])])
    for sign, ra in product([-1.0, 1.0], [90.0, 270.0]):
        points = np.concatenate([points, np.column_stack([np.full_like(base, ra), sign * base])])
    return np.deg2rad(points)


@pytest.fixture(scope="module")
def pts():
    radec = great_circle_points()
    return oracle.radec_to_xyz(radec[:, 0], radec[:, 1])


SINGLE = oracle.radec_to_xyz(np.array([0.0]), np.array([0.0]))


@pytest.mark.parametrize("use_c", [False, True])
class TestTreeCountKAT:
    @pytest.mark.parametrize("ang_max", [1.0, 2.0, 10.0, 89.0])
    def test_count_single(self, pts, ang_max, use_c):  # test_trees.py:181-195
        w = np.full(len(pts), 2.0)
        amax = ang_max + DELTA
        c = oracle.tree_count(pts, w, SINGLE, np.array([2.0]), np.deg2rad(amax - 1.0), np.deg2rad(amax), use_c=use_c)
        assert c == 4 * 2.0**2

    @pytest.mark.parametrize("ang_max", [2.0, 10.0, 89.0])
    def test_count_bins(self, pts, ang_max, use_c):  # test_trees.py:197-212
        w = np.full(len(pts), 2.0)
        amax = np.arange(1.0, ang_max) + DELTA
        c = oracle.tree_count(pts, w, SINGLE, np.array([2.0]), np.deg2rad(amax - 1.0), np.deg2rad(amax), use_c=use_c)
        assert_array_equal(c, np.full_like(amax, 4 * 2.0**2))

    @pytest.mark.parametrize("ang_max", [1.0, 2.0, 10.0, 89.0])
    def test_count_range(self, pts, ang_max, use_c):  # test_trees.py:214-225
        w = np.full(len(pts), 2.0)
        c = oracle.tree_count(pts, w, SINGLE, np.array([2.0]), DELTA, np.deg2rad(ang_max) + DELTA, use_c=use_c)
        assert c == int(ang_max) * 4 * 2.0**2

    @pytest.mark.parametrize("num_bins", [1, 2])
    def test_count_empty(self, num_bins, use_c):  # test_trees.py:227-237
        empty = np.empty((0, 3))
        amin = np.linspace(0.0, 1.0, num_bins) + DELTA
        c = oracle.tree_count(empty, np.empty(0), empty, np.empty(0), amin, amin + 1.0, use_c=use_c)
        assert_array_equal(c, np.zeros(num_bins))

    def test_count_dualtree(self, pts, use_c):  # test_trees.py:239-247
        lims = np.deg2rad([0.0, 1.0]) + DELTA
        c = oracle.tree_count(pts, None, pts, None, lims[0], lims[1], use_c=use_c)
        assert c == 4 * 6 + 2 * (len(pts) - 6)

    def test_count_invalid_ang(self, pts, use_c):  # test_trees.py:249-254
        with pytest.raises(ValueError):
            oracle.tree_count(pts, None, pts, None, [-1.0], [1.0], use_c=use_c)
        with pytest.raises(ValueError):
            oracle.tree_count(pts, None, pts, None, [1.0], [np.pi + DELTA], use_c=use_c)


def test_helpers_match_reference_tests():
    # test_trees.py:14-131 restated on the helper functions
    assert_array_equal(oracle.parse_ang_limits([0.0, 1.0], [1.0, np.pi]), [[0.0, 1.0], [1.0, np.pi]])
    with pytest.raises(ValueError):
        oracle.parse_ang_limits([1.0], [0.5])
    bins = oracle.get_ang_bins(np.array([[0.1, 1.0]]), None, 50)
    assert_allclose(bins, [0.1, 1.0])
    bins = oracle.get_ang_bins(np.array([[0.01, 1.0]]), -1.0, 2)
    assert_allclose(bins, [0.01, 0.1, 1.0])
    assert_allclose(oracle.logarithmic_mid(np.array([0.01, 1.0, 100.0])), [0.1, 10.0])
    counts = np.array([1.0, 2.0, 3.0, 4.0])
    ang_bins = np.array([1.0, 2.0, 3.0, 4.0, 5.0])
    got = oracle.get_counts_for_limits(counts, ang_bins, np.array([[1.0, 5.0], [2.0, 4.0]]))
    assert_array_equal(got, [10.0, 5.0])


def patches_from(cat: dict):
    out = []
    n_patch = len(cat["radii"])
    for p in range(n_patch):
        m = cat["patch"] == p
        out.append(
            oracle.OraclePatch(
                cat["ra"][m], cat["dec"][m],
                None if cat["w"] is None else cat["w"][m],
                None if cat["z"] is None else cat["z"][m],
            )
        )
    return out


def check_counts(g, tag, kind, sw1, sw2, counts, exact):
    assert_array_equal(sw1, g[f"{tag}_{kind}_sw1"]) if exact else assert_allclose(
        sw1, g[f"{tag}_{kind}_sw1"], rtol=RTOL_WEIGHTED)
    assert_array_equal(sw2, g[f"{tag}_{kind}_sw2"]) if exact else assert_allclose(
        sw2, g[f"{tag}_{kind}_sw2"], rtol=RTOL_WEIGHTED)
    for s in range(counts.shape[0]):
        want = g[f"{tag}_{kind}_counts_s{s}"]
        if exact:
            assert_array_equal(counts[s], want)
        else:
            assert_allclose(counts[s], want, rtol=RTOL_WEIGHTED, atol=0.0)
        assert want.sum() > 0


@pytest.mark.parametrize("name", ["cross_unweighted", "cross_weighted_multiscale"])
def test_golden_crosscorrelate(name):
    g = golden_io.load(name)
    cfg = golden_io.config_of(g)
    links = golden_io.links_of(g)
    cats = {k: patches_from(golden_io.catalog_arrays(g, k)) for k in ("ref", "unk", "ref_rand", "unk_rand")}
    kw = dict(zedges=cfg["zedges"], closed=cfg["closed"], ang_min=cfg["ang_min"], ang_max=cfg["ang_max"],
              rweight=cfg["rweight"], resolution=cfg["resolution"])
    exact = name == "cross_unweighted"
    for kind, (a, b) in dict(dd=("ref", "unk"), dr=("ref", "unk_rand"), rd=("ref_rand", "unk"),
                             rr=("ref_rand", "unk_rand")).items():
        sw1, sw2, counts = oracle.count_pairs(cats[a], cats[b], links, **kw)
        check_counts(g, "cross", kind, sw1, sw2, counts, exact and kind in ("dd", "dr", "rd", "rr"))


@pytest.mark.parametrize("name", ["auto_unweighted", "auto_rweight_polewrap"])
def test_golden_autocorrelate(name):
    g = golden_io.load(name)
    cfg = golden_io.config_of(g)
    links = golden_io.links_of(g)
    data = patches_from(golden_io.catalog_arrays(g, "data"))
    rand = patches_from(golden_io.catalog_arrays(g, "rand"))
    kw = dict(zedges=cfg["zedges"], closed=cfg["closed"], ang_min=cfg["ang_min"], ang_max=cfg["ang_max"],
              rweight=cfg["rweight"], resolution=cfg["resolution"])
    exact = name == "auto_unweighted"
    check_counts(g, "auto", "dd", *oracle.count_pairs(data, None, links, **kw), exact)
    check_counts(g, "auto", "dr", *oracle.count_pairs(data, (rand, "binned"), links, **kw), exact)
    check_counts(g, "auto", "rr", *oracle.count_pairs(rand, None, links, **kw), exact)


def test_golden_linkage():
    # PatchLinkage.from_catalogs, measurements.py:220-235: centres/radii of the
    # catalog that sorts first by `get_num_records()` (a tuple!) in reverse order
    for name, keys in (("cross_unweighted", ("ref", "unk", "ref_rand", "unk_rand")),
                       ("auto_rweight_polewrap", ("data", "rand"))):
        g = golden_io.load(name)
        cfg = golden_io.config_of(g)
        cats = [golden_io.catalog_arrays(g, k) for k in keys]
        nrec = [tuple(int((c["patch"] == p).sum()) for p in range(len(c["radii"]))) for c in cats]
        order = sorted(range(len(cats)), key=lambda i: nrec[i], reverse=True)
        ref = cats[order[0]]
        links = oracle.compute_linkage(ref["centers"], ref["radii"], cfg["max_angle"])
        assert links == golden_io.links_of(g)


@pytest.mark.parametrize("use_c", [False, True])
def test_golden_edge_adversarial(use_c):
    g = golden_io.load("edge_adversarial")
    a, b = g["a_xyz"], g["b_xyz"]  # exact doubles of the reference trees
    for key in ("upper", "lower", "multi"):
        got = oracle.tree_count(a, None, b, None, g[f"{key}_ang_min"], g[f"{key}_ang_max"], use_c=use_c)
        assert_array_equal(got, g[f"{key}_counts"])


def test_c_and_numpy_agree_weighted():
    rng = np.random.default_rng(5)
    a = rng.normal(size=(700, 3)); a /= np.linalg.norm(a, axis=1)[:, None]
    b = rng.normal(size=(900, 3)); b /= np.linalg.norm(b, axis=1)[:, None]
    w1, w2 = rng.uniform(0.5, 1.5, 700), rng.uniform(0.5, 1.5, 900)
    r2 = oracle.chord_sq_edges(np.array([0.05, 0.1, 0.3, 0.8, 1.5]))
    h_np = oracle.pair_histogram(a, b, w1, w2, r2, use_c=False)
    h_c = oracle.pair_histogram(a, b, w1, w2, r2, use_c=True)
    assert_allclose(h_c, h_np, rtol=1e-13)
    assert_array_equal(oracle.pair_histogram(a, b, None, None, r2, use_c=False),
                       oracle.pair_histogram(a, b, None, None, r2, use_c=True))


@pytest.mark.parametrize("name,workers", [("cross_unweighted", 1), ("cross_weighted_multiscale", 2)])
def test_cpu_port_counts_equal_reference(name, workers):
    """`oracle/cpu_port.py` (the CPU arm of bench.py when the reference itself is not installed: scipy cKDTree per
    patch and z-bin + a task farm over patch pairs, trees built on the worker pool) against the per-patch-pair
    counts the UNMODIFIED reference wrote into the golden vectors -- all four count types, serial and with a pool"""
    import cpu_port
    from yet_another_wizz_b200.measurements import PatchLinkage, _angles_per_bin, _as_binning, prepare_catalog_arrays

    g = golden_io.load(name)
    config = golden_cases.config_from_golden(g)
    cats = {k: golden_cases.catalog_from_golden(g, k) for k in ("ref", "unk", "ref_rand", "unk_rand")}
    binning = _as_binning(config)
    arrays = {k: prepare_catalog_arrays(c, binning if k in ("ref", "ref_rand") else None) for k, c in cats.items()}
    links = PatchLinkage.from_catalogs(config, *cats.values(), engine=object())
    pair_i, pair_j = links.get_patch_id_pairs(auto=False)
    pairs = [(int(i), int(j)) for i, j in zip(pair_i, pair_j)]
    amin, amax = _angles_per_bin(config)
    n_bins, n_patch = len(binning), len(cats["ref"])

    def trees_of(key, binned):
        a = arrays[key]
        rows = []
        for p in range(n_patch):
            s, e = a["patch_off"][p], a["patch_off"][p + 1]
            rows.append((a["xyz"][s:e], None if a["weights"] is None else a["weights"][s:e],
                         a["zbin"][s:e].astype(np.int32) if binned else None))
        built, _ = cpu_port.build_catalog_trees(rows, n_bins if binned else None, workers=workers)
        return dict(enumerate(built))

    trees = {k: trees_of(k, k in ("ref", "ref_rand")) for k in arrays}
    weighted = any(a["weights"] is not None for a in arrays.values())
    for tag, (a, b) in dict(dd=("ref", "unk"), dr=("ref", "unk_rand"), rd=("ref_rand", "unk"), rr=("ref_rand", "unk_rand")).items():
        counts, _ = cpu_port.count_pairs(trees[a], trees[b], pairs, amin, amax, rweight=config.scales.rweight,
                                         resolution=config.scales.resolution, workers=workers)
        for s in range(config.scales.num_scales):
            want = g[f"cross_{tag}_counts_s{s}"]
            got = np.zeros_like(want)
            for (i, j), c in counts.items():
                got[:, i, j] = c[s]
            if weighted:
                assert_allclose(got, want, rtol=1e-12, atol=0)
            else:
                assert_array_equal(got, want)
            assert want.sum() > 0


def _brute_binned(xyz1, patch1, zbin1, xyz2, patch2, pairs, r2, w1, w2, zbin2=None, label1=None, label2=None,
                  n_labels=1):
    """`binned_pair_counts` spelled out: one `pair_histogram` per (label, patch pair, z-bin)"""
    out_i = np.zeros((n_labels, len(pairs), r2.shape[0], r2.shape[1] - 1), dtype=np.int64)
    out_f = np.zeros(out_i.shape)
    lab2 = np.zeros(len(xyz2), dtype=int) if label2 is None else label2
    for ell in range(n_labels):
        for k, (i, j) in enumerate(pairs):
            for b in range(r2.shape[0]):
                m1 = (patch1 == i) & (zbin1 == b) & (True if label1 is None else label1 == ell)
                m2 = (patch2 == j) & (lab2 == ell) & (True if zbin2 is None else zbin2 == b)
                args = (xyz1[m1], xyz2[m2], None if w1 is None else w1[m1], None if w2 is None else w2[m2], r2[b])
                out_i[ell, k, b] = oracle.pair_histogram(*args[:2], None, None, r2[b])
                out_f[ell, k, b] = oracle.pair_histogram(*args)
    return out_i, out_f


@pytest.mark.parametrize("weights", ["none", "first", "second", "both"])
@pytest.mark.parametrize("mode", ["unbinned", "binned", "labels", "binned_labels"])
def test_binned_pair_counts_equal_pair_histogram(weights, mode):
    """the k-d-tree-pruned oracle (`binned_pair_counts`) against `pair_histogram` per (label, patch pair, z-bin):
    dropped rows, duplicated rows (d2 = 0 against a lower edge of 0), equal neighbouring edges, an empty z-bin
    (hi == lo), thresholds that differ per z-bin, patch pairs that are not in the list"""
    rng = np.random.default_rng(["none", "first", "second", "both"].index(weights) * 7 + len(mode))
    n_patch, n_bins, n_labels = 3, 4, 3
    n1, n2 = 900, 1100
    def rows(n):
        ra = rng.uniform(0.0, 0.06, n); dec = np.arcsin(rng.uniform(-0.02, 0.02, n))
        return oracle.radec_to_xyz(ra, dec), np.minimum((ra / 0.02).astype(int), n_patch - 1)
    xyz1, patch1 = rows(n1)
    xyz2, patch2 = rows(n2)
    xyz2[:150], patch2[:150] = xyz1[:150], patch1[:150]  # duplicates
    zbin1 = rng.integers(-1, n_bins, n1)
    zbin2 = rng.integers(-1, n_bins, n2) if mode in ("binned", "binned_labels") else None
    label1 = rng.integers(0, n_labels, n1) if mode == "binned_labels" else None
    label2 = rng.integers(-1, n_labels, n2) if mode in ("labels", "binned_labels") else None
    w1 = rng.uniform(0.5, 1.5, n1) if weights in ("first", "both") else None
    w2 = rng.uniform(0.5, 1.5, n2) if weights in ("second", "both") else None
    r2 = oracle.chord_sq_edges(np.array([0.0, 1e-3, 2e-3, 2e-3, 4e-3, 6e-3]))
    r2 = np.array([r2, r2 * 1.3, np.full(6, r2[3]), r2 * 0.7])
    r2[1, 0] = 1e-7
    pairs = [(0, 0), (0, 1), (1, 0), (1, 1), (2, 1), (1, 2), (2, 2)]  # (0, 2) and (2, 0) are not linked
    pi, pj = np.array(pairs).T
    L = n_labels if label2 is not None else 1
    got_i, got_f = oracle.binned_pair_counts(xyz1, patch1, zbin1, xyz2, patch2, pi, pj, r2, w1=w1, w2=w2,
                                             zbin2=zbin2, label1=label1, label2=label2, n_labels=L)
    want_i, want_f = _brute_binned(xyz1, patch1, zbin1, xyz2, patch2, pairs, r2, w1, w2, zbin2, label1, label2, L)
    assert_array_equal(got_i, want_i)
    assert_allclose(got_f, want_f, rtol=1e-13, atol=0)  # pair_histogram sums in plain order
    assert want_i.sum() > 1000 and not want_i[:, :, 2].any()


@pytest.mark.parametrize("weights", ["none", "both"])
def test_binned_pair_counts_on_edge_adversarial(weights):
    """rows within a few ulp of the bin edges: the pruned oracle decides them as `pair_histogram` does"""
    g = golden_io.load("edge_adversarial")
    a, b = g["a_xyz"], g["b_xyz"]
    rng = np.random.default_rng(8)
    w1 = rng.uniform(0.5, 1.5, len(a)) if weights == "both" else None
    w2 = rng.uniform(0.5, 1.5, len(b)) if weights == "both" else None
    for key in ("upper", "lower", "multi"):
        lim = oracle.parse_ang_limits(g[f"{key}_ang_min"], g[f"{key}_ang_max"])
        r2 = oracle.chord_sq_edges(oracle.get_ang_bins(lim, None, 50))
        got_i, got_f = oracle.binned_pair_counts(a, np.zeros(len(a)), np.zeros(len(a)), b, np.zeros(len(b)), [0], [0],
                                                 r2, w1=w1, w2=w2)
        assert_array_equal(got_i[0, 0, 0], oracle.pair_histogram(a, b, None, None, r2))
        assert_allclose(got_f[0, 0, 0], oracle.pair_histogram(a, b, w1, w2, r2), rtol=1e-14, atol=0)
        assert got_i.sum() > 0
