"""
CPU tests of the deterministic spherical k-means: the numpy restatement in `oracle/kmeans.py` on hand-built
inputs (bisection order, axis tie-break, child ids, empty-cluster relocation), its invariants, and the host
plumbing of `patch_num` in the catalog constructors with a test double whose `kmeans` is the oracle.
"""

import numpy as np
import pytest
from numpy.testing import assert_array_equal
from scipy.cluster import vq

import kmeans as km_oracle

import yet_another_wizz_b200 as yb
from yet_another_wizz_b200 import catalog as catalog_mod
from yet_another_wizz_b200 import measurements
from yet_another_wizz_b200.measurements import PatchLinkage


class KmeansEngine:
    """TEST DOUBLE: the `kmeans` of `Engine`, answered by the oracle; records its inputs."""

    def __init__(self):
        self.calls = []

    def kmeans(self, xyz, k, *, weights=None, max_iter=500):
        self.calls.append((np.array(xyz), None if weights is None else np.array(weights), k))
        return km_oracle.kmeans(xyz, k, weights=weights, max_iter=max_iter)


def on_x(*xs):
    """rows on the x axis (exact multiples of 2^-32, so q is x 2^32)"""
    return np.array([[x, 0.0, 0.0] for x in xs])


def box_xyz(n, seed=1):
    g = yb.BoxRandoms(0, 40, -12.5, 12.5, seed=seed)(n)
    return yb.AngularCoordinates(np.column_stack([g["ra"], g["dec"]])).to_3d()


# ---- the algorithm ---------------------------------------------------------------------------------------------
def test_bisection_splits_most_populated_cell_first():
    # round 1 splits cell 0 at the mean (0.15): {0.5, 0.75, 0.75} -> child 1; round 2 (k - c = 1) splits the
    # larger cell 1 at its mean: {0.75, 0.75} -> child 2
    q = km_oracle.fixed_point(on_x(-0.75, -0.5, 0.5, 0.75, 0.75))
    trace = []
    assert_array_equal(km_oracle.bisect(q, 3, trace), [0, 0, 1, 2, 2])
    assert trace == [(0, 0, 1), (1, 0, 2)]


def test_bisection_ties_go_to_lower_cell_and_children_take_ids_in_order():
    q = km_oracle.fixed_point(on_x(-0.75, -0.5, 0.5, 0.75))
    trace = []
    assert_array_equal(km_oracle.bisect(q, 3, trace), [0, 2, 1, 1])  # cells 0 and 1 both hold 2 rows: 0 splits
    assert trace == [(0, 0, 1), (0, 0, 2)]
    trace = []
    assert_array_equal(km_oracle.bisect(q, 4, trace), [0, 2, 1, 3])  # both split; children 2, 3 in id order
    assert trace == [(0, 0, 1), (0, 0, 2), (1, 0, 3)]


def test_bisection_axis_tie_break_and_unsplittable_cells():
    for rows, axis in (([[0.25, 0.25, 0.0], [0.5, 0.5, 0.0]], 0), ([[0.0, 0.25, 0.25], [0.0, 0.5, 0.5]], 1),
                       ([[0.0, 0.0, 0.25], [0.0, 0.0, 0.5]], 2)):
        trace = []
        km_oracle.bisect(km_oracle.fixed_point(np.array(rows)), 2, trace)
        assert trace == [(0, axis, 1)]
    # cell 1 = three copies of one position cannot be split although it is the largest
    trace = []
    labels = km_oracle.bisect(km_oracle.fixed_point(on_x(0.5, 0.5, 0.5, -0.5, -0.25)), 3, trace)
    assert_array_equal(labels, [1, 1, 1, 0, 2])
    assert trace == [(0, 0, 1), (0, 0, 2)]


def test_duplicates_and_too_few_distinct_positions():
    xyz = np.array([[1.0, 0.0, 0.0]] * 3 + [[0.0, 1.0, 0.0]] * 2 + [[0.0, 0.0, 1.0]])
    C, L, n_iter, converged = km_oracle.kmeans(xyz, 3)
    assert converged
    assert_array_equal(C[L], xyz)  # every distinct position is a patch
    with pytest.raises(ValueError, match="fewer distinct positions than patches"):
        km_oracle.kmeans(xyz, 4)


def test_empty_cluster_relocation():
    # unweighted bisection: {-0.75, -0.5} | {0.5, 0.75}; weight 0 makes cluster 1 empty in iteration 1.  Its
    # rows are 0.0625, 0.25, 0.25, 0.0625 from their own centres (-1, 0, 0), (1, 0, 0): rows 1 and 2 tie, row 1 wins
    xyz = on_x(-0.75, -0.5, 0.5, 0.75)
    stats = {}
    C, L, n_iter, converged = km_oracle.kmeans(xyz, 2, weights=np.array([1.0, 1.0, 0.0, 0.0]), max_iter=1, stats=stats)
    assert stats["relocated"] == [(1, 1, 1)]
    assert_array_equal(C, [[-1.0, 0.0, 0.0], [-0.5, 0.0, 0.0]])
    assert_array_equal(L, [0, 1, 1, 1])  # row 0 is equally far from both centres: the first wins
    assert n_iter == 1 and not converged


def test_relocation_takes_distinct_rows():
    rng = np.random.default_rng(3)

    def blob(n, ra, s):
        r, d = np.deg2rad(ra) + rng.normal(0, s, n), rng.normal(0, s, n)
        return np.column_stack([np.cos(r) * np.cos(d), np.sin(r) * np.cos(d), np.sin(d)])

    xyz = np.concatenate([blob(3000, 10, 0.05), blob(300, 100, 0.01)])
    w = np.concatenate([np.ones(3000), np.zeros(300)])
    stats = {}
    C, L, _, _ = km_oracle.kmeans(xyz, 8, weights=w, max_iter=3, stats=stats)
    first = [(j, row) for it, j, row in stats["relocated"] if it == 1]
    assert len(first) >= 2
    assert len({row for _, row in first}) == len(first)
    assert [j for j, _ in first] == sorted(j for j, _ in first)
    assert_array_equal(L, vq.vq(xyz, C)[0])


@pytest.mark.parametrize("weighted", [False, True])
def test_oracle_invariants(weighted):
    xyz = box_xyz(20000)
    w = np.random.default_rng(5).uniform(0.5, 2.0, len(xyz)) if weighted else None
    C, L, n_iter, converged = km_oracle.kmeans(xyz, 8, weights=w)
    assert converged and 0 < n_iter < 500
    assert_array_equal(L, vq.vq(xyz, C)[0])
    s = km_oracle.int_sums(L, km_oracle.fixed_point(xyz, w), 8)
    assert_array_equal(C, km_oracle.centre(s))
    assert np.all(np.bincount(L, minlength=8) > 0)
    C0, L0, n0, c0 = km_oracle.kmeans(xyz, 8, weights=w, max_iter=0)
    assert n0 == 0 and not c0
    assert_array_equal(L0, vq.vq(xyz, C0)[0])


def test_int_sums_are_exact():
    q = np.array([[2**32, -(2**32), 1]] * 5 + [[3, 3, 3]], dtype=np.int64)
    s = km_oracle.int_sums(np.array([1, 1, 1, 1, 1, 0]), q, 3)
    assert_array_equal(s, [[3, 3, 3], [5 * 2**32, -5 * 2**32, 5], [0, 0, 0]])


# ---- host plumbing ---------------------------------------------------------------------------------------------
def _radec(n, seed=1):
    g = yb.BoxRandoms(0, 40, -12.5, 12.5, seed=seed)(n)
    return np.rad2deg(g["ra"]), np.rad2deg(g["dec"])


def _assert_same_catalog(a, b):
    assert list(a.keys()) == list(b.keys())
    assert_array_equal(a.get_centers().data, b.get_centers().data)
    for pid in a:
        assert_array_equal(a[pid].load_data(), b[pid].load_data())


def test_from_arrays_patch_num_equals_explicit_centres():
    ra, dec = _radec(5000)
    w = np.random.default_rng(2).uniform(0.5, 1.5, len(ra))
    eng = KmeansEngine()
    cat = yb.Catalog.from_arrays(ra, dec, patch_num=6, weights=w, engine=eng)
    assert len(cat) == 6 and len(eng.calls) == 1
    xyz, weights, k = eng.calls[0]
    want = yb.AngularCoordinates(np.deg2rad(np.column_stack([ra, dec]))).to_3d()
    assert k == 6
    assert_array_equal(xyz, want)
    assert_array_equal(weights, w)  # the catalog's weights go into the k-means
    C, _, _, _ = km_oracle.kmeans(want, 6, weights=w)
    assert_array_equal(cat.get_centers().data, yb.AngularCoordinates.from_3d(C).data)
    again = yb.Catalog.from_arrays(ra, dec, patch_centers=cat, weights=w, engine=eng)
    assert len(eng.calls) == 1
    _assert_same_catalog(cat, again)


def test_probe_size_takes_every_ceil_n_over_probe_row():
    ra, dec = _radec(1000)
    w = np.arange(1000, dtype=np.float64) + 1.0
    eng = KmeansEngine()
    centres = catalog_mod.create_patch_centers(np.deg2rad(ra), np.deg2rad(dec), 4, weights=w, probe_size=300,
                                               engine=eng)
    xyz, weights, _ = eng.calls[0]
    full = yb.AngularCoordinates(np.deg2rad(np.column_stack([ra, dec]))).to_3d()
    assert len(xyz) == 250  # ceil(1000 / 300) = 4
    assert_array_equal(xyz, full[::4])
    assert_array_equal(weights, w[::4])
    assert isinstance(centres, yb.AngularCoordinates) and len(centres) == 4
    catalog_mod.create_patch_centers(np.deg2rad(ra), np.deg2rad(dec), 4, probe_size=1000, engine=eng)
    assert len(eng.calls[1][0]) == 1000
    catalog_mod.create_patch_centers(np.deg2rad(ra), np.deg2rad(dec), 4, probe_size=-1, engine=eng)
    assert len(eng.calls[2][0]) == 1000


def test_create_patch_centers_uses_the_default_engine(monkeypatch):
    eng = KmeansEngine()
    monkeypatch.setattr(measurements, "get_default_engine", lambda: eng)
    ra, dec = _radec(500)
    centres = catalog_mod.create_patch_centers(np.deg2rad(ra), np.deg2rad(dec), 3)
    assert len(eng.calls) == 1 and len(centres) == 3


def test_from_dataframe_patch_num_and_precedence():
    ra, dec = _radec(3000)
    frame = {"ra": ra, "dec": dec, "z": np.linspace(0.1, 1.0, len(ra)), "pid": np.arange(len(ra)) % 3}
    eng = KmeansEngine()
    cat = yb.Catalog.from_dataframe("df", frame, ra_name="ra", dec_name="dec", redshift_name="z", patch_num=5,
                                    probe_size=1000, engine=eng)
    assert len(cat) == 5 and cat.has_redshifts
    assert len(eng.calls) == 1 and len(eng.calls[0][0]) == 1000
    _assert_same_catalog(cat, yb.Catalog.from_dataframe("df2", frame, ra_name="ra", dec_name="dec",
                                                        redshift_name="z", patch_centers=cat, engine=eng))
    # patch_centers, then patch_name, then patch_num
    by_centres = yb.Catalog.from_dataframe("a", frame, ra_name="ra", dec_name="dec", patch_centers=cat,
                                           patch_name="pid", patch_num=7, engine=eng)
    by_name = yb.Catalog.from_dataframe("b", frame, ra_name="ra", dec_name="dec", patch_name="pid", patch_num=7,
                                        engine=eng)
    assert len(eng.calls) == 1
    assert len(by_centres) == 5 and len(by_name) == 3
    assert [len(p) for p in by_name.values()] == [1000, 1000, 1000]


def test_patch_num_errors():
    ra, dec = _radec(100)
    eng = KmeansEngine()
    for bad in (0, -3):
        with pytest.raises(ValueError, match="patch_num"):
            yb.Catalog.from_arrays(ra, dec, patch_num=bad, engine=eng)
        with pytest.raises(ValueError, match="patch_num"):
            yb.Catalog.from_random("r", yb.BoxRandoms(0, 1, 0, 1), 100, patch_num=bad, engine=eng)
    with pytest.raises(ValueError, match="must be provided"):
        yb.Catalog.from_arrays(ra, dec, engine=eng)
    with pytest.raises(ValueError, match="must be provided"):
        yb.Catalog.from_dataframe("c", {"ra": ra, "dec": dec}, ra_name="ra", dec_name="dec", engine=eng)
    # a patch_num that is not used is not checked (precedence as above)
    cat = yb.Catalog.from_arrays(ra, dec, patch_ids=np.arange(100) % 2, patch_num=0, engine=eng)
    assert len(cat) == 2 and not eng.calls


def test_from_random_patch_num_links_with_its_randoms():
    eng = KmeansEngine()
    data = yb.Catalog.from_random("d", yb.BoxRandoms(0, 40, -12.5, 12.5, seed=1), 8000, patch_num=8, engine=eng)
    rand = yb.Catalog.from_random("r", yb.BoxRandoms(0, 40, -12.5, 12.5, seed=2), 16000, patch_centers=data,
                                  engine=eng)
    assert len(eng.calls) == 1 and len(data) == 8
    assert list(rand.keys()) == list(data.keys())
    assert_array_equal(rand.get_centers().data, data.get_centers().data)
    config = yb.Configuration.create(rmin=100, rmax=1000, zmin=0.1, zmax=1.0, num_bins=4)
    links = PatchLinkage.from_catalogs(config, data, rand)
    assert set(links.patch_links) == set(data.keys())
    assert all(p in links.patch_links[p] for p in data)
