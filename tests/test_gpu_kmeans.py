"""
GPU tests of the deterministic spherical k-means (`yawb_kmeans`, `Engine.kmeans`, `patch_num=`): bit-exact against
the numpy restatement in `oracle/kmeans.py`, and independent checks at catalog sizes the oracle cannot reach.
"""

import numpy as np
import pytest
from numpy.testing import assert_array_equal
from scipy.cluster import vq

import kmeans as km_oracle

import yet_another_wizz_b200 as yb

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    eng = yb.Engine(0)
    yield eng
    eng.close()


def box_xyz(n, seed=1):
    g = yb.BoxRandoms(0, 40, -12.5, 12.5, seed=seed)(n)
    return yb.AngularCoordinates(np.column_stack([g["ra"], g["dec"]])).to_3d()


def blobs_xyz(n_per, centres_deg, sigma_deg, seed=4):
    rng = np.random.default_rng(seed)
    parts = []
    for ra, dec in centres_deg:
        r = np.deg2rad(ra + rng.normal(0, sigma_deg, n_per))
        d = np.deg2rad(np.clip(dec + rng.normal(0, sigma_deg, n_per), -89.0, 89.0))
        parts.append(np.column_stack([np.cos(r) * np.cos(d), np.sin(r) * np.cos(d), np.sin(d)]))
    return np.concatenate(parts)


def check_vs_oracle(engine, xyz, k, weights=None, max_iter=500, stats=None):
    got = engine.kmeans(xyz, k, weights=weights, max_iter=max_iter)
    want = km_oracle.kmeans(xyz, k, weights=weights, max_iter=max_iter, stats=stats)
    assert_array_equal(got[0], want[0])
    assert_array_equal(got[1], want[1])
    assert got[2:] == tuple(want[2:])
    return got


def test_uniform_50k_k16_converged(engine):
    C, L, n_iter, converged = check_vs_oracle(engine, box_xyz(50_000), 16)
    assert converged


def test_uniform_200k_k64_converged(engine):
    C, L, n_iter, converged = check_vs_oracle(engine, box_xyz(200_000), 64)
    assert converged
    print(f"2e5 x 64: {n_iter} iterations")


def test_clustered(engine):
    rng = np.random.default_rng(8)
    centres = np.column_stack([rng.uniform(0, 360, 20), np.rad2deg(np.arcsin(rng.uniform(-1, 1, 20)))])
    check_vs_oracle(engine, blobs_xyz(5000, centres, 3.0), 32, max_iter=50)


def test_weighted(engine):
    xyz = box_xyz(100_000, seed=2)
    w = np.random.default_rng(3).uniform(0.0, 3.0, len(xyz))
    check_vs_oracle(engine, xyz, 16, weights=w, max_iter=50)


def test_single_patch(engine):
    C, L, n_iter, converged = check_vs_oracle(engine, box_xyz(100_000, seed=3), 1, max_iter=5)
    assert converged and n_iter == 1 and not L.any()


def test_sorted_rows(engine):
    # rows in RA order: whole warps share a label, the warp-aggregated path of the accumulators
    xyz = box_xyz(100_000, seed=5)
    xyz = xyz[np.argsort(np.arctan2(xyz[:, 1], xyz[:, 0]), kind="stable")]
    check_vs_oracle(engine, xyz, 16, max_iter=30)


def test_many_centre_blocks(engine):
    check_vs_oracle(engine, box_xyz(30_000, seed=6), 2500, max_iter=5)


def test_empty_cluster_relocation(engine):
    # zero-weight rows form clusters whose weighted sum is (0, 0, 0)
    xyz = blobs_xyz(3000, [(10, 0)], 2.9, seed=3)
    xyz = np.concatenate([xyz, blobs_xyz(300, [(100, 0)], 0.6, seed=9)])
    w = np.concatenate([np.ones(3000), np.zeros(300)])
    stats = {}
    check_vs_oracle(engine, xyz, 8, weights=w, max_iter=20, stats=stats)
    assert len(stats["relocated"]) >= 2


def test_not_converged_and_initial(engine):
    xyz = box_xyz(50_000, seed=7)
    C, L, n_iter, converged = check_vs_oracle(engine, xyz, 16, max_iter=3)
    assert n_iter == 3 and not converged
    C, L, n_iter, converged = check_vs_oracle(engine, xyz, 16, max_iter=0)
    assert n_iter == 0 and not converged


def test_2e6_rows_20_iterations(engine):
    check_vs_oracle(engine, box_xyz(2_000_000, seed=8), 64, max_iter=20)


def test_1e7_rows_self_consistent_and_repeatable(engine):
    xyz = box_xyz(10_000_000, seed=9)
    C, L, n_iter, converged = engine.kmeans(xyz, 64)
    assert_array_equal(L, vq.vq(xyz, C)[0])
    C2, L2, n2, c2 = engine.kmeans(xyz, 64)
    assert_array_equal(C2, C)
    assert_array_equal(L2, L)
    assert (n2, c2) == (n_iter, converged)
    print(f"1e7 x 64: {n_iter} iterations, converged={converged}")


def test_recovers_separated_blobs(engine):
    centres = [(45 + 90 * i, s * 35) for i in range(4) for s in (1, -1)]  # the corners of a cube
    xyz = blobs_xyz(2000, centres, 2.0, seed=11)
    C, L, n_iter, converged = engine.kmeans(xyz, 8)
    assert converged
    blob_labels = L.reshape(8, 2000)
    assert np.all(blob_labels == blob_labels[:, :1])
    assert len(set(blob_labels[:, 0].tolist())) == 8


def test_balance_uniform_box(engine):
    C, L, n_iter, converged = engine.kmeans(box_xyz(200_000), 16)
    counts = np.bincount(L, minlength=16)
    assert converged and counts.min() > 0
    ratio = counts.max() / counts.min()
    print(f"2e5 x 16: max/min rows per patch {ratio:.3f} after {n_iter} iterations")
    assert ratio <= 1.6


def test_patch_num_end_to_end(engine):
    pool = np.random.default_rng(7).uniform(0.1, 1.0, 100000)

    def gen(seed, z=True):
        return yb.BoxRandoms(0, 10, -2.5, 2.5, redshifts=pool if z else None, seed=seed)

    ref = yb.Catalog.from_random("ref", gen(1), 20000, patch_num=16, engine=engine)
    assert len(ref) == 16
    unk = yb.Catalog.from_random("unk", gen(2, False), 30000, patch_centers=ref, engine=engine)
    rand = yb.Catalog.from_random("rand", gen(3), 40000, patch_centers=ref, engine=engine)
    centres = ref.get_centers()
    ref2 = yb.Catalog.from_random("ref2", gen(1), 20000, patch_centers=centres, engine=engine)
    unk2 = yb.Catalog.from_random("unk2", gen(2, False), 30000, patch_centers=centres, engine=engine)
    rand2 = yb.Catalog.from_random("rand2", gen(3), 40000, patch_centers=centres, engine=engine)
    config = yb.Configuration.create(rmin=100, rmax=1000, zmin=0.1, zmax=1.0, num_bins=5)
    (a,) = yb.crosscorrelate(config, ref, unk, ref_rand=rand, engine=engine)
    (b,) = yb.crosscorrelate(config, ref2, unk2, ref_rand=rand2, engine=engine)
    for kind in ("dd", "rd"):
        assert_array_equal(getattr(a, kind).counts.counts, getattr(b, kind).counts.counts)
    assert a.dd.counts.counts.sum() > 0
    (a,) = yb.autocorrelate(config, ref, rand, engine=engine)
    (b,) = yb.autocorrelate(config, ref2, rand2, engine=engine)
    for kind in ("dd", "dr", "rr"):
        assert_array_equal(getattr(a, kind).counts.counts, getattr(b, kind).counts.counts)


def test_errors_leave_engine_usable(engine):
    xyz = box_xyz(1000, seed=12)
    bad_nan = xyz.copy()
    bad_nan[17, 1] = np.nan
    bad_big = xyz.copy()
    bad_big[3, 2] = 1.0 + 1e-12
    w_neg = np.ones(len(xyz))
    w_neg[5] = -1.0
    cases = [
        (dict(xyz=bad_nan, k=4), "not finite"),
        (dict(xyz=bad_big, k=4), "outside"),
        (dict(xyz=xyz, k=4, weights=w_neg), "negative"),
        (dict(xyz=xyz[:3], k=4), "more patches"),
        (dict(xyz=xyz, k=4097), "k must be"),
        (dict(xyz=np.repeat(xyz[:2], 50, axis=0), k=3), "fewer distinct positions"),
    ]
    for kw, msg in cases:
        with pytest.raises(yb.YawbError, match=msg):
            engine.kmeans(**kw)
    check_vs_oracle(engine, xyz, 4, max_iter=10)
