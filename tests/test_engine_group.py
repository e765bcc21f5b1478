"""`EngineGroup` on the CPU: the share plan of a call, and every measurement function on groups of 1, 2 and 3
oracle-backed engine doubles that hold only their share of the catalogs (a partial upload and a second-role row mask,
restated here on top of the existing doubles).  The golden results, or what a single double returns, must come out."""

import numpy as np
import pytest

import golden_cases
import golden_io
from fake_engine import OracleEngine, _FakeDeviceCatalog
from test_autocorrelate_tomographic import BinnedLabelOracleEngine, split_catalog
from test_tomographic import LabelOracleEngine, assert_same

from yet_another_wizz_b200.sharding import Shard, plan_shares

N_TOMO = 3


class _Shares:
    """`upload_catalog(keep=, second_rows=)` as the library does it: only the rows of the kept patches (unkept patches
    empty), and a second-role view holding the masked rows; every count takes the second catalog's view"""

    def upload_catalog(self, xyz, patch_off, *, keep=None, second_rows=None, **kw):
        self.partial_uploads = getattr(self, "partial_uploads", 0) + 1
        xyz = np.asarray(xyz).reshape(-1, 3)
        sizes = np.diff(patch_off)
        rows = np.concatenate([np.arange(patch_off[p], patch_off[p + 1]) for p in range(len(sizes)) if keep[p]] or
                              [np.zeros(0, dtype=np.int64)]).astype(np.int64)
        off = np.concatenate([[0], np.cumsum(np.where(np.asarray(keep) != 0, sizes, 0))])
        cols = {k: (v[rows] if isinstance(v, np.ndarray) and len(v) == len(xyz) else v) for k, v in kw.items()}
        cat = super().upload_catalog(xyz[rows], off, **cols)
        m = np.asarray(second_rows) != 0
        assert len(m) == len(rows)
        patch = np.repeat(np.arange(len(sizes)), np.diff(off))
        off2 = np.concatenate([[0], np.cumsum(np.bincount(patch[m], minlength=len(sizes)))])
        cols2 = {k: (v[m] if isinstance(v, np.ndarray) and len(v) == len(rows) else v) for k, v in cols.items()}
        cat.second = super().upload_catalog(xyz[rows][m], off2, **cols2)
        return cat

    def count(self, cat1, cat2, *args, **kw):
        return super().count(cat1, getattr(cat2, "second", cat2), *args, **kw)

    def count2(self, cat1a, cat1b, cat2, *args, **kw):
        return super().count2(cat1a, cat1b, getattr(cat2, "second", cat2), *args, **kw)


class ShareOracle(_Shares, LabelOracleEngine):
    pass


class ShareBinnedOracle(_Shares, BinnedLabelOracleEngine):
    pass


def _group(n, cls=ShareOracle):
    from yet_another_wizz_b200 import EngineGroup

    return EngineGroup([cls() for _ in range(n)])


def test_plan_owns_every_row_once_and_keeps_every_partner():
    rng = np.random.default_rng(3)
    n_patch = 24
    ra, dec = rng.uniform(0, 0.6, n_patch), rng.uniform(-0.3, 0.3, n_patch)
    centers = np.column_stack([np.cos(ra) * np.cos(dec), np.sin(ra) * np.cos(dec), np.sin(dec)])
    d2 = ((centers[:, None] - centers[None]) ** 2).sum(-1)
    pi, pj = np.nonzero(d2 < 0.04)
    sizes = rng.integers(0, 400, n_patch)
    sizes[5] = 0  # an empty patch still has an owner
    patch_off = np.concatenate([[0], np.cumsum(sizes)])
    xyz = np.repeat(centers, sizes, axis=0) + rng.normal(0, 0.01, (patch_off[-1], 3))
    for n_dev in (1, 2, 3, 8):
        plan = plan_shares([(pi, pj, sizes, sizes), (pj, pi, sizes, sizes)], np.full(n_patch, 0.05), centers, n_dev)
        owned = np.zeros(patch_off[-1], dtype=int)
        for d in range(n_dev):
            keep = plan.keep[d].astype(bool)
            rows = np.concatenate([np.arange(patch_off[p], patch_off[p + 1]) for p in np.flatnonzero(keep)] or [[]])
            mask = plan.mask(d, xyz, patch_off)
            assert len(mask) == len(rows)
            owned[rows.astype(int)[mask == 1]] += 1
            # every patch linked to an owned second patch, either way round, is uploaded
            assert keep[pi[plan.second[d][pj]]].all() and keep[pj[plan.second[d][pi]]].all()
            assert not (mask[np.isin(np.repeat(np.flatnonzero(keep), sizes[keep]), np.flatnonzero(~plan.second[d]))]).any()
        assert (owned == 1).all()
        assert sum(s.sum() for s in plan.second) >= n_patch  # every patch has at least one owner


@pytest.mark.parametrize("n_dev", [1, 2, 3])
@pytest.mark.parametrize("name", ["cross_unweighted", "cross_weighted_multiscale"])
def test_crosscorrelate(name, n_dev):
    g = golden_io.load(name)
    grp = _group(n_dev)
    corrs = golden_cases.run_cross(g, grp)
    golden_cases.check_corrfunc(g, "cross", corrs, ("dd", "dr", "rd", "rr"), exact=name == "cross_unweighted")
    assert all(e.partial_uploads == 4 for e in grp.engines)


@pytest.mark.parametrize("n_dev", [1, 2, 3])
@pytest.mark.parametrize("name", ["auto_unweighted", "auto_rweight_polewrap"])
def test_autocorrelate(name, n_dev):
    g = golden_io.load(name)
    corrs = golden_cases.run_auto(g, _group(n_dev))
    golden_cases.check_corrfunc(g, "auto", corrs, ("dd", "dr", "rr"), exact=name == "auto_unweighted")


@pytest.mark.parametrize("n_dev", [1, 2, 3])
@pytest.mark.parametrize("name", ["scalar_unweighted", "scalar_weighted"])
def test_scalar(name, n_dev):
    g = golden_io.load(name)
    golden_cases.check_scalar(g, golden_cases.run_scalar(g, _group(n_dev)), exact_numbers=name == "scalar_unweighted")


@pytest.mark.parametrize("n_dev", [1, 2, 3])
def test_crosscorrelate_tomographic(n_dev):
    import yet_another_wizz_b200 as yb

    g = golden_io.load("cross_weighted_multiscale")
    config = golden_cases.config_from_golden(g)
    cats = {k: golden_cases.catalog_from_golden(g, k) for k in ("ref", "ref_rand", "unk_rand")}
    unknowns = split_catalog(g, "unk")
    kw = dict(ref_rand=cats["ref_rand"], unk_rand=cats["unk_rand"])
    got = yb.crosscorrelate_tomographic(config, cats["ref"], unknowns, engine=_group(n_dev), **kw)
    want = yb.crosscorrelate_tomographic(config, cats["ref"], unknowns, engine=LabelOracleEngine(), **kw)
    for a, b in zip(got, want):
        assert_same(a, b, exact=False)


@pytest.mark.parametrize("n_dev", [1, 2, 3])
@pytest.mark.parametrize("rand_form", ["shared", "per_bin"])
def test_autocorrelate_tomographic(rand_form, n_dev):
    import yet_another_wizz_b200 as yb

    g = golden_io.load("auto_unweighted")
    config = golden_cases.config_from_golden(g)
    data = split_catalog(g, "data")
    rand = golden_cases.catalog_from_golden(g, "rand") if rand_form == "shared" else split_catalog(g, "rand", seed=12)
    got = yb.autocorrelate_tomographic(config, data, rand, engine=_group(n_dev, ShareBinnedOracle))
    want = yb.autocorrelate_tomographic(config, data, rand, engine=BinnedLabelOracleEngine())
    for a, b in zip(got, want):
        assert_same(a, b, exact=True)


def test_group_with_active_shard_raises():
    import yet_another_wizz_b200 as yb

    g = golden_io.load("cross_unweighted")
    config = golden_cases.config_from_golden(g)
    ref, unk, rand = (golden_cases.catalog_from_golden(g, k) for k in ("ref", "unk", "unk_rand"))
    with pytest.raises(ValueError, match="shard"):
        yb.crosscorrelate(config, ref, unk, unk_rand=rand, engine=_group(2), shard=Shard(0, 2))


def test_an_engine_object_appears_once():
    from yet_another_wizz_b200 import EngineGroup

    eng = ShareOracle()
    with pytest.raises(ValueError):
        EngineGroup([eng, eng])
