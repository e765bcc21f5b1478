"""`autocorrelate_tomographic` on the CPU: every tomographic bin must get exactly what its own `autocorrelate` call
returns.  The counts come from a test double of the engine that understands binned labels (`BinnedLabelOracleEngine`,
the oracle behind `Engine.count` with catalogs uploaded with `n_labels`), so this checks the host logic: the labelled
uploads, the union of the bins' pair lists, the swapped DR against shared randoms, the per-bin packaging, RR counted
once, the errors, the multi-rank reduce and the labelled-upload cache."""

import gc
import os
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp
from numpy.testing import assert_array_equal

import golden_cases
import golden_io
from fake_engine import OracleEngine, _FakeDeviceCatalog
from test_tomographic import LabelOracleEngine, assert_same, catalog_rows

HERE = os.path.dirname(os.path.abspath(__file__))
N_TOMO = 3


class _CachingUploads:
    """uploads counted in `uploads`; with `cache=True` device catalogs are kept by the engine's own cache code"""

    from yet_another_wizz_b200.engine import Engine as _E

    cache_lookup, cache_store, _cache_drop = _E.cache_lookup, _E.cache_store, _E._cache_drop
    _cache_identity = _E.__dict__["_cache_identity"]
    del _E

    def __init__(self, cache=False):
        super().__init__()
        self.log = []
        self.uploads = 0
        self.cache_catalogs = cache
        self.cache_bytes = 1 << 40
        self._cat_cache = {}
        self._cat_cache_tick = 0

    def upload_catalog(self, xyz, patch_off, *, weights=None, zbin=None, n_bins=1, n_labels=None):
        self.uploads += 1
        cat = _FakeDeviceCatalog(xyz, patch_off, weights, zbin, n_bins)
        cat.n_labels = n_labels
        cat._h = object()  # a live handle, as the engine's cache expects
        cat.info = lambda: (len(cat.xyz), cat.xyz.nbytes)
        return cat


class BinnedLabelOracleEngine(_CachingUploads, OracleEngine):
    """`OracleEngine` that also answers counts of catalogs with binned labels (id = label * B + z-bin): label l of
    the second catalog is cut out as a z-binned catalog and counted by the oracle against label l of the first
    catalog (rule a) or against the whole, unlabelled first catalog (rule b).  `log` records every count as
    (first, second)."""

    @staticmethod
    def _label_view(cat, label, n_z):
        ids = cat.zbin.astype(np.int64)
        m = (ids >= label * n_z) & (ids < (label + 1) * n_z)
        off = np.concatenate([[0], np.cumsum(np.bincount(cat.patch[m], minlength=cat.n_patch))])
        return _FakeDeviceCatalog(cat.xyz[m], off, None if cat.w is None else cat.w[m], ids[m] - label * n_z, n_z)

    def count(self, cat1, cat2, pair_i, pair_j, r2_edges, *, exact=False, labels=False):
        self.log.append((cat1, cat2))
        l1, l2 = getattr(cat1, "n_labels", None), getattr(cat2, "n_labels", None)
        if l2 is None:
            assert l1 is None, "a labelled first catalog needs a labelled second one"
            return OracleEngine.count(self, cat1, cat2, pair_i, pair_j, r2_edges)
        n_z = cat2.n_bins // l2
        assert (l1 == l2 and cat1.n_bins == cat2.n_bins) if l1 is not None else (cat1.binned and cat1.n_bins == n_z)
        assert r2_edges.shape[0] == n_z
        outs = [OracleEngine.count(self, cat1 if l1 is None else self._label_view(cat1, lab, n_z),
                                   self._label_view(cat2, lab, n_z), pair_i, pair_j, r2_edges) for lab in range(l2)]
        return np.stack([o[0] for o in outs]), np.stack([o[1] for o in outs]), outs[0][2]


def split_catalog(g, prefix, n_tomo=N_TOMO, seed=11):
    """the rows of a golden catalog split into `n_tomo` catalogs by a seeded label"""
    c = golden_io.catalog_arrays(g, prefix)
    lab = np.random.default_rng(seed).integers(0, n_tomo, len(c["ra"]))
    return [catalog_rows(c, lab == i) for i in range(n_tomo)]


def _inputs(name):
    g = golden_io.load(name)
    config = golden_cases.config_from_golden(g)
    rand = golden_cases.catalog_from_golden(g, "rand")
    return g, config, rand, split_catalog(g, "data")


def per_bin(config, data, rands, engine, count_rr=True):
    import yet_another_wizz_b200 as yb

    return [yb.autocorrelate(config, d, r, count_rr=count_rr, engine=engine) for d, r in zip(data, rands)]


NAMES = ["auto_unweighted", "auto_rweight_polewrap"]


@pytest.mark.parametrize("count_rr", [True, False])
@pytest.mark.parametrize("rand_form", ["shared", "per_bin"])
@pytest.mark.parametrize("name", NAMES)
def test_equals_per_bin_calls(name, rand_form, count_rr):
    import yet_another_wizz_b200 as yb

    g, config, rand, data = _inputs(name)
    if rand_form == "shared":
        arg, rands = rand, [rand] * N_TOMO
    else:
        arg = rands = split_catalog(g, "rand", seed=12)
    eng = BinnedLabelOracleEngine()
    got = yb.autocorrelate_tomographic(config, data, arg, count_rr=count_rr, engine=eng)
    want = per_bin(config, data, rands, BinnedLabelOracleEngine(), count_rr=count_rr)
    for a, b in zip(got, want):
        assert_same(a, b, exact=name == "auto_unweighted")
        assert all((c.rr is None) == (not count_rr) for c in a)
    assert got[0][0].dd.counts.counts.sum() > 0 and got[-1][0].dr.counts.counts.sum() > 0
    # DD, DR (and RR): one count each, the data as one catalog with binned labels
    assert len(eng.log) == 2 + count_rr
    dd1, dd2 = eng.log[0]
    assert dd1 is dd2 and dd1.n_labels == N_TOMO and dd1.n_bins == N_TOMO * len(config.binning.binning)
    dr1, dr2 = eng.log[1]
    if rand_form == "shared":  # swapped: the randoms (binned, unlabelled) first
        assert dr1.n_labels is None and dr1.binned and dr2 is dd1
    else:
        assert dr1 is dd1 and dr2.n_labels == N_TOMO
    if count_rr:
        rr1, rr2 = eng.log[2]
        assert rr1 is rr2 is (dr1 if rand_form == "shared" else dr2)
    assert set(yb.measurements.last_stats()) == ({"DD", "DR", "RR"} if count_rr else {"DD", "DR"})


def test_bins_with_different_links():
    """a bin larger than the randoms, with wider patches, decides its own (larger) link set; the other bins keep
    theirs, RR over the shared randoms is still exact per bin, and no pair outside a bin's linkage appears"""
    import yet_another_wizz_b200 as yb
    from yet_another_wizz_b200.measurements import PatchLinkage

    g, config, rand, data = _inputs("auto_rweight_polewrap")
    c, cr = golden_io.catalog_arrays(g, "data"), golden_io.catalog_arrays(g, "rand")
    ctr = c["centers"]
    push = lambda a, i: ctr[c["patch"], i] + 1.6 * (a - ctr[c["patch"], i])  # noqa: E731
    wide = {k: np.concatenate([c[k], cr[k], push(c[k], i)]) for k, i in (("ra", 0), ("dec", 1))}
    for k in ("patch", "z", "w"):
        wide[k] = np.concatenate([c[k], np.ones(len(cr["ra"])) if k == "w" else cr[k], c[k]])
    wide.update(centers=ctr)
    big = catalog_rows(wide, np.ones(len(wide["ra"]), dtype=bool))
    data = [big, *data[1:]]
    links = [PatchLinkage.from_catalogs(config, d, rand).patch_links for d in data]
    assert links[0] != links[1]
    eng = BinnedLabelOracleEngine()
    got = yb.autocorrelate_tomographic(config, data, rand, engine=eng)
    want = per_bin(config, data, [rand] * N_TOMO, BinnedLabelOracleEngine())
    for a, b, lk in zip(got, want, links):
        assert_same(a, b, exact=False)
        for kind in ("dd", "dr", "rr"):
            counted = getattr(a[0], kind).counts.counts.sum(axis=0) != 0
            for i, j in zip(*np.nonzero(counted)):
                assert j in lk[i]
    assert len(eng.log) == 3  # RR once over the union of the bins' pair lists


def test_errors_are_raised_before_counting():
    import yet_another_wizz_b200 as yb
    from yet_another_wizz_b200 import AngularCoordinates, Catalog, InconsistentPatchesError

    g, config, rand, data = _inputs("auto_rweight_polewrap")
    c = golden_io.catalog_arrays(g, "data")
    eng = BinnedLabelOracleEngine()
    run = lambda d, r=rand, **kw: yb.autocorrelate_tomographic(config, d, r, engine=eng, **kw)  # noqa: E731
    with pytest.raises(ValueError, match="at least one catalog"):
        run([])
    with pytest.raises(ValueError, match="254"):
        run([data[0]] * 255)
    with pytest.raises(ValueError, match="holds 2 catalogs"):
        run(data, split_catalog(g, "rand", n_tomo=2))
    with pytest.raises(ValueError, match="cache directory"):
        run([data[0], rand])
    with pytest.raises(ValueError, match="cache directory"):
        run(data, [rand, rand, data[2]])
    no_z = Catalog.from_arrays(c["ra"], c["dec"], patch_ids=c["patch"], patch_centers=AngularCoordinates(c["centers"]),
                               degrees=False)
    with pytest.raises(ValueError, match="redshifts"):
        run([data[0], no_z])
    with pytest.raises(ValueError, match="redshifts"):
        run(data, [split_catalog(g, "rand")[0], no_z, split_catalog(g, "rand")[2]])
    unweighted = catalog_rows(c, np.arange(len(c["ra"])) % 2 == 0, weights=False)
    with pytest.raises(ValueError, match="weights"):
        run([data[0], unweighted])
    rands = [catalog_rows(c, np.arange(len(c["ra"])) % 3 == i, weights=i != 1) for i in range(3)]
    with pytest.raises(ValueError, match="per-bin randoms"):
        run(data, rands)
    no_patch0 = catalog_rows(c, c["patch"] != 0)
    with pytest.raises(InconsistentPatchesError):
        run([data[0], no_patch0])
    assert eng.log == [] and eng.calls == 0 and eng.uploads == 0


def test_second_call_uploads_nothing_and_cache_follows_its_members():
    import yet_another_wizz_b200 as yb

    g, config, rand, data = _inputs("auto_unweighted")
    rands = split_catalog(g, "rand", seed=12)
    eng = BinnedLabelOracleEngine(cache=True)
    first = yb.autocorrelate_tomographic(config, data, rands, engine=eng)
    assert eng.uploads == 2  # the bins and their randoms, each as one labelled catalog
    second = yb.autocorrelate_tomographic(config, data, rands, engine=eng)
    assert eng.uploads == 2
    for a, b in zip(first, second):
        assert_same(a, b, exact=True)
    # a shared random catalog is kept as a single catalog; the labelled data catalog is reused
    yb.autocorrelate_tomographic(config, data, rand, engine=eng)
    assert eng.uploads == 3
    assert len(eng._cat_cache) == 3
    # an entry goes when any of its members dies
    del rands[1]
    gc.collect()
    assert len(eng._cat_cache) == 2
    # YAWB_CACHE=0: nothing stays
    off = BinnedLabelOracleEngine(cache=False)
    yb.autocorrelate_tomographic(config, data, rand, engine=off)
    yb.autocorrelate_tomographic(config, data, rand, engine=off)
    assert off.uploads == 4 and off._cat_cache == {}


def test_crosscorrelate_tomographic_reuses_labelled_uploads():
    import yet_another_wizz_b200 as yb
    from test_tomographic import _inputs as cross_inputs

    g, config, ref, ref_rand, unk_rand, unknowns = cross_inputs("cross_unweighted")
    per = split_catalog(g, "unk_rand", seed=12)
    eng = type("CachingLabelOracleEngine", (_CachingUploads, LabelOracleEngine), {})(cache=True)
    first = yb.crosscorrelate_tomographic(config, ref, unknowns, ref_rand=ref_rand, unk_rand=per, engine=eng)
    n = eng.uploads
    second = yb.crosscorrelate_tomographic(config, ref, unknowns, ref_rand=ref_rand, unk_rand=per, engine=eng)
    assert eng.uploads == n
    for a, b in zip(first, second):
        assert_same(a, b, exact=True)


@pytest.mark.parametrize("n_tomo", [3, 90])
def test_prepare_labelled_arrays_drops_rows_outside_the_binning(n_tomo):
    from yet_another_wizz_b200.measurements import _as_binning, prepare_catalog_arrays, prepare_labelled_arrays

    g, config, rand, _ = _inputs("auto_unweighted")
    data = split_catalog(g, "data", n_tomo=n_tomo)
    binning = _as_binning(config)
    n_z = len(binning)
    z_all = np.concatenate([np.asarray(d[p].load_data()["redshifts"]) for d in data for p in d.keys()])
    assert np.any(binning.digitize(z_all) < 0) or np.any(binning.digitize(z_all) >= n_z)  # some rows outside
    out = prepare_labelled_arrays(data, binning)
    assert out["n_labels"] == n_tomo and out["n_bins"] == n_tomo * n_z
    ids = out["zbin"].astype(np.int64)
    assert out["zbin"].dtype == (np.uint8 if n_tomo * n_z <= 254 else np.int32)
    drop = 255 if n_tomo * n_z <= 254 else -1
    # per (patch, label): the ids are label * B + the ids prepare_catalog_arrays gives that catalog alone
    pos = 0
    for p in range(len(data[0])):
        for lab, d in enumerate(data):
            own = prepare_catalog_arrays(d, binning)
            s, e = own["patch_off"][p], own["patch_off"][p + 1]
            z = own["zbin"][s:e].astype(np.int64)
            kept = z < n_z if own["zbin"].dtype == np.uint8 else (z >= 0) & (z < n_z)
            assert_array_equal(ids[pos:pos + e - s], np.where(kept, lab * n_z + z, drop))
            assert_array_equal(out["xyz"][pos:pos + e - s], own["xyz"][s:e])
            pos += e - s
    assert pos == len(ids)
    with pytest.raises(ValueError, match="redshifts"):
        prepare_labelled_arrays([catalog_rows({**golden_io.catalog_arrays(g, "data"), "z": None},
                                              np.ones(3000, dtype=bool))], binning)


def _worker(rank, world, port, out_dir, rand_form):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.join(os.path.dirname(HERE), "oracle"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from test_autocorrelate_tomographic import BinnedLabelOracleEngine, _inputs, split_catalog

    import yet_another_wizz_b200 as yb

    g, config, rand, data = _inputs("auto_unweighted")
    arg = rand if rand_form == "shared" else split_catalog(g, "rand", seed=12)
    res = yb.autocorrelate_tomographic(config, data, arg, engine=BinnedLabelOracleEngine())  # shard from torch.distributed
    if rank == 0:
        np.savez(os.path.join(out_dir, "rank0.npz"), **{f"{kind}_{i}": getattr(corrs[0], kind).counts.counts
                                                        for i, corrs in enumerate(res) for kind in ("dd", "dr", "rr")})
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(300)
@pytest.mark.parametrize("rand_form", ["shared", "per_bin"])
def test_two_rank_gloo_reduce_matches_single_rank(tmp_path, rand_form):
    import yet_another_wizz_b200 as yb

    port = 29500 + ((os.getpid() + 991 + 7 * (rand_form == "shared")) % 2000)
    mp.spawn(_worker, args=(2, port, str(tmp_path), rand_form), nprocs=2, join=True)
    g, config, rand, data = _inputs("auto_unweighted")
    arg = rand if rand_form == "shared" else split_catalog(g, "rand", seed=12)
    want = yb.autocorrelate_tomographic(config, data, arg, engine=BinnedLabelOracleEngine())
    got = np.load(tmp_path / "rank0.npz")
    for i, corrs in enumerate(want):
        for kind in ("dd", "dr", "rr"):
            assert_array_equal(got[f"{kind}_{i}"], getattr(corrs[0], kind).counts.counts)
