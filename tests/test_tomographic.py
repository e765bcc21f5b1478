"""`crosscorrelate_tomographic` on the CPU: every tomographic bin must get exactly what its own `crosscorrelate` call
returns.  The counts come from a label-aware test double of the engine (`LabelOracleEngine`, the oracle behind
`Engine.count(..., labels=True)`), so this checks the host logic: one labelled upload, the union of the bins' pair
lists, the per-bin packaging, the shared randoms counted once, the errors and the multi-rank reduce."""

import os
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp
from numpy.testing import assert_allclose, assert_array_equal

import golden_cases
import golden_io
from fake_engine import OracleEngine, _FakeDeviceCatalog

HERE = os.path.dirname(os.path.abspath(__file__))
N_TOMO = 3


class LabelOracleEngine(OracleEngine):
    """`OracleEngine` that also answers `labels=True`: a binned second catalog is split by its ids into unbinned
    catalogs, one per label, each counted by the oracle.  `log` records every count call as (first, second)."""

    def __init__(self):
        super().__init__()
        self.log = []

    @staticmethod
    def _label_view(cat2, label):
        m = cat2.zbin == label
        off = np.concatenate([[0], np.cumsum(np.bincount(cat2.patch[m], minlength=cat2.n_patch))])
        return _FakeDeviceCatalog(cat2.xyz[m], off, None if cat2.w is None else cat2.w[m], None, 1)

    def _count(self, cat1, cat2, pair_i, pair_j, r2_edges, labels):
        if not labels:
            return OracleEngine.count(self, cat1, cat2, pair_i, pair_j, r2_edges)
        views = [self._label_view(cat2, lab) for lab in range(cat2.n_bins)] if cat2.binned else [cat2]
        outs = [OracleEngine.count(self, cat1, v, pair_i, pair_j, r2_edges) for v in views]
        return np.stack([o[0] for o in outs]), np.stack([o[1] for o in outs]), outs[0][2]

    def count(self, cat1, cat2, pair_i, pair_j, r2_edges, *, exact=False, labels=False):
        self.log.append((cat1, cat2))
        return self._count(cat1, cat2, pair_i, pair_j, r2_edges, labels)

    def count2(self, cat1a, cat1b, cat2, pair_i, pair_j, r2_edges, *, labels=False):
        self.log.append(((cat1a, cat1b), cat2))
        ia, fa, st = self._count(cat1a, cat2, pair_i, pair_j, r2_edges, labels)
        ib, fb, _ = self._count(cat1b, cat2, pair_i, pair_j, r2_edges, labels)
        return (ia, fa), (ib, fb), st


def catalog_rows(c, m, weights=True):
    from yet_another_wizz_b200 import AngularCoordinates, Catalog

    return Catalog.from_arrays(
        c["ra"][m], c["dec"][m], patch_ids=c["patch"][m], patch_centers=AngularCoordinates(c["centers"]),
        weights=None if (c["w"] is None or not weights) else c["w"][m],
        redshifts=None if c["z"] is None else c["z"][m], degrees=False,
    )


def split_catalog(g, prefix, n_tomo=N_TOMO, seed=11):
    """the rows of a golden catalog split into `n_tomo` catalogs by a seeded label"""
    c = golden_io.catalog_arrays(g, prefix)
    lab = np.random.default_rng(seed).integers(0, n_tomo, len(c["ra"]))
    return [catalog_rows(c, lab == i) for i in range(n_tomo)]


def assert_same(got, want, exact):
    """`got` / `want`: lists of CorrFunc; unweighted results compare with ==, weighted ones to 1e-12"""
    assert len(got) == len(want)
    for a, b in zip(got, want):
        if exact:
            assert a == b
        for kind in ("dd", "dr", "rd", "rr"):
            x, y = getattr(a, kind), getattr(b, kind)
            assert (x is None) == (y is None), kind
            if x is None:
                continue
            cmp = assert_array_equal if exact else (lambda p, q: assert_allclose(p, q, rtol=golden_cases.RTOL_WEIGHTED))
            cmp(x.counts.counts, y.counts.counts)
            cmp(x.sum_weights.sum_weights1, y.sum_weights.sum_weights1)
            cmp(x.sum_weights.sum_weights2, y.sum_weights.sum_weights2)


def per_bin(config, ref, unknowns, ref_rand, rands, engine):
    import yet_another_wizz_b200 as yb

    return [yb.crosscorrelate(config, ref, unk, ref_rand=ref_rand, unk_rand=rand, engine=engine)
            for unk, rand in zip(unknowns, rands)]


def _inputs(name):
    g = golden_io.load(name)
    config = golden_cases.config_from_golden(g)
    ref, ref_rand, unk_rand = (golden_cases.catalog_from_golden(g, k) for k in ("ref", "ref_rand", "unk_rand"))
    return g, config, ref, ref_rand, unk_rand, split_catalog(g, "unk")


@pytest.mark.parametrize("rand_form", ["shared", "per_bin", "none"])
@pytest.mark.parametrize("name", ["cross_unweighted", "cross_weighted_multiscale"])
def test_equals_per_bin_calls(name, rand_form):
    import yet_another_wizz_b200 as yb

    g, config, ref, ref_rand, unk_rand, unknowns = _inputs(name)
    if rand_form == "shared":
        arg, rands = unk_rand, [unk_rand] * N_TOMO
    elif rand_form == "per_bin":
        arg = rands = split_catalog(g, "unk_rand", seed=12)
    else:
        arg, rands = None, [None] * N_TOMO
    eng = LabelOracleEngine()
    got = yb.crosscorrelate_tomographic(config, ref, unknowns, ref_rand=ref_rand, unk_rand=arg, engine=eng)
    want = per_bin(config, ref, unknowns, ref_rand, rands, LabelOracleEngine())
    for a, b in zip(got, want):
        assert_same(a, b, exact=name == "cross_unweighted")
    assert got[0][0].dd.counts.counts.sum() > 0
    # the bins travel as one labelled catalog; per-bin randoms as another, a shared one unlabelled
    assert eng.log[0][1].binned and eng.log[0][1].n_bins == N_TOMO
    assert all(cat2.binned == (rand_form != "shared" or cat2 is eng.log[0][1]) for _, cat2 in eng.log)
    n_second = 1 + (rand_form != "none")
    fused = bool(ref.has_weights) == bool(ref_rand.has_weights)  # crosscorrelate's decision
    assert len(eng.log) == (n_second if fused else 2 * n_second)


def test_ref_rand_none_takes_the_unfused_path():
    import yet_another_wizz_b200 as yb

    g, config, ref, _, unk_rand, unknowns = _inputs("cross_unweighted")
    eng = LabelOracleEngine()
    got = yb.crosscorrelate_tomographic(config, ref, unknowns, unk_rand=unk_rand, engine=eng)
    want = per_bin(config, ref, unknowns, None, [unk_rand] * N_TOMO, LabelOracleEngine())
    for a, b in zip(got, want):
        assert_same(a, b, exact=True)
        assert a[0].rd is None and a[0].rr is None
    assert len(eng.log) == 2 and all(not isinstance(c1, tuple) for c1, _ in eng.log)  # DD and DR, one call each


def test_shared_randoms_are_counted_once():
    import yet_another_wizz_b200 as yb

    g, config, ref, ref_rand, unk_rand, unknowns = _inputs("cross_unweighted")
    eng = LabelOracleEngine()
    yb.crosscorrelate_tomographic(config, ref, unknowns, ref_rand=ref_rand, unk_rand=unk_rand, engine=eng)
    unlabelled = [cat2 for _, cat2 in eng.log if not cat2.binned]
    assert len(unlabelled) == 1  # DR + RR: one fused count for all bins
    labelled = [cat2 for _, cat2 in eng.log if cat2.binned]
    assert len(labelled) == 1 and labelled[0].n_bins == N_TOMO  # DD + RD: one count over the labelled bins
    stats = yb.measurements.last_stats()
    assert set(stats) == {"DD+RD", "DR+RR"}


def test_bins_with_different_links():
    """a bin larger than every other catalog, with wider patches, decides its own (larger) link set; the other bins
    keep theirs, and no pair outside a bin's linkage appears in its result"""
    import yet_another_wizz_b200 as yb
    from yet_another_wizz_b200.measurements import PatchLinkage

    g, config, ref, ref_rand, unk_rand, unknowns = _inputs("cross_unweighted")
    c = golden_io.catalog_arrays(g, "unk")
    # copies of every row pushed away from the centre of its patch (ra, dec offsets x 1.6), plus the rows of the
    # random catalogs: more rows than any other catalog, and larger radii
    cr = golden_io.catalog_arrays(g, "unk_rand")
    wide = {}
    for k in ("ra", "dec", "patch", "z", "w"):
        parts = [c[k], cr[k]] if c[k] is not None and cr[k] is not None else None
        wide[k] = None if parts is None else np.concatenate(parts)
    ctr = golden_io.catalog_arrays(g, "unk")["centers"]
    push = lambda a, i: ctr[c["patch"], i] + 1.6 * (a - ctr[c["patch"], i])  # noqa: E731
    for k, i in (("ra", 0), ("dec", 1)):
        wide[k] = np.concatenate([wide[k], push(c[k], i)])
    for k in ("patch", "z", "w"):
        if wide[k] is not None:
            wide[k] = np.concatenate([wide[k], c[k]])
    wide["centers"] = ctr
    big = catalog_rows(wide, np.ones(len(wide["ra"]), dtype=bool))
    unknowns = [big, *unknowns[1:]]
    links = [PatchLinkage.from_catalogs(config, ref, u, ref_rand, unk_rand).patch_links for u in unknowns]
    assert links[0] != links[1]
    got = yb.crosscorrelate_tomographic(config, ref, unknowns, ref_rand=ref_rand, unk_rand=unk_rand,
                                        engine=LabelOracleEngine())
    want = per_bin(config, ref, unknowns, ref_rand, [unk_rand] * N_TOMO, LabelOracleEngine())
    for a, b, lk in zip(got, want, links):
        assert_same(a, b, exact=True)
        counted = a[0].dd.counts.counts.sum(axis=0) != 0
        for i, j in zip(*np.nonzero(counted)):
            assert j in lk[i]


def test_errors_are_raised_before_counting():
    import yet_another_wizz_b200 as yb
    from yet_another_wizz_b200 import InconsistentPatchesError

    g, config, ref, ref_rand, unk_rand, unknowns = _inputs("cross_weighted_multiscale")
    c = golden_io.catalog_arrays(g, "unk")
    eng = LabelOracleEngine()
    run = lambda unks, **kw: yb.crosscorrelate_tomographic(config, ref, unks, engine=eng, **kw)  # noqa: E731
    with pytest.raises(ValueError, match="at least one catalog"):
        run([], ref_rand=ref_rand)
    with pytest.raises(ValueError, match="254"):
        run([unknowns[0]] * 255, ref_rand=ref_rand)
    with pytest.raises(ValueError, match="random"):
        run(unknowns)
    with pytest.raises(ValueError, match="holds 2 catalogs"):
        run(unknowns, ref_rand=ref_rand, unk_rand=split_catalog(g, "unk_rand", n_tomo=2))
    with pytest.raises(ValueError, match="cache directory"):
        run([unknowns[0], ref], ref_rand=ref_rand)
    with pytest.raises(ValueError, match="cache directory"):
        run(unknowns, ref_rand=ref_rand, unk_rand=[unk_rand, unk_rand, unknowns[2]])
    unweighted = catalog_rows(c, np.arange(len(c["ra"])) % 2 == 0, weights=False)
    with pytest.raises(ValueError, match="weights"):
        run([unknowns[0], unweighted], ref_rand=ref_rand)
    rands = [catalog_rows(c, np.arange(len(c["ra"])) % 3 == i, weights=i != 1) for i in range(3)]
    with pytest.raises(ValueError, match="per-bin randoms"):
        run(unknowns, ref_rand=ref_rand, unk_rand=rands)
    no_patch0 = catalog_rows(c, c["patch"] != 0)
    with pytest.raises(InconsistentPatchesError):
        run([unknowns[0], no_patch0], ref_rand=ref_rand)
    assert eng.log == [] and eng.calls == 0


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.join(os.path.dirname(HERE), "oracle"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from test_tomographic import LabelOracleEngine, _inputs

    import yet_another_wizz_b200 as yb

    g, config, ref, ref_rand, unk_rand, unknowns = _inputs("cross_unweighted")
    res = yb.crosscorrelate_tomographic(config, ref, unknowns, ref_rand=ref_rand, unk_rand=unk_rand,
                                        engine=LabelOracleEngine())  # shard picked up from torch.distributed
    if rank == 0:
        np.savez(os.path.join(out_dir, "rank0.npz"), **{f"{kind}_{i}": getattr(corrs[0], kind).counts.counts
                                                        for i, corrs in enumerate(res) for kind in ("dd", "dr", "rd", "rr")})
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_rank_gloo_reduce_matches_single_rank(tmp_path):
    import yet_another_wizz_b200 as yb

    port = 29500 + ((os.getpid() + 997) % 2000)
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    g, config, ref, ref_rand, unk_rand, unknowns = _inputs("cross_unweighted")
    want = yb.crosscorrelate_tomographic(config, ref, unknowns, ref_rand=ref_rand, unk_rand=unk_rand,
                                         engine=LabelOracleEngine())
    got = np.load(tmp_path / "rank0.npz")
    for i, corrs in enumerate(want):
        for kind in ("dd", "dr", "rd", "rr"):
            assert_array_equal(got[f"{kind}_{i}"], getattr(corrs[0], kind).counts.counts)
