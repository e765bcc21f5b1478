"""
GPU tests of counting one measurement on several contexts: the second-role row mask (yawb_catalog_set_second_rows),
the partial upload (yawb_upload_catalog_patches), several contexts driven by threads, and `EngineGroup` against
`Engine` for every public measurement function.

Bar: integer counts bit-exact, weighted sums within 1e-12 relative.
"""

import threading

import numpy as np
import pytest
from numpy.testing import assert_allclose, assert_array_equal

import golden_cases
import golden_io
import oracle

pytestmark = pytest.mark.gpu

RTOL = 1e-12


@pytest.fixture(scope="module")
def engine():
    from yet_another_wizz_b200 import Engine

    eng = Engine(0, cache_catalogs=False)
    yield eng
    eng.close()


def _rows(rng, n_patch, n_per, n_bins, weighted):
    """rows grouped by patch: patches of about 1 degree on a 4 x n_patch/4 grid, z-bin ids with some dropped"""
    ras = np.deg2rad(np.repeat(np.arange(n_patch) % 4 * 1.0, n_per) + rng.uniform(0, 1.0, n_patch * n_per))
    decs = np.deg2rad(np.repeat(np.arange(n_patch) // 4 * 1.0, n_per) + rng.uniform(0, 1.0, n_patch * n_per))
    xyz = oracle.radec_to_xyz(ras, decs)
    off = np.arange(n_patch + 1, dtype=np.int64) * n_per
    zbin = rng.integers(-1, n_bins + 1, len(xyz)).astype(np.int32)
    w = rng.uniform(0.5, 1.5, len(xyz)) if weighted else None
    return xyz, off, zbin, w


def _edges(n_bins, n_edges):
    return np.stack([oracle.chord_sq_edges(np.deg2rad(np.geomspace(0.02, 0.8 + 0.05 * b, n_edges)))
                     for b in range(n_bins)])


def _pairs(n_patch):
    pi, pj = np.meshgrid(np.arange(n_patch), np.arange(n_patch), indexing="ij")
    return pi.ravel().astype(np.int32), pj.ravel().astype(np.int32)


def _same(got, want, weighted, what=""):
    for g, w in zip(got, want):
        if weighted:
            assert_allclose(g, w, rtol=RTOL, atol=RTOL * max(np.abs(w).max(), 1e-300), err_msg=what)
        else:
            assert_array_equal(g, w, err_msg=what)


# (n_edges, weighted): Single, SingleWeighted, Cumulative, Histogram, HistogramWeighted
PATHS = [(2, False), (2, True), (5, False), (12, False), (6, True)]


@pytest.mark.parametrize("n_edges,weighted", PATHS)
def test_mask_contract_every_path(engine, n_edges, weighted):
    rng = np.random.default_rng(n_edges + 10 * weighted)
    n_patch, n_bins = 8, 3
    xyz, off, zbin, w = _rows(rng, n_patch, 3000, n_bins, weighted)
    xyz1, off1, zbin1, w1 = _rows(rng, n_patch, 2000, n_bins, weighted)
    edges = _edges(n_bins, n_edges)
    pi, pj = _pairs(n_patch)
    m = (rng.random(len(xyz)) < 0.4).astype(np.uint8)

    def up(x, o, z, ww, mask=None, **kw):
        return engine.upload_catalog(x, o, weights=ww, zbin=z, n_bins=n_bins, second_rows=mask, **kw)

    full, a, b = up(xyz, off, zbin, w), up(xyz, off, zbin, w, m), up(xyz, off, zbin, w, 1 - m)
    c1, c1b = up(xyz1, off1, zbin1, w1), up(xyz1[::-1].copy(), off1, zbin1, w1)
    pick = 1 if weighted else 0

    def plus(x, y):
        return x + y

    # yawb_count; auto counts with the masked upload as the second catalog and the full one (or itself) as the first
    for first_a, first_b, first_full in ((c1, c1, c1), (full, full, full), (a, b, full)):
        ga, gb, gf = (engine.count(f, s, pi, pj, edges) for f, s in ((first_a, a), (first_b, b), (first_full, full)))
        _same([plus(ga[pick], gb[pick]), plus(ga[0], gb[0])], [gf[pick], gf[0]], weighted, "count")
    # exact cross-check path
    ga, gb, gf = (engine.count(c1, s, pi, pj, edges, exact=True) for s in (a, b, full))
    _same([ga[pick] + gb[pick]], [gf[pick]], weighted, "exact")
    # yawb_count2 (fused first-role index) and yawb_count4
    ra, rb, rf = (engine.count2(c1, c1b, s, pi, pj, edges) for s in (a, b, full))
    for t in range(2):
        _same([ra[t][pick] + rb[t][pick]], [rf[t][pick]], weighted, "count2")
    oa, _ = engine.count4(c1, c1b, a, b, pi, pj, edges)
    for t in range(2):
        _same([oa[t][pick] + oa[t + 2][pick]], [rf[t][pick]], weighted, "count4")
    # the second-role mask leaves the first role, the sums of weights (FP64 atomic sums) and the row count alone
    assert_allclose(a.sum_weights(), full.sum_weights(), rtol=RTOL)
    assert a.info()[0] == full.info()[0]
    assert ga[0].sum() > 0 and gb[0].sum() > 0
    # clearing the mask gives the full upload back
    a.set_second_rows(None)
    _same([engine.count(c1, a, pi, pj, edges)[pick]], [gf[pick]], weighted, "cleared")
    for c in (full, a, b, c1, c1b):
        c.free()


@pytest.mark.parametrize("weighted", [False, True])
def test_mask_contract_labelled(engine, weighted):
    rng = np.random.default_rng(40 + weighted)
    n_patch, n_z, n_lab = 8, 2, 3
    xyz, off, zbin, w = _rows(rng, n_patch, 3000, n_z * n_lab, weighted)
    xyz1, off1, zbin1, w1 = _rows(rng, n_patch, 2000, n_z, weighted)
    lab8 = np.where(zbin >= 0, zbin, 255).astype(np.uint8)  # labels 0..5 (YAWB_FLAG_SECOND_LABELS) or binned labels
    pi, pj = _pairs(n_patch)
    m = (rng.random(len(xyz)) < 0.5).astype(np.uint8)
    pick = 1 if weighted else 0
    c1 = engine.upload_catalog(xyz1, off1, weights=w1, zbin=zbin1, n_bins=n_z)
    # YAWB_FLAG_SECOND_LABELS against the unbinned first role
    for mode in ("labels", "binned_labels"):
        kw = dict(n_labels=n_lab) if mode == "binned_labels" else {}
        cats = [engine.upload_catalog(xyz, off, weights=w, zbin=lab8, n_bins=n_z * n_lab, second_rows=mask, **kw)
                for mask in (m, 1 - m, None)]
        edges = _edges(n_z, 7)
        lab = mode == "labels"
        outs = [engine.count(c1, c, pi, pj, edges, labels=lab) for c in cats]
        _same([outs[0][pick] + outs[1][pick]], [outs[2][pick]], weighted, mode)
        if mode == "binned_labels":  # both catalogs labelled: auto count of a binned-label catalog
            autos = [engine.count(first, c, pi, pj, edges) for first, c in ((cats[2], cats[0]), (cats[2], cats[1]),
                                                                             (cats[2], cats[2]))]
            _same([autos[0][pick] + autos[1][pick]], [autos[2][pick]], weighted, "binned-label auto")
            assert autos[2][0].sum() > 0
        for c in cats:
            c.free()
    c1.free()


@pytest.mark.parametrize("column", ["int32", "uint8", "redshifts"])
def test_partial_upload_matches_full(engine, column):
    rng = np.random.default_rng(7)
    n_patch, n_bins = 12, 4
    xyz, off, zbin, w = _rows(rng, n_patch, 2500, n_bins, True)
    keep = np.zeros(n_patch, dtype=np.uint8)
    keep[[0, 1, 2, 5, 9, 10]] = 1  # three runs of consecutive patches
    zedges = np.linspace(0.0, 1.0, n_bins + 1)
    if column == "int32":
        kw = dict(zbin=zbin, n_bins=n_bins)
    elif column == "uint8":
        kw = dict(zbin=np.where(zbin >= 0, zbin, 255).astype(np.uint8), n_bins=n_bins)
    else:
        kw = dict(redshifts=rng.uniform(-0.1, 1.1, len(xyz)), edges=zedges)
    full = engine.upload_catalog(xyz, off, weights=w, **kw)
    part = engine.upload_catalog(xyz, off, weights=w, keep=keep, **kw)
    kept = np.flatnonzero(keep)
    sw_full, sw_part = full.sum_weights(), part.sum_weights()
    assert_allclose(sw_part[:, kept], sw_full[:, kept], rtol=RTOL)
    assert (sw_part[:, keep == 0] == 0).all()
    _, _, num = part.patch_metadata()
    assert_array_equal(num, np.where(keep != 0, np.diff(off), 0))
    pi, pj = (a.ravel().astype(np.int32) for a in np.meshgrid(kept, kept, indexing="ij"))
    edges = _edges(n_bins, 4)
    for first, second in ((part, part), (full, part), (part, full)):
        gi, gf, _ = engine.count(first, second, pi, pj, edges)
        wi, wf, _ = engine.count(full, full, pi, pj, edges)
        assert_array_equal(gi, wi)
        assert_allclose(gf, wf, rtol=RTOL)
    assert wi.sum() > 0
    full.free()
    part.free()


def test_two_contexts_on_one_device_from_two_threads():
    from yet_another_wizz_b200 import Engine

    rng = np.random.default_rng(5)
    n_patch, n_bins = 8, 3
    xyz, off, zbin, w = _rows(rng, n_patch, 20000, n_bins, True)
    pi, pj = _pairs(n_patch)
    edges = _edges(n_bins, 9)
    engines = [Engine(0, cache_catalogs=False) for _ in range(2)]
    try:
        ref = engines[0].upload_catalog(xyz, off, weights=w, zbin=zbin, n_bins=n_bins)
        want = engines[0].count(ref, ref, pi, pj, edges)
        ref.free()
        results = [None, None]
        barrier = threading.Barrier(2)

        def run(k):
            e = engines[k]
            barrier.wait()
            out = []
            for _ in range(3):
                c = e.upload_catalog(xyz, off, weights=w, zbin=zbin, n_bins=n_bins)
                out.append(e.count(c, c, pi, pj, edges))
                c.free()
            results[k] = out

        threads = [threading.Thread(target=run, args=(k,)) for k in range(2)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        for out in results:
            assert out is not None
            for gi, gf, _ in out:
                assert_array_equal(gi, want[0])
                assert_allclose(gf, want[1], rtol=RTOL)
    finally:
        for e in engines:
            e.close()


# ---- EngineGroup against Engine -------------------------------------------------------------------------------
def _arrays(result):
    """(array, float sum) of every count and sum of a measurement result (nested lists of CorrFunc / ScalarCorrFunc);
    scalar-weighted counts are float sums whatever the weights"""
    if isinstance(result, (list, tuple)):
        for r in result:
            yield from _arrays(r)
        return
    for kind in ("dd", "dr", "rd", "rr"):
        nc = getattr(result, kind, None)
        if nc is None:
            continue
        if hasattr(nc, "kappa_counts"):
            yield nc.kappa_counts.counts, True
            yield nc.number_counts.counts, False
        else:
            yield nc.counts.counts, False
            yield nc.sum_weights.sum_weights1, False
            yield nc.sum_weights.sum_weights2, False


def _compare(got, want, exact):
    g, w = list(_arrays(got)), list(_arrays(want))
    assert len(g) == len(w) > 0
    for (a, fa), (b, _) in zip(g, w):
        if exact and not fa:
            assert_array_equal(a, b)
        else:  # signed scalar sums cancel: tolerance relative to the largest entry
            assert_allclose(a, b, rtol=RTOL, atol=RTOL * np.abs(b).max())


def _dense():
    """a denser input of the size of the C1 benchmark (1e5 x 1e5 rows, 1e6 randoms per side, 16 patches), weighted
    data samples, with scalar values on the reference sample"""
    import yet_another_wizz_b200 as yb

    ras, decs = np.arange(4) * 10.0 + 5.0, np.arange(4) * 6.25 - 9.375
    centers = yb.AngularCoordinates(np.deg2rad([[r, d] for d in decs for r in ras]))
    pool = np.random.default_rng(7).uniform(0.1, 1.0, 1_000_000)
    wpool = np.random.default_rng(8).uniform(0.5, 1.5, 1_000_000)
    cats = {}
    for key, n, seed in (("ref", 100_000, 1), ("unk", 100_000, 2), ("ref_rand", 1_000_000, 3), ("unk_rand", 1_000_000, 4)):
        gen = yb.BoxRandoms(0.0, 40.0, -12.5, 12.5, redshifts=pool if key != "unk" else None,
                            weights=wpool if key in ("ref", "unk") else None, seed=seed)
        cats[key] = yb.Catalog.from_random(key, gen, n, patch_centers=centers)
    config = yb.Configuration.create(rmin=100, rmax=1000, zmin=0.1, zmax=1.0, num_bins=10)
    return config, cats


def _run_all(config, cats, engine, *, scalar_ref=None):
    """the six public functions on one input; the tomographic ones on the unknown / data sample split by patch
    parity and by a seeded label"""
    import yet_another_wizz_b200 as yb

    ref, unk, rr, ur = cats["ref"], cats["unk"], cats["ref_rand"], cats["unk_rand"]
    out = dict(
        cross=yb.crosscorrelate(config, ref, unk, ref_rand=rr, unk_rand=ur, engine=engine),
        auto=yb.autocorrelate(config, ref, rr, engine=engine),
        cross_tomo=yb.crosscorrelate_tomographic(config, ref, cats["unk_bins"], ref_rand=rr, unk_rand=ur, engine=engine),
        auto_tomo=yb.autocorrelate_tomographic(config, cats["ref_bins"], rr, engine=engine),
    )
    if scalar_ref is not None:
        out["cross_scalar"] = yb.crosscorrelate_scalar(config, scalar_ref, unk, unk_rand=ur, engine=engine)
        out["auto_scalar"] = yb.autocorrelate_scalar(config, scalar_ref, engine=engine)
    return out


def _golden_inputs(name):
    from test_tomographic import catalog_rows

    g = golden_io.load(name)
    config = golden_cases.config_from_golden(g)
    cats = {k: golden_cases.catalog_from_golden(g, k) for k in ("ref", "unk", "ref_rand", "unk_rand")}
    for key, src, seed in (("unk_bins", "unk", 11), ("ref_bins", "ref", 12)):
        c = golden_io.catalog_arrays(g, src)
        lab = np.random.default_rng(seed).integers(0, 3, len(c["ra"]))
        cats[key] = [catalog_rows(c, lab == i) for i in range(3)]
    return config, cats


def _with_kappa(catalog, seed):
    """the catalog's rows with a seeded scalar value per row"""
    import yet_another_wizz_b200 as yb

    rows = [catalog[p].load_data() for p in catalog.keys()]
    ra = np.concatenate([r["ra"] for r in rows])
    dec = np.concatenate([r["dec"] for r in rows])
    patch = np.concatenate([np.full(len(r), p) for p, r in zip(catalog.keys(), rows)])
    names = rows[0].dtype.names
    w = np.concatenate([r["weights"] for r in rows]) if "weights" in names else None
    z = np.concatenate([r["redshifts"] for r in rows]) if "redshifts" in names else None
    kappa = np.random.default_rng(seed).normal(0.0, 1.0, len(ra))
    return yb.Catalog.from_arrays(ra, dec, patch_ids=patch, patch_centers=catalog.get_centers(), weights=w,
                                  redshifts=z, kappa=kappa, degrees=False)


@pytest.fixture(scope="module")
def single():
    from yet_another_wizz_b200 import Engine

    eng = Engine(0)
    yield eng
    eng.close()


def _check_groups(config, cats, single, groups, exact, scalar_ref):
    from yet_another_wizz_b200 import EngineGroup

    want = _run_all(config, cats, single, scalar_ref=scalar_ref)
    for devices in groups:
        grp = EngineGroup(devices)
        try:
            got = _run_all(config, cats, grp, scalar_ref=scalar_ref)
            again = _run_all(config, cats, grp, scalar_ref=scalar_ref)  # resident shares of the engines' caches
        finally:
            grp.close()
        for key in want:
            _compare(got[key], want[key], exact)
            _compare(again[key], want[key], exact)


@pytest.mark.parametrize("name", ["cross_unweighted", "cross_weighted_multiscale"])
def test_engine_group_golden_inputs(single, name):
    config, cats = _golden_inputs(name)
    _check_groups(config, cats, single, ([0, 0], [0, 0, 0]), name == "cross_unweighted",
                  _with_kappa(cats["ref"], 3))


def test_engine_group_dense_input(single):
    config, cats = _dense()
    # tomographic bins: the unknown sample and the reference sample split by a seeded label
    for key, src, seed in (("unk_bins", "unk", 11), ("ref_bins", "ref", 12)):
        cats[key] = [_subset(cats[src], seed, i) for i in range(3)]
    _check_groups(config, cats, single, ([0, 0], [0, 0, 0]), False, _with_kappa(cats["ref"], 5))


def _subset(catalog, seed, i, n_tomo=3):
    import yet_another_wizz_b200 as yb

    rows = [catalog[p].load_data() for p in catalog.keys()]
    ra = np.concatenate([r["ra"] for r in rows])
    dec = np.concatenate([r["dec"] for r in rows])
    patch = np.concatenate([np.full(len(r), p) for p, r in zip(catalog.keys(), rows)])
    names = rows[0].dtype.names
    w = np.concatenate([r["weights"] for r in rows]) if "weights" in names else None
    z = np.concatenate([r["redshifts"] for r in rows]) if "redshifts" in names else None
    m = np.random.default_rng(seed).integers(0, n_tomo, len(ra)) == i
    return yb.Catalog.from_arrays(ra[m], dec[m], patch_ids=patch[m], patch_centers=catalog.get_centers(),
                                  weights=None if w is None else w[m], redshifts=None if z is None else z[m],
                                  degrees=False)


def test_engine_group_distinct_devices(single):
    import torch

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip(f"needs at least 2 visible GPUs ({n} visible): EngineGroup over distinct devices not run")
    config, cats = _golden_inputs("cross_weighted_multiscale")
    _check_groups(config, cats, single, (list(range(min(n, 4))),), False, _with_kappa(cats["ref"], 3))
