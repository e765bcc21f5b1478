"""
GPU tests of measurement calls counted in passes: the footprint bounds (`yawb_catalog_footprint`,
`yawb_count_footprint`) against the allocator's high-water mark (`yawb_memory_stats`), and every public measurement
function with a memory limit that forces several passes against the same call in one pass, on one engine and on
`EngineGroup([0, 0])`.

Bar: integer counts bit-exact, weighted sums within 1e-12 relative; the high-water mark of a multi-pass call within
its limit.
"""

import numpy as np
import pytest

from test_gpu_engine_group import _compare, _dense, _edges, _golden_inputs, _pairs, _rows, _run_all, _subset, _with_kappa

pytestmark = pytest.mark.gpu

FUNCS = ("cross", "auto", "cross_tomo", "auto_tomo", "cross_scalar", "auto_scalar")


def _fresh(**kw):
    from yet_another_wizz_b200 import Engine

    return Engine(0, cache_catalogs=False, **kw)


# (weighted, how the z-bins travel, labels, mask)
UPLOADS = [(False, None, 0, False), (True, "i32", 0, False), (False, "u8", 0, True), (True, "z", 0, False),
           (False, "u8", 3, True), (True, "i32", 2, False)]


@pytest.mark.parametrize("weighted,zbin,labels,mask", UPLOADS)
def test_catalog_footprint_bounds_the_peak(weighted, zbin, labels, mask):
    rng = np.random.default_rng(5)
    n_patch, n_bins = 12, 6
    xyz, off, z, w = _rows(rng, n_patch, 20_000, n_bins, weighted)
    eng = _fresh()
    try:
        kw = dict(weights=w)
        if zbin == "z":
            edges = np.linspace(0.0, 1.0, n_bins + 1)
            kw.update(redshifts=rng.uniform(-0.1, 1.1, len(xyz)), edges=edges)
        elif zbin is not None:
            kw.update(zbin=(np.where(z < 0, 255, z).astype(np.uint8) if zbin == "u8" else z), n_bins=n_bins)
            if labels:
                kw["n_labels"] = labels
        m = (rng.random(len(xyz)) < 0.5).astype(np.uint8) if mask else None
        cat = eng.upload_catalog(xyz, off, second_rows=m, **kw)
        cat.build_index(1)
        cat.build_index(2)
        eng.sync()
        peak = eng.memory_stats()["peak"]
        bound = eng.footprint(len(xyz), n_patch, n_bins if zbin else 1, weighted=weighted, zbin=zbin,
                              labelled=bool(labels), mask=mask)
        assert 0 < peak <= bound, (peak, bound)
        cat.free()
    finally:
        eng.close()


@pytest.mark.parametrize("kind", ["count", "count2", "count4", "labelled"])
@pytest.mark.parametrize("n_edges,weighted", [(2, False), (6, True)])
def test_count_footprint_bounds_the_peak(kind, n_edges, weighted):
    rng = np.random.default_rng(n_edges)
    n_patch, n_bins = 8, 3
    eng = _fresh()
    try:
        rows = [_rows(rng, n_patch, 15_000, n_bins, weighted) for _ in range(4)]
        labelled = kind == "labelled"
        cats = [eng.upload_catalog(x, o, weights=ww, zbin=z if k < 2 or labelled else None, n_bins=n_bins)
                for k, (x, o, z, ww) in enumerate(rows)]
        n = [len(r[0]) for r in rows]
        zb = ["i32" if k < 2 or labelled else None for k in range(4)]
        nb = [n_bins if k < 2 or labelled else 1 for k in range(4)]

        def index(k, role):  # the index of catalog k a count builds, without the upload
            return eng.footprint(n[k], n_patch, nb[k], weighted=weighted, zbin=zb[k], first=role == 1,
                                 second=role == 2, upload=False)

        edges = _edges(n_bins, n_edges)
        pi, pj = _pairs(n_patch)
        n_items = len(pi) * (max(n) // n_patch // 256 + 1 + n_bins)
        eng.sync()
        eng.memory_reset_peak()
        base = eng.memory_stats()["held"]  # the four uploads
        fused = eng.footprint(n[0] + n[1], n_patch, n_bins, weighted=weighted, second=False, upload=False)
        if kind == "count":
            eng.count(cats[0], cats[2], pi, pj, edges)
            extra = index(0, 1) + index(2, 2) + eng.count_footprint(n_items, len(pi), n_bins, n_edges, weighted=weighted)
        elif kind == "count2":
            eng.count2(cats[0], cats[1], cats[2], pi, pj, edges)
            extra = fused + index(2, 2) + eng.count_footprint(n_items, len(pi), n_bins, n_edges, n_blocks=2,
                                                               weighted=weighted)
        elif kind == "count4":
            eng.count4(cats[0], cats[1], cats[2], cats[3], pi, pj, edges)
            union = not weighted and n_edges == 2  # the single-bin path tiles the union of both second catalogs
            second = (eng.footprint(n[2] + n[3], n_patch, 1, weighted=weighted, first=False, upload=False) if union
                      else index(2, 2) + index(3, 2))
            extra = fused + second + eng.count_footprint(2 * n_items, len(pi), n_bins, n_edges, n_blocks=4,
                                                         weighted=weighted)
        else:
            eng.count(cats[0], cats[2], pi, pj, edges[:, :n_edges], labels=True)
            extra = index(0, 1) + index(2, 2) + eng.count_footprint(n_items, len(pi), n_bins, n_edges,
                                                                     n_blocks=n_bins, weighted=weighted)
        eng.sync()
        peak = eng.memory_stats()["peak"]
        assert base < peak <= base + extra, (peak, base, extra)
    finally:
        eng.close()


def _limits(config, cats, scalar_ref, frac):
    """per function: a memory limit of `frac` of the call's predicted footprint in one pass (at least what one patch
    with its linked patches needs), found by planning the call without running it"""
    from yet_another_wizz_b200 import measurements

    class Planned(Exception):
        pass

    out = {}
    for key in FUNCS:
        seen = []

        def probe(counts, radii, centers, footprint, limits):
            n_patch = len(centers)
            whole = footprint(np.ones(n_patch, dtype=bool))
            floor = 0
            for p in range(n_patch):
                keep = np.zeros(n_patch, dtype=bool)
                keep[p] = True
                for pi, pj, _, _ in counts:
                    keep[np.asarray(pi)[np.asarray(pj) == p]] = True
                    keep[np.asarray(pj)[np.asarray(pi) == p]] = True
                floor = max(floor, footprint(keep))
            limit = max(int(whole * frac), int(floor * 1.01))
            seen.append(limit if limit < whole else None)  # every patch linked to every other: one pass only
            raise Planned

        saved = measurements.plan_passes
        measurements.plan_passes = probe
        try:
            eng = _fresh()
            with pytest.raises(Planned):
                _one(key, config, cats, eng, scalar_ref)
            eng.close()
        finally:
            measurements.plan_passes = saved
        out[key] = seen[0]
    return out


def _one(key, config, cats, engine, scalar_ref):
    import yet_another_wizz_b200 as yb

    ref, unk, rr, ur = cats["ref"], cats["unk"], cats["ref_rand"], cats["unk_rand"]
    if key == "cross":
        return yb.crosscorrelate(config, ref, unk, ref_rand=rr, unk_rand=ur, engine=engine)
    if key == "auto":
        return yb.autocorrelate(config, ref, rr, engine=engine)
    if key == "cross_tomo":
        return yb.crosscorrelate_tomographic(config, ref, cats["unk_bins"], ref_rand=rr, unk_rand=ur, engine=engine)
    if key == "auto_tomo":
        return yb.autocorrelate_tomographic(config, cats["ref_bins"], rr, engine=engine)
    if key == "cross_scalar":
        return yb.crosscorrelate_scalar(config, scalar_ref, unk, unk_rand=ur, engine=engine)
    return yb.autocorrelate_scalar(config, scalar_ref, engine=engine)


def _check_passes(config, cats, exact, scalar_ref, frac=0.55):
    from yet_another_wizz_b200 import EngineGroup, measurements

    single = _fresh()
    try:
        want = _run_all(config, cats, single, scalar_ref=scalar_ref)
    finally:
        single.close()
    limits = _limits(config, cats, scalar_ref, frac)
    for key in FUNCS:
        if limits[key] is None:
            continue
        eng = _fresh(memory_limit=limits[key])
        try:
            eng.memory_reset_peak()
            got = _one(key, config, cats, eng, scalar_ref)
            passes = {st.get("passes", 1) for st in measurements.last_stats().values()}
            assert min(passes) >= 2, (key, passes)
            assert eng.memory_stats()["peak"] <= limits[key], key
            _compare(got, want[key], exact)
        finally:
            eng.close()
        grp = EngineGroup([_fresh(memory_limit=limits[key]), _fresh(memory_limit=limits[key])])
        try:
            got = _one(key, config, cats, grp, scalar_ref)
            _compare(got, want[key], exact)
        finally:
            for e in grp.engines:
                e.close()
            grp.close()
    return [key for key in FUNCS if limits[key] is not None]


@pytest.mark.parametrize("name", ["cross_unweighted", "cross_weighted_multiscale"])
def test_passes_golden_inputs(name):
    config, cats = _golden_inputs(name)
    _check_passes(config, cats, name == "cross_unweighted", _with_kappa(cats["ref"], 3))


def test_passes_dense_input():
    config, cats = _dense()
    for key, src, seed in (("unk_bins", "unk", 11), ("ref_bins", "ref", 12)):
        cats[key] = [_subset(cats[src], seed, i) for i in range(3)]
    assert len(_check_passes(config, cats, False, _with_kappa(cats["ref"], 5))) == len(FUNCS)


def test_engine_counts_again_after_a_pass_cannot_fit():
    import yet_another_wizz_b200 as yb

    config, cats = _golden_inputs("cross_unweighted")
    ref, unk, ur = cats["ref"], cats["unk"], cats["unk_rand"]
    eng = _fresh(memory_limit=1 << 20)
    try:
        with pytest.raises(ValueError, match="bytes of device memory, more than the limit"):
            yb.crosscorrelate(config, ref, unk, unk_rand=ur, engine=eng)
        eng.memory_limit = None
        got = yb.crosscorrelate(config, ref, unk, unk_rand=ur, engine=eng)
    finally:
        eng.close()
    ref_eng = _fresh()
    try:
        want = yb.crosscorrelate(config, ref, unk, unk_rand=ur, engine=ref_eng)
    finally:
        ref_eng.close()
    _compare(got, want, True)
