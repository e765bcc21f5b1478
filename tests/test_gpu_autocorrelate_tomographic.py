"""Binned labels (`Engine.upload_catalog(n_labels=)`, `yawb_catalog_set_labels`) and `autocorrelate_tomographic` on
the device.

ABI level: a catalog with binned labels (id = label * B + z-bin) counted once must give, for every label, exactly what
a z-binned upload of that label's rows gives -- under rule a (both catalogs labelled, the auto case `cat1 is cat2`
included) and rule b (an unlabelled binned first catalog), in every kernel path.  Public level: one
`autocorrelate_tomographic` call against the loop of `autocorrelate` calls it replaces."""

import os
import sys
from ctypes import byref, c_void_p

import numpy as np
import pytest
from numpy.testing import assert_allclose, assert_array_equal

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))

pytestmark = pytest.mark.gpu

RTOL = 1e-12


@pytest.fixture(scope="module")
def engine():
    import yet_another_wizz_b200 as yb

    eng = yb.Engine(0)
    yield eng
    eng.close()


def _rows(rng, n, side, box=0.12):
    """rows in a small box of the sky, grouped by a (side x side) patch grid: (xyz, patch_off, patch of each row)"""
    import oracle

    ra = rng.uniform(0.0, box, n)
    dec = np.arcsin(rng.uniform(-box / 2, box / 2, n))
    px = np.minimum((ra / box * side).astype(int), side - 1)
    py = np.minimum(((np.sin(dec) / box + 0.5) * side).astype(int), side - 1)
    patch = py * side + px
    order = np.argsort(patch, kind="stable")
    off = np.concatenate([[0], np.cumsum(np.bincount(patch, minlength=side**2))])
    return oracle.radec_to_xyz(ra, dec)[order], off, patch[order]


class Setup:
    """a sample D with binned labels (L labels x B z-bins; 5 % dropped rows, and the last label absent from the first
    row of patches), randoms RL with the same binned labels, unlabelled binned randoms R, and z-binned uploads of
    every label's rows (D_l, RL_l)"""

    def __init__(self, engine, *, n_d=30_000, n_r=50_000, side=4, n_bins=6, n_lab=4, weighted=False, seed=0):
        rng = np.random.default_rng(seed)
        self.engine, self.n_lab, self.n_bins, self.side = engine, n_lab, n_bins, side
        w = (lambda n: rng.uniform(0.5, 1.5, n)) if weighted else (lambda n: None)
        self.owned = []

        def labelled(n):
            x, off, patch = _rows(rng, n, side)
            lab, z = rng.integers(0, n_lab, n), rng.integers(0, n_bins, n)
            ids = (lab * n_bins + z).astype(np.uint8)
            ids[rng.random(n) < 0.05] = 255  # dropped rows
            if n_lab > 1:
                ids[(lab == n_lab - 1) & (patch < side)] = 255  # a label with empty patches
            wt = w(n)
            dev = self.up(x, off, weights=wt, zbin=ids, n_bins=n_lab * n_bins, n_labels=n_lab)
            per = []
            for ell in range(n_lab):
                m = (ids >= ell * n_bins) & (ids < (ell + 1) * n_bins)
                o = np.concatenate([[0], np.cumsum(np.bincount(patch[m], minlength=side * side))])
                per.append(self.up(x[m], o, weights=None if wt is None else wt[m],
                                   zbin=(ids[m] - ell * n_bins).astype(np.uint8), n_bins=n_bins))
            return dev, per

        self.D, self.D_l = labelled(n_d)
        self.RL, self.RL_l = labelled(n_r)
        x, off, _ = _rows(rng, n_r, side)
        self.R = self.up(x, off, weights=w(n_r), zbin=rng.integers(0, n_bins, n_r).astype(np.int32), n_bins=n_bins)
        pi, pj = np.meshgrid(np.arange(side * side), np.arange(side * side), indexing="ij")
        self.pi, self.pj = pi.ravel(), pj.ravel()

    def up(self, *args, **kw):
        dev = self.engine.upload_catalog(*args, **kw)
        self.owned.append(dev)
        return dev

    def r2(self, n_edges):
        import oracle

        a0 = np.linspace(2e-4, 6e-4, self.n_bins)
        return np.stack([oracle.chord_sq_edges(np.geomspace(a, 8 * a, n_edges)) for a in a0])

    def free(self):
        for c in self.owned:
            c.free()


def _same(got, want, weighted):
    if weighted:
        assert_allclose(got, want, rtol=RTOL, atol=0)
    else:
        assert_array_equal(got, want)


def _check_rules(engine, s, r2, weighted):
    """rules a (auto and cross) and b against the per-label z-binned uploads"""
    k = 1 if weighted else 0  # weighted sums, integer counts otherwise
    shape = (s.n_lab, len(s.pi), s.n_bins, r2.shape[1] - 1)
    for (c1, c2, pi, pj), per in (
        ((s.D, s.D, s.pi, s.pj), [(u, u) for u in s.D_l]),                    # a: DD, cat1 is cat2
        ((s.D, s.RL, s.pi, s.pj), list(zip(s.D_l, s.RL_l))),                  # a: DR with per-label randoms
        ((s.R, s.D, s.pj, s.pi), [(s.R, u) for u in s.D_l]),                  # b: DR, randoms first, pairs swapped
    ):
        out = engine.count(c1, c2, pi, pj, r2)
        assert out[0].shape == out[1].shape == shape
        naive = 0
        for ell, (u1, u2) in enumerate(per):
            want = engine.count(u1, u2, pi, pj, r2)
            _same(out[k][ell], want[k], weighted)
            assert_array_equal(out[0][ell], want[0])
            naive += want[2]["pair_tests_naive"]
        assert out[2]["pair_tests_naive"] == naive
        assert out[0].sum() > 0
    # rule b is the swapped unlabelled count: (R, D_l) over (pj, pi) == (D_l, R) over (pi, pj)
    for ell, u in enumerate(s.D_l):
        want = engine.count(u, s.R, s.pi, s.pj, r2)
        assert_array_equal(engine.count(s.R, s.D, s.pj, s.pi, r2)[0][ell], want[0])


VARIANTS = {  # name: (weighted, n_edges)
    "single": (False, 2),
    "cumulative": (False, 4),
    "subbins": (False, 24),
    "weighted_single": (True, 2),
    "weighted_multi": (True, 5),
}


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_binned_labels_equal_per_label_uploads(engine, variant):
    weighted, n_edges = VARIANTS[variant]
    s = Setup(engine, weighted=weighted)
    try:
        _check_rules(engine, s, s.r2(n_edges), weighted)
        # the last label holds no row in the first row of patches: its counts there are zero
        dd = engine.count(s.D, s.D, s.pi, s.pj, s.r2(n_edges))[0][s.n_lab - 1]
        assert dd[s.pi < s.side].sum() == 0 and dd.sum() > 0
    finally:
        s.free()


def test_single_label(engine):
    s = Setup(engine, n_lab=1, seed=2)
    try:
        _check_rules(engine, s, s.r2(3), False)
        # L = 1 equals the same ids without labels
        assert_array_equal(engine.count(s.D, s.D, s.pi, s.pj, s.r2(3))[0][0],
                           engine.count(s.D_l[0], s.D_l[0], s.pi, s.pj, s.r2(3))[0])
    finally:
        s.free()


def test_large_64_patches_5_labels_30_bins(engine):
    """1e6 rows, 64 patches, 5 labels x 30 z-bins: the warps' tables stay sized by the 30 z-bins"""
    s = Setup(engine, n_d=1_000_000, n_r=1_000_000, side=8, n_bins=30, n_lab=5, seed=9)
    try:
        import oracle

        r2 = np.tile(oracle.chord_sq_edges(np.array([3e-4, 3e-3])), (s.n_bins, 1))
        for c1, c2, pi, pj, per in ((s.D, s.D, s.pi, s.pj, [(u, u) for u in s.D_l]),
                                    (s.R, s.D, s.pj, s.pi, [(s.R, u) for u in s.D_l])):
            out = engine.count(c1, c2, pi, pj, r2)
            for ell, (u1, u2) in enumerate(per):
                assert_array_equal(out[0][ell], engine.count(u1, u2, pi, pj, r2)[0])
            assert out[0].sum() > 1e6
    finally:
        s.free()


def test_rejected_combinations_leave_the_engine_usable(engine):
    import yet_another_wizz_b200 as yb
    from yet_another_wizz_b200 import _lib

    s = Setup(engine, n_d=5000, n_r=8000, seed=4)
    try:
        r2 = s.r2(2)
        ok = engine.count(s.D, s.D, s.pi, s.pj, r2)[0]
        assert ok.sum() > 0

        def still_ok():
            assert_array_equal(engine.count(s.D, s.D, s.pi, s.pj, r2)[0], ok)

        rng = np.random.default_rng(1)
        x, off, _ = _rows(rng, 4000, s.side)
        two = s.up(x, off, zbin=rng.integers(0, s.n_lab * s.n_bins, 4000).astype(np.uint8),
                   n_bins=s.n_lab * s.n_bins, n_labels=2)
        other_b = s.up(x, off, zbin=rng.integers(0, s.n_bins + 1, 4000).astype(np.uint8), n_bins=s.n_bins + 1)
        r2_lab = np.tile(r2[:1], (s.n_lab * s.n_bins // 2, 1))
        cases = [
            ("swap the roles", lambda: engine.count(s.D, s.R, s.pi, s.pj, r2)),
            ("swap the roles", lambda: engine.count(s.D, s.D_l[0], s.pi, s.pj, r2)),
            ("differ", lambda: engine.count(s.D, two, s.pi, s.pj, r2_lab)),
            ("differ", lambda: engine.count(other_b, s.D, s.pi, s.pj, r2)),
            ("EXACT_BRUTEFORCE", lambda: engine.count(s.D, s.D, s.pi, s.pj, r2, exact=True)),
            ("SECOND_LABELS", lambda: engine.count(s.R, s.D, s.pi, s.pj, r2, labels=True)),
            ("yawb_count2", lambda: engine.count2(s.R, s.RL_l[0], s.D, s.pi, s.pj, r2)),
            ("yawb_count4", lambda: engine.count4(s.R, s.RL_l[0], s.D, s.RL, s.pi, s.pj, r2)),
        ]
        for msg, call in cases:
            with pytest.raises(yb.YawbError, match=msg):
                call()
            still_ok()
        # the setter: unbinned, device-digitised, n_labels < 1 or not dividing n_bins
        plain = s.up(x, off)
        zcat = s.up(x, off, redshifts=rng.uniform(0, 1, 4000), edges=np.linspace(0, 1, 5))
        for cat, n in ((plain, 1), (zcat, 2), (s.R, 0), (s.R, 4)):
            assert engine.lib.yawb_catalog_set_labels(cat._h, n) != 0
            still_ok()
        with pytest.raises(yb.YawbError, match="divide"):
            engine.upload_catalog(x, off, zbin=np.zeros(4000, dtype=np.uint8), n_bins=6, n_labels=4)
        still_ok()
        assert engine.lib.yawb_version() >= _lib.BINNED_LABELS_MIN_VERSION
        # the C ABI directly: a labelled first catalog against an unlabelled second one
        pi = np.ascontiguousarray(s.pi, dtype=np.int32)
        pj = np.ascontiguousarray(s.pj, dtype=np.int32)
        out = np.zeros((len(pi), s.n_bins, 1), dtype=np.int64)
        stats = _lib.YawbStats()
        rc = engine.lib.yawb_count(engine._h, s.D._h, s.R._h, pi.ctypes.data_as(c_void_p), pj.ctypes.data_as(c_void_p),
                                   len(pi), r2.ctypes.data_as(c_void_p), 2, 0, None, out.ctypes.data_as(c_void_p),
                                   byref(stats))
        assert rc != 0 and b"swap" in engine.lib.yawb_last_error()
        still_ok()
    finally:
        s.free()


def _c1_auto(n_tomo=5, weighted=False):
    """C1-sized BoxRandoms catalogs (16 patches, 10 z-bins): a sample with redshifts split into `n_tomo` bins by a
    seeded label, one shared random catalog and one random catalog per bin"""
    import yet_another_wizz_b200 as yb

    box = (0.0, 10.0, -2.5, 2.5)
    ras = (np.arange(4) + 0.5) * 10.0 / 4
    decs = -2.5 + (np.arange(4) + 0.5) * 5.0 / 4
    centers = yb.AngularCoordinates(np.deg2rad([[r, d] for d in decs for r in ras]))
    pool = np.random.default_rng(7).uniform(0.05, 1.05, 100_000)  # some rows outside the binning
    wpool = np.random.default_rng(8).uniform(0.5, 1.5, 100_000) if weighted else None
    mk = lambda name, n, seed, w=None: yb.Catalog.from_random(  # noqa: E731
        name, yb.BoxRandoms(*box, redshifts=pool, weights=w, seed=seed), n, patch_centers=centers)
    sample = mk("sample", 100_000, 2, w=wpool)
    shared = mk("rand", 1_000_000, 4)
    rows = {p: sample[p].load_data() for p in sample}
    lab = {p: np.random.default_rng(100 + p).integers(0, n_tomo, len(rows[p])) for p in sample}
    data = []
    for i in range(n_tomo):
        parts = {p: rows[p][lab[p] == i] for p in sample}
        cat = lambda k: np.concatenate([parts[p][k] for p in sample])  # noqa: E731
        ids = np.concatenate([np.full(len(parts[p]), p) for p in sample])
        data.append(yb.Catalog.from_arrays(cat("ra"), cat("dec"), patch_ids=ids, patch_centers=centers,
                                           weights=cat("weights") if weighted else None, redshifts=cat("redshifts"),
                                           degrees=False))
    per_bin = [mk(f"rand_{i}", 200_000, 40 + i) for i in range(n_tomo)]
    config = yb.Configuration.create(rmin=100, rmax=1000, zmin=0.1, zmax=1.0, num_bins=10)
    return config, data, shared, per_bin


@pytest.mark.parametrize("weighted", [False, True])
def test_autocorrelate_tomographic_vs_loop(engine, weighted):
    import yet_another_wizz_b200 as yb

    config, data, shared, per_bin = _c1_auto(weighted=weighted)
    for arg, rands in ((shared, [shared] * len(data)), (per_bin, per_bin)):
        got = yb.autocorrelate_tomographic(config, data, arg, engine=engine)
        for i, (d, rand) in enumerate(zip(data, rands)):
            want = yb.autocorrelate(config, d, rand, engine=engine)
            for a, b in zip(got[i], want):
                if not weighted:
                    assert a == b
                for kind in ("dd", "dr", "rr"):
                    x, y = getattr(a, kind), getattr(b, kind)
                    assert_allclose(x.counts.counts, y.counts.counts, rtol=RTOL, atol=0)
                    assert_allclose(x.sum_weights.sum_weights1, y.sum_weights.sum_weights1, rtol=RTOL, atol=0)
                    assert_allclose(x.sum_weights.sum_weights2, y.sum_weights.sum_weights2, rtol=RTOL, atol=0)
        assert got[0][0].dd.counts.counts.sum() > 0 and got[-1][0].rr.counts.counts.sum() > 0
        # a warm second call finds every catalog in the engine's cache
        again = yb.autocorrelate_tomographic(config, data, arg, engine=engine)
        if not weighted:
            assert all(a == b for x, y in zip(got, again) for a, b in zip(x, y))
