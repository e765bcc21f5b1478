"""Labelled second catalogs (`YAWB_FLAG_SECOND_LABELS`) and `crosscorrelate_tomographic` on the device.

ABI level: a labelled upload counted once must give, for every label, exactly what an unbinned upload of that
label's rows gives -- through `count`, `count2` and `count4`, in every kernel variant.  Public level: one
`crosscorrelate_tomographic` call against the loop of `crosscorrelate` calls it replaces."""

import ctypes
import os
import sys

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


def _rows(rng, n, n_patch_side, box=0.12):
    """rows in a small box of the sky, grouped by a (side x side) patch grid: (xyz, patch_off, patch of each row)"""
    import oracle

    ra = rng.uniform(0.0, box, n)
    dec = np.arcsin(rng.uniform(-box / 2, box / 2, n))
    px = np.minimum((ra / box * n_patch_side).astype(int), n_patch_side - 1)
    py = np.minimum(((np.sin(dec) / box + 0.5) * n_patch_side).astype(int), n_patch_side - 1)
    patch = py * n_patch_side + px
    order = np.argsort(patch, kind="stable")
    off = np.concatenate([[0], np.cumsum(np.bincount(patch, minlength=n_patch_side**2))])
    return oracle.radec_to_xyz(ra, dec)[order], off, patch[order]


class Setup:
    """a z-binned first catalog (and its randoms), a labelled second catalog with some dropped rows (255), an
    unbinned second catalog, and per-label unbinned uploads of the labelled one"""

    def __init__(self, engine, *, n1=30_000, n2=50_000, side=4, n_bins=6, n_lab=4, weighted=False, seed=0):
        rng = np.random.default_rng(seed)
        self.engine, self.n_lab = engine, n_lab
        x1, o1, _ = _rows(rng, n1, side)
        x1b, o1b, _ = _rows(rng, n1 // 2, side)
        x2, o2, p2 = _rows(rng, n2, side)
        x3, o3, _ = _rows(rng, n2 // 2, side)
        w = (lambda n: rng.uniform(0.5, 1.5, n)) if weighted else (lambda n: None)
        lab = rng.integers(0, n_lab, n2).astype(np.uint8)
        lab[rng.random(n2) < 0.05] = 255  # dropped rows
        w2 = w(n2)
        self.c1a = engine.upload_catalog(x1, o1, weights=w(n1), zbin=rng.integers(0, n_bins, n1).astype(np.uint8),
                                         n_bins=n_bins)
        self.c1b = engine.upload_catalog(x1b, o1b, zbin=rng.integers(0, n_bins, n1 // 2).astype(np.int32), n_bins=n_bins)
        self.lab = engine.upload_catalog(x2, o2, weights=w2, zbin=lab, n_bins=n_lab)
        self.rand = engine.upload_catalog(x3, o3, weights=w(n2 // 2))
        self.per_label = []
        for ell in range(n_lab):
            m = lab == ell
            off = np.concatenate([[0], np.cumsum(np.bincount(p2[m], minlength=side * side))])
            self.per_label.append(engine.upload_catalog(x2[m], off, weights=None if w2 is None else w2[m]))
        pi, pj = np.meshgrid(np.arange(side * side), np.arange(side * side), indexing="ij")
        self.pi, self.pj = pi.ravel(), pj.ravel()
        self.n_bins = n_bins

    def r2(self, n_edges):
        import oracle

        a0 = np.linspace(2e-4, 6e-4, self.n_bins)
        return np.stack([oracle.chord_sq_edges(np.geomspace(a, 8 * a, n_edges)) for a in a0])

    def free(self):
        for c in (self.c1a, self.c1b, self.lab, self.rand, *self.per_label):
            c.free()


def _same(got, want, weighted):
    if weighted:
        assert_allclose(got, want, rtol=RTOL, atol=0)
    else:
        assert_array_equal(got, want)


VARIANTS = {  # name: (weighted, n_edges)
    "single": (False, 2),
    "cumulative": (False, 4),
    "subbins": (False, 24),
    "weighted_single": (True, 2),
    "weighted_multi": (True, 5),
}


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_labelled_equals_per_label_uploads(engine, variant):
    weighted, n_edges = VARIANTS[variant]
    s = Setup(engine, weighted=weighted)
    try:
        r2 = s.r2(n_edges)
        k = 1 if weighted else 0  # weighted sums, integer counts otherwise
        # count: one labelled pass against one unbinned pass per label
        out = engine.count(s.c1a, s.lab, s.pi, s.pj, r2, labels=True)
        assert out[0].shape == (s.n_lab, len(s.pi), s.n_bins, n_edges - 1)
        for ell, u in enumerate(s.per_label):
            want = engine.count(s.c1a, u, s.pi, s.pj, r2)
            _same(out[k][ell], want[k], weighted)
            assert_array_equal(out[0][ell], want[0])
        assert out[0].sum() > 0
        # count2: two first catalogs against the labels
        a, b, _ = engine.count2(s.c1a, s.c1b, s.lab, s.pi, s.pj, r2, labels=True)
        for ell, u in enumerate(s.per_label):
            _same(a[k][ell], engine.count(s.c1a, u, s.pi, s.pj, r2)[k], weighted)
            assert_array_equal(b[0][ell], engine.count(s.c1b, u, s.pi, s.pj, r2)[0])
        # count4: labelled cat2a with an unbinned cat2b, in one launch
        outs, _ = engine.count4(s.c1a, s.c1b, s.lab, s.rand, s.pi, s.pj, r2, labels=True)
        assert outs[0][0].shape[0] == s.n_lab and outs[2][0].shape[0] == 1
        for ell, u in enumerate(s.per_label):
            _same(outs[0][k][ell], a[k][ell], weighted)
            assert_array_equal(outs[1][0][ell], b[0][ell])
        _same(outs[2][k][0], engine.count(s.c1a, s.rand, s.pi, s.pj, r2)[k], weighted)
        assert_array_equal(outs[3][0][0], engine.count(s.c1b, s.rand, s.pi, s.pj, r2)[0])
        # and the reverse order: unbinned cat2a, labelled cat2b
        outs2, _ = engine.count4(s.c1a, s.c1b, s.rand, s.lab, s.pi, s.pj, r2, labels=True)
        _same(outs2[0][k][0], outs[2][k][0], weighted)
        for ell in range(s.n_lab):
            _same(outs2[2][k][ell], outs[0][k][ell], weighted)
            assert_array_equal(outs2[3][0][ell], outs[1][0][ell])
    finally:
        s.free()


def test_out_device_and_stats(engine):
    import torch

    s = Setup(engine, seed=3)
    try:
        r2 = s.r2(2)
        (ia, _), (ib, _), st = engine.count2(s.c1a, s.c1b, s.lab, s.pi, s.pj, r2, labels=True)
        shape = (s.n_lab, len(s.pi), s.n_bins, 1)
        bufs = [torch.zeros(shape, dtype=dt, device="cuda:0") for dt in (torch.float64, torch.int64) * 2]
        engine.count2(s.c1a, s.c1b, s.lab, s.pi, s.pj, r2, labels=True, out_device=tuple(b.data_ptr() for b in bufs))
        torch.cuda.synchronize()
        assert_array_equal(bufs[1].cpu().numpy(), ia)
        assert_array_equal(bufs[3].cpu().numpy(), ib)
        assert_array_equal(bufs[0].cpu().numpy(), ia.astype(np.float64))
        # a labelled catalog's naive tests count the rows of all its labels, as an unbinned catalog's do
        naive = sum(engine.count2(s.c1a, s.c1b, u, s.pi, s.pj, r2)[2]["pair_tests_naive"] for u in s.per_label)
        assert st["pair_tests_naive"] == naive
    finally:
        s.free()


def test_single_label_equals_unbinned(engine):
    rng = np.random.default_rng(5)
    x1, o1, _ = _rows(rng, 20_000, 4)
    x2, o2, _ = _rows(rng, 30_000, 4)
    c1 = engine.upload_catalog(x1, o1, zbin=rng.integers(0, 5, 20_000).astype(np.uint8), n_bins=5)
    one = engine.upload_catalog(x2, o2, zbin=np.zeros(30_000, dtype=np.uint8), n_bins=1)
    plain = engine.upload_catalog(x2, o2)
    try:
        import oracle

        r2 = np.tile(oracle.chord_sq_edges(np.array([2e-4, 1.5e-3])), (5, 1))
        pi, pj = np.meshgrid(np.arange(16), np.arange(16), indexing="ij")
        got = engine.count(c1, one, pi.ravel(), pj.ravel(), r2, labels=True)
        want = engine.count(c1, plain, pi.ravel(), pj.ravel(), r2)
        assert got[0].shape[0] == 1
        assert_array_equal(got[0][0], want[0])
        assert_array_equal(got[1][0], want[1])
        # an unbinned second catalog under the flag: L = 1
        assert_array_equal(engine.count(c1, plain, pi.ravel(), pj.ravel(), r2, labels=True)[0][0], want[0])
    finally:
        for c in (c1, one, plain):
            c.free()


def test_large_many_labels_share_warps(engine):
    """1e6 rows per catalog, 64 patches, 5 labels: items of many labels are interleaved in every warp's stream"""
    s = Setup(engine, n1=1_000_000, n2=1_000_000, side=8, n_bins=10, n_lab=5, seed=9)
    try:
        import oracle

        r2 = np.tile(oracle.chord_sq_edges(np.array([3e-4, 3e-3])), (s.n_bins, 1))
        outs, st = engine.count4(s.c1a, s.c1b, s.lab, s.rand, s.pi, s.pj, r2, labels=True)
        for ell, u in enumerate(s.per_label):
            assert_array_equal(outs[0][0][ell], engine.count(s.c1a, u, s.pi, s.pj, r2)[0])
            assert_array_equal(outs[1][0][ell], engine.count(s.c1b, u, s.pi, s.pj, r2)[0])
        assert outs[0][0].sum() > 1e6 and st["work_items"] > 0
    finally:
        s.free()


def test_rejected_flags_leave_the_engine_usable(engine):
    from ctypes import byref, c_void_p

    import yet_another_wizz_b200 as yb
    from yet_another_wizz_b200 import _lib

    s = Setup(engine, n1=5000, n2=8000, seed=4)
    try:
        r2 = s.r2(2)
        with pytest.raises(yb.YawbError, match="EXACT_BRUTEFORCE"):
            engine.count(s.c1a, s.lab, s.pi, s.pj, r2, exact=True, labels=True)
        ok = engine.count(s.c1a, s.lab, s.pi, s.pj, r2, labels=True)
        assert ok[0].sum() > 0
        pi = np.ascontiguousarray(s.pi, dtype=np.int32)
        pj = np.ascontiguousarray(s.pj, dtype=np.int32)
        out = np.zeros((len(pi), s.n_bins, 1), dtype=np.int64)
        stats = _lib.YawbStats()
        rc = engine.lib.yawb_count(engine._h, s.c1a._h, s.per_label[0]._h, pi.ctypes.data_as(c_void_p),
                                   pj.ctypes.data_as(c_void_p), len(pi), r2.ctypes.data_as(c_void_p), 2, 8, None,
                                   out.ctypes.data_as(c_void_p), byref(stats))
        assert rc != 0 and b"unknown flag" in engine.lib.yawb_last_error()
        again = engine.count(s.c1a, s.lab, s.pi, s.pj, r2, labels=True)
        assert_array_equal(again[0], ok[0])
    finally:
        s.free()


def _c1_tomographic(n_tomo=5, weighted=False):
    """C1-sized BoxRandoms catalogs (16 patches, 10 z-bins), the unknown sample split by a seeded label"""
    import yet_another_wizz_b200 as yb

    box = (0.0, 10.0, -2.5, 2.5)
    ras = (np.arange(4) + 0.5) * 10.0 / 4
    decs = -2.5 + (np.arange(4) + 0.5) * 5.0 / 4
    centers = yb.AngularCoordinates(np.deg2rad([[r, d] for d in decs for r in ras]))
    pool = np.random.default_rng(7).uniform(0.1, 1.0, 100_000)
    wpool = np.random.default_rng(8).uniform(0.5, 1.5, 100_000) if weighted else None
    mk = lambda name, n, seed, z=False, w=None: yb.Catalog.from_random(  # noqa: E731
        name, yb.BoxRandoms(*box, redshifts=pool if z else None, weights=w, seed=seed), n, patch_centers=centers)
    ref = mk("ref", 100_000, 1, z=True, w=wpool)
    ref_rand = mk("ref_rand", 1_000_000, 3, z=True)
    unk_rand = mk("unk_rand", 1_000_000, 4)
    unk = mk("unk", 100_000, 2, w=wpool)
    rows = {p: unk[p].load_data() for p in unk}
    lab = {p: np.random.default_rng(100 + p).integers(0, n_tomo, len(rows[p])) for p in unk}
    unknowns = []
    for i in range(n_tomo):
        parts = {p: rows[p][lab[p] == i] for p in unk}
        ra = np.concatenate([parts[p]["ra"] for p in unk])
        dec = np.concatenate([parts[p]["dec"] for p in unk])
        w = np.concatenate([parts[p]["weights"] for p in unk]) if weighted else None
        ids = np.concatenate([np.full(len(parts[p]), p) for p in unk])
        unknowns.append(yb.Catalog.from_arrays(ra, dec, patch_ids=ids, patch_centers=centers, weights=w, degrees=False))
    per_bin_rand = [mk(f"unk_rand_{i}", 200_000, 40 + i) for i in range(n_tomo)]
    config = yb.Configuration.create(rmin=100, rmax=1000, zmin=0.1, zmax=1.0, num_bins=10)
    return config, ref, ref_rand, unknowns, unk_rand, per_bin_rand


@pytest.mark.parametrize("weighted", [False, True])
def test_crosscorrelate_tomographic_vs_loop(engine, weighted):
    import yet_another_wizz_b200 as yb

    config, ref, ref_rand, unknowns, unk_rand, per_bin_rand = _c1_tomographic(weighted=weighted)
    for arg, rands in ((unk_rand, [unk_rand] * len(unknowns)), (per_bin_rand, per_bin_rand),
                       (None, [None] * len(unknowns))):
        got = yb.crosscorrelate_tomographic(config, ref, unknowns, ref_rand=ref_rand, unk_rand=arg, engine=engine)
        for i, (unk, rand) in enumerate(zip(unknowns, rands)):
            want = yb.crosscorrelate(config, ref, unk, ref_rand=ref_rand, unk_rand=rand, engine=engine)
            for a, b in zip(got[i], want):
                if not weighted:
                    assert a == b
                for kind in ("dd", "dr", "rd", "rr"):
                    x, y = getattr(a, kind), getattr(b, kind)
                    assert (x is None) == (y is None)
                    if x is not None:
                        assert_allclose(x.counts.counts, y.counts.counts, rtol=RTOL, atol=0)
                        assert_allclose(x.sum_weights.sum_weights2, y.sum_weights.sum_weights2, rtol=RTOL, atol=0)
        assert got[0][0].dd.counts.counts.sum() > 0
