"""Measurement calls counted in passes, on the CPU: the pass planner (every second-catalog row owned by exactly one
pass, every linked partner kept, every pass within its limit, one pass when the call fits, ValueError when one patch
with its partners cannot fit) and every measurement function on oracle doubles with a memory limit that forces
several passes, on one engine and on a group of two, against the golden results or a double without a limit."""

import numpy as np
import pytest

import golden_cases
import golden_io
from test_autocorrelate_tomographic import BinnedLabelOracleEngine
from test_autocorrelate_tomographic import split_catalog as split_auto
from test_engine_group import _Shares
from test_tomographic import LabelOracleEngine, assert_same, split_catalog

import yet_another_wizz_b200 as yb
from yet_another_wizz_b200 import measurements
from yet_another_wizz_b200.sharding import plan_passes


class _Memory:
    """a memory model for the doubles: 1000 bytes per catalog plus 100 per row, nothing for a count"""

    def __init__(self, limit=None):
        super().__init__()
        self.memory_limit = limit
        self.plain_uploads = 0
        self.released = 0

    def upload_catalog(self, xyz, patch_off, *, keep=None, second_rows=None, **kw):
        if keep is None:  # the path of a call that fits: a whole upload
            self.plain_uploads += 1
            return super(_Shares, self).upload_catalog(xyz, patch_off, **kw)
        return super().upload_catalog(xyz, patch_off, keep=keep, second_rows=second_rows, **kw)

    def footprint(self, n_rows, n_patch, n_bins=1, **kw):
        return 1000 + 100 * int(n_rows)

    def count_footprint(self, *args, **kw):
        return 0

    def memory_available(self):
        return self.memory_limit if self.memory_limit is not None else 1 << 62

    def memory_release(self):
        self.released += 1


class PassOracle(_Memory, _Shares, LabelOracleEngine):
    pass


class PassBinnedOracle(_Memory, _Shares, BinnedLabelOracleEngine):
    pass


def _centers(n_patch, seed=3):
    rng = np.random.default_rng(seed)
    ra, dec = rng.uniform(0, 0.6, n_patch), rng.uniform(-0.3, 0.3, n_patch)
    return np.column_stack([np.cos(ra) * np.cos(dec), np.sin(ra) * np.cos(dec), np.sin(dec)])


def _toy(n_patch=24, seed=3):
    rng = np.random.default_rng(seed)
    centers = _centers(n_patch, seed)
    d2 = ((centers[:, None] - centers[None]) ** 2).sum(-1)
    pi, pj = np.nonzero(d2 < 0.04)
    sizes = rng.integers(0, 400, n_patch)
    sizes[5] = 0
    patch_off = np.concatenate([[0], np.cumsum(sizes)])
    xyz = np.repeat(centers, sizes, axis=0) + rng.normal(0, 0.01, (patch_off[-1], 3))
    return centers, pi, pj, sizes, patch_off, xyz


def _fp(sizes):
    return lambda keep: 1000 + 100 * int(sizes[keep].sum())


def test_passes_own_every_row_once_keep_every_partner_and_fit():
    centers, pi, pj, sizes, patch_off, xyz = _toy()
    counts = [(pi, pj, sizes, sizes), (pj, pi, sizes, sizes)]
    whole = _fp(sizes)(np.ones(len(sizes), dtype=bool))
    # the smallest pass: one patch with its partners
    floor = max(_fp(sizes)(np.isin(np.arange(len(sizes)), np.r_[pi[pj == p], pj[pi == p], p])) for p in range(len(sizes)))
    for n_dev in (1, 2, 3):
        for frac in (0.9, 0.6, 0.4, 0.0):
            limits = [max(int(whole * frac), floor)] * n_dev
            steps = plan_passes(counts, np.full(len(sizes), 0.05), centers, _fp(sizes), limits)
            owned = np.zeros(patch_off[-1], dtype=int)
            for plan in steps:
                assert plan.n_devices == n_dev
                for d in range(n_dev):
                    keep = plan.keep[d].astype(bool)
                    assert _fp(sizes)(keep) <= limits[d]
                    rows = np.concatenate([np.arange(patch_off[p], patch_off[p + 1]) for p in np.flatnonzero(keep)]
                                          or [[]]).astype(int)
                    mask = plan.mask(d, xyz, patch_off)
                    owned[rows[mask == 1]] += 1
                    assert keep[pi[plan.second[d][pj]]].all() and keep[pj[plan.second[d][pi]]].all()
            assert (owned == 1).all()
            if n_dev == 1 and limits[0] < whole:
                assert len(steps) > 1


def test_one_pass_when_the_call_fits_and_error_when_one_patch_cannot():
    centers, pi, pj, sizes, _, _ = _toy()
    counts = [(pi, pj, sizes, sizes)]
    whole = _fp(sizes)(np.ones(len(sizes), dtype=bool))
    assert len(plan_passes(counts, np.full(len(sizes), 0.05), centers, _fp(sizes), [whole])) == 1
    assert len(plan_passes(counts, np.full(len(sizes), 0.05), centers, _fp(sizes), [whole, whole])) == 1
    with pytest.raises(ValueError, match=r"needs \d+ bytes of device memory, more than the limit of 2000 bytes"):
        plan_passes(counts, np.full(len(sizes), 0.05), centers, _fp(sizes), [2000])


class _Planned(Exception):
    pass


def _limit_for(run, cls, target, monkeypatch):
    """the largest limit (in steps of 4 % from 16 MB) under which the call `run(engine)` is planned in at least `target` passes"""
    seen = []

    def probe(*args, **kw):
        steps = plan_passes(*args, **kw)
        seen.append(len(steps))
        raise _Planned

    with monkeypatch.context() as m:
        m.setattr(measurements, "plan_passes", probe)
        limit = 1 << 24
        while limit > 1000:
            try:
                run(cls(limit))
            except _Planned:
                pass
            except ValueError:  # no smaller pass is possible
                break
            if seen[-1] >= target:
                return limit
            limit = int(limit * 0.96)
    pytest.skip(f"no limit gives {target} passes")


def _engines(cls, limit, n_dev):
    if n_dev == 1:
        return cls(limit)
    return yb.EngineGroup([cls(limit) for _ in range(n_dev)])


def _passes(engine):
    stats = measurements.last_stats()
    assert stats and all(st.get("passes", 1) > 1 for st in stats.values())
    members = engine.engines if isinstance(engine, yb.EngineGroup) else [engine]
    assert all(e.plain_uploads == 0 and e.released >= 2 for e in members)


@pytest.mark.parametrize("n_dev", [1, 2])
@pytest.mark.parametrize("target", [2, 3, 5])
@pytest.mark.parametrize("name", ["cross_unweighted", "cross_weighted_multiscale"])
def test_crosscorrelate(name, target, n_dev, monkeypatch):
    g = golden_io.load(name)
    limit = _limit_for(lambda e: golden_cases.run_cross(g, e), PassOracle, target, monkeypatch)
    eng = _engines(PassOracle, limit, n_dev)
    corrs = golden_cases.run_cross(g, eng)
    _passes(eng)
    golden_cases.check_corrfunc(g, "cross", corrs, ("dd", "dr", "rd", "rr"), exact=name == "cross_unweighted")


@pytest.mark.parametrize("n_dev", [1, 2])
@pytest.mark.parametrize("target", [2, 3, 5])
@pytest.mark.parametrize("name", ["auto_unweighted", "auto_rweight_polewrap"])
def test_autocorrelate(name, target, n_dev, monkeypatch):
    g = golden_io.load(name)
    limit = _limit_for(lambda e: golden_cases.run_auto(g, e), PassOracle, target, monkeypatch)
    eng = _engines(PassOracle, limit, n_dev)
    corrs = golden_cases.run_auto(g, eng)
    _passes(eng)
    golden_cases.check_corrfunc(g, "auto", corrs, ("dd", "dr", "rr"), exact=name == "auto_unweighted")


@pytest.mark.parametrize("n_dev", [1, 2])
@pytest.mark.parametrize("target", [2, 3, 5])
@pytest.mark.parametrize("name", ["scalar_unweighted", "scalar_weighted"])
def test_scalar(name, target, n_dev, monkeypatch):
    g = golden_io.load(name)
    limit = _limit_for(lambda e: golden_cases.run_scalar(g, e), PassOracle, target, monkeypatch)
    eng = _engines(PassOracle, limit, n_dev)
    golden_cases.check_scalar(g, golden_cases.run_scalar(g, eng), exact_numbers=name == "scalar_unweighted")
    _passes(eng)


@pytest.mark.parametrize("n_dev", [1, 2])
@pytest.mark.parametrize("target", [2, 3, 5])
def test_crosscorrelate_tomographic(target, n_dev, monkeypatch):
    g = golden_io.load("cross_weighted_multiscale")
    config = golden_cases.config_from_golden(g)
    cats = {k: golden_cases.catalog_from_golden(g, k) for k in ("ref", "ref_rand", "unk_rand")}
    unknowns = split_catalog(g, "unk")
    kw = dict(ref_rand=cats["ref_rand"], unk_rand=cats["unk_rand"])

    def run(e):
        return yb.crosscorrelate_tomographic(config, cats["ref"], unknowns, engine=e, **kw)

    limit = _limit_for(run, PassOracle, target, monkeypatch)
    eng = _engines(PassOracle, limit, n_dev)
    got = run(eng)
    _passes(eng)
    for a, b in zip(got, run(LabelOracleEngine())):
        assert_same(a, b, exact=False)


@pytest.mark.parametrize("n_dev", [1, 2])
@pytest.mark.parametrize("target", [2, 3, 5])
@pytest.mark.parametrize("rand_form", ["shared", "per_bin"])
def test_autocorrelate_tomographic(rand_form, target, n_dev, monkeypatch):
    g = golden_io.load("auto_unweighted")
    config = golden_cases.config_from_golden(g)
    data = split_auto(g, "data")
    rand = golden_cases.catalog_from_golden(g, "rand") if rand_form == "shared" else split_auto(g, "rand", seed=12)

    def run(e):
        return yb.autocorrelate_tomographic(config, data, rand, engine=e)

    limit = _limit_for(run, PassBinnedOracle, target, monkeypatch)
    eng = _engines(PassBinnedOracle, limit, n_dev)
    got = run(eng)
    _passes(eng)
    for a, b in zip(got, run(BinnedLabelOracleEngine())):
        assert_same(a, b, exact=True)


def test_a_call_that_fits_uploads_whole_catalogs():
    g = golden_io.load("cross_unweighted")
    eng = PassOracle(1 << 40)
    corrs = golden_cases.run_cross(g, eng)
    golden_cases.check_corrfunc(g, "cross", corrs, ("dd", "dr", "rd", "rr"), exact=True)
    assert eng.plain_uploads == 4 and eng.released == 0
    assert all("passes" not in st for st in measurements.last_stats().values())


def test_a_pass_that_cannot_fit_raises_before_any_upload():
    g = golden_io.load("cross_unweighted")
    eng = PassOracle(1500)
    with pytest.raises(ValueError, match="more than the limit of 1500 bytes"):
        golden_cases.run_cross(g, eng)
    assert eng.plain_uploads == 0 and not getattr(eng, "partial_uploads", 0)
