"""Host side of the memory model of a call counted in passes: the work-item bound of `yawb_count_footprint` across the
count at which the planner switches to the longer lists of a small job, the default memory limit of an `Engine` and
the catalogs it drops from its cache to make room, and the one-patch-per-pass fallback with unequal limits."""

import numpy as np
import pytest

from yet_another_wizz_b200.sharding import plan_passes

ITEM = 96  # bytes of a work item (yawb_internal.cuh)


def _count_bound(lib, sms, n_items, n_pairs=100, n_bins=4, n_edges=8):
    from ctypes import byref, c_int64

    from yet_another_wizz_b200 import _lib

    out = c_int64()
    _lib.check(lib.yawb_count_footprint(sms, n_items, n_pairs, n_bins, n_edges, 1, 1, byref(out)))
    return out.value


def test_count_bound_covers_both_sides_of_the_small_job_threshold():
    from yet_another_wizz_b200 import _lib
    from yet_another_wizz_b200.csrc import build

    build.build()
    lib = _lib.load()
    sms = 148
    threshold = 30 * sms * 4 * 4  # SMALL_JOB_ITEMS x warps of the persistent grid
    largest_small = 7 * (4 * (threshold - 1) + 2048) * ITEM  # the lists a real count just below the threshold gets
    bounds = [_count_bound(lib, sms, n) for n in range(threshold - 3, threshold + 4)]
    assert bounds == sorted(bounds)  # an overestimate of the items never lowers the bound
    assert bounds[2] >= largest_small and bounds[-1] >= largest_small
    assert _count_bound(lib, sms, 20 * threshold) >= (4 * 20 * threshold + 2048) * ITEM


class _Dev:
    def __init__(self, nbytes):
        self.nbytes, self._h, self.freed = nbytes, 1, False

    def info(self):
        return 0, self.nbytes

    def free(self):
        self.freed, self._h = True, None


class _Cat:
    pass


def _engine(limit=None):
    from yet_another_wizz_b200 import Engine

    class MemoryEngine(Engine):  # the cache and limit logic of Engine over a fake device
        def memory_stats(self):
            return dict(held=0, peak=0, device_free=100)

        def memory_parked(self):
            return 50

    eng = object.__new__(MemoryEngine)
    eng._h = None
    eng.memory_limit = limit
    eng._cat_cache = {}
    return eng


def test_default_limit_counts_cached_catalogs_and_make_room_drops_unused_ones_lru():
    eng = _engine()
    old, newer, used = _Cat(), _Cat(), _Cat()
    devs = {}
    for tick, (cat, nbytes) in enumerate(((old, 300), (newer, 300), (used, 400))):
        devs[id(cat)] = _Dev(nbytes)
        eng._cat_cache[(("id", id(cat)), False)] = [None, devs[id(cat)], 0, [], tick]
    assert eng.memory_available() == 100 + 50 + 1000
    eng.make_room(800, [used])  # free + parked + the call's own catalog: 550; the oldest unrelated entry is enough
    assert devs[id(old)].freed and not devs[id(newer)].freed and not devs[id(used)].freed
    eng.make_room(10_000, [used])  # never the call's own catalogs
    assert devs[id(newer)].freed and not devs[id(used)].freed


def test_explicit_limit_drops_nothing():
    eng = _engine(limit=123)
    cat = _Cat()
    dev = _Dev(300)
    eng._cat_cache[(("id", id(cat)), False)] = [None, dev, 0, [], 0]
    assert eng.memory_available() == 123
    eng.make_room(10_000, [])
    assert not dev.freed


def test_a_fitting_call_makes_room_for_its_footprint():
    import golden_cases
    import golden_io
    from test_passes import PassOracle

    class Recording(PassOracle):
        def make_room(self, nbytes, catalogs=()):
            self.room = (nbytes, len(catalogs))

    g = golden_io.load("cross_unweighted")
    eng = Recording(1 << 40)
    golden_cases.run_cross(g, eng)
    assert eng.plain_uploads == 4 and eng.room[0] > 0 and eng.room[1] == 4


def test_empty_passes_of_the_fallback_need_no_memory():
    # three unlinked patches on four devices: the fourth device has no patch, and a limit below a catalog's base cost
    centers = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [0.0, 0.0, 1.0]])
    pi = pj = np.arange(3)
    sizes = np.array([100, 100, 100])
    fp = lambda keep: 5000 + 100 * int(sizes[keep].sum())  # noqa: E731
    steps = plan_passes([(pi, pj, sizes, sizes)], np.full(3, 0.1), centers, fp, [20000] * 3 + [4000])
    owned = sum(np.array([s.second[d] for d in range(4)]).sum(0) for s in steps)
    assert (owned == 1).all()
    with pytest.raises(ValueError, match="more than the limit"):
        plan_passes([(pi, pj, sizes, sizes)], np.full(3, 0.1), centers, fp, [4000] * 4)
