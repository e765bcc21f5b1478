"""
`crosscorrelate` / `autocorrelate` -- the drop-in for the reference's measurement
driver (`src/yaw/correlation/measurements.py`), with the pair counting moved to the
GPU engine.

Kept from the reference, line for line in behaviour: the patch linkage
(`PatchLinkage.from_catalogs` :193-237, `get_max_angle` :152-168,
`check_patch_conistency` :131-149), the visited pair set (`iter_patch_id_pairs`
:258-289), the scatter of results with the 0.5 on auto diagonals (:354-364), the
error behaviour (:432-448, :588-589) and the public signatures (:455-463, :529-538).
Replaced: `process_patch_pair` + `parallel.iter_unordered` (:88-128, :344-350) by one
`yawb_count` call per count type, and the tree build by one catalog upload.

Both this package's `Configuration` / `Catalog` and genuine `yaw.Configuration` /
`yaw.Catalog` objects are accepted (duck typing on the attributes listed in
`config.py` / `catalog.py`).
"""

from __future__ import annotations

import functools
import logging
import os
import threading
from collections.abc import Sequence
from copy import deepcopy
from itertools import compress

import numpy as np

from .angular import AngularBinPlan
from .binning import Binning
from .catalog import InconsistentPatchesError
from .coordinates import AngularCoordinates, AngularDistances
from .corrfunc import CorrFunc, ScalarCorrFunc
from .paircounts import NormalisedCounts, NormalisedScalarCounts, PatchedCounts, PatchedSumWeights
from .sharding import Shard, assign_pairs_lpt, current_shard, pair_costs, plan_passes, plan_shares

__all__ = ["PatchLinkage", "autocorrelate", "autocorrelate_scalar", "autocorrelate_tomographic",
           "compute_scalar_normalisation", "crosscorrelate", "crosscorrelate_scalar", "crosscorrelate_tomographic",
           "get_default_engine", "last_stats"]

logger = logging.getLogger("yaw_b200")

_default_engine = None
_last_stats: dict[str, dict] = {}


def get_default_engine():
    """Process-wide engine on `cuda:LOCAL_RANK` (created on first use; raises without a GPU)."""
    global _default_engine
    if _default_engine is None:
        from .engine import Engine

        _default_engine = Engine(int(os.environ.get("LOCAL_RANK", "0")))
    return _default_engine


def last_stats() -> dict[str, dict]:
    """Engine statistics of the most recent `crosscorrelate` / `autocorrelate` call, per count type."""
    return dict(_last_stats)


# ---- duck-typed accessors shared by this package's and the reference's objects -------------------
def _coords_data(obj) -> np.ndarray:
    return np.asarray(obj.data, dtype=np.float64)


def _as_binning(config) -> Binning:
    b = config.binning.binning
    return b if isinstance(b, Binning) else Binning(np.asarray(b.edges, dtype=np.float64), closed=str(b.closed))


def _patch_rows(patch):
    data = patch.load_data()
    names = data.dtype.names
    ra = np.asarray(data["ra"], dtype=np.float64)
    dec = np.asarray(data["dec"], dtype=np.float64)
    weights = np.asarray(data["weights"], dtype=np.float64) if "weights" in names else None
    redshifts = np.asarray(data["redshifts"], dtype=np.float64) if "redshifts" in names else None
    kappa = np.asarray(data["kappa"], dtype=np.float64) if "kappa" in names else None
    return ra, dec, weights, redshifts, kappa


_ANGLE_CACHE: dict = {}  # (id(cosmology), scales, z-bin centres) -> (cosmology, result): a few entries per process


def _angles_per_bin(config) -> tuple[np.ndarray, np.ndarray]:
    """`get_angle_radian(zmid)` of every z-bin, evaluated once (the reference re-evaluates it
    for every patch pair, `measurements.py:110-112`).  The conversion integrates the cosmology numerically per
    redshift (a third of the host time of a call whose catalogs are already on the device), so the result is kept
    per (cosmology object, scales, z-bin centres): a loop of calls over tomographic bins with the same
    configuration (`cli/tasks.py:536-550`) evaluates it once.  Identical inputs, identical doubles."""
    zmids = _as_binning(config).mids
    scales = config.scales.scales
    cosmology = config.cosmology
    key = None
    try:
        key = (id(cosmology), str(getattr(scales, "unit", None)), tuple(np.atleast_1d(scales.scale_min).tolist()),
               tuple(np.atleast_1d(scales.scale_max).tolist()), tuple(np.asarray(zmids, dtype=np.float64).tolist()))
        hit = _ANGLE_CACHE.get(key)
        if hit is not None and hit[0] is cosmology:
            return hit[1][0].copy(), hit[1][1].copy()
    except Exception:  # foreign scales objects without these attributes: no caching
        key = None
    amin, amax = [], []
    for z in zmids:
        lo, hi = config.scales.scales.get_angle_radian(z, cosmology=config.cosmology)
        amin.append(np.atleast_1d(lo))
        amax.append(np.atleast_1d(hi))
    out = np.array(amin, dtype=np.float64), np.array(amax, dtype=np.float64)
    if key is not None:
        if len(_ANGLE_CACHE) > 16:
            _ANGLE_CACHE.clear()
        _ANGLE_CACHE[key] = (cosmology, (out[0].copy(), out[1].copy()))
    return out


def prepare_catalog_arrays(catalog, binning: Binning | None, *, kappa: bool = False,
                           workers: int | None = None, alloc=None, device_digitize: bool = False) -> dict:
    """Host preparation of one catalog for the C ABI: load every patch once, convert to unit
    vectors with the reference's formula (`AngularCoordinates.to_3d`: numpy cos / sin in double, so the
    device sees the doubles the reference's trees hold), digitise the redshifts (`trees.py:408-414`).
    Returns the keyword arguments of `Engine.upload_catalog`.

    The patches are processed by a small thread pool (numpy releases the GIL inside its loops) that
    writes straight into the preallocated output arrays: for C3-sized inputs this is what an end-to-end
    call spends most of its time on, not the GPU.

    `kappa=True` prepares the "k" side of a scalar-field count: the per-row pair weight is
    kappa x weight (kappa alone without weights), `AngularTree.get_pair_weights`, `trees.py:270-301`.
    `alloc(shape, dtype)` supplies the output arrays (page-locked staging of the engine; default numpy)."""
    alloc = alloc or np.empty
    has_w = bool(catalog.has_weights) or kappa
    if binning is not None and not catalog.has_redshifts:
        raise ValueError("patch has no 'redshifts' attached")  # trees.py:397-398
    patch_ids = list(catalog.keys())
    if patch_ids != list(range(len(patch_ids))):
        raise InconsistentPatchesError("patch IDs must be 0..num_patches-1")
    sizes = [int(n) for n in catalog.get_num_records()]
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    n = int(off[-1])
    xyz = alloc((n, 3), np.float64)
    ws = alloc(n, np.float64) if has_w else None
    # z-bin ids travel as bytes when they fit (255 = outside the binning): a quarter of the PCIe traffic;
    # with `device_digitize` the raw redshifts travel instead and the device assigns the bins (same comparisons
    # as np.digitize, `yawb_upload_catalog_z`): 8 bytes per row over PCIe against a host pass over the redshifts
    small_bins = binning is not None and len(binning) <= 254
    zb = zr = None
    if binning is not None and device_digitize:
        zr = alloc(n, np.float64)
    elif binning is not None:
        zb = alloc(n, np.uint8 if small_bins else np.int32)

    def fill(pid: int) -> None:
        ra, dec, weights, redshifts, kappa_vals = _patch_rows(catalog[pid])
        s, e = int(off[pid]), int(off[pid + 1])
        if kappa:
            if kappa_vals is None:
                raise ValueError("missing required 'kappa'")
            weights = kappa_vals if weights is None else kappa_vals * weights
        _fill_rows(xyz, ws, s, e, pid, ra, dec, weights)
        if zr is not None:
            zr[s:e] = redshifts
        elif binning is not None:
            ids = binning.digitize(redshifts)  # -1 below, len(binning) above the binning
            if small_bins:
                ids[ids < 0] = 255
            zb[s:e] = ids

    _run_fill(fill, patch_ids, n, workers)
    out = dict(xyz=xyz, patch_off=off, weights=ws, zbin=zb, n_bins=len(binning) if binning is not None else 1)
    if zr is not None:
        out.update(redshifts=zr, edges=np.asarray(binning.edges, dtype=np.float64), closed=str(binning.closed))
    return out


def _fill_rows(xyz, ws, s: int, e: int, pid: int, ra, dec, weights) -> None:
    """rows `s:e` of the output arrays from the rows of patch `pid`: unit vectors with the reference's formula and, when
    the catalog is weighted (`ws` is not None), the weights"""
    if len(ra) != e - s:
        raise InconsistentPatchesError(f"patch {pid} holds {len(ra)} rows, its meta data says {e - s}")
    cos_dec = np.cos(dec)  # same operations, same order as coordinates.py:134-147
    np.multiply(np.cos(ra), cos_dec, out=xyz[s:e, 0])
    np.multiply(np.sin(ra), cos_dec, out=xyz[s:e, 1])
    np.sin(dec, out=xyz[s:e, 2])
    if ws is not None:
        ws[s:e] = weights


def _run_fill(fill, tasks, n_rows: int, workers: int | None) -> None:
    """`fill(task)` for every task; by a small thread pool (numpy releases the GIL) when the rows are many"""
    if workers is None:
        workers = min(16, os.cpu_count() or 1)
    if workers > 1 and len(tasks) > 1 and n_rows > 200_000:
        from concurrent.futures import ThreadPoolExecutor

        with ThreadPoolExecutor(max_workers=workers) as pool:
            list(pool.map(fill, tasks))
    else:
        for task in tasks:
            fill(task)


def prepare_labelled_arrays(catalogs, binning: Binning | None = None, *, workers: int | None = None,
                            alloc=None) -> dict:
    """Host preparation of ONE labelled catalog from several (`YAWB_FLAG_SECOND_LABELS`): per patch the rows of
    `catalogs[0]`, `catalogs[1]`, ..., each row labelled with the position of its catalog (byte-sized ids, at
    most 254 catalogs).  The rows and their unit vectors are those `prepare_catalog_arrays` gives each catalog.
    Returns the keyword arguments of `Engine.upload_catalog`.

    With `binning` the ids are binned labels (`n_labels` = number of catalogs): `label * B + z-bin`, the z-bins
    digitised as `prepare_catalog_arrays` does.  A row outside the binning is dropped (id 255 when `L * B <= 254`,
    else -1), never given a neighbouring label's id."""
    alloc = alloc or np.empty
    catalogs = list(catalogs)
    if not 1 <= len(catalogs) <= 254:
        raise ValueError("a labelled catalog holds 1 to 254 catalogs")
    has_w = bool(catalogs[0].has_weights)
    if any(bool(c.has_weights) != has_w for c in catalogs):
        raise ValueError("the catalogs of a labelled upload must all have weights or all have none")
    if binning is not None and not all(c.has_redshifts for c in catalogs):
        raise ValueError("patch has no 'redshifts' attached")  # as prepare_catalog_arrays
    n_zbins = len(binning) if binning is not None else 1
    n_ids = len(catalogs) * n_zbins
    small_ids = n_ids <= 254
    n_patch = len(catalogs[0])
    for c in catalogs:
        if list(c.keys()) != list(range(n_patch)):
            raise InconsistentPatchesError("patch IDs must be 0..num_patches-1")
    sizes = np.array([[int(n) for n in c.get_num_records()] for c in catalogs], dtype=np.int64)  # (label, patch)
    # row offset of (patch, label): patch-major, the labels of a patch one after the other
    start = np.concatenate([[0], np.cumsum(sizes.T.ravel())]).astype(np.int64)
    off = np.ascontiguousarray(start[:: len(catalogs)])
    n = int(off[-1])
    xyz = alloc((n, 3), np.float64)
    ws = alloc(n, np.float64) if has_w else None
    lab = alloc(n, np.uint8 if small_ids else np.int32)

    def fill(task) -> None:
        label, pid = task
        ra, dec, weights, redshifts, _ = _patch_rows(catalogs[label][pid])
        s = int(start[pid * len(catalogs) + label])
        e = s + int(sizes[label, pid])
        _fill_rows(xyz, ws, s, e, pid, ra, dec, weights)
        if binning is None:
            lab[s:e] = label
        else:
            z = binning.digitize(redshifts)  # -1 below, len(binning) above the binning
            lab[s:e] = np.where((z >= 0) & (z < n_zbins), label * n_zbins + z, 255 if small_ids else -1)

    _run_fill(fill, [(label, pid) for pid in range(n_patch) for label in range(len(catalogs))], n, workers)
    out = dict(xyz=xyz, patch_off=off, weights=ws, zbin=lab, n_bins=n_ids)
    if binning is not None:
        out["n_labels"] = len(catalogs)
    return out


def _prepare_for(engine, catalog, binning: Binning | None, kappa: bool) -> dict:
    # opt-in (`Engine(staging=True)`): large catalogs are prepared straight into the engine's page-locked
    # staging cache; the copy is then asynchronous and overlaps with the preparation of the next catalog
    staged = getattr(engine, "staging", False) and sum(catalog.get_num_records()) >= engine.staging_min_rows
    return prepare_catalog_arrays(catalog, binning, kappa=kappa, alloc=engine.staging_empty if staged else None,
                                  device_digitize=bool(getattr(engine, "device_digitize", False)))


class _Uploads:
    """Device catalogs of one measurement call, uploaded once and shared by DD/DR/RD/RR.

    `enqueue` takes the catalogs of the call in the order they should travel: their host preparation
    (numpy releases the GIL) runs one catalog ahead on a helper thread, so preparing catalog k + 1
    overlaps with the copy of catalog k, which for pageable host memory blocks the calling thread.

    On an `EngineGroup` every catalog is prepared once on the host and uploaded in shares: `plan` (the call's
    `SharePlan`) says which patches and rows each device holds."""

    def __init__(self, engine, plan=None) -> None:
        self.engine = engine
        self.plan = plan
        self.run = _current_run()  # a call counted in passes: host arrays prepared once, no resident catalogs
        self._resident: set = set()  # keys whose device catalog belongs to the engine's cache (not freed here)
        self._cache: dict[tuple[int, bool, bool], object] = {}
        self._pending: dict[tuple[int, bool, bool], object] = {}
        self._pool = None

    @staticmethod
    def _key(catalog, binning, kappa):
        return (id(catalog), binning is not None, bool(kappa))

    @staticmethod
    def _signature(catalog, binning):
        """what a resident device catalog depends on besides the catalog object: the z-binning (the reference's
        `binning` file) and, as a guard against catalogs refilled in place, the rows per patch"""
        if isinstance(catalog, tuple):  # a labelled upload: the signatures of its members
            return tuple(_Uploads._signature(c, binning) for c in catalog)
        rows = tuple(int(n) for n in catalog.get_num_records())
        if binning is None:
            return (rows, None)
        return (rows, tuple(np.asarray(binning.edges, dtype=np.float64).tolist()), str(binning.closed))

    def _resident_lookup(self, key, catalog, binning, kappa) -> bool:
        if self.run is not None:
            return False
        lookup = getattr(self.engine, "cache_lookup", None)
        if self._group():  # the parts stay with their engines' caches: the GroupCatalog itself is not resident
            dev = self.engine.cache_lookup(catalog, self._signature(catalog, binning), kappa, self.plan)
            if dev is not None:
                self._cache[key] = dev
            return dev is not None
        dev = lookup(catalog, self._signature(catalog, binning), kappa) if lookup else None
        if dev is None:
            return False
        self._cache[key] = dev
        self._resident.add(key)
        return True

    def _group(self) -> bool:
        from .engine import EngineGroup

        if not isinstance(self.engine, EngineGroup):
            return False
        if self.plan is None:
            raise ValueError("an EngineGroup counts through the measurement functions, which plan its shares")
        return True

    def _upload(self, key, catalog, binning, kappa, arrays):
        if self._group():
            cache = None if self.run is not None else (catalog, self._signature(catalog, binning), kappa)
            dev = self.engine.upload_catalog(arrays, self.plan, cache=cache)
            if self.run is not None:
                dev.sums_hook = self.run.sums
            self._cache[key] = dev
            return dev
        dev = self.engine.upload_catalog(arrays.pop("xyz"), arrays.pop("patch_off"), **arrays)
        return self._store(key, catalog, binning, kappa, dev)

    def _store(self, key, catalog, binning, kappa, dev):
        self._cache[key] = dev
        store = getattr(self.engine, "cache_store", None)
        if store and store(catalog, self._signature(catalog, binning), kappa, dev):
            self._resident.add(key)
        return dev

    def enqueue(self, requests) -> None:
        """`requests`: iterable of (catalog or None, binning or None[, kappa])."""
        from concurrent.futures import ThreadPoolExecutor

        todo = []
        for req in requests:
            catalog, binning, kappa = (*req, False)[:3]
            key = self._key(catalog, binning, kappa)
            if catalog is not None and key not in self._cache and key not in self._pending:
                if not self._resident_lookup(key, catalog, binning, kappa):
                    todo.append((key, catalog, binning, kappa))
        if not todo:
            return
        if self._pool is None:
            self._pool = ThreadPoolExecutor(max_workers=1)
        for key, catalog, binning, kappa in todo:
            self._pending[key] = (self._pool.submit(self._prepare, key, catalog, binning, kappa), catalog, binning, kappa)
        for key, *_ in todo:  # upload in order; each wait overlaps with the preparation of the next catalog
            self._resolve(key)

    def _resolve(self, key):
        fut, catalog, binning, kappa = self._pending.pop(key)
        return self._upload(key, catalog, binning, kappa, fut.result())

    def _prepare(self, key, catalog, binning, kappa, make=None):
        """host arrays of one catalog; in a call counted in passes prepared once and kept for every pass"""
        make = make or (lambda: _prepare_for(self.engine, catalog, binning, kappa))
        if self.run is None:
            return make()
        with self.run.lock:
            if key not in self.run.prepared:
                self.run.prepared[key] = make()
            return self.run.prepared[key]

    def get(self, catalog, binning: Binning | None, kappa: bool = False):
        key = self._key(catalog, binning, kappa)
        if key in self._pending:
            return self._resolve(key)
        if key not in self._cache and not self._resident_lookup(key, catalog, binning, kappa):
            self._upload(key, catalog, binning, kappa, self._prepare(key, catalog, binning, kappa))
        return self._cache[key]

    def get_labelled(self, catalogs, binning: Binning | None = None):
        """ONE device catalog holding the rows of `catalogs`, labelled by position (`prepare_labelled_arrays`; with
        `binning`, binned labels).  Kept in the engine's cache like a single catalog, keyed by the tuple of its
        members, and dropped there as soon as any member dies."""
        catalogs = tuple(catalogs)
        key = (("labelled", *map(id, catalogs)), binning is not None, False)
        if key not in self._cache and not self._resident_lookup(key, catalogs, binning, False):
            arrays = self._prepare(key, catalogs, binning, False, lambda: prepare_labelled_arrays(catalogs, binning))
            self._upload(key, catalogs, binning, False, arrays)
        return self._cache[key]

    def free(self) -> None:
        for fut, *_ in self._pending.values():
            fut.cancel()
        self._pending.clear()
        if self._pool is not None:
            self._pool.shutdown(wait=True)
            self._pool = None
        for key, dev in self._cache.items():
            if key not in self._resident:  # resident catalogs stay with the engine for the next call
                dev.free()
        self._cache.clear()
        self._resident.clear()
        if getattr(self.engine, "staging", False):  # every upload of this call has been consumed or dropped
            self.engine.sync()
            self.engine.staging_release()


# ---- patch linkage ----------------------------------------------------------------------------------
# The functions and methods from here to `PatchLinkage.get_patch_id_pairs` (`check_patch_conistency`,
# `get_max_angle`, `PatchLinkage.from_catalogs` and its properties, `iter_patch_id_pairs`) restate the reference's
# decisions step by step (yet_another_wizz v3.1.1, `src/yaw/correlation/measurements.py:131-168, 193-289`,
# Copyright (C) Jan Luca van den Busch, GPL-3.0-or-later): the engine must visit exactly the reference's set of
# patch pairs, including the order in which `set.pop()` yields them, so this block follows that code closely
# and is covered by the same licence terms.
def check_patch_conistency(catalog, *catalogs, rtol: float = 0.5) -> None:
    centers = AngularCoordinates(_coords_data(catalog.get_centers()))
    radii = _coords_data(catalog.get_radii())
    for cat in catalogs:
        distance = centers.distance(AngularCoordinates(_coords_data(cat.get_centers())))
        if np.any(distance.data / radii > rtol):
            raise InconsistentPatchesError("patch centers are not aligned")


def get_max_angle(config, redshift_limit: float = 0.05) -> AngularDistances:
    min_redshift = max(config.binning.zmin, redshift_limit)
    _, ang_max = config.scales.scales.get_angle_radian(min_redshift, cosmology=config.cosmology)
    return AngularDistances(np.max(ang_max))


class PatchLinkage:
    """Which patch pairs are counted (`patch_links`: id -> set of linked ids) and the count driver."""

    def __init__(self, config, patch_links: dict[int, set[int]], *, engine=None, shard: Shard | None = None) -> None:
        self.config = config
        self.patch_links = patch_links
        self.engine = engine
        self.shard = shard
        self._plan: AngularBinPlan | None = None
        self._uploads: _Uploads | None = None

    @classmethod
    def from_catalogs(cls, config, catalog, *catalogs, engine=None, shard: Shard | None = None) -> "PatchLinkage":
        if any(set(cat.keys()) != catalog.keys() for cat in catalogs):
            raise InconsistentPatchesError("patch IDs do not match")
        max_scale_angle = get_max_angle(config)
        # largest catalog = best constrained centres/radii; compares `get_num_records()` tuples
        ref_cat, *other_cats = sorted([catalog, *catalogs], key=lambda cat: cat.get_num_records(), reverse=True)
        check_patch_conistency(ref_cat, *other_cats)

        patch_ids = list(ref_cat.keys())
        centers = AngularCoordinates(_coords_data(ref_cat.get_centers()))
        radii = AngularDistances(_coords_data(ref_cat.get_radii()))
        patch_links = {}
        for patch_id, patch_center, patch_radius in zip(patch_ids, centers, radii):
            distances = centers.distance(AngularCoordinates(np.broadcast_to(patch_center.data, centers.data.shape)))
            linked = distances.data < (radii.data + patch_radius.data + max_scale_angle.data)
            patch_links[patch_id] = set(compress(patch_ids, linked))
        return cls(config, patch_links, engine=engine, shard=shard)

    @property
    def num_total(self) -> int:
        return len(self.patch_links) ** 2

    @property
    def num_links(self) -> int:
        return sum(len(links) for links in self.patch_links.values())

    @property
    def density(self) -> float:
        return self.num_links / self.num_total

    def __repr__(self) -> str:
        return f"{type(self).__name__}(num_links={self.num_links}, density={self.density:.0%})"

    def iter_patch_id_pairs(self, *, auto: bool):
        """Same set and order as the reference: all (i, i) first, then round-robin over the links."""
        patch_links = deepcopy(self.patch_links)
        for i, links in patch_links.items():
            links.remove(i)
            yield (i, i)
        while len(patch_links) > 0:
            exhausted = set()
            for i, links in patch_links.items():
                try:
                    j = links.pop()
                except KeyError:
                    exhausted.add(i)
                    continue
                if not auto or j > i:
                    yield (i, j)
            for i in exhausted:
                patch_links.pop(i)

    def get_patch_id_pairs(self, *, auto: bool) -> tuple[np.ndarray, np.ndarray]:
        """the pair list as two arrays; walked once per linkage and `auto` (every count of a call asks for it)"""
        cache = self.__dict__.setdefault("_pair_cache", {})
        hit = cache.get(bool(auto))
        if hit is not None and hit[0] == self.num_links:
            return hit[1].copy(), hit[2].copy()
        pairs = list(self.iter_patch_id_pairs(auto=auto))
        if not pairs:
            return np.empty(0, dtype=np.int32), np.empty(0, dtype=np.int32)
        arr = np.array(pairs, dtype=np.int32)
        cache[bool(auto)] = (self.num_links, arr[:, 0].copy(), arr[:, 1].copy())
        return arr[:, 0].copy(), arr[:, 1].copy()

    # ---- the count driver --------------------------------------------------------------------------
    def _get_plan(self) -> AngularBinPlan:
        if self._plan is None:
            ang_min, ang_max = _angles_per_bin(self.config)
            self._plan = AngularBinPlan(ang_min, ang_max, self.config.scales.rweight, self.config.scales.resolution)
        return self._plan

    def count_pairs(self, main_catalog, *optional_catalog, progress: bool = False, max_workers=None,
                    mode: str = "nn", count_type_info: str | None = None, binned_second: bool | None = None
                    ) -> list[NormalisedCounts]:
        """Pair counts between the patches of two catalogs; omit `optional_catalog` for an
        autocorrelation.  `binned_second` states whether the second catalog is paired bin by bin
        (autocorrelate DR) or as a whole with every z-bin (crosscorrelate's unknown sample)."""
        if mode not in ("nn", "nk", "kn", "kk"):
            raise ValueError(f"invalid count mode '{mode}'")
        kappa1, kappa2 = mode[0] == "k", mode[1] == "k"
        if count_type_info is not None:
            logger.info("counting %s from patch pairs", count_type_info)
        auto = len(optional_catalog) == 0
        second = main_catalog if auto else optional_catalog[0]
        if binned_second is None:
            binned_second = auto
        engine = self.engine or get_default_engine()
        shard = self.shard or current_shard()
        uploads = self._uploads or _Uploads(engine)

        binning = _as_binning(self.config)
        plan = self._get_plan()
        ij = self.get_patch_id_pairs(auto=auto)
        # the "k" side of a scalar-field count carries kappa x weight per row (trees.py:270-301)
        has1, has2 = _has_kappa(main_catalog), _has_kappa(second)
        if kappa1 and kappa2 and not (has1 and has2):
            raise ValueError("missing required 'kappa' for both tree.")
        if kappa1 and not has1:
            raise ValueError("missing required 'kappa' for first tree.")
        if kappa2 and not has2:
            raise ValueError("missing required 'kappa' for second tree.")

        try:
            bins2 = binning if binned_second else None
            dev1 = uploads.get(main_catalog, binning, kappa1)
            dev2 = dev1 if (auto and kappa1 == kappa2) else uploads.get(second, bins2, kappa2)
            # the reported sums are always the plain sum of weights (`AngularTree.sum_weights`)
            sw1_all = (uploads.get(main_catalog, binning) if kappa1 else dev1).sum_weights()
            sw2_all = (uploads.get(second, bins2) if kappa2 else dev2).sum_weights()

            own = _own_pairs(shard, ij, main_catalog.get_num_records(), second.get_num_records(),
                             main_catalog.get_radii().data)
            hist = _count(engine, shard, count_type_info or ("auto" if auto else "cross"), dev1, dev2, ij, own, plan.r2)
        finally:
            if self._uploads is None:
                uploads.free()
        return self._package(hist, plan, binning, len(main_catalog), *ij, sw1_all, sw2_all, auto)

    @staticmethod
    def _package(hist, plan, binning, num_patches, pair_i, pair_j, sw1_all, sw2_all, auto) -> list[NormalisedCounts]:
        """sub-bin histograms of the patch pairs -> one `NormalisedCounts` per scale (`measurements.py:354-367`)"""
        num_bins = len(binning)
        counts = plan.finish(hist)  # (n_scales, n_pairs, n_bins)
        sum_weights1 = np.zeros((num_bins, num_patches))
        sum_weights2 = np.zeros((num_bins, num_patches))
        ids1, ids2 = np.unique(pair_i), np.unique(pair_j)
        sum_weights1[:, ids1] = sw1_all[:, ids1]
        # an unbinned second catalog reports the same total for every z-bin (trees.py:600-601)
        sum_weights2[:, ids2] = sw2_all[:, ids2] if sw2_all.shape[0] == num_bins else np.broadcast_to(
            sw2_all[0, ids2], (num_bins, len(ids2)))

        result = []
        sum_weights = PatchedSumWeights(binning, sum_weights1, sum_weights2, auto=auto)
        for s in range(plan.n_scales):
            patched = PatchedCounts.zeros(binning, num_patches, auto=auto)
            vals = counts[s]  # (n_pairs, n_bins)
            if auto:
                vals = np.where((pair_i == pair_j)[:, None], vals * 0.5, vals)  # pairs counted twice
            patched.counts[:, pair_i, pair_j] = vals.T
            result.append(NormalisedCounts(patched, sum_weights))
        return result

    def count_pairs_fused(self, main_a, main_b, second, *, count_type_info: tuple[str, str] = ("DD", "RD")
                          ) -> tuple[list[NormalisedCounts], list[NormalisedCounts]]:
        """`count_pairs(main_a, second)` and `count_pairs(main_b, second)` of a cross-correlation in ONE pass of
        the engine (`yawb_count2`: the two z-binned catalogs share one sky-cell index, every register tile of
        the unbinned `second` catalog is set up once).  Same results as the two separate calls."""
        logger.info("counting %s and %s from patch pairs", *count_type_info)
        engine = self.engine or get_default_engine()
        shard = self.shard or current_shard()
        uploads = self._uploads or _Uploads(engine)
        binning = _as_binning(self.config)
        plan = self._get_plan()
        ij = self.get_patch_id_pairs(auto=False)
        try:
            dev_a, dev_b = uploads.get(main_a, binning), uploads.get(main_b, binning)
            dev2 = uploads.get(second, None)
            sw_a, sw_b, sw2 = dev_a.sum_weights(), dev_b.sum_weights(), dev2.sum_weights()
            larger = main_a if sum(main_a.get_num_records()) >= sum(main_b.get_num_records()) else main_b
            own = _own_pairs(shard, ij, larger.get_num_records(), second.get_num_records(), larger.get_radii().data)
            hist_a, hist_b = _count(engine, shard, "+".join(count_type_info), (dev_a, dev_b), dev2, ij, own, plan.r2)
        finally:
            if self._uploads is None:
                uploads.free()
        return (self._package(hist_a, plan, binning, len(main_a), *ij, sw_a, sw2, False),
                self._package(hist_b, plan, binning, len(main_a), *ij, sw_b, sw2, False))

    def count_pairs_optional(self, main_catalog, *optional_catalog, **kwargs):
        if any(cat is None for cat in (main_catalog, *optional_catalog)):
            return [None for _ in range(self.config.scales.num_scales)]
        return self.count_pairs(main_catalog, *optional_catalog, **kwargs)


    def count_scalar_pairs(self, main_catalog, *optional_catalog, progress: bool = False, max_workers=None,
                           mode: str = "nn", count_type_info: str | None = None,
                           binned_second: bool | None = None) -> list[NormalisedScalarCounts]:
        """Scalar-field pair counts: one pass in `mode` ("kn" / "kk"), one in "nn" over the same patch
        pairs, combined per scale (`PatchLinkage.count_scalar_pairs`, `measurements.py:394-429`)."""
        own_uploads = self._uploads is None
        if own_uploads:
            self._uploads = _Uploads(self.engine or get_default_engine())
        try:
            counts = {
                m: self.count_pairs(main_catalog, *optional_catalog, mode=m, count_type_info=count_type_info,
                                    binned_second=binned_second)
                for m in (mode, "nn")
            }
        finally:
            if own_uploads:
                self._uploads.free()
                self._uploads = None
        return [NormalisedScalarCounts(kk.counts, nn.counts) for kk, nn in zip(counts[mode], counts["nn"])]


# ---- the count step of every measurement --------------------------------------------------------------
def _own_pairs(shard: Shard, ij, n1_per_patch, n2_per_patch, radii1) -> np.ndarray:
    """rows of the pair list `ij = (pair_i, pair_j)` counted by this rank (all of them without sharding)"""
    if not shard.active:
        return np.arange(len(ij[0]))
    costs = pair_costs(*ij, n1_per_patch, n2_per_patch, radii1=np.asarray(radii1))
    return assign_pairs_lpt(costs, shard.world_size)[shard.rank]


def _share_plan(engine, shard: Shard | None, catalogs, counts, footprint=None):
    """The `SharePlan` of a call on an `EngineGroup` (None on a single engine).  `catalogs`: the catalogs of the
    linkage (the largest gives the patch centres and radii, as for the links); `counts`: `(pair_i, pair_j, first,
    second)` of every pair count of the call, `pair_j` the patches of the second catalog, `first` / `second` rows per
    patch; `footprint`: a `_Footprint` of the call's uploads.

    When the predicted footprint of the call exceeds the memory of an engine (`Engine.memory_available`), the call
    is planned in passes (`sharding.plan_passes`) and `_PassesNeeded` hands them to `_in_passes`, before anything is
    uploaded; while a pass runs, this returns that pass's plan."""
    from .engine import EngineGroup

    run = _current_run()
    if run is not None:
        return run.steps[run.k]
    group = isinstance(engine, EngineGroup)
    if (shard or current_shard()).active:
        if group:
            raise ValueError("an EngineGroup splits a call over the GPUs of one process; it cannot be combined with an "
                             "active shard (one process per GPU)")
        return None
    eng = engine if engine is not None else get_default_engine()
    members = eng.engines if group else [eng]
    ref = max(catalogs, key=lambda c: tuple(c.get_num_records()))
    centers = AngularCoordinates(_coords_data(ref.get_centers())).to_3d()
    counts = [(pi, pj, np.asarray(n1, dtype=np.float64), np.asarray(n2, dtype=np.float64)) for pi, pj, n1, n2 in counts]
    radii = _coords_data(ref.get_radii())
    if footprint is None or not all(hasattr(e, "memory_available") for e in members):
        return plan_shares(counts, radii, centers, len(members)) if group else None
    fp = footprint.bind(members[0], counts, bool(getattr(eng, "device_digitize", False)))
    steps = plan_passes(counts, radii, centers, fp, [e.memory_available() for e in members])
    if len(steps) == 1:
        # the default limit counted the engines' cached catalogs as obtainable: drop the ones this call does not use
        # (least recently used first) until its footprint fits
        for d, e in enumerate(members):
            if hasattr(e, "make_room"):
                e.make_room(fp(steps[0].keep[d].astype(bool)), catalogs)
        return steps[0] if group else None
    raise _PassesNeeded(eng, steps, default_limit=any(e.memory_limit is None for e in members))


class _Footprint:
    """The device memory model of one call: its uploads, as `_Uploads` makes them (with a second-role row mask and
    both indexes), the fused first-role indexes of `Engine.count2`, and the workspace of every count."""

    def __init__(self, links: "PatchLinkage") -> None:
        r2 = links._get_plan().r2
        self.n_bins, self.n_edges = r2.shape
        self.uploads: list[tuple[np.ndarray, int, dict]] = []
        self.fused: list[np.ndarray] = []
        self.n_labels = 1

    def upload(self, catalog, binning: Binning | None, kappa: bool = False):
        # how binned ids travel depends on the engine (`bind`): "binned" stands for byte / int32 ids or raw redshifts
        zbin = None if binning is None else "binned" if len(binning) <= 254 else "i32"
        self.uploads.append((_rows(catalog), len(binning) if binning is not None else 1,
                             dict(weighted=bool(catalog.has_weights) or kappa, zbin=zbin)))
        return self

    def labelled(self, catalogs, binning: Binning | None = None):
        catalogs = list(catalogs)
        n_ids = len(catalogs) * (len(binning) if binning is not None else 1)
        self.uploads.append((np.sum([_rows(c) for c in catalogs], axis=0), n_ids,
                             dict(weighted=bool(catalogs[0].has_weights), zbin="u8" if n_ids <= 254 else "i32",
                                  labelled=binning is not None)))
        self.n_labels = max(self.n_labels, len(catalogs))
        return self

    def fuse(self, *catalogs):
        self.fused.append(np.sum([_rows(c) for c in catalogs], axis=0))
        return self

    def bind(self, engine, counts, device_digitize: bool):
        """`footprint(keep)` for `sharding.plan_passes`: device bytes of a pass keeping the patches `keep`.
        `device_digitize`: the engine ships raw redshifts (`_prepare_for`)"""
        n_edges = self.n_edges
        uploads = [(rows, nb, dict(kw, zbin=("z" if device_digitize else "u8") if kw["zbin"] == "binned" else kw["zbin"]))
                   for rows, nb, kw in self.uploads]
        b2 = max(nb for _, nb, _ in uploads) if uploads else 1

        def footprint(keep: np.ndarray) -> int:
            n_patch = len(keep)
            total = sum(engine.footprint(int(rows[keep].sum()), n_patch, nb, mask=True, **kw)
                        for rows, nb, kw in uploads)
            total += sum(engine.footprint(int(rows[keep].sum()), n_patch, self.n_bins, weighted=True, second=False,
                                          upload=False) for rows in self.fused)
            for pi, pj, _, n2 in counts:  # tiles of a second patch: at most rows / 256 + one per segment
                pj = np.asarray(pj)
                mine = keep[pj]
                n_items = int(np.sum(np.ceil(n2[pj[mine]] / 256.0) + b2))
                total += engine.count_footprint(n_items, int(mine.sum()), self.n_bins, n_edges,
                                                n_blocks=2 * self.n_labels, weighted=True)
            return total

        return footprint


class _PassesNeeded(Exception):
    """raised by `_share_plan` before anything is uploaded: the call does not fit and runs in these passes"""

    def __init__(self, engine, steps, default_limit: bool) -> None:
        super().__init__(f"{len(steps)} passes")
        self.engine, self.steps, self.default_limit = engine, steps, default_limit


_pass_state = threading.local()


def _current_run():
    return getattr(_pass_state, "run", None)


class _PassRun:
    """One call counted in passes.  The body of a measurement function runs once per pass and makes the same
    requests in the same order every time, so the n-th count of a pass adds to the n-th count of the passes before
    (histograms placed in the full pair axis, summed in pass order; counters and times summed), and the n-th sums of
    weights take every patch from the first pass that kept it.  What the last pass returns is the whole call."""

    def __init__(self, steps) -> None:
        self.steps = steps
        self.k = 0
        self.prepared: dict = {}  # host arrays of every catalog, prepared once for all passes
        self.lock = threading.Lock()
        self._counts: list = []
        self._sums: list = []
        self._nc = self._ns = 0

    def begin(self, k: int) -> None:
        self.k, self._nc, self._ns = k, 0, 0

    def counts(self, hists: list, stats: dict) -> tuple[list, dict]:
        i, self._nc = self._nc, self._nc + 1
        if i == len(self._counts):
            self._counts.append(([h.copy() for h in hists], dict(stats)))
        else:
            acc, st = self._counts[i]
            for a, h in zip(acc, hists):
                a += h
            for key, v in stats.items():
                st[key] = st.get(key, 0) + v
        acc, st = self._counts[i]
        st["passes"] = self.k + 1
        return [a.copy() for a in acc], dict(st)

    def sums(self, sw, kept: np.ndarray):
        i, self._ns = self._ns, self._ns + 1
        if i == len(self._sums):
            self._sums.append((sw.copy(), kept.copy()))
        else:
            acc, done = self._sums[i]
            take = kept & ~done
            acc[:, take] = sw[:, take]
            done |= take
        return self._sums[i][0].copy()


def _in_passes(fn):
    """A measurement function that runs in passes when `_share_plan` finds that its call does not fit: the body runs
    once per pass on an `EngineGroup` (a single engine is wrapped in a group of one), every pass uploads its share of
    the catalogs and frees it before the next one, and the allocator returns its parked blocks to the driver so the
    next pass starts from the same memory.  A call that fits runs the body once, as it is."""

    @functools.wraps(fn)
    def call(*args, **kw):
        from .engine import EngineGroup

        try:
            return fn(*args, **kw)
        except _PassesNeeded as need:
            engine, steps, default_limit = need.engine, need.steps, need.default_limit
        group = engine if isinstance(engine, EngineGroup) else EngineGroup([engine])
        run = _PassRun(steps)
        try:
            if default_limit:  # the default limit counts the memory of the engine's cached catalogs as available
                group._map(lambda d, e: e.cache_clear() if hasattr(e, "cache_clear") else None)
            _pass_state.run = run
            # blocks parked by earlier calls go back to the driver first, so every pass starts from the same level
            group._map(lambda d, e: e.memory_release() if hasattr(e, "memory_release") else None)
            for k in range(len(steps)):
                run.begin(k)
                result = fn(*args, **{**kw, "engine": group})
                group._map(lambda d, e: e.memory_release() if hasattr(e, "memory_release") else None)
        finally:
            _pass_state.run = None
            if group is not engine:
                group.close()
        return result

    return call


def _rows(catalog):
    return np.asarray(catalog.get_num_records(), dtype=np.float64)


def _reduce(engine, shard: Shard, hist: np.ndarray, own: np.ndarray, n_pairs: int, *, labelled: bool) -> np.ndarray:
    """the histograms of the pairs `own` placed into the full pair axis (behind the leading label axis if `labelled`)
    and summed over the ranks"""
    if not shard.active:
        return hist
    axis = 1 if labelled else 0
    full = np.zeros((*hist.shape[:axis], n_pairs, *hist.shape[axis + 1:]), dtype=hist.dtype)
    full[(slice(None),) * axis + (own,)] = hist
    device = getattr(engine, "device", None)
    return shard.reduce_to_root(full, device=None if device is None else f"cuda:{device}")


def _count(engine, shard: Shard, tag: str, first, second, ij, own: np.ndarray, r2: np.ndarray, *,
           swap: bool = False, labels: bool = False):
    """`first` (a device catalog, or a tuple of two counted in one pass by `Engine.count2`) against `second` over the
    rows `own` of the pair list `ij` (`swap`: `pair_i` and `pair_j` exchanged), statistics recorded under `tag`.
    Returns the histogram of each first catalog, float if any catalog is weighted, summed over the ranks."""
    pi, pj = ij[0][own], ij[1][own]
    if swap:
        pi, pj = pj, pi
    kw = dict(labels=True) if labels else {}
    fused = isinstance(first, tuple)
    if fused:
        *outs, stats = engine.count2(*first, second, pi, pj, r2, **kw)
    else:
        *out, stats = engine.count(first, second, pi, pj, r2, **kw)
        outs = [out]
    weighted = any(c.weighted for c in (*(first if fused else (first,)), second))
    labelled = labels or getattr(second, "n_labels", None) is not None  # a leading label axis
    hists = [_reduce(engine, shard, out[1] if weighted else out[0], own, len(ij[0]), labelled=labelled) for out in outs]
    run = _current_run()
    if run is not None:
        hists, stats = run.counts(hists, stats)
    _last_stats[tag] = stats
    return tuple(hists) if fused else hists[0]


def _fuse(engine, reference, ref_rand) -> bool:
    """whether the reference sample and its randoms are counted against a second catalog in one pass
    (`Engine.count2`): they share patches, z-bins and thresholds, unless only one of them carries weights"""
    return (ref_rand is not None and bool(reference.has_weights) == bool(ref_rand.has_weights)
            and hasattr(engine, "count2"))


def _has_kappa(catalog) -> bool:
    has = getattr(catalog, "has_kappa", None)
    if has is not None:
        return bool(has)
    return all(p.has_kappa for p in catalog.values())


# ---- public API -----------------------------------------------------------------------------------------
def _ensure_unique_catalogs(*catalogs) -> None:
    cats = [c for c in catalogs if c is not None]
    paths = {str(getattr(c, "cache_directory", id(c))) for c in cats}
    if len(paths) != len(cats):
        raise ValueError("each catalog must have a separate cache directory to avoid interference.")


@_in_passes
def autocorrelate(config, data, random, *, count_rr: bool = True, progress: bool = False, max_workers=None,
                  engine=None, shard: Shard | None = None) -> list[CorrFunc]:
    """Angular autocorrelation pair counts (DD, DR, optional RR) of a z-binned sample.
    Signature and result layout of `yaw.autocorrelate` (`measurements.py:455-525`);
    `progress` / `max_workers` are accepted and ignored."""
    _ensure_unique_catalogs(data, random)
    links = PatchLinkage.from_catalogs(config, data, random, engine=engine, shard=shard)
    auto_ij, cross_ij = links.get_patch_id_pairs(auto=True), links.get_patch_id_pairs(auto=False)
    nd, nr = _rows(data), _rows(random)
    binning = _as_binning(config)
    plan = _share_plan(engine, shard, (data, random), [(*auto_ij, nd, nd), (*cross_ij, nd, nr)]
                       + ([(*auto_ij, nr, nr)] if count_rr else []),
                       _Footprint(links).upload(data, binning).upload(random, binning))
    links._uploads = _Uploads(engine or get_default_engine(), plan)
    _last_stats.clear()
    try:
        links._uploads.enqueue(((data, binning), (random, binning)))
        DD = links.count_pairs(data, count_type_info="DD")
        DR = links.count_pairs(data, random, count_type_info="DR", binned_second=True)
        RR = links.count_pairs_optional(random if count_rr else None, count_type_info="RR")
    finally:
        links._uploads.free()
        links._uploads = None
    return [CorrFunc(dd, dr, None, rr) for dd, dr, rr in zip(DD, DR, RR)]


@_in_passes
def crosscorrelate(config, reference, unknown, *, ref_rand=None, unk_rand=None, progress: bool = False,
                   max_workers=None, engine=None, shard: Shard | None = None) -> list[CorrFunc]:
    """Angular cross-correlation pair counts (DD and DR / RD / RR as randoms allow) between the
    z-binned reference sample and the unbinned unknown sample.  Signature and result layout of
    `yaw.crosscorrelate` (`measurements.py:529-628`)."""
    _ensure_unique_catalogs(reference, unknown, ref_rand, unk_rand)
    count_dr = unk_rand is not None
    count_rd = ref_rand is not None
    if not count_dr and not count_rd:
        raise ValueError("at least one random dataset must be provided")
    randoms = [cat for cat in (ref_rand, unk_rand) if cat is not None]

    links = PatchLinkage.from_catalogs(config, reference, unknown, *randoms, engine=engine, shard=shard)
    ij = links.get_patch_id_pairs(auto=False)
    binning = _as_binning(config)
    fp = _Footprint(links).upload(reference, binning).upload(unknown, None)
    for cat, bins in ((ref_rand, binning), (unk_rand, None)):
        if cat is not None:
            fp.upload(cat, bins)
    if ref_rand is not None:
        fp.fuse(reference, ref_rand)
    plan = _share_plan(engine, shard, (reference, unknown, *randoms),
                       [(*ij, _rows(c1), _rows(c2)) for c1 in (reference, ref_rand) if c1 is not None
                        for c2 in (unknown, unk_rand) if c2 is not None], fp)
    links._uploads = _Uploads(engine or get_default_engine(), plan)
    _last_stats.clear()
    kw = dict(binned_second=False)
    try:
        # uploads are asynchronous: enqueue every catalog first, the data samples before the randoms, and
        # count in the order in which the inputs become complete -- DD gets the GPU going a few ms into the
        # transfer, RD / DR follow, and only RR waits for the last catalog (same schedule as
        # `pipeline.count_cross_pipelined`)
        links._uploads.enqueue(((reference, binning), (unknown, None), (ref_rand, binning), (unk_rand, None)))
        if _fuse(links.engine or get_default_engine(), reference, ref_rand):
            DD, RD = links.count_pairs_fused(reference, ref_rand, unknown, count_type_info=("DD", "RD"))
            if unk_rand is not None:
                DR, RR = links.count_pairs_fused(reference, ref_rand, unk_rand, count_type_info=("DR", "RR"))
            else:
                DR = RR = [None for _ in range(config.scales.num_scales)]
        else:
            DD = links.count_pairs(reference, unknown, count_type_info="DD", **kw)
            RD = links.count_pairs_optional(ref_rand, unknown, count_type_info="RD", **kw)
            DR = links.count_pairs_optional(reference, unk_rand, count_type_info="DR", **kw)
            RR = links.count_pairs_optional(ref_rand, unk_rand, count_type_info="RR", **kw)
    finally:
        links._uploads.free()
        links._uploads = None
    return [CorrFunc(dd, dr, rd, rr) for dd, dr, rd, rr in zip(DD, DR, RD, RR)]


@_in_passes
def crosscorrelate_tomographic(config, reference, unknowns, *, ref_rand=None, unk_rand=None, progress: bool = False,
                               max_workers=None, engine=None, shard: Shard | None = None) -> list[list[CorrFunc]]:
    """`crosscorrelate` of the reference sample with every tomographic bin of the unknown sample in one pass:
    `result[i]` is `crosscorrelate(config, reference, unknowns[i], ref_rand=ref_rand, unk_rand=<randoms of bin
    i>)`, the loop of the reference CLI's `CrossCorrTask` (`cli/tasks.py:536-550`) as one call.

    `unknowns`: 1 to 254 catalogs, one per bin, all with weights or all without.  `unk_rand`: None, one catalog
    shared by every bin, or a sequence of one catalog per bin.  The bins travel to the device as ONE labelled
    catalog (`YAWB_FLAG_SECOND_LABELS`), per-bin randoms likewise, and stay in the engine's cache like single
    catalogs; every count runs once over the union of the bins' patch-pair lists, and each bin is packaged from its
    own linkage.  A shared `unk_rand` is counted once
    (DR and RR) for all bins.  Everything a per-bin call would raise is raised before any counting.
    `progress` / `max_workers` are accepted and ignored."""
    unknowns, rands, shared = _check_tomographic(unknowns, unk_rand, "unknowns", "unk_rand", (reference, ref_rand))
    if ref_rand is None and unk_rand is None:
        raise ValueError("at least one random dataset must be provided")
    _check_tomographic_weights(unknowns, rands, shared)
    # the linkage of every bin, exactly as its own call would build it: the largest catalog decides the links
    links = [PatchLinkage.from_catalogs(config, reference, unknown, *[c for c in (ref_rand, rand) if c is not None],
                                        engine=engine, shard=shard) for unknown, rand in zip(unknowns, rands)]
    bin_pairs = [lk.get_patch_id_pairs(auto=False) for lk in links]
    ij, bin_rows = _union_pairs(bin_pairs)

    eng = engine or get_default_engine()
    shard = shard or current_shard()
    binning = _as_binning(config)
    plan = links[0]._get_plan()
    num_patches = len(reference)
    _last_stats.clear()
    uploads = _Uploads(eng)

    # a pair's cost sums the rows of every bin
    first = reference if ref_rand is None or sum(reference.get_num_records()) >= sum(ref_rand.get_num_records()) \
        else ref_rand
    own = _own_pairs(shard, ij, first.get_num_records(), np.sum([u.get_num_records() for u in unknowns], axis=0),
                     first.get_radii().data)
    n_unk = np.sum([_rows(u) for u in unknowns], axis=0)
    n_ur = None if unk_rand is None else _rows(unk_rand) if shared else np.sum([_rows(r) for r in rands], axis=0)
    fp = _Footprint(links[0]).upload(reference, binning).labelled(unknowns)
    if ref_rand is not None:
        fp.upload(ref_rand, binning).fuse(reference, ref_rand)
    if unk_rand is not None:
        fp.upload(unk_rand, None) if shared else fp.labelled(rands)
    uploads.plan = _share_plan(engine, shard, (reference, *unknowns, *[c for c in (ref_rand, *rands) if c is not None]),
                               [(*ij, _rows(c1), n2) for c1 in (reference, ref_rand) if c1 is not None
                                for n2 in (n_unk, n_ur) if n2 is not None], fp)
    fuse = _fuse(eng, reference, ref_rand)
    counts: dict[str, tuple] = {}
    try:
        uploads.enqueue(((reference, binning), (ref_rand, binning), (unk_rand if shared else None, None)))
        dev_ref = uploads.get(reference, binning)
        dev_rr = uploads.get(ref_rand, binning) if ref_rand is not None else None
        dev_unk = uploads.get_labelled(unknowns)
        dev_ur = None
        if unk_rand is not None:
            dev_ur = uploads.get(unk_rand, None) if shared else uploads.get_labelled(rands)
        # sums of weights with a leading label axis: (1, z-bins, patches) for the reference sample and its randoms,
        # (labels, 1, patches) for the unknown side
        sw_ref, sw_unk = dev_ref.sum_weights()[None], dev_unk.sum_weights()[:, None]
        sw_rr = dev_rr.sum_weights()[None] if dev_rr is not None else None
        sw_ur = dev_ur.sum_weights()[:, None] if dev_ur is not None else None
        for second, sw2, kinds in ((dev_unk, sw_unk, ("DD", "RD")), (dev_ur, sw_ur, ("DR", "RR"))):
            if second is None:
                continue
            if fuse:
                hists = _count(eng, shard, "+".join(kinds), (dev_ref, dev_rr), second, ij, own, plan.r2, labels=True)
            else:
                hists = [None if dev1 is None else _count(eng, shard, kind, dev1, second, ij, own, plan.r2, labels=True)
                         for kind, dev1 in zip(kinds, (dev_ref, dev_rr))]
            counts.update((kind, (h, sw1, sw2)) for kind, h, sw1 in zip(kinds, hists, (sw_ref, sw_rr)) if h is not None)
    finally:
        uploads.free()

    result = []
    for i, (pairs, rows) in enumerate(zip(bin_pairs, bin_rows)):
        DD, DR, RD, RR = (_package_bin(counts.get(kind), i, rows, pairs, False, plan, binning, num_patches)
                          for kind in ("DD", "DR", "RD", "RR"))
        result.append([CorrFunc(dd, dr, rd, rr) for dd, dr, rd, rr in zip(DD, DR, RD, RR)])
    return result


def _check_tomographic(bins, rand, bins_name: str, rand_name: str, others=(), *, rand_required: bool = False
                       ) -> tuple[list, list, bool]:
    """`bins`: 1 to 254 catalogs; `rand`: None (unless `rand_required`), one catalog shared by every bin or one per
    bin; no catalog twice among a bin, its randoms and `others`.  Returns (bins, randoms of every bin, shared)."""
    bins = list(bins)
    n_tomo = len(bins)
    if n_tomo == 0:
        raise ValueError(f"'{bins_name}' must hold at least one catalog")
    if n_tomo > 254:
        raise ValueError(f"at most 254 tomographic bins are supported (got {n_tomo})")
    per_bin = isinstance(rand, Sequence)
    rands = list(rand) if per_bin else [rand] * n_tomo
    if len(rands) != n_tomo:
        raise ValueError(f"'{rand_name}' holds {len(rands)} catalogs for {n_tomo} tomographic bins")
    if (per_bin or rand_required) and any(r is None for r in rands):
        raise ValueError(f"'{rand_name}' must hold a catalog for every bin")
    for b, r in zip(bins, rands):
        _ensure_unique_catalogs(*others, b, r)
    return bins, rands, rand is not None and not per_bin


def _check_tomographic_weights(bins, rands, shared: bool) -> None:
    """the bins, and per-bin randoms, travel as one labelled catalog each: all with weights or all without"""
    if len({bool(c.has_weights) for c in bins}) > 1:
        raise ValueError("the tomographic bins must all have weights or all have none")
    if not shared and rands[0] is not None and len({bool(c.has_weights) for c in rands}) > 1:
        raise ValueError("the per-bin randoms must all have weights or all have none")


def _union_pairs(bin_pairs) -> tuple[tuple[np.ndarray, np.ndarray], list[np.ndarray]]:
    """union of the bins' patch-pair lists (first appearance order) and, per bin, the rows of the union that make up
    its own list, in its order"""
    union: dict[tuple[int, int], int] = {}
    for pi, pj in bin_pairs:
        for pair in zip(pi.tolist(), pj.tolist()):
            union.setdefault(pair, len(union))
    union_ij = np.array(list(union), dtype=np.int32).reshape(-1, 2)
    rows = [np.array([union[p] for p in zip(pi.tolist(), pj.tolist())], dtype=np.int64) for pi, pj in bin_pairs]
    return (union_ij[:, 0], union_ij[:, 1]), rows


def _package_bin(count, i: int, rows: np.ndarray, pairs, auto: bool, plan, binning, num_patches: int
                 ) -> list[NormalisedCounts | None]:
    """bin `i`'s share of a count over the union of the bins' pair lists: `rows` of the union are its own `pairs`.
    `count`: (histogram, sums of weights of the first and second catalog), each with a leading axis of one entry per
    bin or one shared by every bin; None: a count not made."""
    if count is None:
        return [None] * plan.n_scales
    hist, sw1, sw2 = (x[i if len(x) > 1 else 0] for x in count)
    return PatchLinkage._package(hist[rows], plan, binning, num_patches, *pairs, sw1, sw2, auto)


@_in_passes
def autocorrelate_tomographic(config, data, random, *, count_rr: bool = True, progress: bool = False,
                              max_workers=None, engine=None, shard: Shard | None = None) -> list[list[CorrFunc]]:
    """`autocorrelate` of every tomographic bin of a sample in one pass: `result[i]` is `autocorrelate(config,
    data[i], <randoms of bin i>, count_rr=count_rr)`, the per-bin unknown autocorrelation of the reference CLI
    (`auto_unk`) as one call.

    `data`: 1 to 254 z-binned catalogs, one per bin, all with weights or all without.  `random`: one catalog shared
    by every bin, or a sequence of one catalog per bin.  The bins travel to the device as ONE catalog with binned
    labels (id = bin * B + z-bin, `Engine.upload_catalog(n_labels=)`), per-bin randoms likewise.  DD is one
    labelled autocount; DR one labelled count, or with shared randoms one count with the randoms as the first
    catalog (pair counts are symmetric); RR one count, with shared randoms a plain z-binned autocount for all bins.
    Every count runs once over the union of the bins' patch-pair lists, and each bin is packaged from its own
    linkage.  Everything a per-bin call would raise is raised before any counting.  The labelled uploads stay in
    the engine's cache like single catalogs.  `progress` / `max_workers` are accepted and ignored."""
    data, rands, shared = _check_tomographic(data, random, "data", "random", rand_required=True)
    n_tomo = len(data)
    # the linkage of every bin, exactly as its own call would build it
    links = [PatchLinkage.from_catalogs(config, d, r, engine=engine, shard=shard) for d, r in zip(data, rands)]
    if not all(c.has_redshifts for c in (*data, *rands)):
        raise ValueError("patch has no 'redshifts' attached")
    _check_tomographic_weights(data, rands, shared)
    binning = _as_binning(config)
    n_zbins = len(binning)
    if n_tomo * n_zbins > 4096:
        raise ValueError(f"bins x z-bins must not exceed 4096 (got {n_tomo} x {n_zbins})")

    auto_pairs = [lk.get_patch_id_pairs(auto=True) for lk in links]
    cross_pairs = [lk.get_patch_id_pairs(auto=False) for lk in links]
    auto_ij, auto_rows = _union_pairs(auto_pairs)
    cross_ij, cross_rows = _union_pairs(cross_pairs)

    eng = engine or get_default_engine()
    shard = shard or current_shard()
    plan = links[0]._get_plan()
    num_patches = len(data[0])
    _last_stats.clear()
    uploads = _Uploads(eng)

    n_data = np.sum([d.get_num_records() for d in data], axis=0)
    n_rand = rands[0].get_num_records() if shared else np.sum([r.get_num_records() for r in rands], axis=0)
    radii = rands[0].get_radii().data
    own_auto_dd = _own_pairs(shard, auto_ij, n_data, n_data, radii)
    own_cross = _own_pairs(shard, cross_ij, n_data, n_rand, radii)
    own_auto_rr = _own_pairs(shard, auto_ij, n_rand, n_rand, radii)
    # with shared randoms DR is counted with the pair lists swapped: the data sample is the second catalog
    dr_pairs = (cross_ij[1], cross_ij[0], n_rand, n_data) if shared else (*cross_ij, n_data, n_rand)
    fp = _Footprint(links[0]).labelled(data, binning)
    fp.upload(random, binning) if shared else fp.labelled(rands, binning)
    uploads.plan = _share_plan(engine, shard, (*data, *rands), [(*auto_ij, n_data, n_data), dr_pairs]
                               + ([(*auto_ij, n_rand, n_rand)] if count_rr else []), fp)

    counts: dict[str, tuple] = {}
    try:
        dev_d = uploads.get_labelled(data, binning)
        dev_r = uploads.get(random, binning) if shared else uploads.get_labelled(rands, binning)
        sw_d = dev_d.sum_weights().reshape(n_tomo, n_zbins, num_patches)
        sw_r = dev_r.sum_weights().reshape(-1, n_zbins, num_patches)
        dd = _count(eng, shard, "DD", dev_d, dev_d, auto_ij, own_auto_dd, plan.r2)
        if shared:  # the randoms as the first catalog, every bin's rows against their z-bin: pair lists swapped
            dr = _count(eng, shard, "DR", dev_r, dev_d, cross_ij, own_cross, plan.r2, swap=True)
        else:
            dr = _count(eng, shard, "DR", dev_d, dev_r, cross_ij, own_cross, plan.r2)
        counts.update(DD=(dd, sw_d, sw_d), DR=(dr, sw_d, sw_r))
        if count_rr:
            rr = _count(eng, shard, "RR", dev_r, dev_r, auto_ij, own_auto_rr, plan.r2)
            counts["RR"] = (rr[None] if shared else rr, sw_r, sw_r)
    finally:
        uploads.free()

    result = []
    for i in range(n_tomo):
        DD = _package_bin(counts["DD"], i, auto_rows[i], auto_pairs[i], True, plan, binning, num_patches)
        DR = _package_bin(counts["DR"], i, cross_rows[i], cross_pairs[i], False, plan, binning, num_patches)
        RR = _package_bin(counts.get("RR"), i, auto_rows[i], auto_pairs[i], True, plan, binning, num_patches)
        result.append([CorrFunc(dd, dr, None, rr) for dd, dr, rr in zip(DD, DR, RR)])
    return result

# ---- scalar-field correlations (NK / KK) ----------------------------------------------------------------
def compute_scalar_normalisation(catalog, binning: Binning, *, engine=None, uploads: "_Uploads | None" = None
                                 ) -> NormalisedScalarCounts:
    """Mean-kappa correction per patch and z-bin: sum(kappa x w) and sum(w) on the diagonal of two
    `PatchedCounts` (`compute_scalar_normalisation`, `measurements.py:634-648`).  Both sums are the
    per-(bin, patch) weight sums the device already computes for its catalogs."""
    from .engine import EngineGroup

    own = uploads is None
    if own and isinstance(engine, EngineGroup):  # per-patch sums need no share of the devices
        engine = engine.engines[0]
    uploads = uploads or _Uploads(engine or get_default_engine())
    try:
        num_bins, num_patches = len(binning), len(catalog)
        sum_kappa = np.zeros((num_bins, num_patches, num_patches))
        sum_weights = np.zeros_like(sum_kappa)
        diag = np.arange(num_patches)
        sum_kappa[:, diag, diag] = uploads.get(catalog, binning, True).sum_weights()
        sum_weights[:, diag, diag] = uploads.get(catalog, binning).sum_weights()
    finally:
        if own:
            uploads.free()
    return NormalisedScalarCounts(PatchedCounts(binning, sum_kappa, auto=False),
                                  PatchedCounts(binning, sum_weights, auto=False))


@_in_passes
def autocorrelate_scalar(config, data, *, progress: bool = False, max_workers=None, engine=None,
                         shard: Shard | None = None) -> list[ScalarCorrFunc]:
    """Angular autocorrelation of a scalar field in z-bins: KK and NN counts of the data sample.
    Signature and result layout of `yaw.autocorrelate_scalar` (`measurements.py:651-705`)."""
    links = PatchLinkage.from_catalogs(config, data, engine=engine, shard=shard)
    nd = _rows(data)
    binning = _as_binning(config)
    plan = _share_plan(engine, shard, (data,), [(*links.get_patch_id_pairs(auto=True), nd, nd)],
                       _Footprint(links).upload(data, binning, kappa=True).upload(data, binning))
    links._uploads = _Uploads(engine or get_default_engine(), plan)
    _last_stats.clear()
    try:
        DD = links.count_scalar_pairs(data, mode="kk", count_type_info="DD")
    finally:
        links._uploads.free()
        links._uploads = None
    return [ScalarCorrFunc(dd) for dd in DD]


@_in_passes
def crosscorrelate_scalar(config, reference, unknown, *, unk_rand=None, progress: bool = False,
                          max_workers=None, engine=None, shard: Shard | None = None) -> list[ScalarCorrFunc]:
    """Angular cross-correlation between a z-binned scalar-field sample (`reference`, carries
    `kappa`) and the unbinned `unknown` sample: KN and NN counts for DD and, with `unk_rand`,
    for DR; without it DR is the per-patch mean-kappa normalisation.  Signature and result layout
    of `yaw.crosscorrelate_scalar` (`measurements.py:708-794`)."""
    _ensure_unique_catalogs(reference, unknown, unk_rand)
    randoms = [unk_rand] if unk_rand is not None else []
    links = PatchLinkage.from_catalogs(config, reference, unknown, *randoms, engine=engine, shard=shard)
    ij = links.get_patch_id_pairs(auto=False)
    binning = _as_binning(config)
    fp = _Footprint(links).upload(reference, binning, kappa=True).upload(reference, binning)
    for cat in (unknown, *randoms):
        fp.upload(cat, None)
    plan = _share_plan(engine, shard, (reference, unknown, *randoms),
                       [(*ij, _rows(reference), _rows(c2)) for c2 in (unknown, *randoms)], fp)
    links._uploads = _Uploads(engine or get_default_engine(), plan)
    _last_stats.clear()
    kw = dict(binned_second=False, mode="kn")
    try:
        DD = links.count_scalar_pairs(reference, unknown, count_type_info="DD", **kw)
        if unk_rand is None:
            DR = [compute_scalar_normalisation(reference, _as_binning(config), uploads=links._uploads)] * len(DD)
        else:
            DR = links.count_scalar_pairs(reference, unk_rand, count_type_info="DR", **kw)
    finally:
        links._uploads.free()
        links._uploads = None
    return [ScalarCorrFunc(dd, dr) for dd, dr in zip(DD, DR)]
