"""
Thin object wrappers over the C ABI: `Engine` (one context on one GPU),
`DeviceCatalog` (one patch-partitioned catalog resident in HBM) and
`EngineGroup` (several engines driven from one process, each holding its share of
a measurement's catalogs).

These are the B200 counterparts of the reference's worker pool
(`src/yaw/utils/parallel.py:318-343`) and of its per-patch `BinnedTrees` cache
(`src/yaw/catalog/trees.py:432-601`).  All arithmetic happens in libyawb.so.
"""

from __future__ import annotations

import ctypes
import os
import weakref
from concurrent.futures import ThreadPoolExecutor
from ctypes import byref, c_double, c_int, c_int64, c_void_p

import numpy as np

from . import _lib


def _ptr(a: np.ndarray | None):
    return None if a is None else a.ctypes.data_as(c_void_p)


def _pairs_and_edges(pair_i, pair_j, r2_edges, n_bins: int) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """the pair lists as contiguous int32 and `r2_edges` as contiguous `(n_bins, n_edges)` doubles (one row of
    thresholds stands for every z-bin)"""
    pair_i = np.ascontiguousarray(pair_i, dtype=np.int32)
    pair_j = np.ascontiguousarray(pair_j, dtype=np.int32)
    r2_edges = np.ascontiguousarray(r2_edges, dtype=np.float64)
    if r2_edges.ndim == 1:
        r2_edges = np.ascontiguousarray(np.broadcast_to(r2_edges, (n_bins, len(r2_edges))))
    if r2_edges.shape[0] != n_bins:
        raise ValueError(f"r2_edges must have shape (n_bins={n_bins}, n_edges)")
    return pair_i, pair_j, r2_edges


class DeviceCatalog:
    """Handle of a catalog uploaded with `Engine.upload_catalog`."""

    def __init__(self, engine: "Engine", handle: c_void_p, n_patch: int, n_bins: int, binned: bool, weighted: bool):
        self.engine = engine
        self._h = handle
        self.n_patch = n_patch
        self.n_bins = n_bins
        self.binned = binned
        self.weighted = weighted
        self.n_labels = None  # binned labels (`Engine.upload_catalog(n_labels=)`): id = label * (n_bins // n_labels) + z-bin

    def sum_weights(self) -> np.ndarray:
        """`(n_bins, n_patch)` sum of weights (row counts if unweighted)."""
        out = np.empty((self.n_bins, self.n_patch), dtype=np.float64)
        _lib.check(self.engine.lib.yawb_sum_weights(self._h, _ptr(out)))
        return out

    def patch_metadata(self) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """`(center_xyz (n_patch, 3), radius (n_patch,) in radian, num_records (n_patch,))` computed on the device
        from the uploaded rows: the quantities of the reference's `Metadata.compute`
        (`src/yaw/catalog/patch.py:104-147`; centres agree with numpy's to ~1e-15, the sums run in another order)."""
        center = np.empty((self.n_patch, 3), dtype=np.float64)
        chord = np.empty(self.n_patch, dtype=np.float64)
        num = np.empty(self.n_patch, dtype=np.int64)
        _lib.check(self.engine.lib.yawb_patch_metadata(self._h, _ptr(center), _ptr(chord), _ptr(num)))
        return center, 2.0 * np.arcsin(np.minimum(chord / 2.0, 1.0)), num

    def set_second_rows(self, mask: np.ndarray | None) -> None:
        """Rows of the second-role index (`yawb_catalog_set_second_rows`): one byte per uploaded row (for a partial
        upload the rows of the kept patches, in patch order), 0 = left out; None clears the mask.  The first role,
        `sum_weights` and `info` keep every row."""
        if mask is not None:
            mask = np.ascontiguousarray(mask, dtype=np.uint8)
            n_rows = self._n_uploaded
            if len(mask) != n_rows:
                raise ValueError(f"the mask needs one byte per uploaded row ({n_rows}), got {len(mask)}")
        _lib.check(self.engine.lib.yawb_catalog_set_second_rows(self._h, _ptr(mask)))

    def info(self) -> tuple[int, int]:
        n, nbytes = c_int64(), c_int64()
        _lib.check(self.engine.lib.yawb_catalog_info(self._h, byref(n), byref(nbytes)))
        return n.value, nbytes.value

    def build_index(self, role: int) -> float:
        ms = c_double()
        _lib.check(self.engine.lib.yawb_build_index(self._h, role, byref(ms)))
        return ms.value

    def drop_index(self) -> None:
        _lib.check(self.engine.lib.yawb_drop_index(self._h))

    def free(self) -> None:
        # a closed engine has already released every device block of its catalogs (and its streams are gone)
        if self._h is not None and self.engine._h is not None:
            self.engine.lib.yawb_free_catalog(self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Engine:
    """One context on one CUDA device.  Raises if the device or library is missing."""

    def __init__(self, device: int = 0, *, staging: bool | None = None, cache_catalogs: bool | None = None,
                 cache_bytes: int | None = None, memory_limit: int | None = None):
        """`cache_catalogs` (default on; YAWB_CACHE=0 turns it off): device catalogs uploaded by the measurement
        functions stay resident, with their indexes, keyed by (catalog, z-binning) -- the counterpart of the
        reference's on-disk tree cache (`BinnedTrees.build` skips the rebuild while the `binning` file matches,
        `src/yaw/catalog/trees.py:515-526`).  A loop of `crosscorrelate` calls over tomographic bins then uploads and
        indexes only the catalogs that changed.  A labelled upload of several catalogs (`crosscorrelate_tomographic`,
        `autocorrelate_tomographic`) is kept the same way, keyed by the tuple of its members and dropped as soon as
        any of them dies.  Least recently used entries are dropped beyond `cache_bytes` of device memory (default
        64 GB, YAWB_CACHE_GB).

        `staging=True` (or YAWB_STAGING=1): measurement calls prepare large catalogs straight into a
        cache of page-locked buffers, so their copies are asynchronous and run at full PCIe rate.  Worth it
        for loops of many calls (C3: 225 -> 118 ms per call), not for a single one: page-locking the cache
        costs ~1.5 s per GB once.

        `memory_limit` (bytes): the device memory a measurement call may plan for.  A call whose predicted footprint
        (`footprint`, `count_footprint`) exceeds it is counted in several passes over shares of its patches, one
        after the other, each uploading only its share (`sharding.plan_passes`).  Default: what the context can
        obtain when the call starts (`memory_available`): the device's free bytes, the allocator's parked blocks and
        the engine's cached catalogs.  Under the default a call that fits drops the cached catalogs it does not use,
        least recently used first, until it fits (`make_room`); a call that needs passes drops the whole cache."""
        self.memory_limit = None if memory_limit is None else int(memory_limit)
        self.staging = bool(int(os.environ.get("YAWB_STAGING", "0"))) if staging is None else bool(staging)
        self.staging_min_rows = 1_000_000  # smaller catalogs are not worth a page-locked detour
        # YAWB_DEVICE_DIGITIZE=1: measurement calls ship raw redshifts and the device assigns the z-bins
        # (`yawb_upload_catalog_z`); default: byte-sized ids assigned on the host (1/8 of the PCIe traffic)
        self.device_digitize = bool(int(os.environ.get("YAWB_DEVICE_DIGITIZE", "0")))
        self.lib = _lib.load()
        h = c_void_p()
        _lib.check(self.lib.yawb_create(int(device), byref(h)))
        self._h = h
        self.device = int(device)
        self._catalogs = weakref.WeakSet()  # live device catalogs: freed before the context goes away
        self.cache_catalogs = (os.environ.get("YAWB_CACHE", "1") != "0") if cache_catalogs is None else bool(cache_catalogs)
        self.cache_bytes = int(float(os.environ.get("YAWB_CACHE_GB", "64")) * 2**30) if cache_bytes is None else int(cache_bytes)
        self._cat_cache: dict = {}  # (identity, kappa) -> [signature of the binning, DeviceCatalog, bytes, weakrefs, tick]
        self._cat_cache_tick = 0
        self._pinned: list[c_void_p] = []
        self._stage_free: list[tuple[c_void_p, int]] = []
        self._stage_used: list[tuple[c_void_p, int]] = []

    @property
    def num_sms(self) -> int:
        return self.lib.yawb_device_sms(self._h)

    # ---- device memory --------------------------------------------------------------------------------
    def footprint(self, n_rows: int, n_patch: int, n_bins: int = 1, *, weighted: bool = False, zbin: str | None = None,
                  labelled: bool = False, mask: bool = False, first: bool = True, second: bool = True,
                  upload: bool = True) -> int:
        """Upper bound on the device bytes of one catalog (`yawb_catalog_footprint`, host arithmetic): `zbin` is how
        the z-bin ids travel, None (unbinned), "i32", "u8" or "z" (raw redshifts); `mask` a second-role row mask;
        `first` / `second` the indexes to cover; `upload=False` an index over rows uploaded by other catalogs (fused
        first-role index, union second-role index)."""
        what = ((_lib.FOOT_WEIGHTED if weighted else 0) | (_lib.FOOT_LABELLED if labelled else 0)
                | (_lib.FOOT_MASK if mask else 0) | (_lib.FOOT_FIRST if first else 0) | (_lib.FOOT_SECOND if second else 0)
                | (0 if upload else _lib.FOOT_NO_UPLOAD)
                | {None: 0, "i32": _lib.FOOT_BINNED, "u8": _lib.FOOT_U8, "z": _lib.FOOT_Z}[zbin])
        out = c_int64()
        _lib.check(self.lib.yawb_catalog_footprint(int(n_rows), int(n_patch), int(n_bins), what, byref(out)))
        return out.value

    def count_footprint(self, n_items: int, n_pairs: int, n_bins: int, n_edges: int, *, n_blocks: int = 1,
                        weighted: bool = False) -> int:
        """Upper bound on the workspace of one count call (`yawb_count_footprint`): `n_items` (patch pair, tile)
        combinations, `n_blocks` = first catalogs x labels of the second catalogs."""
        out = c_int64()
        _lib.check(self.lib.yawb_count_footprint(self.num_sms, int(n_items), int(n_pairs), int(n_bins), int(n_edges),
                                                 int(n_blocks), int(bool(weighted)), byref(out)))
        return out.value

    def memory_stats(self) -> dict:
        """`held`: bytes the allocator holds (parked blocks included), `peak`: its high-water mark since the last
        `memory_reset_peak`, `device_free`: free bytes of the device"""
        held, peak, free = c_int64(), c_int64(), c_int64()
        _lib.check(self.lib.yawb_memory_stats(self._h, byref(held), byref(peak), byref(free)))
        return dict(held=held.value, peak=peak.value, device_free=free.value)

    def memory_reset_peak(self) -> None:
        _lib.check(self.lib.yawb_memory_reset_peak(self._h))

    def memory_release(self) -> None:
        """blocks parked by the allocator go back to the driver"""
        _lib.check(self.lib.yawb_memory_release(self._h))

    def memory_parked(self) -> int:
        """bytes of the blocks the allocator holds parked for reuse (they go back to the driver when it runs out)"""
        out = c_int64()
        _lib.check(self.lib.yawb_memory_parked(self._h, byref(out)))
        return out.value

    def _cache_entry_bytes(self, entry) -> int:
        dev = entry[1]
        return max(dev.info()[1], 0) if dev._h is not None else 0

    def memory_available(self) -> int:
        """The bytes a measurement call plans for: `memory_limit`, or what the context can obtain for it -- the
        device's free bytes, the parked blocks of the allocator and the catalogs in the engine's cache (those the
        call uses are part of its footprint, the others are dropped by `make_room` when the call needs their
        memory).  Catalogs uploaded outside the cache are not counted."""
        if self.memory_limit is not None:
            return self.memory_limit
        return (self.memory_stats()["device_free"] + self.memory_parked()
                + sum(self._cache_entry_bytes(e) for e in self._cat_cache.values()))

    def make_room(self, nbytes: int, catalogs=()) -> None:
        """Under the default limit: drop cached catalogs that are none of `catalogs` (and no labelled upload of
        them), least recently used first, until the free bytes, the parked blocks and the cached catalogs of
        `catalogs` add up to `nbytes`.  With an explicit `memory_limit` nothing is dropped."""
        if self.memory_limit is not None or not self._cat_cache:
            return
        mine = {id(c) for c in catalogs}

        def used(key) -> bool:
            kind, ident = key[0]
            return ident in mine if kind == "id" else any(i in mine for i in ident)

        have = self.memory_stats()["device_free"] + self.memory_parked()
        have += sum(self._cache_entry_bytes(e) for k, e in self._cat_cache.items() if used(k))
        for key in sorted((k for k in self._cat_cache if not used(k)), key=lambda k: self._cat_cache[k][4]):
            if have >= nbytes:
                break
            have += self._cache_entry_bytes(self._cat_cache[key])
            self._cache_drop(key)

    def upload_catalog(
        self,
        xyz: np.ndarray,
        patch_off: np.ndarray,
        *,
        weights: np.ndarray | None = None,
        zbin: np.ndarray | None = None,
        n_bins: int = 1,
        redshifts: np.ndarray | None = None,
        edges: np.ndarray | None = None,
        closed: str = "right",
        n_labels: int | None = None,
        keep: np.ndarray | None = None,
        second_rows: np.ndarray | None = None,
    ) -> DeviceCatalog:
        """`zbin` (+ `n_bins`): z-bin ids assigned on the host; or `redshifts` + `edges` (+ `closed`): the raw
        redshifts travel and the device assigns the bins with np.digitize's comparisons (`yawb_upload_catalog_z`,
        reference `src/yaw/catalog/trees.py:408-414`).

        `n_labels` (with `zbin`): binned labels (`yawb_catalog_set_labels`), the ids are `label * B + z-bin` with
        `B = n_bins // n_labels`, e.g. the tomographic bins of a sample, each z-binned (`prepare_labelled_arrays`
        with a binning).  `count` then pairs label by label; see there.

        `keep` (one flag per patch): only the rows of the kept patches travel (`yawb_upload_catalog_patches`), straight
        from these arrays; an unkept patch is an empty patch.  `second_rows`: the mask of `DeviceCatalog.set_second_rows`,
        one byte per row that travels."""
        if n_labels is not None:
            if zbin is None:
                raise ValueError("'n_labels' needs z-bin ids ('zbin')")
            version = self.lib.yawb_version()
            if version < _lib.BINNED_LABELS_MIN_VERSION:
                raise _lib.YawbError(f"n_labels needs libyawb version >= {_lib.BINNED_LABELS_MIN_VERSION} "
                                     f"(loaded: {version})")
        xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
        patch_off = np.ascontiguousarray(patch_off, dtype=np.int64)
        n = len(xyz)
        if patch_off[-1] != n:
            raise ValueError("patch_off[-1] must equal the number of rows")
        if weights is not None:
            weights = np.ascontiguousarray(weights, dtype=np.float64)
            if len(weights) != n:
                raise ValueError("shape of 'xyz' and 'weights' does not match")
        upload = self.lib.yawb_upload_catalog
        if zbin is not None:
            if np.asarray(zbin).dtype == np.uint8:  # byte-sized ids (255 = dropped row): a quarter of the traffic
                zbin = np.ascontiguousarray(zbin)
                upload = self.lib.yawb_upload_catalog_u8
            else:
                zbin = np.ascontiguousarray(zbin, dtype=np.int32)
            if len(zbin) != n:
                raise ValueError("shape of 'xyz' and 'zbin' does not match")
        h = c_void_p()
        if redshifts is not None:
            if zbin is not None or edges is None:
                raise ValueError("pass either 'zbin' or 'redshifts' with 'edges'")
            redshifts = np.ascontiguousarray(redshifts, dtype=np.float64)
            edges = np.ascontiguousarray(edges, dtype=np.float64)
            if len(redshifts) != n:
                raise ValueError("shape of 'xyz' and 'redshifts' does not match")
            n_bins = len(edges) - 1
        n_rows = n
        if keep is not None:
            keep = np.ascontiguousarray(keep, dtype=np.uint8)
            if len(keep) != len(patch_off) - 1:
                raise ValueError("'keep' needs one flag per patch")
            n_rows = int(np.diff(patch_off)[keep != 0].sum())
            z8 = zbin is not None and zbin.dtype == np.uint8
            _lib.check(
                self.lib.yawb_upload_catalog_patches(
                    self._h, _ptr(xyz), _ptr(weights), None if z8 else _ptr(zbin), _ptr(zbin) if z8 else None,
                    _ptr(redshifts), _ptr(edges), int(str(closed) == "right"), _ptr(patch_off), len(patch_off) - 1,
                    int(n_bins), _ptr(keep), byref(h),
                )
            )
        elif redshifts is not None:
            _lib.check(
                self.lib.yawb_upload_catalog_z(
                    self._h, _ptr(xyz), _ptr(weights), _ptr(redshifts), _ptr(edges), int(str(closed) == "right"),
                    _ptr(patch_off), len(patch_off) - 1, int(n_bins), byref(h),
                )
            )
        else:
            _lib.check(
                upload(
                    self._h, _ptr(xyz), _ptr(weights), _ptr(zbin), _ptr(patch_off),
                    len(patch_off) - 1, int(n_bins), byref(h),
                )
            )
        binned = zbin is not None or redshifts is not None
        cat = DeviceCatalog(self, h, len(patch_off) - 1, int(n_bins) if binned else 1, binned, weights is not None)
        cat._n_uploaded = n_rows
        try:
            if n_labels is not None:
                _lib.check(self.lib.yawb_catalog_set_labels(h, int(n_labels)))
                cat.n_labels = int(n_labels)
            if second_rows is not None:
                cat.set_second_rows(second_rows)
        except Exception:
            cat.free()
            raise
        # the upload is asynchronous: keep the host buffers alive as long as the handle
        cat._keepalive = (xyz, weights, zbin, redshifts, patch_off)
        self._catalogs.add(cat)
        return cat

    def sample_patch_sum(self, values: np.ndarray, pair_i: np.ndarray, pair_j: np.ndarray,
                         n_patch: int) -> tuple[np.ndarray, np.ndarray]:
        """Sum over the linked patch pairs and its leave-one-patch-out jackknife samples on the device
        (`yawb_jackknife`): `values` is `(n_pairs, n_bins)`; returns `(total (n_bins,), samples (n_patch, n_bins))`,
        the `data` / `samples` of the reference's `SampledPatchSum` (`src/yaw/correlation/paircounts.py:113-141`)."""
        values = np.ascontiguousarray(values, dtype=np.float64)
        pair_i = np.ascontiguousarray(pair_i, dtype=np.int32)
        pair_j = np.ascontiguousarray(pair_j, dtype=np.int32)
        n_pairs, n_bins = values.shape
        total = np.empty(n_bins, dtype=np.float64)
        samples = np.empty((int(n_patch), n_bins), dtype=np.float64)
        _lib.check(self.lib.yawb_jackknife(self._h, _ptr(values), _ptr(pair_i), _ptr(pair_j), int(n_pairs), int(n_patch),
                                           int(n_bins), _ptr(total), _ptr(samples)))
        return total, samples

    def _labels_flag(self, labels: bool) -> int:
        if not labels:
            return 0
        version = self.lib.yawb_version()
        if version < _lib.LABELS_MIN_VERSION:
            raise _lib.YawbError(f"labels=True needs libyawb version >= {_lib.LABELS_MIN_VERSION} (loaded: {version})")
        return _lib.FLAG_SECOND_LABELS

    @staticmethod
    def _shape(cat2: DeviceCatalog, labels: bool, n_pairs: int, n_bins: int, n_edges: int) -> tuple:
        """result shape of one (first, second) catalog combination: a leading label axis with `labels` or with the
        binned labels of `cat2`"""
        shape = (n_pairs, n_bins, n_edges - 1)
        n_labels = getattr(cat2, "n_labels", None)
        if n_labels is not None:
            return (n_labels, *shape)
        return ((cat2.n_bins if cat2.binned else 1), *shape) if labels else shape

    def count(
        self,
        cat1: DeviceCatalog,
        cat2: DeviceCatalog,
        pair_i: np.ndarray,
        pair_j: np.ndarray,
        r2_edges: np.ndarray,
        *,
        exact: bool = False,
        labels: bool = False,
    ) -> tuple[np.ndarray, np.ndarray, dict]:
        """
        Returns `(counts_i64, sums_f64, stats)`, both arrays shaped
        `(n_pairs, n_bins, n_edges - 1)`.

        `labels=True` (`YAWB_FLAG_SECOND_LABELS`): the z-bin ids of a binned `cat2` are sample labels 0..L-1 (L =
        `cat2.n_bins`, 1 for an unbinned `cat2`); every row is paired with every z-bin of `cat1` and the arrays
        gain a leading label axis, `(L, n_pairs, n_bins, n_edges - 1)`: entry l is the count against the rows of
        label l alone.

        Binned labels (`cat2` uploaded with `n_labels=L`, `B = cat2.n_bins // L` z-bins per label): `r2_edges` is
        `(B, n_edges)` and the arrays are `(L, n_pairs, B, n_edges - 1)`, also for L = 1.  Entry l is the z-binned
        count of label l of `cat2` against label l of `cat1` when `cat1` carries the same binned labels (`cat1` may
        be `cat2`), or against the whole of `cat1` when `cat1` is binned with B z-bins and unlabelled.  A labelled
        `cat1` needs a labelled `cat2`: pair counts are symmetric, swap the catalogs and the pair lists.
        """
        lab = cat2 if getattr(cat2, "n_labels", None) else cat1  # binned labels: r2_edges per z-bin of a label
        n_bins = lab.n_bins // lab.n_labels if getattr(lab, "n_labels", None) else cat1.n_bins
        pair_i, pair_j, r2_edges = _pairs_and_edges(pair_i, pair_j, r2_edges, n_bins)
        n_edges = r2_edges.shape[1]
        n_pairs = len(pair_i)
        shape = self._shape(cat2, labels, n_pairs, n_bins, n_edges)
        out_i = np.zeros(shape, dtype=np.int64)
        out_f = np.zeros(shape, dtype=np.float64)
        stats = _lib.YawbStats()
        flags = (_lib.FLAG_EXACT_BRUTEFORCE if exact else 0) | self._labels_flag(labels)
        _lib.check(
            self.lib.yawb_count(
                self._h, cat1._h, cat2._h, _ptr(pair_i), _ptr(pair_j), n_pairs, _ptr(r2_edges), n_edges,
                flags, _ptr(out_f), _ptr(out_i), byref(stats),
            )
        )
        return out_i, out_f, stats.as_dict()

    def count2(
        self,
        cat1a: DeviceCatalog,
        cat1b: DeviceCatalog,
        cat2: DeviceCatalog,
        pair_i: np.ndarray,
        pair_j: np.ndarray,
        r2_edges: np.ndarray,
        *,
        out_device: tuple[int, int, int, int] | None = None,
        labels: bool = False,
    ) -> tuple[tuple[np.ndarray, np.ndarray], tuple[np.ndarray, np.ndarray], dict]:
        """`count(cat1a, cat2)` and `count(cat1b, cat2)` in one pass over a fused index of the two first
        catalogs (`yawb_count2`): returns `((counts_a, sums_a), (counts_b, sums_b), stats)`.

        `out_device = (sums_a, counts_a, sums_b, counts_b)`: raw device pointers (0 = not wanted) of
        caller-owned buffers shaped `(n_pairs, n_bins, n_edges - 1)`; the results stay on the device
        (`YAWB_FLAG_OUT_DEVICE`, e.g. for an NCCL reduce) and the arrays returned are `None`.
        `labels`: as in `count`; the results (and device buffers) gain the leading label axis of `cat2`."""
        n_bins = cat1a.n_bins
        pair_i, pair_j, r2_edges = _pairs_and_edges(pair_i, pair_j, r2_edges, n_bins)
        n_edges = r2_edges.shape[1]
        shape = self._shape(cat2, labels, len(pair_i), n_bins, n_edges)
        stats = _lib.YawbStats()
        lab = self._labels_flag(labels)
        if out_device is not None:
            ptrs = [c_void_p(p) if p else None for p in out_device]
            _lib.check(
                self.lib.yawb_count2(
                    self._h, cat1a._h, cat1b._h, cat2._h, _ptr(pair_i), _ptr(pair_j), len(pair_i), _ptr(r2_edges), n_edges,
                    _lib.FLAG_OUT_DEVICE | lab, *ptrs, byref(stats),
                )
            )
            return (None, None), (None, None), stats.as_dict()
        out = [(np.zeros(shape, dtype=np.int64), np.zeros(shape, dtype=np.float64)) for _ in range(2)]
        _lib.check(
            self.lib.yawb_count2(
                self._h, cat1a._h, cat1b._h, cat2._h, _ptr(pair_i), _ptr(pair_j), len(pair_i), _ptr(r2_edges), n_edges, lab,
                _ptr(out[0][1]), _ptr(out[0][0]), _ptr(out[1][1]), _ptr(out[1][0]), byref(stats),
            )
        )
        return out[0], out[1], stats.as_dict()

    def count4(
        self,
        cat1a: DeviceCatalog,
        cat1b: DeviceCatalog,
        cat2a: DeviceCatalog,
        cat2b: DeviceCatalog,
        pair_i: np.ndarray,
        pair_j: np.ndarray,
        r2_edges: np.ndarray,
        *,
        out_device: tuple | None = None,
        labels: bool = False,
    ):
        """The four counts of a cross-correlation in ONE launch (`yawb_count4`): `count(cat1a, cat2a)`,
        `count(cat1b, cat2a)`, `count(cat1a, cat2b)`, `count(cat1b, cat2b)` -- DD, RD, DR, RR for (reference, its
        randoms, unknown, its randoms), `src/yaw/correlation/measurements.py:623-626`.  Returns
        `([(counts, sums)] * 4, stats)` in that order.

        `out_device = (sums_0, counts_0, ..., sums_3, counts_3)`: raw device pointers (0 = not wanted); the results
        stay on the device and the arrays returned are `None`.
        `labels`: as in `count`; each output gains the leading label axis of its own second catalog (e.g. a
        labelled unknown sample as `cat2a` with a shared, unbinned random catalog as `cat2b`)."""
        n_bins = cat1a.n_bins
        pair_i, pair_j, r2_edges = _pairs_and_edges(pair_i, pair_j, r2_edges, n_bins)
        n_edges = r2_edges.shape[1]
        shapes = [self._shape(c2, labels, len(pair_i), n_bins, n_edges) for c2 in (cat2a, cat2a, cat2b, cat2b)]
        stats = _lib.YawbStats()
        tab_f, tab_i = (c_void_p * 4)(), (c_void_p * 4)()
        out = None
        if out_device is not None:
            for t in range(4):
                tab_f[t] = out_device[2 * t] or None
                tab_i[t] = out_device[2 * t + 1] or None
            flags = _lib.FLAG_OUT_DEVICE
        else:
            out = [(np.zeros(s, dtype=np.int64), np.zeros(s, dtype=np.float64)) for s in shapes]
            for t in range(4):
                tab_i[t] = out[t][0].ctypes.data
                tab_f[t] = out[t][1].ctypes.data
            flags = 0
        flags |= self._labels_flag(labels)
        _lib.check(
            self.lib.yawb_count4(
                self._h, cat1a._h, cat1b._h, cat2a._h, cat2b._h, _ptr(pair_i), _ptr(pair_j), len(pair_i), _ptr(r2_edges),
                n_edges, flags, tab_f, tab_i, byref(stats),
            )
        )
        if out is None:
            return [(None, None)] * 4, stats.as_dict()
        return out, stats.as_dict()

    def count_into_device(self, cat1, cat2, pair_i, pair_j, r2_edges, out_f64_ptr: int, out_i64_ptr: int):
        """Variant writing into caller-owned device buffers (raw pointers)."""
        pair_i, pair_j, r2_edges = _pairs_and_edges(pair_i, pair_j, r2_edges, cat1.n_bins)
        stats = _lib.YawbStats()
        _lib.check(
            self.lib.yawb_count(
                self._h, cat1._h, cat2._h, _ptr(pair_i), _ptr(pair_j), len(pair_i), _ptr(r2_edges),
                r2_edges.shape[1], _lib.FLAG_OUT_DEVICE,
                c_void_p(out_f64_ptr) if out_f64_ptr else None,
                c_void_p(out_i64_ptr) if out_i64_ptr else None, byref(stats),
            )
        )
        return stats.as_dict()

    def assign_patches(self, xyz: np.ndarray, centers_xyz: np.ndarray) -> np.ndarray:
        """Index of the nearest patch centre of every row (`scipy.cluster.vq.vq` arithmetic on the device;
        replaces `assign_patch_centers`, reference `src/yaw/catalog/catalog.py:229-249`)."""
        xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
        centers_xyz = np.ascontiguousarray(centers_xyz, dtype=np.float64).reshape(-1, 3)
        out = np.empty(len(xyz), dtype=np.int32)
        _lib.check(self.lib.yawb_assign_patches(self._h, _ptr(xyz), len(xyz), _ptr(centers_xyz), len(centers_xyz),
                                                _ptr(out)))
        return out

    def kmeans(self, xyz: np.ndarray, k: int, *, weights: np.ndarray | None = None,
               max_iter: int = 500) -> tuple[np.ndarray, np.ndarray, int, bool]:
        """Deterministic spherical k-means on the device (`yawb_kmeans`, DESIGN.md section 4.4): patch centres for
        `k` patches from rows `xyz` (`(n, 3)`, as `AngularCoordinates.to_3d` gives them), optionally weighted.
        Returns `(centers_xyz (k, 3), labels (n,) int32, n_iter, converged)`; `labels` is the nearest centre of
        every row (`scipy.cluster.vq.vq` arithmetic).  With `max_iter=0` the initial centres are returned."""
        xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
        if weights is not None:
            weights = np.ascontiguousarray(weights, dtype=np.float64)
            if len(weights) != len(xyz):
                raise ValueError("shape of 'xyz' and 'weights' does not match")
        centers = np.empty((max(int(k), 0), 3), dtype=np.float64)
        labels = np.empty(len(xyz), dtype=np.int32)
        n_iter, converged = c_int(), c_int()
        _lib.check(self.lib.yawb_kmeans(self._h, _ptr(xyz), _ptr(weights), len(xyz), int(k), int(max_iter),
                                        _ptr(centers), _ptr(labels), byref(n_iter), byref(converged)))
        return centers, labels, n_iter.value, bool(converged.value)

    # ---- resident catalogs across measurement calls -------------------------------------------------
    @staticmethod
    def _cache_identity(catalog):
        # the catalog OBJECT (an entry lives exactly as long as it does); a cache directory is only a label for
        # this package's in-memory catalogs, and on disk it can be overwritten, so paths are not identities.  A
        # labelled upload (`prepare_labelled_arrays`) is keyed by the tuple of its member catalogs.
        if isinstance(catalog, tuple):
            return ("labelled", tuple(id(c) for c in catalog))
        return ("id", id(catalog))

    def cache_lookup(self, catalog, signature, kappa: bool):
        """Device catalog kept for `catalog` with this z-binning, or None.  An entry built for another binning
        is dropped (the reference rebuilds its trees in that case, `trees.py:519-526`)."""
        if not self.cache_catalogs:
            return None
        key = (self._cache_identity(catalog), bool(kappa))
        entry = self._cat_cache.get(key)
        if entry is None:
            return None
        if entry[0] != signature or entry[1]._h is None:
            self._cache_drop(key)
            return None
        self._cat_cache_tick += 1
        entry[4] = self._cat_cache_tick
        return entry[1]

    def cache_store(self, catalog, signature, kappa: bool, dev: DeviceCatalog) -> bool:
        if not self.cache_catalogs:
            return False
        ident = self._cache_identity(catalog)
        key = (ident, bool(kappa))
        members = catalog if isinstance(catalog, tuple) else (catalog,)
        try:  # the entry is dropped as soon as any member dies
            ref = [weakref.ref(c, lambda _r, k=key: self._cache_drop(k)) for c in members]
        except TypeError:
            return False
        self._cache_drop(key)
        nbytes = max(dev.info()[1], 0) * 3  # raw rows now, the indexes built later are about twice that
        self._cat_cache_tick += 1
        self._cat_cache[key] = [signature, dev, nbytes, ref, self._cat_cache_tick]
        total = sum(e[2] for e in self._cat_cache.values())
        while total > self.cache_bytes and len(self._cat_cache) > 1:  # least recently used first, never the new one
            victim = min((k for k in self._cat_cache if k != key), key=lambda k: self._cat_cache[k][4])
            total -= self._cat_cache[victim][2]
            self._cache_drop(victim)
        return True

    def _cache_drop(self, key) -> None:
        entry = self._cat_cache.pop(key, None)
        if entry is not None:
            try:
                entry[1].free()
            except Exception:
                pass

    def cache_clear(self) -> None:
        for key in list(self._cat_cache):
            self._cache_drop(key)

    def timer_start(self) -> None:
        _lib.check(self.lib.yawb_timer_start(self._h))

    def timer_stop(self) -> float:
        """milliseconds of device time since `timer_start` (CUDA events on the engine's stream)"""
        ms = c_double()
        _lib.check(self.lib.yawb_timer_stop(self._h, byref(ms)))
        return ms.value

    def pinned_empty(self, shape, dtype) -> np.ndarray:
        """numpy array backed by page-locked host memory (freed with the engine)"""
        dtype = np.dtype(dtype)
        nbytes = int(np.prod(shape)) * dtype.itemsize
        ptr = c_void_p()
        _lib.check(self.lib.yawb_host_alloc(byref(ptr), nbytes))
        self._pinned.append(ptr)
        buf = (ctypes.c_char * max(nbytes, 1)).from_address(ptr.value)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    # ---- staging buffers for repeated measurement calls ----------------------------------------------
    def staging_empty(self, shape, dtype) -> np.ndarray:
        """Page-locked array from the engine's staging cache (new blocks are allocated on demand and kept;
        `staging_release` makes every block handed out so far available again).  Page-locking costs a few
        hundred ms per GB once; afterwards a measurement call prepares its catalogs straight into pinned
        memory and the copies run asynchronously at full PCIe rate."""
        dtype = np.dtype(dtype)
        count = int(np.prod(shape))
        nbytes = max(count * dtype.itemsize, 1)
        best = None
        for k, (ptr, size) in enumerate(self._stage_free):
            if nbytes <= size <= nbytes + nbytes // 2 + (1 << 20) and (best is None or size < self._stage_free[best][1]):
                best = k
        if best is not None:
            ptr, size = self._stage_free.pop(best)
        else:
            size = (nbytes + (1 << 20) - 1) & ~((1 << 20) - 1)
            ptr = c_void_p()
            _lib.check(self.lib.yawb_host_alloc(byref(ptr), size))
            self._pinned.append(ptr)
        self._stage_used.append((ptr, size))
        buf = (ctypes.c_char * size).from_address(ptr.value)
        return np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)

    def staging_release(self) -> None:
        """Hand every staging block back to the cache; call when the uploads that used them are complete."""
        self._stage_free.extend(self._stage_used)
        self._stage_used.clear()

    def sync(self) -> None:
        _lib.check(self.lib.yawb_sync(self._h))

    def close(self) -> None:
        if self._h is not None:
            self.cache_clear()
            for cat in list(self._catalogs):
                cat.free()
            for ptr in self._pinned:
                self.lib.yawb_host_free(ptr)
            self._pinned.clear()
            self._stage_free.clear()
            self._stage_used.clear()
            self.lib.yawb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class GroupCatalog:
    """One catalog of a measurement call on the devices of an `EngineGroup`: `parts[d]` is device d's upload (its kept
    patches, second-role rows masked to its strips), `plan` the `SharePlan` it was made for."""

    def __init__(self, parts: list, plan, resident: list[bool]) -> None:
        self.parts = parts
        self.plan = plan
        self._resident = resident  # parts owned by their engine's catalog cache (not freed here)
        self.sums_hook = None  # a call counted in passes: sum_weights goes through it (sums over the passes)
        first = parts[0]
        self.n_patch, self.n_bins, self.binned, self.weighted = first.n_patch, first.n_bins, first.binned, first.weighted
        self.n_labels = getattr(first, "n_labels", None)

    def sum_weights(self) -> np.ndarray:
        """`(n_bins, n_patch)`, every patch from the first device that uploaded it"""
        out = None
        done = np.zeros(self.n_patch, dtype=bool)
        for part, keep in zip(self.parts, self.plan.keep):
            take = keep.astype(bool) & ~done
            if not take.any():
                continue
            sw = part.sum_weights()
            if out is None:
                out = np.zeros_like(sw)
            out[:, take] = sw[:, take]
            done |= take
        return out if self.sums_hook is None else self.sums_hook(out, done)

    def free(self) -> None:
        for part, resident in zip(self.parts, self._resident):
            if not resident:
                part.free()


class EngineGroup:
    """Several engines driven from one process: a measurement function called with `engine=EngineGroup([0, 1, ...])`
    splits its pair counts over the devices and returns what the same call on one `Engine` returns.

    Every call cuts the patches of its second catalogs into one share per device (`sharding.plan_shares`: the exact
    fractional split of the pair costs, a patch at a cut shared as two compact strips of rows).  Each device uploads,
    of every catalog of the call, only its own patches and the patches linked to them, counts the pairs whose second
    patch it owns against its strips, and the histograms are summed on the host in device order (integers exactly,
    float sums to rounding).  No device holds a whole catalog, so a measurement larger than one GPU's memory fits on
    several.

    `devices`: CUDA device ids (a device may repeat, e.g. `[0, 0]`) or existing engine objects.  One worker thread per
    engine uploads and counts; the library releases the GIL.  Patch centres (`kmeans`, `assign_patches`) stay on
    `Engine`.  Not combined with `shard=` (one process per GPU under torchrun)."""

    def __init__(self, devices) -> None:
        devices = list(devices)
        if not devices:
            raise ValueError("an EngineGroup needs at least one device")
        created = []
        try:
            for d in devices:
                if isinstance(d, (int, np.integer)):
                    created.append(Engine(int(d)))
            it = iter(created)
            self.engines = [next(it) if isinstance(d, (int, np.integer)) else d for d in devices]
        except Exception:
            for e in created:
                e.close()
            raise
        self._own = created
        # raw redshifts travel when every engine asks for it (`Engine.device_digitize`), as on a single engine
        self.device_digitize = all(getattr(e, "device_digitize", False) for e in self.engines)
        if len({id(e) for e in self.engines}) != len(self.engines):
            raise ValueError("an engine object may appear only once in an EngineGroup (a context serves one thread)")
        self._pool = ThreadPoolExecutor(max_workers=len(self.engines), thread_name_prefix="yawb-group")

    def __len__(self) -> int:
        return len(self.engines)

    def _map(self, fn):
        """fn(d, engine) for every device, concurrently; results in device order"""
        futures = [self._pool.submit(fn, d, e) for d, e in enumerate(self.engines)]
        return [f.result() for f in futures]

    # ---- uploads --------------------------------------------------------------------------------------
    def cache_lookup(self, catalog, signature, kappa: bool, plan):
        """a `GroupCatalog` if every engine keeps this catalog uploaded for its share of `plan`, else None"""
        parts = []
        for d, e in enumerate(self.engines):
            lookup = getattr(e, "cache_lookup", None)
            dev = lookup(catalog, (signature, plan.signature(d)), kappa) if lookup else None
            if dev is None:
                return None
            parts.append(dev)
        return GroupCatalog(parts, plan, [True] * len(parts))

    def upload_catalog(self, arrays: dict, plan, cache=None) -> GroupCatalog:
        """`arrays`: the keyword arguments of `Engine.upload_catalog` for the whole catalog (`xyz`, `patch_off`, ...);
        device d uploads the patches `plan.keep[d]` with the second-role rows of its strips.  `cache = (catalog,
        signature, kappa)`: each part is kept in its engine's catalog cache under the signature and its share."""
        arrays = dict(arrays)
        xyz, patch_off = arrays.pop("xyz"), arrays.pop("patch_off")

        def one(d, e):
            dev = e.upload_catalog(xyz, patch_off, keep=plan.keep[d], second_rows=plan.mask(d, xyz, patch_off), **arrays)
            store = getattr(e, "cache_store", None)
            resident = bool(cache is not None and store and store(cache[0], (cache[1], plan.signature(d)), cache[2], dev))
            return dev, resident

        parts = self._map(one)
        return GroupCatalog([p for p, _ in parts], plan, [r for _, r in parts])

    # ---- counts ---------------------------------------------------------------------------------------
    @staticmethod
    def _merge(n_pairs: int, results, n_out: int):
        """per device (rows, [(counts, sums)] * n_out, stats) -> the outputs over the full pair list, summed in device
        order; counters summed, times of the slowest device"""
        outs, stats = [], {}
        for t in range(n_out):
            full = [None, None]
            for rows, dev_outs, _ in results:
                for k, arr in enumerate(dev_outs[t]):
                    if full[k] is None:
                        shape = list(arr.shape)
                        shape[arr.ndim - 3] = n_pairs  # the pair axis, behind a leading label axis if any
                        full[k] = np.zeros(shape, dtype=arr.dtype)
                    idx = (slice(None),) * (arr.ndim - 3) + (rows,)
                    full[k][idx] += arr
            outs.append(tuple(full))
        for _, _, st in results:
            for key, v in st.items():
                stats[key] = max(stats.get(key, 0), v) if key.endswith("_ms") else stats.get(key, 0) + v
        return outs, stats

    def _fan_out(self, second: GroupCatalog, pair_i, pair_j, count_one):
        """`count_one(d, engine, pair_i, pair_j) -> ([(counts, sums), ...], stats)` on every device over the pairs whose
        second patch it owns; returns (n_pairs, [(rows, outputs, stats)] in device order)"""
        pair_i = np.ascontiguousarray(pair_i, dtype=np.int32)
        pair_j = np.ascontiguousarray(pair_j, dtype=np.int32)

        def one(d, e):
            rows = np.flatnonzero(second.plan.second[d][pair_j])
            outs, stats = count_one(d, e, pair_i[rows], pair_j[rows])
            return rows, outs, stats

        return len(pair_i), self._map(one)

    def count(self, cat1: GroupCatalog, cat2: GroupCatalog, pair_i, pair_j, r2_edges, **kw):
        """`Engine.count` over the devices: each counts the pairs whose second patch it owns"""
        def one(d, e, pi, pj):
            counts, sums, stats = e.count(cat1.parts[d], cat2.parts[d], pi, pj, r2_edges, **kw)
            return [(counts, sums)], stats

        n, res = self._fan_out(cat2, pair_i, pair_j, one)
        (out,), stats = self._merge(n, res, 1)
        return (*out, stats)

    def count2(self, cat1a: GroupCatalog, cat1b: GroupCatalog, cat2: GroupCatalog, pair_i, pair_j, r2_edges, **kw):
        """`Engine.count2` over the devices"""
        def one(d, e, pi, pj):
            a, b, stats = e.count2(cat1a.parts[d], cat1b.parts[d], cat2.parts[d], pi, pj, r2_edges, **kw)
            return [a, b], stats

        n, res = self._fan_out(cat2, pair_i, pair_j, one)
        (a, b), stats = self._merge(n, res, 2)
        return a, b, stats

    def sync(self) -> None:
        self._map(lambda d, e: e.sync())

    def close(self) -> None:
        """shut the worker threads down and close the engines the group created (engines passed in stay open)"""
        if self._pool is not None:
            self._pool.shutdown(wait=True)
            self._pool = None
        for e in self._own:
            e.close()
        self._own = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
