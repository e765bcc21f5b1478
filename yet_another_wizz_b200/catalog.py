"""
Patch-partitioned catalogs on the host -- the input side of the pair-count path.

Mirrors the attribute surface of `yaw.Catalog` / `yaw.catalog.Patch` that
`crosscorrelate` / `autocorrelate` consume (reference
`src/yaw/catalog/catalog.py:911-1460`, `src/yaw/catalog/patch.py:41-147, 321-440`):
a `Mapping[int, Patch]` with `get_centers()`, `get_radii()`, `get_num_records()`,
`has_weights`, `has_redshifts`; a patch yields its rows through `load_data()`
as a structured array with fields `ra`, `dec`, `weights`, `redshifts`.

The reference's ingest pipeline (chunked FITS/HDF5/Parquet readers, writer
processes) is out of scope (SURVEY.md section 2, row 6).  Patches here are built in
memory from arrays, or opened from a cache directory written by the reference
(`data.bin` + `meta.yml`, byte-compatible read-only access).  Patch centres can be
given, or computed from a number of patches by the device k-means
(`create_patch_centers`, in place of the reference's treecorr k-means).
Real `yaw.Catalog` objects can be handed to the engine directly; both kinds are
read through the same duck-typed accessors in `measurements.py`.
"""

from __future__ import annotations

import os
from collections.abc import Mapping
from pathlib import Path

import numpy as np

from .coordinates import AngularCoordinates, AngularDistances

__all__ = ["Catalog", "InconsistentPatchesError", "Metadata", "Patch", "create_patch_centers"]

ATTR_ORDER = ("ra", "dec", "weights", "redshifts", "patch_ids", "kappa")  # src/yaw/datachunk.py:44


class InconsistentPatchesError(Exception):
    """Raised when the patches of two catalogs do not line up."""


class Metadata:
    """Patch meta data: `num_records`, `sum_weights`, `center`, `radius`
    (reference `Metadata.compute`, `src/yaw/catalog/patch.py:104-147`)."""

    __slots__ = ("num_records", "sum_weights", "center", "radius")

    def __init__(self, *, num_records, sum_weights, center, radius) -> None:
        self.num_records = int(num_records)
        self.sum_weights = float(sum_weights)
        self.center = center
        self.radius = radius

    @classmethod
    def compute(cls, coords: AngularCoordinates, *, weights=None, center: AngularCoordinates | None = None):
        num = len(coords)
        sum_weights = float(num) if weights is None else float(np.sum(weights))
        if center is not None:
            if len(center) != 1:
                raise ValueError("'center' must be one single coordinate")
            center = center.copy()
        else:
            center = coords.mean(weights)
        radius = coords.distance(center).max()
        return cls(num_records=num, sum_weights=sum_weights, center=center, radius=radius)

    def __repr__(self) -> str:
        return (f"Metadata(num_records={self.num_records}, sum_weights={self.sum_weights}, "
                f"center={self.center.data[0]}, radius={self.radius.data[0]})")


def _structured(ra, dec, weights, redshifts, kappa=None) -> np.ndarray:
    fields = [("ra", "f8"), ("dec", "f8")]
    if weights is not None:
        fields.append(("weights", "f8"))
    if redshifts is not None:
        fields.append(("redshifts", "f8"))
    if kappa is not None:
        fields.append(("kappa", "f8"))
    data = np.empty(len(ra), dtype=np.dtype(fields))
    data["ra"] = ra
    data["dec"] = dec
    if weights is not None:
        data["weights"] = weights
    if redshifts is not None:
        data["redshifts"] = redshifts
    if kappa is not None:
        data["kappa"] = kappa
    return data


class Patch:
    """One spatial patch: rows + meta data."""

    __slots__ = ("_data", "_path", "meta")

    def __init__(self, data: np.ndarray | None, meta: Metadata | None = None, *, center=None, path=None) -> None:
        self._data = data
        self._path = path
        if meta is None:
            rows = self.load_data()
            coords = AngularCoordinates(np.column_stack([rows["ra"], rows["dec"]]))
            weights = rows["weights"] if "weights" in rows.dtype.names else None
            meta = Metadata.compute(coords, weights=weights, center=center)
        self.meta = meta

    def load_data(self) -> np.ndarray:
        if self._data is not None:
            return self._data
        return read_patch_data(self._path)

    @property
    def has_weights(self) -> bool:
        return "weights" in self.load_data().dtype.names if self._data is not None else _cache_flags(self._path)[0]

    @property
    def has_redshifts(self) -> bool:
        return "redshifts" in self.load_data().dtype.names if self._data is not None else _cache_flags(self._path)[1]

    @property
    def has_kappa(self) -> bool:
        return "kappa" in self.load_data().dtype.names

    @property
    def coords(self) -> AngularCoordinates:
        rows = self.load_data()
        return AngularCoordinates(np.column_stack([rows["ra"], rows["dec"]]))

    def __len__(self) -> int:
        return self.meta.num_records

    def __repr__(self) -> str:
        return f"Patch(num_records={self.meta.num_records})"


def _cache_flags(path) -> tuple[bool, bool]:
    with open(path, "rb") as f:
        state = int.from_bytes(f.read(1), byteorder="big")
    return bool(state & (1 << 2)), bool(state & (1 << 3))


def read_patch_data(path) -> np.ndarray:
    """Read a `data.bin` written by the reference: one flag byte, then packed
    float64 records (`src/yaw/catalog/patch.py:164-178`, `src/yaw/datachunk.py:74-112`)."""
    with open(path, "rb") as f:
        state = int.from_bytes(f.read(1), byteorder="big")
        attrs = ["ra", "dec"] + [a for i, a in enumerate(ATTR_ORDER) if i >= 2 and state & (1 << i)]
        raw = np.fromfile(f, dtype=np.byte)
    return raw.view(np.dtype([(a, "f8") for a in attrs]))


def _nearest_center(xyz: np.ndarray, centers_xyz: np.ndarray, engine=None) -> np.ndarray:
    """index of the nearest patch centre in Euclidean xyz (what
    `scipy.cluster.vq.vq` computes in `assign_patch_centers`,
    `src/yaw/catalog/catalog.py:229-249`); with an `engine` the same arithmetic runs on the device
    (`yawb_assign_patches`)"""
    if engine is not None and hasattr(engine, "assign_patches"):
        return engine.assign_patches(xyz, centers_xyz)
    from scipy.cluster import vq

    ids, _ = vq.vq(xyz, centers_xyz)
    return ids.astype(np.int32)


def create_patch_centers(ra, dec, patch_num: int, *, weights=None, probe_size: int = -1,
                         engine=None) -> AngularCoordinates:
    """Centres of `patch_num` patches for the rows `(ra, dec)` (radian): the deterministic spherical k-means of
    `Engine.kmeans` on their `to_3d` positions, with `weights` if given.  It takes the place of the reference's
    treecorr k-means (`create_patch_centers`, `src/yaw/catalog/catalog.py:183-226`) but does not reproduce its centres.

    `probe_size > 0` runs the k-means on every `ceil(n / probe_size)`-th row in input order (this package's
    subsampling rule); the default uses every row.  `engine=None` uses `measurements.get_default_engine()`;
    there is no CPU fallback."""
    patch_num = int(patch_num)
    if patch_num < 1:
        raise ValueError(f"'patch_num' must be at least 1 (got {patch_num})")
    if engine is None:
        from .measurements import get_default_engine

        engine = get_default_engine()
    xyz = AngularCoordinates(np.column_stack([np.asarray(ra, dtype=np.float64), np.asarray(dec, dtype=np.float64)])).to_3d()
    if weights is not None:
        weights = np.asarray(weights, dtype=np.float64)
    if probe_size > 0:
        step = -(-len(xyz) // int(probe_size))
        xyz = xyz[::step]
        weights = None if weights is None else weights[::step]
    centers, _, _, _ = engine.kmeans(xyz, patch_num, weights=weights)
    return AngularCoordinates.from_3d(centers)


class Catalog(Mapping):
    """Mapping patch id -> `Patch`; patch ids are 0..P-1 and iterate in sorted order
    (the reference uses them as array indices, `src/yaw/correlation/measurements.py:358-364`)."""

    _anon_counter = 0

    def __init__(self, patches: dict[int, Patch], cache_directory=None) -> None:
        self._patches = dict(sorted(patches.items()))
        if cache_directory is None:
            Catalog._anon_counter += 1
            cache_directory = f"<memory:{id(self)}:{Catalog._anon_counter}>"
        self.cache_directory = Path(cache_directory)

    # ---- constructors -----------------------------------------------------------------------
    @classmethod
    def from_arrays(cls, ra, dec, *, patch_centers=None, patch_ids=None, patch_num=None, probe_size: int = -1,
                    weights=None, redshifts=None, kappa=None, degrees: bool = True, cache_directory=None,
                    engine=None) -> "Catalog":
        """Patches from `patch_centers` (rows go to the nearest centre), else from `patch_ids`, else from
        `patch_num`: centres of `create_patch_centers` (with the catalog's weights and `probe_size`), then used
        exactly as if they had been passed as `patch_centers`.  `engine`: assign rows to the nearest patch
        centre on the device instead of scipy's vq, and run the k-means there (default: the default engine)."""
        ra = np.asarray(ra, dtype=np.float64)
        dec = np.asarray(dec, dtype=np.float64)
        if degrees:
            ra, dec = np.deg2rad(ra), np.deg2rad(dec)
        weights = None if weights is None else np.asarray(weights, dtype=np.float64)
        redshifts = None if redshifts is None else np.asarray(redshifts, dtype=np.float64)
        kappa = None if kappa is None else np.asarray(kappa, dtype=np.float64)
        if patch_centers is None and patch_ids is None:
            if patch_num is None:
                raise ValueError("one of 'patch_centers', 'patch_ids' and 'patch_num' must be provided")
            patch_centers = create_patch_centers(ra, dec, patch_num, weights=weights, probe_size=probe_size,
                                                 engine=engine)
        centers = None
        if patch_centers is not None:
            if isinstance(patch_centers, Mapping):  # another catalog
                patch_centers = patch_centers.get_centers()
            centers = patch_centers if isinstance(patch_centers, AngularCoordinates) else AngularCoordinates(
                getattr(patch_centers, "data", patch_centers))
            if patch_ids is None:  # with both given, the ids assign rows and the centres fix the meta data
                xyz = AngularCoordinates(np.column_stack([ra, dec])).to_3d()
                patch_ids = _nearest_center(xyz, centers.to_3d(), engine)
        patch_ids = np.asarray(patch_ids)
        order = np.argsort(patch_ids, kind="stable")
        sorted_ids = patch_ids[order]
        uniq, starts = np.unique(sorted_ids, return_index=True)
        ends = np.append(starts[1:], len(order))
        patches = {}
        for pid, s, e in zip(uniq.tolist(), starts, ends):
            sel = order[s:e]
            data = _structured(ra[sel], dec[sel], None if weights is None else weights[sel],
                               None if redshifts is None else redshifts[sel],
                               None if kappa is None else kappa[sel])
            center = None if centers is None else centers[int(pid)]
            patches[int(pid)] = Patch(data, center=center)
        return cls(patches, cache_directory)

    @classmethod
    def from_dataframe(cls, cache_directory, dataframe, *, ra_name, dec_name, weight_name=None,
                       redshift_name=None, patch_centers=None, patch_name=None, patch_num=None,
                       kappa_name=None, degrees: bool = True, probe_size: int = -1, engine=None,
                       **_ignored) -> "Catalog":
        """Signature of `yaw.Catalog.from_dataframe` (`src/yaw/catalog/catalog.py:980-1108`); patches come from
        `patch_centers`, else `patch_name`, else `patch_num` (see `from_arrays`)."""
        get = lambda name: None if name is None else np.asarray(dataframe[name])  # noqa: E731
        return cls.from_arrays(
            get(ra_name), get(dec_name), patch_centers=patch_centers,
            patch_ids=None if patch_centers is not None else get(patch_name),
            patch_num=patch_num, probe_size=probe_size, weights=get(weight_name), redshifts=get(redshift_name),
            kappa=get(kappa_name), degrees=degrees, cache_directory=cache_directory, engine=engine,
        )

    @classmethod
    def from_random(cls, cache_directory, generator, num_randoms: int, *, patch_centers=None, patch_num=None,
                    probe_size: int = -1, engine=None, **_ignored) -> "Catalog":
        """Signature of `yaw.Catalog.from_random` (`src/yaw/catalog/catalog.py:1245-1343`); patches come from
        `patch_centers`, else `patch_num` (see `from_arrays`)."""
        chunk = generator(int(num_randoms))
        return cls.from_arrays(chunk["ra"], chunk["dec"], patch_centers=patch_centers, patch_num=patch_num,
                               probe_size=probe_size,
                               weights=chunk.get("weights"), redshifts=chunk.get("redshifts"),
                               degrees=False, cache_directory=cache_directory, engine=engine)

    @classmethod
    def from_cache(cls, cache_directory) -> "Catalog":
        """Open a catalog cache written by the reference (`patch_ids.bin`,
        `patch_<id>/{data.bin,meta.yml}`, `src/yaw/catalog/catalog.py:70-73, 325-386`)."""
        import yaml

        root = Path(cache_directory)
        info = root / "patch_ids.bin"
        if not info.exists():
            raise InconsistentPatchesError("patch info file not found")
        patches = {}
        for pid in np.fromfile(info, dtype="i2").tolist():
            pdir = root / f"patch_{pid:d}"
            meta = None
            if (pdir / "meta.yml").exists():
                with open(pdir / "meta.yml") as f:
                    d = yaml.safe_load(f)
                meta = Metadata(num_records=d["num_records"], sum_weights=d["sum_weights"],
                                center=AngularCoordinates(d["center"]), radius=AngularDistances(d["radius"]))
            patches[int(pid)] = Patch(None, meta, path=pdir / "data.bin")
        return cls(patches, root)

    # ---- mapping --------------------------------------------------------------------------------
    def __len__(self) -> int:
        return len(self._patches)

    def __getitem__(self, patch_id: int) -> Patch:
        return self._patches[patch_id]

    def __iter__(self):
        yield from sorted(self._patches.keys())

    def __repr__(self) -> str:
        return (f"Catalog(num_patches={self.num_patches}, weights={self.has_weights}, "
                f"redshifts={self.has_redshifts}) @ {self.cache_directory}")

    @property
    def num_patches(self) -> int:
        return len(self)

    @property
    def has_weights(self) -> bool:
        return all(p.has_weights for p in self.values())

    @property
    def has_redshifts(self) -> bool:
        return all(p.has_redshifts for p in self.values())

    @property
    def has_kappa(self) -> bool:
        return all(p.has_kappa for p in self.values())

    def get_num_records(self) -> tuple[int, ...]:
        return tuple(p.meta.num_records for p in self.values())

    def get_sum_weights(self) -> tuple[float, ...]:
        return tuple(p.meta.sum_weights for p in self.values())

    def get_centers(self) -> AngularCoordinates:
        return AngularCoordinates.from_coords(p.meta.center for p in self.values())

    def get_radii(self) -> AngularDistances:
        return AngularDistances(np.concatenate([p.meta.radius.data for p in self.values()]))

    def build_trees(self, binning=None, *, closed: str = "right", **_ignored) -> None:
        """Kept for API compatibility (`src/yaw/catalog/catalog.py:1406-1460`): there are no
        trees to build, the device index is created when the catalog is uploaded."""
        return None
