"""
ORACLE -- TEST INFRASTRUCTURE ONLY.  Not imported by the product package.

CPU restatement (numpy / plain C brute force) of the reference's pair-counting
hot path.  Only `tests/`, `__graft_entry__.smoke()` and the `cpu_baseline` leg
of `bench.py` may import this module; the product path
(`yet_another_wizz_b200`) never does and fails loudly without its CUDA library.

Parity status: PINNED.  The restatement is checked against
  * the reference's own known-answer tests `tests/catalog/test_trees.py:181-254`
    (restated in `tests/test_oracle.py`),
  * golden vectors produced by running the unmodified reference in the build
    container (`tests/golden/make_golden.py` -> `tests/golden/*.npz`),
  * the live reference when `/root/reference` is present
    (`tests/test_vs_reference.py::test_oracle_against_live_reference`).

The arithmetic that the reference delegates to scipy's compiled
`cKDTree.count_neighbors` (scipy 1.18.1 in this image; unpinned in the
reference's `pyproject.toml:25`) is restated from its published contract and
from probes of its behaviour (SURVEY.md section 7, hard parts 2-3):

    a pair (a, b) falls into sub-bin k  iff  r2[k-1] < d2 <= r2[k]
    d2 = (dx*dx + dy*dy) + dz*dz     IEEE double, no FMA, summed x->y->z
    r2[k] = pow(r[k], 2.0)           libm pow, not r*r

Each function cites the reference file:line it follows (paths relative to
`/root/reference/`).
"""

from __future__ import annotations

import ctypes
import math
import os
from itertools import compress

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_CLIB_PATH = os.path.join(_HERE, "_build", "libpaircount_ref.so")
_clib = None


# --------------------------------------------------------------------------- #
# geometry helpers
# --------------------------------------------------------------------------- #
def radec_to_xyz(ra: np.ndarray, dec: np.ndarray) -> np.ndarray:
    """`AngularCoordinates.to_3d`, src/yaw/coordinates.py:134-147."""
    cos_dec = np.cos(dec)
    return np.column_stack([np.cos(ra) * cos_dec, np.sin(ra) * cos_dec, np.sin(dec)])


def xyz_to_radec(xyz: np.ndarray) -> np.ndarray:
    """`AngularCoordinates.from_3d`, src/yaw/coordinates.py:110-132."""
    x, y, z = np.transpose(np.atleast_2d(xyz))
    r_d2 = np.sqrt(x * x + y * y)
    r_d3 = np.sqrt(x * x + y * y + z * z)
    x_normed = np.ones_like(x)
    np.divide(x, r_d2, where=r_d2 > 0.0, out=x_normed)
    sgn = np.where(y == 0.0, 1.0, np.sign(y))  # src/yaw/coordinates.py `sgn`: sign with 0 -> +1
    ra = np.arccos(x_normed) * sgn % (2.0 * np.pi)
    dec = np.arcsin(z / r_d3)
    return np.column_stack([ra, dec])


def angle_to_chord(theta: np.ndarray) -> np.ndarray:
    """`AngularDistances.to_3d`, src/yaw/coordinates.py:270-277."""
    return 2.0 * np.sin(np.asarray(theta, dtype=np.float64) / 2.0)


def chord_to_angle(chord: np.ndarray) -> np.ndarray:
    """`AngularDistances.from_3d`, src/yaw/coordinates.py:245-268."""
    return 2.0 * np.arcsin(np.asarray(chord, dtype=np.float64) / 2.0)


def angular_distance(radec1: np.ndarray, radec2: np.ndarray) -> np.ndarray:
    """`AngularCoordinates.distance`, src/yaw/coordinates.py:183-205."""
    a = radec_to_xyz(radec1[:, 0], radec1[:, 1])
    b = radec_to_xyz(radec2[:, 0], radec2[:, 1])
    return chord_to_angle(np.sqrt(((a - b) ** 2).sum(axis=1)))


# --------------------------------------------------------------------------- #
# angular bin bookkeeping (src/yaw/catalog/trees.py:46-160)
# --------------------------------------------------------------------------- #
def parse_ang_limits(ang_min, ang_max) -> np.ndarray:
    """src/yaw/catalog/trees.py:46-81."""
    ang_min = np.atleast_1d(ang_min).astype(np.float64)
    ang_max = np.atleast_1d(ang_max).astype(np.float64)
    if ang_min.ndim != 1 or ang_max.ndim != 1:
        raise ValueError("'ang_min' and 'ang_max' must be 1-dim")
    if len(ang_min) != len(ang_max):
        raise ValueError("length of 'ang_min' and 'ang_max' does not match")
    if np.any(ang_min >= ang_max):
        raise ValueError("'ang_min' < 'ang_max' not satisfied")
    ang_range = np.column_stack((ang_min, ang_max))
    if np.any(ang_range < 0.0) or np.any(ang_range > np.pi):
        raise ValueError("'ang_min' and 'ang_max' not in range [0.0, pi]")
    return ang_range


def get_ang_bins(ang_range: np.ndarray, weight_scale, weight_res) -> np.ndarray:
    """src/yaw/catalog/trees.py:84-117."""
    with np.errstate(divide="ignore"):
        log_range = np.log10(ang_range)
    if weight_scale is not None:
        log_bins = np.linspace(log_range.min(), log_range.max(), weight_res + 1)
        log_bins = np.concatenate([log_bins, log_range.flatten()])
    else:
        log_bins = log_range.flatten()
    return 10.0 ** np.sort(np.unique(log_bins))


def logarithmic_mid(edges: np.ndarray) -> np.ndarray:
    """src/yaw/catalog/trees.py:120-124."""
    log_edges = np.log10(edges)
    return 10.0 ** ((log_edges[:-1] + log_edges[1:]) / 2.0)


def get_counts_for_limits(counts, ang_bins, ang_limits) -> np.ndarray:
    """src/yaw/catalog/trees.py:134-160."""
    final = np.empty(len(ang_limits), dtype=counts.dtype)
    for i, (ang_min, ang_max) in enumerate(ang_limits):
        idx_min = np.argmin(np.abs(ang_bins - ang_min))
        idx_max = np.argmin(np.abs(ang_bins - ang_max))
        final[i] = counts[idx_min:idx_max].sum()
    return final


def chord_sq_edges(ang_bins: np.ndarray) -> np.ndarray:
    """Squared chord thresholds exactly as scipy forms them: libm pow(r, 2.0)
    of `AngularDistances(ang_bins).to_3d()` (src/yaw/catalog/trees.py:350)."""
    r = angle_to_chord(ang_bins)
    return np.array([math.pow(float(x), 2.0) for x in r], dtype=np.float64)


# --------------------------------------------------------------------------- #
# the pair-count primitive (scipy cKDTree.count_neighbors restated)
# --------------------------------------------------------------------------- #
def _load_clib():
    global _clib
    if _clib is None and os.path.exists(_CLIB_PATH):
        lib = ctypes.CDLL(_CLIB_PATH)
        dp = ctypes.POINTER(ctypes.c_double)
        lib.paircount_ref.restype = None
        lib.paircount_ref.argtypes = [
            dp, ctypes.c_int64, dp, dp, ctypes.c_int64, dp, dp, ctypes.c_int,
            ctypes.POINTER(ctypes.c_int64), dp,
        ]
        _clib = lib
    return _clib


def _as_dp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double)) if a is not None else None


def pair_histogram(xyz1, xyz2, w1, w2, r2, *, use_c: bool | None = None):
    """
    Sub-bin histogram of all pairs between two point sets.

    Returns `(n_edges - 1,)`: int64 if both sides are unweighted, else float64
    (mirrors scipy: `weights=(None, None)` -> integer counts,
    src/yaw/catalog/trees.py:348-353; SURVEY.md Appendix A.4).

    hist[k-1] += w1[a] * w2[b]   for   r2[k-1] < d2 <= r2[k],  1 <= k < len(r2)
    """
    xyz1 = np.ascontiguousarray(xyz1, dtype=np.float64).reshape(-1, 3)
    xyz2 = np.ascontiguousarray(xyz2, dtype=np.float64).reshape(-1, 3)
    r2 = np.ascontiguousarray(r2, dtype=np.float64)
    nsub = len(r2) - 1
    weighted = (w1 is not None) or (w2 is not None)
    n1, n2 = len(xyz1), len(xyz2)
    if n1 == 0 or n2 == 0:
        return np.zeros(nsub, dtype=np.float64 if weighted else np.int64)

    if w1 is not None:
        w1 = np.ascontiguousarray(w1, dtype=np.float64)
    if w2 is not None:
        w2 = np.ascontiguousarray(w2, dtype=np.float64)

    lib = _load_clib() if use_c in (None, True) else None
    if use_c is True and lib is None:
        raise RuntimeError("oracle C library not built (run `make -C oracle`)")
    if lib is not None:
        hi = np.zeros(nsub, dtype=np.int64)
        hf = np.zeros(nsub, dtype=np.float64)
        lib.paircount_ref(
            _as_dp(xyz1), n1, _as_dp(w1), _as_dp(xyz2), n2, _as_dp(w2),
            _as_dp(r2), len(r2), hi.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), _as_dp(hf),
        )
        return hf if weighted else hi

    # numpy path: chunk rows of set 1 so a block holds <= ~4e6 pairs
    hist = np.zeros(nsub, dtype=np.float64 if weighted else np.int64)
    step = max(1, 4_000_000 // n2)
    x2, y2, z2 = xyz2[:, 0], xyz2[:, 1], xyz2[:, 2]
    for lo in range(0, n1, step):
        a = xyz1[lo : lo + step]
        dx = a[:, 0:1] - x2[None, :]
        dy = a[:, 1:2] - y2[None, :]
        dz = a[:, 2:3] - z2[None, :]
        d2 = (dx * dx + dy * dy) + dz * dz  # separate roundings, x->y->z
        k = np.searchsorted(r2, d2.ravel(), side="left")
        keep = (k >= 1) & (k <= nsub)
        if weighted:
            wa = np.ones(len(a)) if w1 is None else w1[lo : lo + step]
            wb = np.ones(n2) if w2 is None else w2
            ww = (wa[:, None] * wb[None, :]).ravel()
            hist += np.bincount(k[keep] - 1, weights=ww[keep], minlength=nsub)[:nsub]
        else:
            hist += np.bincount(k[keep] - 1, minlength=nsub)[:nsub]
    return hist


def binned_pair_counts(
    xyz1, patch1, zbin1, xyz2, patch2, pair_i, pair_j, r2, *,
    w1=None, w2=None, zbin2=None, label1=None, label2=None, n_labels: int = 1,
):
    """
    `pair_histogram` of every (patch pair, z-bin) of a pair list at once, for catalogs far too large for a brute
    force per (pair, z-bin): the layout of `yawb_count`'s results, `(n_labels, n_pairs, n_bins, n_edges - 1)`.

    Row a of the first catalog (patch `patch1[a]`, z-bin `zbin1[a]`; < 0 = dropped) meets row b of the second one
    iff `zbin2` is None (unbinned) or `zbin2[b] == zbin1[a]`, and `label1` is None or `label1[a] == label2[b]`.
    The pair goes to output block `label2[b]` (0 without labels; < 0 = dropped), patch pair k with
    `(pair_i[k], pair_j[k]) == (patch1[a], patch2[b])`, z-bin `zbin1[a]`, and sub-bin k with
    `r2[z][k-1] < d2 <= r2[z][k]` (`r2`: `(n_bins, n_edges)`).

    A k-d tree only SELECTS candidate pairs, with the search radius of the device kernel
    (`sqrt(max r2) (1 + 1e-9) + 1e-14`, far beyond the rounding of its own distances); every candidate is then
    decided by the reference expression `(dx*dx + dy*dy) + dz*dz` in float64 and `searchsorted(..., "left")`, as in
    `pair_histogram`.  Returns `(counts int64, sums float64)`: counts exact, sums of `w1[a] * w2[b]` correctly
    rounded (`math.fsum` per entry; the counts as floats if neither catalog is weighted).
    """
    from scipy.spatial import cKDTree

    xyz1 = np.ascontiguousarray(xyz1, dtype=np.float64).reshape(-1, 3)
    xyz2 = np.ascontiguousarray(xyz2, dtype=np.float64).reshape(-1, 3)
    r2 = np.atleast_2d(np.asarray(r2, dtype=np.float64))
    n_bins, n_edges = r2.shape
    nsub = n_edges - 1
    pair_i = np.asarray(pair_i, dtype=np.int64)
    pair_j = np.asarray(pair_j, dtype=np.int64)
    n_pairs = len(pair_i)
    patch1 = np.asarray(patch1, dtype=np.int64)
    patch2 = np.asarray(patch2, dtype=np.int64)
    zb1 = np.asarray(zbin1, dtype=np.int64)
    lab2 = np.zeros(len(xyz2), dtype=np.int64) if label2 is None else np.asarray(label2, dtype=np.int64)
    shape = (n_labels, n_pairs, n_bins, nsub)
    counts = np.zeros(int(np.prod(shape)), dtype=np.int64)
    weighted = w1 is not None or w2 is not None
    sums = np.zeros(counts.shape, dtype=np.float64)
    if n_pairs == 0 or len(xyz1) == 0 or len(xyz2) == 0:
        return counts.reshape(shape), sums.reshape(shape)

    n_patch = int(max(patch1.max(initial=0), patch2.max(initial=0), pair_i.max(), pair_j.max())) + 1
    pair_of = np.full((n_patch, n_patch), -1, dtype=np.int64)
    if len(set(zip(pair_i.tolist(), pair_j.tolist()))) != n_pairs:
        raise ValueError("pair list has repeated patch pairs")
    pair_of[pair_i, pair_j] = np.arange(n_pairs)

    # rows that can meet share a group key: (z-bin if the second catalog is binned, label if the first is labelled)
    live1 = (zb1 >= 0) & (zb1 < n_bins)
    if label1 is not None:
        live1 &= np.asarray(label1) >= 0
    live2 = (lab2 >= 0) & (lab2 < n_labels)
    g1 = np.zeros(len(xyz1), dtype=np.int64)
    g2 = np.zeros(len(xyz2), dtype=np.int64)
    if zbin2 is not None:
        zb2 = np.asarray(zbin2, dtype=np.int64)
        live2 &= zb2 >= 0
        g1 = g1 * (n_bins + 1) + zb1
        g2 = g2 * (n_bins + 1) + zb2
    if label1 is not None:
        g1 = g1 * (n_labels + 1) + np.asarray(label1, dtype=np.int64)
        g2 = g2 * (n_labels + 1) + lab2
    rmax = math.sqrt(float(r2[:, -1].max())) * (1.0 + 1e-9) + 1e-14

    flat_all, prod_all = [], []
    for g in np.intersect1d(g1[live1], g2[live2]):
        ia = np.flatnonzero(live1 & (g1 == g))
        ib = np.flatnonzero(live2 & (g2 == g))
        cand = cKDTree(xyz1[ia]).sparse_distance_matrix(cKDTree(xyz2[ib]), rmax, output_type="coo_matrix")
        a, b = ia[cand.row], ib[cand.col]
        kp = pair_of[patch1[a], patch2[b]]
        a, b, kp = a[kp >= 0], b[kp >= 0], kp[kp >= 0]
        d = xyz1[a] - xyz2[b]
        dx, dy, dz = d[:, 0], d[:, 1], d[:, 2]
        d2 = (dx * dx + dy * dy) + dz * dz  # separate roundings, x -> y -> z
        z = zb1[a]
        k = np.zeros(len(a), dtype=np.int64)
        for zz in np.unique(z):
            m = z == zz
            k[m] = np.searchsorted(r2[zz], d2[m], side="left")
        keep = (k >= 1) & (k <= nsub)
        a, b, kp, z, k = a[keep], b[keep], kp[keep], z[keep], k[keep]
        flat = ((lab2[b] * n_pairs + kp) * n_bins + z) * nsub + (k - 1)
        counts += np.bincount(flat, minlength=len(counts))
        if weighted:
            flat_all.append(flat)
            prod_all.append((np.ones(len(a)) if w1 is None else np.asarray(w1)[a]) *
                            (np.ones(len(b)) if w2 is None else np.asarray(w2)[b]))
    if weighted and flat_all:
        flat, prod = np.concatenate(flat_all), np.concatenate(prod_all)
        order = np.argsort(flat, kind="stable")
        flat, prod = flat[order], prod[order]
        cells, start = np.unique(flat, return_index=True)
        sums[cells] = [math.fsum(c) for c in np.split(prod, start[1:])]
    elif not weighted:
        sums = counts.astype(np.float64)
    return counts.reshape(shape), sums.reshape(shape)


def tree_count(
    xyz1, w1, xyz2, w2, ang_min, ang_max, *, weight_scale=None, weight_res=50, use_c=None
) -> np.ndarray:
    """
    `AngularTree.count`, src/yaw/catalog/trees.py:303-362, with the cKDTree
    query replaced by the brute-force histogram.  Returns float64 `(n_scales,)`.
    """
    ang_limits = parse_ang_limits(ang_min, ang_max)
    ang_bins = get_ang_bins(ang_limits, weight_scale, weight_res)
    if len(xyz1) == 0 or len(xyz2) == 0:  # trees.py:344-345
        return np.zeros(len(ang_limits))
    r2 = chord_sq_edges(ang_bins)
    counts = pair_histogram(xyz1, xyz2, w1, w2, r2, use_c=use_c).astype(np.float64)
    if weight_scale is not None:  # trees.py:358-360
        ang_weights = logarithmic_mid(ang_bins) ** weight_scale
        counts *= ang_weights / ang_weights.sum()
    return get_counts_for_limits(counts, ang_bins, ang_limits)


# --------------------------------------------------------------------------- #
# patch level (src/yaw/correlation/measurements.py)
# --------------------------------------------------------------------------- #
class OraclePatch:
    """Plain-array stand-in for a reference `Patch` (+ its `BinnedTrees`)."""

    def __init__(self, ra, dec, weights=None, redshifts=None):
        self.ra = np.asarray(ra, dtype=np.float64)
        self.dec = np.asarray(dec, dtype=np.float64)
        self.weights = None if weights is None else np.asarray(weights, dtype=np.float64)
        self.redshifts = None if redshifts is None else np.asarray(redshifts, dtype=np.float64)
        self.xyz = radec_to_xyz(self.ra, self.dec)

    def __len__(self):
        return len(self.ra)

    # `Metadata.compute`, src/yaw/catalog/patch.py:104-147
    def center_radius(self):
        mean_xyz = np.average(self.xyz, weights=self.weights, axis=0)
        center = xyz_to_radec(mean_xyz)
        radius = angular_distance(
            np.column_stack([self.ra, self.dec]), np.broadcast_to(center, (len(self), 2))
        ).max()
        return center[0], float(radius)

    def bin_slices(self, zedges, closed):
        """`build_trees`, src/yaw/catalog/trees.py:402-427: list of
        (xyz, w, sum_weights) per z-bin, or a single entry if `zedges` is None."""
        if zedges is None:
            sw = float(len(self)) if self.weights is None else float(self.weights.sum())
            return [(self.xyz, self.weights, sw)]
        if self.redshifts is None:
            raise ValueError("patch has no 'redshifts' attached")
        idx = np.digitize(self.redshifts, zedges, right=(closed == "right"))
        out = []
        for b in range(1, len(zedges)):
            m = idx == b
            w = None if self.weights is None else self.weights[m]
            # empty bins: AngularTree.empty -> sum_weights 0.0 (trees.py:249-258)
            sw = float(m.sum()) if w is None else float(w.sum())
            out.append((self.xyz[m], w, sw))
        return out


def compute_linkage(centers_radec, radii, max_angle) -> dict[int, set[int]]:
    """`PatchLinkage.from_catalogs`, src/yaw/correlation/measurements.py:226-235
    (centres/radii of the reference catalog chosen by the caller)."""
    n = len(radii)
    ids = list(range(n))
    links = {}
    for i in range(n):
        d = angular_distance(centers_radec, np.broadcast_to(centers_radec[i], (n, 2)))
        linked = d < (radii + radii[i] + max_angle)
        links[i] = set(compress(ids, linked))
    return links


def linked_pairs(links: dict[int, set[int]], auto: bool) -> list[tuple[int, int]]:
    """Set of pairs visited by `iter_patch_id_pairs`,
    src/yaw/correlation/measurements.py:258-289 (order is irrelevant)."""
    out = []
    for i, js in links.items():
        for j in sorted(js):
            if i == j or (not auto) or j > i:
                out.append((i, j))
    return out


def count_pairs(
    patches1, patches2, links, *, zedges, closed, ang_min, ang_max,
    rweight=None, resolution=None, use_c=None,
):
    """
    `PatchLinkage.count_pairs` + `process_patch_pair`,
    src/yaw/correlation/measurements.py:88-128, 307-367.

    `patches2=None` -> autocorrelation (`auto=True`).  `ang_min/ang_max` have
    shape `(n_bins, n_scales)` (the reference's `get_angle_radian(zmid[b])`).
    The first catalog is always z-binned; the second is binned iff auto or
    `binned2` patches carry redshifts AND the caller passes them binned -- the
    reference only ever uses (binned, binned) [autocorrelate :508-510] and
    (binned, unbinned) [crosscorrelate :597-607].

    Returns `(sum_weights1, sum_weights2, counts)` with shapes
    `(n_bins, P)`, `(n_bins, P)`, `(n_scales, n_bins, P, P)`.
    """
    auto = patches2 is None
    binned2 = auto
    if isinstance(patches2, tuple):  # (patches, "binned")
        patches2, flag = patches2
        binned2 = flag == "binned"
    if auto:
        patches2 = patches1
    P = len(patches1)
    n_bins = len(zedges) - 1
    ang_min = np.asarray(ang_min, dtype=np.float64).reshape(n_bins, -1)
    ang_max = np.asarray(ang_max, dtype=np.float64).reshape(n_bins, -1)
    n_scales = ang_min.shape[1]

    slices1 = [p.bin_slices(zedges, closed) for p in patches1]
    if binned2:
        slices2 = slices1 if auto else [p.bin_slices(zedges, closed) for p in patches2]
    else:
        slices2 = [p.bin_slices(None, closed) * n_bins for p in patches2]

    sw1 = np.zeros((n_bins, P))
    sw2 = np.zeros((n_bins, P))
    counts = np.zeros((n_scales, n_bins, P, P))
    for i, j in linked_pairs(links, auto):
        for b in range(n_bins):
            xyz1, w1, s1 = slices1[i][b]
            xyz2, w2, s2 = slices2[j][b]
            c = tree_count(
                xyz1, w1, xyz2, w2, ang_min[b], ang_max[b],
                weight_scale=rweight, weight_res=resolution, use_c=use_c,
            )
            if auto and i == j:
                c = c * 0.5  # measurements.py:362-363
            counts[:, b, i, j] = c
            sw1[b, i] = s1
            sw2[b, j] = s2
    return sw1, sw2, counts
