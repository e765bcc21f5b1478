"""
ORACLE (test infrastructure only; the product never imports it): numpy restatement of the deterministic
spherical k-means behind `yawb_kmeans` (contract: DESIGN.md section 4.4, include/yawb.h).  Every step is integer
arithmetic or correctly rounded float64 elementwise operations, so the device result is reproduced bit for bit.

    kmeans(xyz, k, weights=None, max_iter=500) -> (centers (k, 3), labels (n,) int32, n_iter, converged)
"""

from __future__ import annotations

import numpy as np
from scipy.cluster import vq

SCALE = 2.0**32
MAX_K = 4096


def fixed_point(xyz: np.ndarray, weights: np.ndarray | None = None) -> np.ndarray:
    """q = rint(x 2^32) or, weighted, rint((w x) 2^(32 - e)) with e = frexp(max w)[1]; |q| <= 2^32."""
    if weights is None:
        return np.rint(xyz * SCALE).astype(np.int64)
    e = int(np.frexp(np.max(weights))[1])
    return np.rint((weights[:, None] * xyz) * 2.0 ** (32 - e)).astype(np.int64)


def int_sums(labels: np.ndarray, q: np.ndarray, k: int) -> np.ndarray:
    """(k, 3) exact int64 sums of q per label (sort + reduceat; np.bincount would sum in float64)."""
    order = np.argsort(labels, kind="stable")
    lab = labels[order]
    uniq, starts = np.unique(lab, return_index=True)
    out = np.zeros((k, q.shape[1]), dtype=np.int64)
    if len(uniq):
        out[uniq] = np.add.reduceat(q[order], starts, axis=0)
    return out


def centre(s: np.ndarray) -> np.ndarray:
    """c = s / sqrt((s_x s_x + s_y s_y) + s_z s_z) of the int64 sums, every operation correctly rounded."""
    s = s.astype(np.float64)
    norm = np.sqrt((s[:, 0] * s[:, 0] + s[:, 1] * s[:, 1]) + s[:, 2] * s[:, 2])
    with np.errstate(invalid="ignore", divide="ignore"):
        return s / norm[:, None]


def assign(xyz: np.ndarray, centers: np.ndarray) -> np.ndarray:
    return vq.vq(xyz, centers, check_finite=False)[0].astype(np.int32)


def sq_dist(xyz: np.ndarray, centers: np.ndarray, labels: np.ndarray) -> np.ndarray:
    """the squared distance vq minimises (differences centre - row, summed x -> y -> z) to the own centre"""
    d = centers[labels] - xyz
    return (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]


def bisect(q: np.ndarray, k: int, trace: list | None = None) -> np.ndarray:
    """cell labels of the deterministic bisection; `trace` collects (parent, axis, child) per split"""
    n = len(q)
    lab = np.zeros(n, dtype=np.int64)
    c = 1
    while c < k:
        cnt = np.bincount(lab, minlength=c)
        lo = np.full((c, 3), np.iinfo(np.int64).max, dtype=np.int64)
        hi = np.full((c, 3), np.iinfo(np.int64).min, dtype=np.int64)
        for a in range(3):
            np.minimum.at(lo[:, a], lab, q[:, a])
            np.maximum.at(hi[:, a], lab, q[:, a])
        ext = hi - lo
        splittable = [j for j in range(c) if ext[j].max() > 0]
        chosen = sorted(sorted(splittable, key=lambda j: (-cnt[j], j))[: min(c, k - c)])
        if not chosen:
            raise ValueError("fewer distinct positions than patches")
        s = int_sums(lab, q, c)
        new = lab.copy()
        for r, j in enumerate(chosen):
            axis = int(np.argmax(ext[j]))  # first maximum: ties go to x, then y, then z
            high = (lab == j) & (q[:, axis] * cnt[j] > s[j, axis])
            new[high] = c + r
            if trace is not None:
                trace.append((j, axis, c + r))
        lab = new
        c += len(chosen)
    return lab


def kmeans(xyz, k: int, weights=None, max_iter: int = 500, stats: dict | None = None):
    """`stats` (optional dict) receives `relocated`: list of (iteration, cluster, row) of empty-cluster moves."""
    xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
    n = len(xyz)
    if not (1 <= k <= MAX_K and k <= n < 2**30 and max_iter >= 0):
        raise ValueError("need 1 <= k <= 4096, k <= n < 2^30 and max_iter >= 0")
    if not np.all(np.abs(xyz) <= 1.0):
        raise ValueError("rows must be finite with |coordinate| <= 1")
    if weights is not None:
        weights = np.ascontiguousarray(weights, dtype=np.float64)
        if not (np.all(np.isfinite(weights)) and np.all(weights >= 0.0) and weights.max() >= 2.0**-992):
            raise ValueError("weights must be finite, >= 0, and the largest at least 2^-992")
    relocated = []
    q_init = fixed_point(xyz)
    q = q_init if weights is None else fixed_point(xyz, weights)
    C = centre(int_sums(bisect(q_init, k), q_init, k))
    L = assign(xyz, C)
    it, converged = 0, False
    while it < max_iter:
        s = int_sums(L, q, k)
        Cn = centre(s)
        empty = np.flatnonzero(~s.any(axis=1))
        if len(empty):
            d = sq_dist(xyz, C, L)
            order = np.lexsort((np.arange(n), -d))  # largest distance first, ties: lowest row
            for j, row in zip(empty, order):
                Cn[j] = xyz[row]
                relocated.append((it + 1, int(j), int(row)))
        Ln = assign(xyz, Cn)
        it += 1
        changed = np.count_nonzero(Ln != L)
        C, L = Cn, Ln
        if changed == 0:
            converged = True
            break
    if stats is not None:
        stats["relocated"] = relocated
    return C, L, it, converged
