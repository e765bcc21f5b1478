"""
Multi-GPU partitioning of patch-pair work (replaces the dynamic master/worker queue of
`yaw.utils.parallel`, reference `src/yaw/utils/parallel.py:251-343`).

One process per GPU (`torch.distributed`, NCCL over NVLink on the B200 box, gloo in CPU
tests).  Work units are patch pairs; they are independent (the reference only scatters
their results, `src/yaw/correlation/measurements.py:354-364`), so the pairs are assigned
statically by longest-processing-time-first on a cost model, every rank counts its share
into a zero-initialised result tensor and ONE sum-reduce to rank 0 finishes the job.
Every element has exactly one non-zero contributor, so the reduction is exact and
deterministic for integers and floats alike.
"""

from __future__ import annotations

import heapq
import os

import numpy as np

__all__ = ["SharePlan", "Shard", "assign_pairs_lpt", "assign_patches_contiguous", "assign_patch_fractions", "split_rows",
           "current_shard", "pair_costs", "plan_passes", "plan_shares"]


def pair_costs(pair_i, pair_j, n1_per_patch, n2_per_patch, radii1=None) -> np.ndarray:
    """Predicted cost of each patch pair after pruning: diagonal pairs carry nearly all of the work (SURVEY.md
    section 3.1: ~95 %), neighbours only a boundary strip.  The executed pair tests of a pair scale with the rows
    of the second patch times the surface DENSITY of the first one (every tile of the second catalog meets the rows
    of the first inside its search box), so with the patch radii of the first catalog the cost is
    n1(i) / radius(i)^2 * n2(j); without them n1(i) * n2(j), which overrates large patches (measured on the C3
    benchmark, 8 ranks: most loaded rank 12 % above the mean with the product, 3 % with the density)."""
    pair_i = np.asarray(pair_i)
    pair_j = np.asarray(pair_j)
    w1 = np.asarray(n1_per_patch, dtype=np.float64)
    if radii1 is not None:
        r = np.asarray(radii1, dtype=np.float64)
        area = np.where(r > 0.0, r * r, np.inf)
        w1 = w1 / area
        w1 = w1 / max(float(w1.max()), 1e-300) * float(np.max(n1_per_patch))  # keep the scale of a row count
    cost = w1[pair_i] * np.asarray(n2_per_patch, dtype=np.float64)[pair_j]
    off = pair_i != pair_j
    cost[off] *= 0.05
    return cost + 1.0


def assign_pairs_lpt(costs: np.ndarray, world_size: int) -> list[np.ndarray]:
    """Longest-processing-time-first bin packing; returns the pair indices of every rank."""
    order = np.argsort(-np.asarray(costs), kind="stable")
    heap = [(0.0, r) for r in range(world_size)]
    heapq.heapify(heap)
    owned: list[list[int]] = [[] for _ in range(world_size)]
    for k in order:
        load, r = heapq.heappop(heap)
        owned[r].append(int(k))
        heapq.heappush(heap, (load + float(costs[k]), r))
    return [np.array(sorted(o), dtype=np.int64) for o in owned]


def _morton_order(centers_xyz: np.ndarray) -> np.ndarray:
    """patches ordered along a Morton curve of their centres (longitude unwrapped around the mean direction, z)"""
    xyz = np.asarray(centers_xyz, dtype=np.float64)
    lon = np.arctan2(xyz[:, 1], xyz[:, 0])
    # unwrap around the mean direction so a field that straddles RA = 0 stays contiguous
    mean_lon = np.arctan2(xyz[:, 1].sum(), xyz[:, 0].sum())
    lon = (lon - mean_lon + np.pi) % (2 * np.pi)
    def quant(v):
        span = v.max() - v.min()
        return np.zeros(len(v), dtype=np.uint64) if span <= 0 else ((v - v.min()) / span * 1023).astype(np.uint64)
    qx, qy = quant(lon), quant(xyz[:, 2])
    code = np.zeros(len(xyz), dtype=np.uint64)
    for bit in range(10):
        code |= ((qx >> np.uint64(bit)) & np.uint64(1)) << np.uint64(2 * bit)
        code |= ((qy >> np.uint64(bit)) & np.uint64(1)) << np.uint64(2 * bit + 1)
    return np.argsort(code, kind="stable")


def assign_patches_contiguous(patch_costs: np.ndarray, centers_xyz: np.ndarray, world_size: int) -> list[np.ndarray]:
    """Deal patches to ranks as spatially compact groups of about equal cost: patches are ordered along a
    Morton curve of their centres (longitude, z) and the order is cut where the running cost crosses
    k / world_size of the total.  A rank then needs few first-catalog patches beyond its own (only the
    neighbours across the cut), which keeps per-rank uploads and index builds ~1/world_size."""
    patch_costs = np.asarray(patch_costs, dtype=np.float64)
    order = _morton_order(centers_xyz)
    csum = np.cumsum(patch_costs[order])
    total = csum[-1] if len(csum) else 0.0
    bounds = [0]
    for r in range(1, world_size):
        bounds.append(min(len(order), int(np.searchsorted(csum, total * r / world_size * (1 - 1e-12), side="left")) + 1))
    bounds.append(len(order))
    bounds = np.maximum.accumulate(bounds)
    return [np.sort(order[bounds[r]:bounds[r + 1]]) for r in range(world_size)]


def assign_patch_fractions(patch_costs: np.ndarray, centers_xyz: np.ndarray, world_size: int,
                           min_fraction: float = 0.03) -> list[list[tuple[int, float, float]]]:
    """The same compact groups, cut EXACTLY at k / world_size of the total cost: the patch a cut falls into is
    shared by the two ranks, each taking a fraction [f0, f1) of its second-catalog rows (work items are tiles of the
    second catalog, so any subset of a patch's rows is a valid share; `split_rows` makes the subsets compact).
    With 64 patches on 8 ranks whole patches leave the most loaded rank 12 % above the mean (C3 benchmark);
    fractions bring that to the accuracy of the cost model.  Slivers below `min_fraction` of a patch are not
    worth a second copy of its first-catalog neighbours: such a cut snaps to the patch boundary.
    Returns, per rank, a list of (patch, f0, f1)."""
    patch_costs = np.asarray(patch_costs, dtype=np.float64)
    order = _morton_order(centers_xyz)
    cost = patch_costs[order]
    total = float(cost.sum())
    hi = np.cumsum(cost)
    lo = hi - cost
    cuts = [0.0]
    for r in range(1, world_size):
        c = total * r / world_size
        k = int(np.searchsorted(hi, c, side="right"))  # the patch the cut falls into
        if k < len(order) and cost[k] > 0.0:
            f = (c - lo[k]) / cost[k]
            if f < min_fraction:
                c = lo[k]
            elif f > 1.0 - min_fraction:
                c = hi[k]
        cuts.append(max(c, cuts[-1]))
    cuts.append(total)
    shares: list[list[tuple[int, float, float]]] = []
    for r in range(world_size):
        a, b = cuts[r], cuts[r + 1]
        mine = []
        for k, p in enumerate(order):
            if cost[k] <= 0.0:
                if a <= lo[k] < b or (r == world_size - 1 and lo[k] >= b):
                    mine.append((int(p), 0.0, 1.0))  # empty patches travel with their position on the curve
                continue
            f0 = min(max((a - lo[k]) / cost[k], 0.0), 1.0)
            f1 = min(max((b - lo[k]) / cost[k], 0.0), 1.0)
            if f1 - f0 > 1e-12:
                mine.append((int(p), float(f0), float(f1)))
        shares.append(mine)
    return shares


def split_rows(xyz: np.ndarray, f0: float, f1: float) -> np.ndarray:
    """Indices of the rows of ONE patch that make up its fraction [f0, f1): the rows are ordered along the longer
    axis of the patch (longitude or latitude), so every share is a compact strip.  Deterministic: every rank
    derives the same strips."""
    n = len(xyz)
    if f0 <= 0.0 and f1 >= 1.0:
        return np.arange(n)
    xyz = np.asarray(xyz, dtype=np.float64)
    lat = np.arcsin(np.clip(xyz[:, 2], -1.0, 1.0))
    mean_lon = np.arctan2(xyz[:, 1].sum(), xyz[:, 0].sum())
    lon = (np.arctan2(xyz[:, 1], xyz[:, 0]) - mean_lon + np.pi) % (2 * np.pi)
    span_lon = (lon.max() - lon.min()) * np.cos(lat.mean()) if n else 0.0
    key = lon if span_lon >= (lat.max() - lat.min() if n else 0.0) else lat
    order = np.argsort(key, kind="stable")
    return np.sort(order[int(round(f0 * n)):int(round(f1 * n))])


class SharePlan:
    """Which device of an `EngineGroup` holds and counts what in one measurement call.

    `shares[d]`: the (patch, f0, f1) of `assign_patch_fractions` -- device d counts the pairs whose second patch is one of
    these, against the `split_rows` strip [f0, f1) of that patch's rows (a patch split between two devices is counted
    by both, each on its own strip).  `keep[d]`: the patches device d uploads, its own plus every patch linked to one of
    them in a pair list of the call, so that one upload per catalog and device serves as first and as second catalog."""

    def __init__(self, shares: list[list[tuple[int, float, float]]], keep: list[np.ndarray]) -> None:
        self.shares = shares
        self.keep = keep
        n_patch = len(keep[0]) if keep else 0
        self.second = []  # per device: (n_patch,) bool, the second patches it counts
        for mine in shares:
            own = np.zeros(n_patch, dtype=bool)
            own[[p for p, _, _ in mine]] = True
            self.second.append(own)

    @property
    def n_devices(self) -> int:
        return len(self.shares)

    def mask(self, d: int, xyz: np.ndarray, patch_off: np.ndarray) -> np.ndarray:
        """second-role rows of device d: one byte per row of its kept patches (in patch order), 1 for the rows of its
        strips.  `xyz` / `patch_off`: the whole catalog."""
        keep = self.keep[d].astype(bool)
        sizes = np.diff(patch_off)
        dev_off = np.concatenate([[0], np.cumsum(np.where(keep, sizes, 0))])
        out = np.zeros(int(dev_off[-1]), dtype=np.uint8)
        for p, f0, f1 in self.shares[d]:
            s, e = int(patch_off[p]), int(patch_off[p + 1])
            out[dev_off[p] + split_rows(xyz[s:e], f0, f1)] = 1
        return out

    def signature(self, d: int) -> tuple:
        """what device d's uploads depend on besides the catalog: its kept patches and strips (they fix the mask)"""
        return (self.keep[d].tobytes(), tuple(self.shares[d]))


def plan_shares(counts, radii1, centers_xyz, n_devices: int) -> SharePlan:
    """The share plan of one call.  `counts`: the pair counts of the call, each `(pair_i, pair_j, n1_per_patch,
    n2_per_patch)` with `pair_j` the patches of the second catalog.  The cost of a second patch is the sum of
    `pair_costs` over every pair that names it; `assign_patch_fractions` cuts the patches, ordered along the curve of
    their centres, into `n_devices` parts of equal cost."""
    n_patch = len(centers_xyz)
    cost = np.zeros(n_patch)
    for pi, pj, n1, n2 in counts:
        np.add.at(cost, np.asarray(pj), pair_costs(pi, pj, n1, n2, radii1=radii1))
    shares = assign_patch_fractions(cost, centers_xyz, n_devices)
    keep = [_keep_for(counts, n_patch, [p for p, _, _ in mine]) for mine in shares]
    return SharePlan(shares, keep)


def plan_passes(counts, radii1, centers_xyz, footprint, limits) -> list[SharePlan]:
    """The passes of one call whose catalogs may not fit its devices at once.  `counts`, `radii1`, `centers_xyz`: as
    for `plan_shares`; `footprint(keep)`: predicted device bytes of a pass that uploads the patches flagged in `keep`
    (`(n_patch,)` bool) of every catalog of the call and counts there; `limits`: bytes per device.

    The second patches are cut into `n_devices x K` shares of equal cost (`plan_shares`) and device d takes the K
    consecutive shares d K .. d K + K - 1, one per pass; K grows until every pass fits its device.  Past one share
    per patch the cuts stop helping (a pass keeps every patch linked to a patch it owns, whole), and the passes are
    one second patch each, device d taking the patches of its share of `plan_shares`.  Returns one `SharePlan` per
    pass step: share d of step k is device d's k-th pass (K = 1: the plan of `plan_shares`; a device with fewer
    passes has empty shares at the end).  If one patch with its linked patches exceeds a device's limit,
    ValueError is raised."""
    limits = [int(x) for x in limits]
    n_dev, n_patch = len(limits), len(centers_xyz)

    def steps_of(plan, k):
        return [SharePlan([plan.shares[d * k + s] for d in range(n_dev)], [plan.keep[d * k + s] for d in range(n_dev)])
                for s in range(k)]

    k = 1
    while k < n_patch:
        plan = plan_shares(counts, radii1, centers_xyz, n_dev * k)
        need = [int(footprint(keep.astype(bool))) for keep in plan.keep]
        if all(b <= limits[i // k] for i, b in enumerate(need)):
            return steps_of(plan, k)
        k = min(k + max(1, k // 4), n_patch)
    # the smallest passes there are: one second patch each, with its linked patches
    whole = plan_shares(counts, radii1, centers_xyz, n_dev)
    seen: set = set()  # a patch cut between two devices goes to the first
    own = [[p for p, _, _ in mine if not (p in seen or seen.add(p))] for mine in whole.shares]
    k = max(len(o) for o in own)
    shares, keep = [], []
    for d in range(n_dev):
        for s in range(k):
            mine = [(own[d][s], 0.0, 1.0)] if s < len(own[d]) else []
            one = _keep_for(counts, n_patch, [p for p, _, _ in mine])
            b = int(footprint(one.astype(bool))) if mine else 0  # an empty pass uploads nothing
            if b > limits[d]:
                raise ValueError(f"one pass over patch {mine[0][0]} and its linked patches needs {b} bytes of device "
                                 f"memory, more than the limit of {limits[d]} bytes")
            shares.append(mine)
            keep.append(one)
    return steps_of(SharePlan(shares, keep), k)


def _keep_for(counts, n_patch: int, own_patches) -> np.ndarray:
    """the patches a device uploads to count the second patches `own_patches`: those and every patch linked to one"""
    own = np.zeros(n_patch, dtype=bool)
    own[list(own_patches)] = True
    k = own.copy()
    for pi, pj, _, _ in counts:
        pi, pj = np.asarray(pi), np.asarray(pj)
        k[pi[own[pj]]] = True
        k[pj[own[pi]]] = True
    return k.astype(np.uint8)


class Shard:
    """Rank / world size of this process and the reduce used to combine results."""

    def __init__(self, rank: int = 0, world_size: int = 1, group=None) -> None:
        self.rank = rank
        self.world_size = world_size
        self.group = group

    @property
    def active(self) -> bool:
        return self.world_size > 1

    def reduce_to_root(self, array: np.ndarray, device: str | None = None) -> np.ndarray:
        """Sum `array` over the ranks.  Every element has exactly one non-zero contributor, so the sum is exact.
        The result is delivered to EVERY rank (an all-reduce: the tensors are a few hundred KB), so that
        `crosscorrelate` / `autocorrelate` return complete counts wherever they are called.  `device`: where the
        collective runs with the NCCL backend -- the engine's GPU (`cuda:<engine.device>`), not whatever
        `torch.cuda.current_device()` happens to be; ignored for CPU backends (gloo in the tests)."""
        if not self.active:
            return array
        import torch
        import torch.distributed as dist

        backend = dist.get_backend(self.group)
        if backend == "nccl":
            dev = device or f"cuda:{int(os.environ.get('LOCAL_RANK', '0'))}"
        else:
            dev = "cpu"
        t = torch.from_numpy(np.ascontiguousarray(array)).to(dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return t.cpu().numpy()


def current_shard() -> Shard:
    """The shard of this process if `torch.distributed` is initialised, else a single shard.
    torch is imported only when a launcher (torchrun) has set up the environment."""
    if "RANK" not in os.environ and "WORLD_SIZE" not in os.environ:
        return Shard()
    try:
        import torch.distributed as dist
    except Exception:
        return Shard()
    if dist.is_available() and dist.is_initialized():
        return Shard(dist.get_rank(), dist.get_world_size())
    return Shard()
