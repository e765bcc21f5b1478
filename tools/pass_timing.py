"""Time the public `crosscorrelate` counted in passes, and compare the predicted device footprint with the measured
high-water mark of the allocator.

    python tools/pass_timing.py [--workloads C3 C5] [--passes 1 2 4 8] [--c5-fraction 0.25] [--out FILE]

For every workload (the catalogs of `bench.py`) the call's one-pass footprint F is predicted with the model of
`measurements._share_plan` (planning only, nothing uploaded).  C3 runs with memory limits that plan 1, 2, 4 and 8
passes (the largest limit, in steps of 2 % of F, that gives at least that many), C5 in one pass and at
`--c5-fraction` of F.  Each call runs on a fresh engine without a catalog cache and is timed with the host clock
around a call that ends in a device synchronise (host preparation, uploads, index builds, counts).  Recorded: the
time, the passes, the allocator's peak against the limit, and whether the counts equal the one-pass counts bit for
bit.  Then, for every catalog of C3 (upload and both indexes) and every count path (`count`, `count2`, `count4`
with its union index, a labelled count), the predicted footprint against the measured peak.  The card's name and
power limit are read in the same run.  Writes one JSON file.
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from engine_group_timing import counts_of, gpu_info, make_catalogs  # noqa: E402


class _Planned(Exception):
    pass


def planner(config, cats):
    """(footprint(keep), counts, radii, centers) of the call, captured from its planning; `engine` (which the
    footprint asks for count workspaces) is closed by the caller"""
    import yet_another_wizz_b200 as yb
    from yet_another_wizz_b200 import measurements

    got = {}

    def probe(counts, radii, centers, footprint, limits):
        got.update(footprint=footprint, counts=counts, radii=radii, centers=centers)
        raise _Planned

    saved = measurements.plan_passes
    measurements.plan_passes = probe
    eng = yb.Engine(0, cache_catalogs=False)
    try:
        call(config, cats, eng)
    except _Planned:
        pass
    finally:
        measurements.plan_passes = saved
    got["engine"] = eng
    return got


def call(config, cats, engine):
    import yet_another_wizz_b200 as yb

    return yb.crosscorrelate(config, cats["ref"], cats["unk"], ref_rand=cats["ref_rand"], unk_rand=cats["unk_rand"],
                             engine=engine)


def limit_for(plan, target, whole) -> tuple[int, int]:
    """the largest limit (steps of 2 % of the one-pass footprint) planned in at least `target` passes"""
    from yet_another_wizz_b200.sharding import plan_passes

    for k in range(100, 0, -2):
        limit = int(whole * k / 100)
        try:
            n = len(plan_passes(plan["counts"], plan["radii"], plan["centers"], plan["footprint"], [limit]))
        except ValueError:
            break
        if n >= target:
            return limit, n
    return None, None


def timed(config, cats, limit):
    import yet_another_wizz_b200 as yb
    from yet_another_wizz_b200 import measurements

    eng = yb.Engine(0, cache_catalogs=False, memory_limit=limit)
    try:
        eng.memory_reset_peak()
        t0 = time.perf_counter()
        corrs = call(config, cats, eng)
        eng.sync()
        ms = (time.perf_counter() - t0) * 1e3
        stats = measurements.last_stats()
        peak = eng.memory_stats()["peak"]
    finally:
        eng.close()
    passes = max(st.get("passes", 1) for st in stats.values())
    return ms, passes, peak, counts_of(corrs)


def paths(config, cats) -> list[dict]:
    """predicted footprint against the measured peak for every catalog of the call and every count path"""
    import yet_another_wizz_b200 as yb
    from yet_another_wizz_b200.measurements import _as_binning, prepare_catalog_arrays

    binning = _as_binning(config)
    arrays = {k: prepare_catalog_arrays(cats[k], binning if k in ("ref", "ref_rand") else None) for k in cats}
    n_patch = len(arrays["ref"]["patch_off"]) - 1
    out = []

    def rows(k):
        return len(arrays[k]["xyz"])

    def zb(k):
        return "u8" if arrays[k]["zbin"] is not None else None

    def nb(k):
        return arrays[k]["n_bins"]

    for k in arrays:  # one catalog: upload and both indexes
        eng = yb.Engine(0, cache_catalogs=False)
        try:
            a = dict(arrays[k])
            cat = eng.upload_catalog(a.pop("xyz"), a.pop("patch_off"), **a)
            cat.build_index(1)
            cat.build_index(2)
            eng.sync()
            pred = eng.footprint(rows(k), n_patch, nb(k), weighted=False, zbin=zb(k))
            out.append(dict(path=f"catalog {k}", rows=rows(k), predicted=pred, peak=eng.memory_stats()["peak"]))
        finally:
            eng.close()
    edges = np.ascontiguousarray(np.broadcast_to([0.0, 1e-6], (nb("ref"), 2)))  # one sub-bin, single-bin path
    pi, pj = np.meshgrid(np.arange(n_patch), np.arange(n_patch), indexing="ij")
    pi, pj = pi.ravel(), pj.ravel()
    for kind in ("count", "count2", "count4", "labelled"):
        eng = yb.Engine(0, cache_catalogs=False)
        try:
            dev = {}
            for k in arrays:
                a = dict(arrays[k])
                if kind == "labelled" and k == "unk":  # the unknown sample as one label of a labelled catalog
                    a.update(zbin=np.zeros(rows(k), dtype=np.uint8), n_bins=1)
                dev[k] = eng.upload_catalog(a.pop("xyz"), a.pop("patch_off"), **a)
            eng.sync()
            eng.memory_reset_peak()
            base = eng.memory_stats()["held"]

            def index(k, role, n=None, bins=None):
                return eng.footprint(n or rows(k), n_patch, bins or nb(k), zbin=zb(k), first=role == 1,
                                     second=role == 2, upload=False)

            def work(seconds, blocks):  # tiles of the second catalogs per pair: at most rows / 256 + one per segment
                n_items = int(sum(np.sum(np.ceil(np.diff(arrays[k2]["patch_off"])[pj] / 256.0) + nb(k2)) for k2 in seconds))
                return eng.count_footprint(n_items, len(pi), nb("ref"), 2, n_blocks=blocks)

            fused = index("ref", 1, rows("ref") + rows("ref_rand"))
            if kind == "count":
                eng.count(dev["ref"], dev["unk"], pi, pj, edges)
                pred = index("ref", 1) + index("unk", 2) + work(["unk"], 1)
            elif kind == "count2":
                eng.count2(dev["ref"], dev["ref_rand"], dev["unk"], pi, pj, edges)
                pred = fused + index("unk", 2) + work(["unk"], 2)
            elif kind == "count4":
                eng.count4(dev["ref"], dev["ref_rand"], dev["unk"], dev["unk_rand"], pi, pj, edges)
                pred = fused + index("unk", 2, rows("unk") + rows("unk_rand"), 1) + work(["unk", "unk_rand"], 4)
            else:
                eng.count(dev["ref"], dev["unk"], pi, pj, edges, labels=True)
                pred = index("ref", 1) + index("unk", 2) + work(["unk"], 1)
            eng.sync()
            out.append(dict(path=kind, predicted=pred, peak=eng.memory_stats()["peak"] - base))
        finally:
            eng.close()
    for r in out:
        r["predicted_over_peak"] = round(r["predicted"] / max(r["peak"], 1), 3)
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["C3", "C5"])
    ap.add_argument("--passes", nargs="+", type=int, default=[1, 2, 4, 8])
    ap.add_argument("--c5-fraction", type=float, default=0.25)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_pass_timing.json"))
    args = ap.parse_args()
    result = dict(gpus=gpu_info(), runs=[], footprint_vs_peak=[])
    for name in args.workloads:
        t0 = time.perf_counter()
        config, cats = make_catalogs(name)
        print(f"{name}: catalogs in {time.perf_counter() - t0:.1f} s", file=sys.stderr, flush=True)
        plan = planner(config, cats)
        whole = int(plan["footprint"](np.ones(len(plan["centers"]), dtype=bool)))
        if name == "C5":
            settings = [(1, whole), ("fraction", int(whole * args.c5_fraction))]
        else:
            settings = [(k, whole if k == 1 else limit_for(plan, k, whole)[0]) for k in args.passes]
        want = None
        for target, limit in settings:
            if limit is None:
                result["runs"].append(dict(workload=name, target=target, not_run="no limit plans that many passes"))
                continue
            try:
                ms, passes, peak, got = timed(config, cats, limit)
            except ValueError as exc:
                result["runs"].append(dict(workload=name, target=target, limit=limit, not_run=str(exc)))
                continue
            if want is None:
                want = got
            run = dict(workload=name, target_passes=target, limit=limit, one_pass_footprint=whole, passes=passes,
                       ms=round(ms, 1), peak=peak, peak_within_limit=bool(peak <= limit),
                       equal_to_one_pass=bool(all(np.array_equal(got[k], want[k]) for k in want)))
            print(json.dumps(run), file=sys.stderr, flush=True)
            result["runs"].append(run)
        plan["engine"].close()
        if name == "C3":
            result["footprint_vs_peak"] = paths(config, cats)
            print(json.dumps(result["footprint_vs_peak"]), file=sys.stderr, flush=True)
        del cats
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
