"""Time the public `crosscorrelate` on an `EngineGroup` of 1 / 2 / 4 / 8 GPUs against one `Engine`.

    python tools/engine_group_timing.py [--workloads C3 C5] [--devices 1 2 4 8] [--warm 3] [--out FILE]

For every workload (the catalogs of `bench.py`) and device count: one cold call (fresh engines: host preparation,
partial uploads, index builds, counts) and `--warm` calls with the shares resident in the engines' caches, each timed
with the host clock around a call that ends with every device synchronised.  Every result is compared with the
one-device result (integer counts bit for bit).  Device counts above the number of visible GPUs are listed as not
run.  The card's name and power limit are read in the same run.  Writes one JSON file.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info() -> list[str]:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout
        return [line.strip() for line in out.splitlines() if line.strip()]
    except Exception as exc:  # the numbers are still worth keeping
        return [f"unknown ({exc})"]


def make_catalogs(name: str):
    import bench
    import yet_another_wizz_b200 as yb

    spec = bench.WORKLOADS[name]
    nx, ny = spec["grid"]
    ras = bench.BOX[0] + (np.arange(nx) + 0.5) * (bench.BOX[1] - bench.BOX[0]) / nx
    decs = bench.BOX[2] + (np.arange(ny) + 0.5) * (bench.BOX[3] - bench.BOX[2]) / ny
    centers = yb.AngularCoordinates(np.deg2rad([[r, d] for d in decs for r in ras]))
    pool = np.random.default_rng(7).uniform(spec["zmin"], spec["zmax"], 1_000_000)
    config = yb.Configuration.create(rmin=100, rmax=1000, zmin=spec["zmin"], zmax=spec["zmax"], num_bins=spec["bins"])
    cats = {}
    for key, n in zip(("ref", "unk", "ref_rand", "unk_rand"), spec["n"]):
        gen = yb.BoxRandoms(*bench.BOX, redshifts=pool if key in ("ref", "ref_rand") else None, seed=bench.SEEDS[key])
        cats[key] = yb.Catalog.from_random(key, gen, n, patch_centers=centers)
    return config, cats


def counts_of(corrs) -> dict:
    return {k: getattr(corrs[0], k).counts.counts for k in ("dd", "dr", "rd", "rr")}


def timed_call(config, cats, engine) -> tuple[float, dict]:
    import yet_another_wizz_b200 as yb

    t0 = time.perf_counter()
    corrs = yb.crosscorrelate(config, cats["ref"], cats["unk"], ref_rand=cats["ref_rand"], unk_rand=cats["unk_rand"],
                              engine=engine)
    engine.sync()
    return (time.perf_counter() - t0) * 1e3, counts_of(corrs)


def main() -> None:
    import torch

    import yet_another_wizz_b200 as yb

    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["C3", "C5"])
    ap.add_argument("--devices", nargs="+", type=int, default=[1, 2, 4, 8])
    ap.add_argument("--warm", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_engine_group_timing.json"))
    args = ap.parse_args()
    visible = torch.cuda.device_count()
    result = dict(gpus=gpu_info(), visible_gpus=visible, runs=[], not_run=[])
    for name in args.workloads:
        t0 = time.perf_counter()
        config, cats = make_catalogs(name)
        print(f"{name}: catalogs in {time.perf_counter() - t0:.1f} s", file=sys.stderr, flush=True)
        want = None
        for n_dev in args.devices:
            if n_dev > visible:
                result["not_run"].append(dict(workload=name, devices=n_dev, reason=f"{visible} GPU(s) visible"))
                continue
            engine = yb.Engine(0) if n_dev == 1 else yb.EngineGroup(list(range(n_dev)))
            try:
                cold, got = timed_call(config, cats, engine)
                warm = [timed_call(config, cats, engine)[0] for _ in range(args.warm)]
            finally:
                engine.close()
            if want is None:
                want = got
            equal = all(np.array_equal(got[k], want[k]) for k in want)
            run = dict(workload=name, devices=n_dev, cold_ms=round(cold, 1), warm_ms=[round(t, 1) for t in warm],
                       equal_to_one_device=bool(equal))
            print(json.dumps(run), file=sys.stderr, flush=True)
            result["runs"].append(run)
        del cats
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
