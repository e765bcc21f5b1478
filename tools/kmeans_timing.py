"""Device time of `yawb_kmeans` (patch centres by spherical k-means) on uniform randoms in the C3 box; prints one
JSON line and writes it to --out (default profiles/r03_kmeans_timing.json).

    python tools/kmeans_timing.py [--out PATH] [--small]

For 1e7 rows x 64 patches and 1e8 rows x 256 patches (the latter also on a 1e6-row probe, `probe_size=1e6`):
device time of a whole call (`yawb_timer_start` / `yawb_timer_stop`, after a warm-up call), of the same call with
`max_iter=0` (upload, validation, bisection, first assignment), the iteration count, and (row x centre)
evaluations per second of the Lloyd iterations (their time = the difference of the two).  Also the wall time
of `Catalog.from_random(..., patch_num=64)` for 1e7 rows, and the GPU name and power limit.  `--small` runs
1e5 / 1e6 rows instead (a rehearsal).
"""

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import yet_another_wizz_b200 as yb  # noqa: E402

BOX = (0.0, 40.0, -12.5, 12.5)  # bench.py's C3 box


def gpu_info() -> str:
    try:
        res = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30)
        return res.stdout.strip().splitlines()[0] if res.returncode == 0 and res.stdout.strip() else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def box_xyz(n, seed):
    g = yb.BoxRandoms(*BOX, seed=seed)(n)
    return yb.AngularCoordinates(np.column_stack([g["ra"], g["dec"]])).to_3d()


def timed(eng, xyz, k, max_iter=500):
    eng.timer_start()
    _, _, n_iter, converged = eng.kmeans(xyz, k, max_iter=max_iter)
    return eng.timer_stop(), n_iter, converged


def case(eng, xyz, k):
    eng.kmeans(xyz, k, max_iter=1)  # warm-up: module load, device buffers
    ms, n_iter, converged = timed(eng, xyz, k)
    ms0, _, _ = timed(eng, xyz, k, max_iter=0)
    iter_ms = ms - ms0
    evals = float(n_iter) * len(xyz) * k
    return dict(rows=len(xyz), k=k, call_ms=round(ms, 2), init_ms=round(ms0, 2), n_iter=n_iter, converged=converged,
                ms_per_iter=round(iter_ms / max(n_iter, 1), 4),
                evals_per_s=evals / (iter_ms * 1e-3) if iter_ms > 0 else None,
                fp64_tflops=8.0 * evals / (iter_ms * 1e-3) / 1e12 if iter_ms > 0 else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_kmeans_timing.json"))
    ap.add_argument("--small", action="store_true")
    args = ap.parse_args()
    n1, n2 = (100_000, 1_000_000) if args.small else (10_000_000, 100_000_000)
    probe = n2 // 100
    eng = yb.Engine(0)
    out = dict(gpu=gpu_info(), cases=[])
    out["cases"].append(case(eng, box_xyz(n1, 1), 64))
    xyz = box_xyz(n2, 2)
    out["cases"].append(case(eng, xyz, 256))
    step = -(-len(xyz) // probe)
    sub = dict(case(eng, np.ascontiguousarray(xyz[::step]), 256), probe_size=probe)
    out["cases"].append(sub)
    del xyz
    t0 = time.perf_counter()
    cat = yb.Catalog.from_random("t", yb.BoxRandoms(*BOX, seed=3), n1, patch_num=64, engine=eng)
    out["from_random_patch_num_64"] = dict(rows=n1, patches=len(cat), wall_s=round(time.perf_counter() - t0, 3))
    line = json.dumps(out)
    print(line, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    eng.close()


if __name__ == "__main__":
    main()
