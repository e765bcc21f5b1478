"""A loop of `crosscorrelate` calls over tomographic bins against one `crosscorrelate_tomographic` call (`--mode
cross`), or a loop of `autocorrelate` calls against one `autocorrelate_tomographic` call (`--mode auto`); prints one
JSON line and writes it to --out (default profiles/r05_<mode>_tomographic_timing.json).

    python tools/tomographic_timing.py [--mode cross|auto] [--out PATH] [--small] [--repeats R]

Inputs (seeded `BoxRandoms` in the benchmark's C3 box, 64 patches, 30 z-bins, 100-1000 kpc): reference 1e6 rows,
its randoms 1e7, an unknown sample of 1e7 rows split into N = 5 bins by a seeded label.  Cases: (A) one shared
`unk_rand` of 1e7 rows, (B) per-bin randoms of 2e6 rows each, (C) no `unk_rand`.  Per case: wall clock of warm
calls (the first call of each form is a warm-up; the reference catalogs stay resident in the engine's cache either
way), the sums of `kernel_ms`, `index_ms` and `pair_tests` from `last_stats()`, and a check that both forms give
equal results.  Also the GPU name and power limit, read in the same run.  `--small` divides every size by 100 (a
rehearsal).

Auto mode: the unknown sample of 1e7 rows carries redshifts and is split into the same N = 5 bins; cases (A) one
shared random catalog of 1e7 rows with redshifts, (B) per-bin randoms of 2e6 rows each with redshifts.
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
from yet_another_wizz_b200 import measurements  # noqa: E402

BOX = (0.0, 40.0, -12.5, 12.5)  # bench.py's C3 box
N_TOMO = 5


def gpu_info() -> str:
    try:
        res = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30)
        return res.stdout.strip().splitlines()[0] if res.returncode == 0 and res.stdout.strip() else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def inputs(scale: float):
    nx, ny = 8, 8
    ras = BOX[0] + (np.arange(nx) + 0.5) * (BOX[1] - BOX[0]) / nx
    decs = BOX[2] + (np.arange(ny) + 0.5) * (BOX[3] - BOX[2]) / ny
    centers = yb.AngularCoordinates(np.deg2rad([[r, d] for d in decs for r in ras]))
    pool = np.random.default_rng(7).uniform(0.07, 1.42, 1_000_000)

    def box(name, n, seed, z=False):
        gen = yb.BoxRandoms(*BOX, redshifts=pool if z else None, seed=seed)
        return yb.Catalog.from_random(name, gen, max(int(n * scale), 1000), patch_centers=centers)

    ref, ref_rand = box("ref", 1e6, 1, z=True), box("ref_rand", 1e7, 3, z=True)
    unk, unk_rand = box("unk", 1e7, 2), box("unk_rand", 1e7, 4)
    per_bin_rand = [box(f"unk_rand_{i}", 2e6, 40 + i) for i in range(N_TOMO)]
    # the unknown sample split by a seeded label
    rows = {p: unk[p].load_data() for p in unk}
    lab = {p: np.random.default_rng(1000 + p).integers(0, N_TOMO, len(rows[p])) for p in unk}
    unknowns = []
    for i in range(N_TOMO):
        ra = np.concatenate([rows[p]["ra"][lab[p] == i] for p in unk])
        dec = np.concatenate([rows[p]["dec"][lab[p] == i] for p in unk])
        ids = np.concatenate([np.full(int((lab[p] == i).sum()), p) for p in unk])
        unknowns.append(yb.Catalog.from_arrays(ra, dec, patch_ids=ids, patch_centers=centers, degrees=False,
                                               cache_directory=f"unk_{i}"))
    config = yb.Configuration.create(rmin=100, rmax=1000, zmin=0.07, zmax=1.42, num_bins=30)
    return config, ref, ref_rand, unknowns, dict(A=unk_rand, B=per_bin_rand, C=None)


def auto_inputs(scale: float):
    """the unknown sample with redshifts, split into N_TOMO bins, and its randoms with redshifts (shared, per bin)"""
    nx, ny = 8, 8
    ras = BOX[0] + (np.arange(nx) + 0.5) * (BOX[1] - BOX[0]) / nx
    decs = BOX[2] + (np.arange(ny) + 0.5) * (BOX[3] - BOX[2]) / ny
    centers = yb.AngularCoordinates(np.deg2rad([[r, d] for d in decs for r in ras]))
    pool = np.random.default_rng(7).uniform(0.07, 1.42, 1_000_000)

    def box(name, n, seed):
        gen = yb.BoxRandoms(*BOX, redshifts=pool, seed=seed)
        return yb.Catalog.from_random(name, gen, max(int(n * scale), 1000), patch_centers=centers)

    unk, shared = box("unk", 1e7, 2), box("unk_rand", 1e7, 4)
    per_bin_rand = [box(f"unk_rand_{i}", 2e6, 40 + i) for i in range(N_TOMO)]
    rows = {p: unk[p].load_data() for p in unk}
    lab = {p: np.random.default_rng(1000 + p).integers(0, N_TOMO, len(rows[p])) for p in unk}
    data = []
    for i in range(N_TOMO):
        col = lambda k: np.concatenate([rows[p][k][lab[p] == i] for p in unk])  # noqa: E731
        ids = np.concatenate([np.full(int((lab[p] == i).sum()), p) for p in unk])
        data.append(yb.Catalog.from_arrays(col("ra"), col("dec"), patch_ids=ids, patch_centers=centers,
                                           redshifts=col("redshifts"), degrees=False, cache_directory=f"unk_{i}"))
    config = yb.Configuration.create(rmin=100, rmax=1000, zmin=0.07, zmax=1.42, num_bins=30)
    return config, data, dict(A=shared, B=per_bin_rand)


def stat_sums():
    st = measurements.last_stats()
    return {k: sum(s[k] for s in st.values()) for k in ("kernel_ms", "index_ms", "pair_tests")}


def add(total, part):
    for k, v in part.items():
        total[k] = total.get(k, 0) + v


def run_loop(eng, config, ref, ref_rand, unknowns, unk_rand):
    rands = unk_rand if isinstance(unk_rand, list) else [unk_rand] * len(unknowns)
    sums, out = {}, []
    t0 = time.perf_counter()
    for unk, rand in zip(unknowns, rands):
        out.append(yb.crosscorrelate(config, ref, unk, ref_rand=ref_rand, unk_rand=rand, engine=eng))
        add(sums, stat_sums())
    return time.perf_counter() - t0, sums, out


def run_one(eng, config, ref, ref_rand, unknowns, unk_rand):
    t0 = time.perf_counter()
    out = yb.crosscorrelate_tomographic(config, ref, unknowns, ref_rand=ref_rand, unk_rand=unk_rand, engine=eng)
    return time.perf_counter() - t0, stat_sums(), out


def run_loop_auto(eng, config, data, random):
    rands = random if isinstance(random, list) else [random] * len(data)
    sums, out = {}, []
    t0 = time.perf_counter()
    for d, rand in zip(data, rands):
        out.append(yb.autocorrelate(config, d, rand, engine=eng))
        add(sums, stat_sums())
    return time.perf_counter() - t0, sums, out


def run_one_auto(eng, config, data, random):
    t0 = time.perf_counter()
    out = yb.autocorrelate_tomographic(config, data, random, engine=eng)
    return time.perf_counter() - t0, stat_sums(), out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", choices=("cross", "auto"), default="cross")
    ap.add_argument("--out", default=None)
    ap.add_argument("--small", action="store_true")
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    out_path = args.out or os.path.join(ROOT, "profiles", f"r05_{args.mode}_tomographic_timing.json")
    scale = 0.01 if args.small else 1.0
    if args.mode == "cross":
        config, ref, ref_rand, unknowns, rand_forms = inputs(scale)
        loop = lambda eng, r: run_loop(eng, config, ref, ref_rand, unknowns, r)  # noqa: E731
        one = lambda eng, r: run_one(eng, config, ref, ref_rand, unknowns, r)  # noqa: E731
        rows = dict(ref=sum(ref.get_num_records()), ref_rand=sum(ref_rand.get_num_records()),
                    unknown=sum(sum(u.get_num_records()) for u in unknowns))
    else:
        config, data, rand_forms = auto_inputs(scale)
        loop = lambda eng, r: run_loop_auto(eng, config, data, r)  # noqa: E731
        one = lambda eng, r: run_one_auto(eng, config, data, r)  # noqa: E731
        rows = dict(unknown=sum(sum(d.get_num_records()) for d in data))
    eng = yb.Engine(0)
    result = dict(gpu=gpu_info(), mode=args.mode, n_tomo=N_TOMO, rows=rows, cases={})
    for case, unk_rand in rand_forms.items():
        # warm-up of both forms, then alternate them: every catalog stays resident in the engine's cache either way
        _, _, loop_out = loop(eng, unk_rand)
        _, _, one_out = one(eng, unk_rand)
        for a, b in zip(loop_out, one_out):
            assert a == b, f"case {case}: the one-call form differs from the loop"
        loop_t, one_t = [], []
        for _ in range(args.repeats):
            t, loop_stats, _ = loop(eng, unk_rand)
            loop_t.append(t)
            t, one_stats, _ = one(eng, unk_rand)
            one_t.append(t)
        result["cases"][case] = dict(
            unk_rand={"A": "shared 1e7", "B": f"per bin {N_TOMO} x 2e6", "C": "none"}[case],
            loop=dict(wall_s_min=round(min(loop_t), 4), wall_s_all=[round(t, 4) for t in loop_t],
                      kernel_ms=round(loop_stats["kernel_ms"], 3), index_ms=round(loop_stats["index_ms"], 3),
                      pair_tests=int(loop_stats["pair_tests"])),
            one_call=dict(wall_s_min=round(min(one_t), 4), wall_s_all=[round(t, 4) for t in one_t],
                          kernel_ms=round(one_stats["kernel_ms"], 3), index_ms=round(one_stats["index_ms"], 3),
                          pair_tests=int(one_stats["pair_tests"])),
            pair_test_ratio=round(loop_stats["pair_tests"] / max(one_stats["pair_tests"], 1), 3),
            wall_ratio=round(min(loop_t) / min(one_t), 3),
            equal=True,
        )
    eng.close()
    line = json.dumps(result)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
