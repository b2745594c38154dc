"""Cost of the public call on surfaces-only domains with the default route (only the Ns surface rows are traced) against the full
trace (trace_volume_rows=True), and bench.py of two builds, alternating, in one process tree.

    python tools/gpu_trace_rows_probe.py --out profiles/r8/r8a_trace_rows_probe.json [--parent-tree DIR]

Domains: square_domain(101, kappa=0) (N = 10 605, Ns = 404) and circle_domain(16, 25, kappa=0) (beta = 0), at --rays rays per call.
Every route is warmed up once, then called --reps times; the medians of the phases the call records (rtm.last_phase_ms: trace,
smoothing) and of the wall time of the whole blocking call are reported, with rtm.F_raw / rtm.F_smooth of both routes compared bit for
bit.  Irregular lists: on cfg3 (N = 10 605) at --rays rays per full trace, DeviceTracer.trace_rows of R = 1 000 rows as one contiguous
run [0, 1 000), as 1 000 rows at a random irregular spacing (seeded; about one launch per row), against the full trace (dense=False);
medians of --reps blocking calls after a warm-up, wall time and the library's kernel time.  With --parent-tree, `bench.py --gpus 1` runs from that tree and from this one, alternating, --bench-reps times each.  The card's
name, power limit and max SM clock are read with nvidia-smi in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rthx                                                    # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in q[0].split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def same(x, y):
    if sp.issparse(x) or sp.issparse(y):
        x, y = sp.csc_matrix(x), sp.csc_matrix(y)
        x.sort_indices(); y.sort_indices()
        return bool(np.array_equal(x.indptr, y.indptr) and np.array_equal(x.indices, y.indices) and np.array_equal(x.data, y.data))
    return bool(np.array_equal(x, y))


def public(rtm, rays, reps, **kw):
    call = lambda: rtm(rays, method="exchange", verbose=False, seed=2024, devices=[0], **kw)   # noqa: E731
    call()                                                     # warm-up: handles, tables, pinned buffers
    trace, smooth, wall = [], [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        call()
        wall.append(1e3 * (time.perf_counter() - t0))
        trace.append(rtm.last_phase_ms["trace"])
        smooth.append(rtm.last_phase_ms["smoothing"])
    return dict(trace_ms=statistics.median(trace), smoothing_ms=statistics.median(smooth), total_ms=statistics.median(wall),
                rows=int(rtm.last_trace_stats["rows"]), kernel_ms=float(rtm.last_trace_stats["kernel_ms"]),
                smooth_path=rtm.last_smooth_stats.get("path")), (rtm.F_raw, rtm.F_smooth)


def bench(tree, steps, warmup):
    r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup)], cwd=tree,
                       capture_output=True, text=True)
    line = [s for s in r.stdout.splitlines() if s.strip().startswith("{")]
    return json.loads(line[-1]) if line else {"error": r.stderr[-2000:]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rays", type=float, default=1e9)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parent-tree", default=None)
    ap.add_argument("--bench-reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    res = {"gpu": gpu_info(), "rays": a.rays, "reps": a.reps, "domains": {}}
    domains = {"square_101_kappa0": lambda: rthx.meshes.square_domain(101, kappa=0.0),
               "circle_16x25_beta0": lambda: rthx.meshes.circle_domain(N_seg=16, Ndim=25, kappa=0.0)}
    for name, make in domains.items():
        rtm = make()
        assert rtm.surfaces_only
        rows, (F_rows, S_rows) = public(rtm, int(a.rays), a.reps)
        full, (F_full, S_full) = public(rtm, int(a.rays), a.reps, trace_volume_rows=True)
        res["domains"][name] = dict(N=rtm.num_elements, Ns=rtm.num_surfaces, surface_rows=rows, all_rows=full,
                                    trace_ratio=full["trace_ms"] / rows["trace_ms"], kernel_ratio=full["kernel_ms"] / rows["kernel_ms"],
                                    identical_F_raw=same(F_rows, F_full), identical_F_smooth=same(S_rows, S_full))
        print(name, json.dumps(res["domains"][name]), flush=True)
    rtm = rthx.meshes.cfg3()
    tr = rthx.DeviceTracer(rthx.flatten_domain(rtm), device=0)
    N = tr.n_elements
    rpe = int(a.rays) // N
    rng = np.random.default_rng(7)
    lists = {"contiguous_1000": np.arange(1000), "irregular_1000": np.sort(rng.choice(N, 1000, replace=False)), "full": None}
    res["irregular"] = {"N": N, "rays_per_emitter": rpe}
    for name, rows in lists.items():
        call = (lambda: tr.trace(rpe, seed=3, dense=False)) if rows is None else (lambda rows=rows: tr.trace_rows(rows, rpe, seed=3, dense=False))
        call()
        wall, kern, launches = [], [], 0
        for _ in range(a.reps):
            t0 = time.perf_counter()
            out = call()
            wall.append(1e3 * (time.perf_counter() - t0))
            kern.append(out["stats"]["kernel_ms"])
            launches = out["stats"]["n_launches"]
        runs = 1 if rows is None else int(1 + np.count_nonzero(np.diff(np.diff(rows)) != 0))
        res["irregular"][name] = dict(wall_ms=statistics.median(wall), kernel_ms=statistics.median(kern), n_launches=launches,
                                      rows=N if rows is None else len(rows), arithmetic_runs_upper_bound=runs)
        print(name, json.dumps(res["irregular"][name]), flush=True)
    del tr
    if a.parent_tree:
        runs = []
        for _ in range(a.bench_reps):
            for label, tree in (("parent", a.parent_tree), ("this", ROOT)):
                b = bench(tree, a.steps, a.warmup)
                runs.append({"build": label, **b})
                print(label, json.dumps(b), flush=True)
        res["bench_ab"] = runs
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
