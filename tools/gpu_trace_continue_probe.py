"""Cost of continuing a resident trace (DeviceTracer.trace_continue) against tracing all rays afresh.

    python tools/gpu_trace_continue_probe.py --out profiles/r7/r7a_trace_continue_probe.json

Meshes, in one process: cfg3 (N = 10 605, dense resident counts), square_domain(260, kappa=40) (N = 68 640) and
square_domain(400, kappa=40) (N = 161 600), both with the hashed row tally.  On each mesh, on one handle:
  * fresh     : one trace of R1 + R2 rays per emitter;
  * first     : a trace of R1 rays, followed by
  * continue  : trace_continue(R2) (for the hashed form: the new rays' tally and reduction, then the merge into the resident set);
  * plain_r2  : a plain trace of the R2 rays alone (ray_id_offset = R1) — what the continuation costs without the merge.
Each step is timed as the wall time of the blocking call (the library's device times too), warm-up once, then `--reps` times; medians
are reported.  After the continuation the CSR read-out is compared with the fresh trace's (`identical`).  Merge: the device time of
the merge kernels (tally_merge_kernel, and the scan of their tile counts) in one extra continuation under torch.profiler.  Peak
memory: the least free device memory seen by a thread that polls cudaMemGetInfo every 0.2 ms while the continuation runs, against
the free memory before it (a sampled peak), beside the model 16 (old + new + merged keys) + 24 pair capacity bytes.  The card's name,
power limit and max SM clock are read with nvidia-smi.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rthx                                                    # noqa: E402
from rthx._lib import release_pinned                           # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in q[0].split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def free_bytes():
    import torch
    return int(torch.cuda.mem_get_info(0)[0])


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return 1e3 * (time.perf_counter() - t0), out


def with_min_free(fn):
    """Run fn while a thread samples the free device memory; returns (fn's result, least free bytes seen)."""
    low, stop = [free_bytes()], threading.Event()

    def poll():
        while not stop.is_set():
            low[0] = min(low[0], free_bytes())
            time.sleep(2e-4)

    th = threading.Thread(target=poll)
    th.start()
    try:
        out = fn()
    finally:
        stop.set()
        th.join()
    return out, min(low[0], free_bytes())


def merge_kernel_ms(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    names = {}
    for e in prof.events():
        if "tally_merge_kernel" in e.name or "DeviceScan" in e.name:
            names[e.name] = names.get(e.name, 0.0) + e.device_time_total / 1e3
    return sum(names.values()), names


def probe(name, rtm, r1, r2, seed, hashed, reps):
    rthx.load_library().rthx_release_cached()
    flat = rthx.flatten_domain(rtm)
    tr = rthx.DeviceTracer(flat, device=0)
    trace = (lambda r, **kw: tr.trace_sparse(r, seed=seed, **kw)) if hashed else (lambda r, **kw: tr.trace(r, seed=seed, dense=False, **kw))
    steps = {k: [] for k in ("fresh", "first", "continue", "plain_r2")}
    stats = {}
    for rep in range(reps + 1):
        ms, out = timed(lambda: trace(r1 + r2))
        fresh_csr = tr.counts_csr(0, values=True, normalised=False)[:3]
        stats["fresh"] = out
        if rep:
            steps["fresh"].append(ms)
        ms, out = timed(lambda: trace(r1))
        stats["first"] = out
        if rep:
            steps["first"].append(ms)
        nnz_old = tr.counts_stats(0)[0]
        free0 = free_bytes()
        (ms, out), low = with_min_free(lambda: timed(lambda: tr.trace_continue(r2)))
        stats["continue"] = out
        if rep:
            steps["continue"].append(ms)
        cont_csr = tr.counts_csr(0, values=True, normalised=False)[:3]
        identical = all(np.array_equal(a, b) for a, b in zip(fresh_csr, cont_csr))
        ms, out = timed(lambda: trace(r2, ray_id_offset=r1))
        stats["plain_r2"] = out
        nnz_new = tr.counts_stats(0)[0]
        if rep:
            steps["plain_r2"].append(ms)
    trace(r1)
    merge_ms, merge_kernels = merge_kernel_ms(lambda: tr.trace_continue(r2))
    r = {"mesh": name, "n": flat.n_elements, "form": "hashed" if hashed else "dense", "r1": r1, "r2": r2, "identical": bool(identical),
         "wall_ms": {k: statistics.median(v) for k, v in steps.items()}, "wall_ms_all": steps,
         "device_total_ms": {k: v["stats"]["total_ms"] for k, v in stats.items()},
         "kernel_ms": {k: v["stats"]["kernel_ms"] for k, v in stats.items()},
         "merge_kernel_ms": merge_ms, "merge_kernels": merge_kernels,
         "continue_peak_extra_bytes_sampled": free0 - low}
    if hashed:
        sst = stats["continue"]["sparse_stats"]
        r.update({"reduce_ms": {k: v["sparse_stats"]["reduce_ms"] for k, v in stats.items()},
                  "nnz_before": int(nnz_old), "nnz_new_set": int(nnz_new), "nnz_after": int(sst["nnz"]),
                  "pairs": int(sst["pairs"]), "pair_capacity": int(sst["pair_capacity"]), "row_groups": int(sst["row_groups"]),
                  "peak_bytes_model": 16 * (int(nnz_old) + int(nnz_new) + int(sst["nnz"])) + 24 * int(sst["pair_capacity"])})
    tr.close()
    release_pinned()
    print(json.dumps(r), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r7/r7a_trace_continue_probe.json")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    info = gpu_info()
    print(json.dumps(info), flush=True)
    runs = [
        probe("cfg3", rthx.meshes.cfg3(), 50_000, 50_000, 91, False, args.reps),
        probe("square_260_kappa40", rthx.meshes.square_domain(260, kappa=40.0), 1000, 1000, 92, True, args.reps),
        probe("square_400_kappa40", rthx.meshes.square_domain(400, kappa=40.0), 1000, 1000, 93, True, args.reps),
    ]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump({"gpu": info, "runs": runs}, f, indent=1)


if __name__ == "__main__":
    main()
