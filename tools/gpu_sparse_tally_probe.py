"""The hashed row tally (DeviceTracer.trace_sparse) beside the dense-matrix traces of the same meshes.

    python tools/gpu_sparse_tally_probe.py --out profiles/r6/r6a_sparse_tally_probe.json

Meshes, in one process:
  * square_domain(260, kappa=40) (N = 68 640): sparse trace, the dense single pass (global atomics: the u32[N] histogram does not
    fit in shared memory) and row_tiles = 4;
  * square_domain(400, kappa=40) (N = 161 600, the dense matrix would be 209 GB): sparse trace and row_tiles = 5;
  * square_domain(260, kappa=1) (optically thin: rays spread over many absorbers, so tables fill and flush often): sparse trace
    and the dense single pass.
Per route: wall time of the trace call (blocking; the library's device times too), wall time of the read-out of F_raw (CSC for
the resident routes, the host merge of the tile CSRs for row tiles), and the device memory the route holds afterwards (free
memory from cudaMemGetInfo before and after, the handle's pooled buffers stay allocated).  Each route runs once to warm up and
then `--reps` times; the median is reported.  The card's name, power limit and max SM clock are read with nvidia-smi.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rthx                                                    # noqa: E402
from rthx._lib import release_pinned, trace_row_tiles          # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in q[0].split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def free_bytes():
    import torch
    return int(torch.cuda.mem_get_info(0)[0])


def route(flat, kind, rpe, seed, reps):
    """One route on a fresh handle: warm-up, then `reps` timed runs.  Returns a dict of medians and the last run's statistics."""
    rthx.load_library().rthx_release_cached()
    free0 = free_bytes()
    tr = rthx.DeviceTracer(flat, device=0)
    N = tr.n_elements
    trace_s, read_s, out = [], [], None
    for rep in range(reps + 1):
        t0 = time.perf_counter()
        if kind.startswith("row_tiles"):
            res = trace_row_tiles(tr, rpe, int(kind.split("=")[1]), seed=seed)
            t1 = time.perf_counter()
            row_ptr, cols, vals = res["csr"][0]
            import scipy.sparse as sp
            F = sp.csr_matrix((vals, cols, row_ptr), shape=(N, N)).tocsc()
            nnz, st, sst = F.nnz, res["stats"], None
        else:
            out = tr.trace_sparse(rpe, seed=seed) if kind == "sparse" else tr.trace(rpe, seed=seed, dense=False)
            t1 = time.perf_counter()
            nnz = tr.counts_stats(0)[0]
            colptr, rowval, _, fv = tr.counts_csc(0, values=False, normalised=True)
            st, sst = out["stats"], out.get("sparse_stats")
        t2 = time.perf_counter()
        if rep:
            trace_s.append(t1 - t0)
            read_s.append(t2 - t1)
    held = free0 - free_bytes()
    r = {"route": kind, "trace_ms": 1e3 * statistics.median(trace_s), "readout_ms": 1e3 * statistics.median(read_s),
         "trace_ms_all": [1e3 * x for x in trace_s], "nnz": int(nnz), "device_bytes_held": held,
         "kernel_ms": st["kernel_ms"], "total_ms": st["total_ms"], "n_blocks": st["n_blocks"], "row_chunks": st["row_chunks"],
         "smem_bytes": st["smem_bytes"]}
    if sst:
        r.update({"pairs": sst["pairs"], "flushes": sst["flushes"], "row_groups": sst["row_groups"], "hash_slots": sst["hash_slots"],
                  "pair_capacity": sst["pair_capacity"], "reduce_ms": sst["reduce_ms"]})
    tr.close()
    del out
    release_pinned()
    print(json.dumps(r), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r6/r6a_sparse_tally_probe.json")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    info = gpu_info()
    print(json.dumps(info), flush=True)
    meshes = [
        ("square_260_kappa40", rthx.meshes.square_domain(260, kappa=40.0), 1000, 81, ["sparse", "dense_global", "row_tiles=4"]),
        ("square_400_kappa40", rthx.meshes.square_domain(400, kappa=40.0), 1000, 82, ["sparse", "row_tiles=5"]),
        ("square_260_kappa1", rthx.meshes.square_domain(260, kappa=1.0), 4096, 83, ["sparse", "dense_global"]),
    ]
    runs = []
    for name, rtm, rpe, seed, kinds in meshes:
        flat = rthx.flatten_domain(rtm)
        for kind in kinds:
            r = route(flat, kind, rpe, seed, args.reps)
            runs.append(dict(r, mesh=name, n=flat.n_elements, rays_per_emitter=rpe))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump({"gpu": info, "runs": runs}, f, indent=1)


if __name__ == "__main__":
    main()
