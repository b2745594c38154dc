"""Sparse reciprocity smoothing on the device (rthx_smooth_sparse) beside the host smooth_F on the same F_raw.

    python tools/gpu_sparse_smooth_probe.py --out profiles/r5/r5a_sparse_smooth_probe.json

Three optically thick meshes, in one process: the diffusion slab of test/test_2d_diffusion.jl (31 x 31, resident counts),
square_domain(101, kappa=40) (resident counts) and square_domain(260, kappa=40) traced in 4 row tiles (host CSC F_raw).  Per mesh:
nnz of F and X, iterations, device time of the whole smoothing (build X + iterations + recover), the build alone (max_iters = 0),
ms per iteration without the build, one scaling pass alone (pass_gbs over 20 nnz_X + 8 (n + 1) bytes), the host smooth_F wall
time and max |F_device - F_host|.  The card's name, power limit and max SM clock are read with a query of nvidia-smi.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rthx                                                    # noqa: E402
from rthx._lib import trace_row_tiles                          # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in q[0].split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def probe(name, rtm, rays_per_emitter, seed, row_tiles):
    flat = rthx.flatten_domain(rtm)
    tr = rthx.DeviceTracer(flat, device=0)
    N, ns = tr.n_elements, flat.n_surfaces
    w = rthx.get_w(rtm)
    wn = w / w.min()
    if row_tiles > 1:
        res = trace_row_tiles(tr, rays_per_emitter, row_tiles, seed=seed)
        row_ptr, cols, vals = res["csr"][0]
        F_raw = sp.csr_matrix((vals, cols, row_ptr), shape=(N, N)).tocsc()
        src = dict(F=F_raw)
    else:
        tr.trace(rays_per_emitter, seed=seed, dense=False)
        colptr, rowval, _, fv = tr.counts_csc(0, values=False, normalised=True)
        F_raw = sp.csc_matrix((fv.copy(), rowval.copy(), colptr.copy()), shape=(N, N))
        src = {}
    tr.smooth_sparse(wn, **src)                                # warm-up: module load, buffer allocation
    _, s0 = tr.smooth_sparse(wn, max_iters=0, **src)           # build X + first row sums + one delta check + recover
    Fd, st = tr.smooth_sparse(wn, measure_pass=True, **src)
    t0 = time.perf_counter()
    Fh = rthx.smoothing.smooth_F(F_raw, w, ns)
    host_s = time.perf_counter() - t0
    Fh.sort_indices()
    d = (Fd - Fh).tocsc()
    it = st["iterations"]
    nnz_x = Fd.nnz
    pass_bytes = 20.0 * nnz_x + 8.0 * (N + 1)
    per_iter = (st["total_ms"] - s0["total_ms"]) / it if it else 0.0
    out = {
        "mesh": name, "n": N, "row_tiles": row_tiles, "rays_per_emitter": rays_per_emitter,
        "nnz_F": int(F_raw.nnz), "nnz_X": int(nnz_x), "density_F": F_raw.nnz / float(N * N),
        "iterations": it, "converged": st["converged"], "delta_init": st["delta_init"], "delta": st["delta"],
        "launches": st["launches"],
        "device_total_ms": st["total_ms"], "device_ms_per_iteration_incl_build": st["ms_per_iteration"],
        "device_build_ms": s0["total_ms"], "device_ms_per_iteration": per_iter,
        "pass_ms": st["pass_ms"], "pass_gbs": st["pass_gbs"], "pass_bytes": pass_bytes,
        "pass_fits_l2_126MB": pass_bytes < 126e6,
        "overhead_per_iteration_ms": per_iter - st["pass_ms"],
        "host_smooth_F_s": host_s, "host_over_device": host_s * 1e3 / st["total_ms"] if st["total_ms"] > 0 else None,
        "max_abs_diff_device_host": float(np.abs(d.data).max()) if d.nnz else 0.0,
        "same_pattern": bool(np.array_equal(Fd.indptr, Fh.indptr) and np.array_equal(Fd.indices, Fh.indices)),
    }
    tr.close()
    print(json.dumps(out), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r5/r5a_sparse_smooth_probe.json")
    args = ap.parse_args()
    info = gpu_info()
    print(json.dumps(info), flush=True)
    runs = [
        probe("diffusion_slab_31", rthx.meshes.diffusion_slab_domain(31), 1000, 71, 1),
        probe("square_101_kappa40", rthx.meshes.square_domain(101, kappa=40.0), 1000, 72, 1),
        probe("square_260_kappa40_row_tiles4", rthx.meshes.square_domain(260, kappa=40.0), 64, 73, 4),
    ]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump({"gpu": info, "runs": runs}, f, indent=1)


if __name__ == "__main__":
    main()
