"""method=:direct on the hashed row tally (rthx_trace_direct_sparse) against the dense direct route, on isothermal enclosures where every
element is a source (R = N).

  python tools/gpu_direct_sparse_probe.py [--out DIR] [--reps 3] [--skip-400]

Both square_domain(Ndim, kappa = 40) meshes have black walls and every gas cell at 1000 K:
  Ndim = 260: N = 68 640, dense counts 37.7 GB: both routes fit, traced alternately on one handle;
  Ndim = 400: N = 161 600, dense counts 209 GB: the hashed route only.
Per route, the median of --reps calls after one warm-up call of each route: kernel time (CUDA events around the trace launches),
sort + reduce time of the pairs, the rest of the call (uploads, the absorbed-power sums, copies; total - kernel - reduce), the whole
call (CUDA events from the first upload to the last copy); and, from one more call per route on a fresh handle with the library's
cached buffers released, the peak device memory the call held (cudaMemGetInfo sampled every millisecond from a second thread, against
the free memory before the call).  The
absorbed powers of the two routes are compared bit for bit.  The card's name, power limit and maximum SM clock are read in the same
run.  Prints one JSON document and writes it to DIR/direct_sparse_probe.json."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import rthx  # noqa: E402
from rthx.direct import direct_sources  # noqa: E402


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def isothermal(ndim):
    rtm = rthx.meshes.square_domain(ndim, kappa=40.0, T_walls=(1000.0,) * 4)
    for c in rtm.fine_mesh[0]:
        c.T_in_g = 1000.0
    return rtm


class PeakMemory:
    """Lowest free device memory seen while the block runs, sampled from a second thread."""

    def __init__(self):
        import torch
        self.torch = torch

    def __enter__(self):
        self.free0 = self.low = self.torch.cuda.mem_get_info(0)[0]
        self.stop = False
        self.t = threading.Thread(target=self.poll)
        self.t.start()
        return self

    def poll(self):
        while not self.stop:
            self.low = min(self.low, self.torch.cuda.mem_get_info(0)[0])
            time.sleep(0.001)

    def __exit__(self, *exc):
        self.stop = True
        self.t.join()
        self.held = self.free0 - min(self.low, self.torch.cuda.mem_get_info(0)[0])


def one_call(tr, src, rays, reemit, w, sparse, seed):
    out = tr.trace_direct(src, rays, reemit, w, sparse=sparse, seed=seed)
    st, sst = out["stats"], out.get("sparse_stats", {})
    reduce_ms = sst.get("reduce_ms", 0.0)
    return dict(kernel_ms=st["kernel_ms"], reduce_ms=reduce_ms, rest_ms=st["total_ms"] - st["kernel_ms"] - reduce_ms, call_ms=st["total_ms"],
                events=out["events"], lost=int(out["lost"].sum()), sparse_stats=sst), out["absorbed"]


def probe(ndim, bundles, reps, routes):
    rtm = isothermal(ndim)
    flat = rthx.flatten_domain(rtm)
    ws, known_T, E, src, rays, w = direct_sources(rtm, bundles)
    reemit = np.zeros(flat.n_elements, np.uint8)
    reemit[:len(known_T)] = ~known_T
    lib = rthx.load_library()
    name = lambda sparse: "sparse" if sparse else "dense"  # noqa: E731
    # peak memory: one call per route on a fresh handle, with the library's cached buffers released first
    peak = {}
    for sparse in routes:
        lib.rthx_release_cached()
        tr = rthx.DeviceTracer(flat, device=0)
        with PeakMemory() as pm:
            tr.trace_direct(src, rays, reemit, w, sparse=sparse, seed=1)
        peak[name(sparse)] = int(pm.held)
        tr.close()
    lib.rthx_release_cached()
    # times: one handle, a warm-up call of each route, then the routes alternately
    tr = rthx.DeviceTracer(flat, device=0)
    for sparse in routes:
        tr.trace_direct(src, rays, reemit, w, sparse=sparse, seed=1)
    runs, absorbed = [], {}
    for r in range(reps):
        for sparse in routes:
            res, ab = one_call(tr, src, rays, reemit, w, sparse, seed=100 + r)
            runs.append(dict(route=name(sparse), rep=r, **res))
            absorbed.setdefault(r, {})[sparse] = ab
    tr.close()
    lib.rthx_release_cached()
    med = {name(s): dict({k: float(np.median([x[k] for x in runs if x["route"] == name(s)])) for k in ("kernel_ms", "reduce_ms", "rest_ms", "call_ms")},
                         peak_bytes=peak[name(s)]) for s in routes}
    out = dict(ndim=ndim, N=flat.n_elements, sources=len(src), bundles=int(rays.sum()), dense_count_bytes=8 * len(src) * flat.n_elements,
               median=med, runs=runs)
    if len(routes) == 2:
        out["absorbed_bit_identical"] = all(np.array_equal(a[False].view(np.uint64), a[True].view(np.uint64)) for a in absorbed.values())
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--bundles-per-source", type=float, default=1000)
    ap.add_argument("--skip-400", action="store_true")
    a = ap.parse_args()
    res = dict(card=card())
    res["square260"] = probe(260, int(a.bundles_per_source * 68_640), a.reps, (False, True))
    if not a.skip_400:
        res["square400"] = probe(400, int(a.bundles_per_source * 161_600), a.reps, (True,))
    doc = json.dumps(res, indent=1, default=float)
    print(doc)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "direct_sparse_probe.json"), "w") as f:
            f.write(doc)


if __name__ == "__main__":
    main()
