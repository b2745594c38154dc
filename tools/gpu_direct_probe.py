"""method=:direct on the device: bundle and event rates of trace_direct_kernel, and the whole call against :exchange + solveEquilibrium.

  python tools/gpu_direct_probe.py [--out DIR] [--bundles 1e9] [--reps 3]

Rates (DeviceTracer.trace_direct, kernel time from CUDA events, after one warm-up call of each kind), without and with the
redirection tally (redirected=True), alternated rep by rep on one handle:
  cs101   101 x 101, kappa = 1, black walls, bottom at 1000 K, gas of zero net emission (the Crosbie & Schrenker set-up);
  refl41  41 x 41, kappa = 1, eps = (1, .5, .5, .5), bottom at 1000 K (a reflecting enclosure), gas of zero net emission.
Whole call on cs101: rtm(B; method=:direct) against rtm(B; method=:exchange) + solveEquilibrium, host wall time of each, and each
route's centre-line S(tau) error against the C&S table (norm-relative, as test_2d_grey.jl:216).  Prints one JSON document and writes it
to DIR/direct_probe.json."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import rthx  # noqa: E402
from oracle import grey_solver as gs  # noqa: E402
from rthx.direct import direct_sources  # noqa: E402


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def domain(name):
    if name == "cs101":
        return rthx.meshes.square_domain(101, kappa=1.0)
    return rthx.meshes.square_domain(41, kappa=1.0, epsilon=(1, .5, .5, .5))


def rates(name, bundles, reps):
    """Each rep traces the same bundles without and with the redirection tally (redirected=True), alternately, on one handle."""
    rtm = domain(name)
    flat = rthx.flatten_domain(rtm)
    ws, known_T, E, src, rays, w = direct_sources(rtm, bundles)
    reemit = np.zeros(flat.n_elements, np.uint8)
    reemit[:len(known_T)] = ~known_T
    tr = rthx.DeviceTracer(flat, device=0)
    for tally in (False, True):
        tr.trace_direct(src, np.minimum(rays, 1000), reemit, w, seed=1, redirected=tally)
    runs = []
    for r in range(reps):
        for tally in (False, True):
            out = tr.trace_direct(src, rays, reemit, w, seed=100 + r, redirected=tally)
            ms = out["stats"]["kernel_ms"]
            runs.append(dict(tally=tally, kernel_ms=ms, total_ms=out["stats"]["total_ms"], bundles=int(rays.sum()), events=out["events"],
                             lost=int(out["lost"].sum()), bundles_per_s=rays.sum() / (ms * 1e-3), events_per_s=out["events"] / (ms * 1e-3)))
    tr.close()
    median = {str(t): {k: float(np.median([x[k] for x in runs if x["tally"] == t])) for k in ("kernel_ms", "bundles_per_s", "events_per_s")}
              for t in (False, True)}
    return dict(domain=name, N=flat.n_elements, sources=len(src), runs=runs, median_without_tally=median["False"], median_with_tally=median["True"],
                tally_cost=median["True"]["kernel_ms"] / median["False"]["kernel_ms"] - 1.0)


def centre_line_error(rtm):
    S = gs.centerline_source_function(rtm, 101, 1000.0)
    A = gs.analytical_centerline(101)
    return float(np.linalg.norm(S - A) / max(np.linalg.norm(S), np.linalg.norm(A)))


def whole_calls(bundles):
    out = {}
    rtm = domain("cs101")
    rtm(10_000_000, method="direct", verbose=False, seed=1, devices=[0])           # warm-up: handle, modules
    rtm = domain("cs101")
    t0 = time.perf_counter()
    rtm(bundles, method="direct", verbose=False, seed=2, devices=[0])
    out["direct"] = dict(seconds=time.perf_counter() - t0, centre_line_rel_error=centre_line_error(rtm), stats=rtm.last_direct_stats)
    rtm = domain("cs101")
    rtm(10_000_000, method="exchange", verbose=False, seed=1, devices=[0])
    rtm = domain("cs101")
    t0 = time.perf_counter()
    rtm(bundles, method="exchange", verbose=False, seed=2, devices=[0])
    t1 = time.perf_counter()
    rthx.solveEquilibrium(rtm, rtm.F_smooth, verbose=False)
    t2 = time.perf_counter()
    out["exchange_plus_solve"] = dict(seconds=t2 - t0, trace_and_smooth_s=t1 - t0, solve_s=t2 - t1, centre_line_rel_error=centre_line_error(rtm))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--bundles", type=float, default=1e9)
    ap.add_argument("--rate-bundles", type=float, default=2e8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--skip-whole", action="store_true")
    a = ap.parse_args()
    res = dict(card=card(), rates=[rates(n, int(a.rate_bundles), a.reps) for n in ("cs101", "refl41")])
    if not a.skip_whole:
        res["whole_call"] = whole_calls(int(a.bundles))
    doc = json.dumps(res, indent=1, default=float)
    print(doc)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "direct_probe.json"), "w") as f:
            f.write(doc)


if __name__ == "__main__":
    main()
