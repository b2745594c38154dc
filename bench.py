#!/usr/bin/env python
"""bench.py — exchange-factor rays/s on BASELINE.json's metric configuration (config 3: 101x101 grey scattering
enclosure, kappa = sigma_s = 0.5, 1e10 rays per step — sharded over the N GPUs, as BASELINE.json names it).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # CPU restatement of the reference on the host cores
    python bench.py --dump-outputs DIR ...                   # also write the last timed step's tallies to DIR/*.npy

A "step" is one full exchange-factor trace of the workload: zero the UInt64 count matrix, trace rays_total rays (every
emitter row, all bands), land the rows of all GPUs in one matrix on rank 0.  `value` is device-resident whole-job rays/s
(strong scaling by default: the SAME 1e10 rays at every N; `--scaling weak` keeps 1e10 rays per GPU, and a short run of the
other mode is reported under `weak` / `strong`).  `e2e` is the same trace through the C ABI with HOST buffers, by the entry
points the drop-in calls from ONE process — rthx_create_multi + rthx_trace_exchange_multi over all N GPUs (mesh upload +
trace + device->host copy of the counts inside the timed region); `e2e_per_rank` is the one-process-per-GPU variant.
One JSON line is printed by rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

_ROOT = os.path.dirname(os.path.abspath(__file__))
if _ROOT not in sys.path:
    sys.path.insert(0, _ROOT)

METRIC = "exchange_factor_rays_per_sec"
UNIT = "rays/s"
# algorithmic FP64 flop per ray by (emitter kind, ending), SURVEY.md §8(d) / BASELINE.md §4
FLOP_SG, FLOP_SW, FLOP_VG, FLOP_VW, FLOP_CROSS = 90.0, 138.0, 98.0, 146.0, 65.0


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="rthx", choices=["rthx", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"])
    ap.add_argument("--rays", type=float, default=None,
                    help="rays per step (strong) or per GPU and step (weak); default: the configuration's named count (1e10 for cfg3)")
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"],
                    help="strong (default) = the named ray count split over the N GPUs, as BASELINE.json words cfg3; weak = that count per GPU")
    ap.add_argument("--cpu-sample-rays", type=float, default=1.0e9,
                    help="rays of the bounded CPU sample: a fifth of it per step of the reference arm and of the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-smoothing", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip public_call / other_configs / the secondary scaling mode")
    ap.add_argument("--block-threads", type=int, default=0)
    ap.add_argument("--row-chunks", type=int, default=0)
    ap.add_argument("--locator", default="auto", choices=["auto", "generic"],
                    help="generic = the reference-faithful grid + point-in-polygon locator everywhere (the path arbitrary, non-affine meshes take)")
    ap.add_argument("--mode", default="first_interaction", choices=["first_interaction", "multi_bounce", "multi_bounce_specular"],
                    help="first_interaction = what method=:exchange computes (the headline); multi_bounce = total-exchange mode, rays followed "
                         "through scattering / wall reflection until absorbed (rthx.h RTHX_MULTI_BOUNCE)")
    ap.add_argument("--reduce", default="fused", choices=["fused", "nccl"],
                    help="N > 1: fused peer-memory flush over NVLink (default) or a private matrix per rank + NCCL reduce")
    ap.add_argument("--cpu-mode", default="faithful", choices=["faithful", "philox"],
                    help="CPU arm: faithful = per-thread xoshiro256++ and a Dict-like row tally, as the reference does (SURVEY.md 8(d)); "
                         "philox = the parity oracle itself (counter-based RNG, dense row)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (float64): lost [bands, N] whole "
                         "and a fixed seeded sample of emitter rows of the count matrix [bands, N, N]; the same arguments give the same "
                         "inputs, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "rthx":
        ap.error("--dump-outputs applies to --impl rthx")
    return args


# DRAM bytes per launch of the trace kernel measured by ncu --set full (dram__bytes_read.sum + dram__bytes_write.sum)
NCU_DRAM_BYTES_PER_LAUNCH = {"cfg3": (893.59e6 + 831.82e6, "profiles/r2/r2p_trace_exchange_sq_metrics.csv"),
                             "cfg5": (None, "profiles/r1y_trace_exchange_queue_metrics.csv")}

# executed warp instructions per 32 rays of the trace kernel (ncu source page, profiles/<capture>_sass_mix.csv, TOTAL row)
NCU_WARP_INSTR_PER_32_RAYS = {"cfg3": (250.8, "profiles/r2/r2p_trace_exchange_sq_sass_mix.csv"),
                              "cfg5": (680.9, "profiles/r1y_trace_exchange_queue_sass_mix.csv")}

DEFAULT_RAYS = {"cfg1": 1e6, "cfg2": 1e8, "cfg3": 1e10, "cfg4": 1e8, "cfg5": 1e9}


def build_workload(name):
    import rthx
    rtm = getattr(rthx.meshes, name)()
    flat = rthx.flatten_domain(rtm)
    if rtm.spectral_mode == "spectral_variable":
        groups, reps, nonuniform = rthx.group_uniform_bins(rtm.uniform_across_bin)
        bins = [b - 1 for b in nonuniform] + [g[0] - 1 for g in groups]
    else:
        bins = [0]
    return rtm, flat, bins


def workload_desc(name):
    return {
        "cfg1": "README Example 1, 1x1 m square, 11x11 grey gas kappa=1, black walls",
        "cfg2": "2D grey reflecting enclosure 41x41, kappa=1",
        "cfg3": "2D grey absorbing+scattering medium kappa=0.5 sigma_s=0.5, 101x101 mesh",
        "cfg4": "2D spectral multi-band gas 51x51, 8 bands batched in the grid",
        "cfg5": "16-wedge circle with transparent interfaces and triangle sub-meshes (11,11)",
    }[name]


def rays_of_job(args, world):
    """Total rays per traced band and step (the reference's `rays_total`, parallelRayTracing.jl:22-25,34-37)."""
    base = float(args.rays) if args.rays else DEFAULT_RAYS[args.workload]
    return base * (world if args.scaling == "weak" else 1)


def workload_config(args, N, nb, world):
    """The `config` object — identical in this repo's arm and in the reference arm (the driver compares them)."""
    rpe = int(rays_of_job(args, world)) // N
    return {"workload": f"{args.workload}: {workload_desc(args.workload)}", "elements": N, "bands": nb,
            "rays_per_step": rpe * N * nb, "rays_per_emitter": rpe, "scaling": args.scaling,
            "l2": "inputs larger than L2: the 8*N*N-byte count matrix is rewritten every step (900 MB for cfg3 against 126 MB of L2), "
                  "and every step uses a fresh Philox seed"}


def flop_per_ray(stats):
    n = stats["n_surface_gas"] + stats["n_surface_wall"] + stats["n_volume_gas"] + stats["n_volume_wall"]
    if n == 0:
        return 100.0
    return (FLOP_SG * stats["n_surface_gas"] + FLOP_SW * stats["n_surface_wall"] + FLOP_VG * stats["n_volume_gas"]
            + FLOP_VW * stats["n_volume_wall"] + FLOP_CROSS * stats["n_crossings"]) / n


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def host_threads():
    # every host core this process may run on, set explicitly: torchrun exports OMP_NUM_THREADS=1 to its workers
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def run_oracle_sample(flat, bins, rays_total, seed, faithful=False):
    """Time the CPU oracle (all host threads) on a bounded sample of the workload.  Threads are NOT pinned: OMP_PROC_BIND / OMP_PLACES
    put every thread on one core inside the GPU box's container (measured: 5.3e6 instead of 7.7e7 rays/s)."""
    from oracle import oracle
    N = flat.n_elements
    rpe = max(1, int(rays_total) // (N * len(bins)))
    t0 = time.perf_counter()
    out = oracle.trace(flat, rpe, seed=seed, bins=bins, n_threads=host_threads(), faithful=faithful)
    dt = time.perf_counter() - t0
    traced = rpe * N * len(bins)
    loop_s = out["stats"].get("loop_seconds") or dt
    return dict(rays_per_s=traced / dt, loop_rays_per_s=traced / loop_s, seconds=dt, loop_seconds=loop_s, rays=traced, rpe=rpe, stats=out["stats"])


def cpu_sample_text(sample, mode, r):
    what = ("reference-faithful C restatement: contiguous emitter ranges per thread, per-thread xoshiro256++, Dict-like row tally "
            "(parallelRayTracing.jl:83-91,104,124)" if mode == "faithful" else
            "the parity oracle: C restatement with the Philox contract and a dense row tally")
    return (f"{int(sample):d} rays per step of the same workload ({what}; OpenMP, Julia absent); wall time of the whole "
            f"call; emitter loop alone: {r['loop_rays_per_s']:.3e} rays/s; cpu: {cpu_model()}")


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons with nvidia-smi while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.rows = []
        self._stop = threading.Event()
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self._stop.is_set():
                    break
                self.rows.append((time.monotonic(), [x.strip() for x in line.split(",")]))
        except Exception:
            pass

    def stop(self):
        self._stop.set()
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass

    def summary(self, t0=None, t1=None):
        """Median SM clock and active throttle reasons over the samples taken inside [t0, t1] (the timed region)."""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, r in self.rows:
            if (t0 is not None and ts < t0) or (t1 is not None and ts > t1):
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except (ValueError, IndexError):
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def run_julia_reference(args, sample, cfg):
    """If a `julia` binary and baseline/_ref exist, time the UNMODIFIED reference (baseline/run_julia_ref.jl).
    Neither exists in this image (SURVEY.md §0.6), so this returns None and the C restatement is timed instead."""
    import shutil
    julia = shutil.which("julia")
    ref = os.path.join(_ROOT, "baseline", "_ref")
    if julia is None or not os.path.isdir(ref):
        return None
    ndim, kappa, sig = {"cfg1": (11, 1.0, 0.0), "cfg2": (41, 1.0, 0.0), "cfg3": (101, 0.5, 0.5)}[args.workload]
    try:
        r = subprocess.run([julia, "-t", "auto", f"--project={ref}", os.path.join(_ROOT, "baseline", "run_julia_ref.jl"),
                            str(ndim), str(kappa), str(sig), str(int(sample)), str(args.steps)],
                           capture_output=True, text=True, timeout=1500)
        line = next(l for l in r.stdout.splitlines() if l.startswith("RTHX_JULIA_REF"))
        kv = dict(x.split("=") for x in line.split()[1:])
    except Exception:
        return None
    value = float(kv["rays_per_s"])
    return {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": float(kv["rays"]) / value * 1e3, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": int(kv["threads"]), "kind": "reference",
                             "sample": f"{kv['rays']} rays per step, parallelRayTracing of the unmodified Julia reference"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}


def main_reference(args):
    """Reference arm: the reference's own algorithm on the host cores.  Julia is absent from the image, so this is the C
    restatement (oracle/rthx_oracle.c, kind "port") in its reference-faithful timing mode with every host thread, on a bounded
    sample per step; the Philox-contract oracle is timed next to it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    rtm, flat, bins = build_workload(args.workload)
    cfg = workload_config(args, flat.n_elements, len(bins), world)
    sample = min(args.cpu_sample_rays / 5.0, cfg["rays_per_step"])
    julia_line = run_julia_reference(args, sample, cfg) if args.workload in ("cfg1", "cfg2", "cfg3") else None
    if julia_line is not None:
        print(json.dumps(julia_line))
        return 0
    faithful = args.cpu_mode == "faithful"
    for _ in range(max(0, args.warmup)):
        run_oracle_sample(flat, bins, sample / 10.0, seed=7, faithful=faithful)
    t0 = time.perf_counter()
    rays = 0
    last = None
    loop_s = 0.0
    for s in range(args.steps):
        last = run_oracle_sample(flat, bins, sample, seed=100 + s, faithful=faithful)
        rays += last["rays"]
        loop_s += last["loop_seconds"]
    dt = time.perf_counter() - t0
    value = rays / dt
    other = run_oracle_sample(flat, bins, sample, seed=99, faithful=not faithful)
    last = dict(last, loop_rays_per_s=rays / loop_s if loop_s > 0 else value)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / max(1, args.steps) * 1e3, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": last["stats"]["n_threads"] if last else 0, "kind": "port",
                         "mode": args.cpu_mode, "sample": cpu_sample_text(sample, args.cpu_mode, last),
                         "other_mode": {"mode": "philox" if faithful else "faithful", "value": other["rays_per_s"],
                                        "loop_value": other["loop_rays_per_s"]}},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def matrix_hash(t):
    """Position-sensitive 64-bit hash of an int64 tensor (wrapping arithmetic): sum_i c_i * (i * K + 1) mod 2^64."""
    import torch
    flat = t.reshape(-1)
    acc = 0
    chunk = 1 << 26
    for a in range(0, flat.numel(), chunk):
        c = flat[a:a + chunk]
        idx = torch.arange(a, a + c.numel(), dtype=torch.int64, device=c.device)
        acc = (acc + int((c * (idx * -7046029254386353131 + 1)).sum().item())) & 0xFFFFFFFFFFFFFFFF
    return acc


DUMP_COUNT_BYTES = 48 << 20     # count-matrix sample of --dump-outputs (900 MB whole for cfg3); lost and the row ids stay small


def dump_outputs(out_dir, counts, lost):
    """Write the last step's `lost` [nb, N] whole and the rows of `counts` [nb, N, N] of a fixed seeded sample of emitters (all
    rows when they fit DUMP_COUNT_BYTES) with their indices, as float64 (exact: every count is below 2^53)."""
    import numpy as np
    import torch
    nb, N, _ = counts.shape
    k = max(1, min(N, DUMP_COUNT_BYTES // (8 * nb * N)))
    rows = np.sort(np.random.default_rng(0).choice(N, size=k, replace=False))
    sample = counts.index_select(1, torch.from_numpy(rows).to(counts.device))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "counts_rows.npy"), sample.cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "counts_row_ids.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "lost.npy"), lost.cpu().numpy().astype(np.float64))


def main():
    args = parse_args()
    if args.impl == "reference":
        return main_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    import rthx
    from rthx.dist import ShardedTracer
    from rthx._lib import create_multi, trace_multi, pinned_empty

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the rthx path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        cpu_group = dist.new_group(backend="gloo")          # host-only barriers while ONE rank drives every GPU
    dev = torch.device("cuda", local_rank)

    rtm, flat, bins = build_workload(args.workload)
    N = flat.n_elements
    nb = len(bins)
    cfg = workload_config(args, N, nb, world)
    rpe = cfg["rays_per_emitter"]
    traced_per_step = cfg["rays_per_step"]

    kw = dict(bins=bins, block_threads=args.block_threads, row_chunks=args.row_chunks, locator=1 if args.locator == "generic" else 0,
              mode={"first_interaction": 0, "multi_bounce": 1, "multi_bounce_specular": 2}[args.mode])
    stream = torch.cuda.current_stream(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def host_barrier():
        if world > 1:
            dist.barrier(group=cpu_group)

    def timed_resident(sh, rpe_, steps, warmup, seed0, sampler=None):
        """W warm-up + K timed steps of the device-resident sharded trace; returns (ms_per_step, kernel_ms, last stats, window)."""
        st = None
        for w in range(warmup):
            sh.enqueue(rpe_, seed=seed0 + w, **kw); sh.finish()
        barrier()
        kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t_win0 = time.monotonic()
        e0.record(stream)
        for s in range(steps):
            kev[s][0].record(stream)
            st = sh.enqueue(rpe_, seed=seed0 + 1000 + s, **kw)      # zero (own rows) + trace kernel (+ fused peer flush) + step flag
            kev[s][1].record(stream)
            sh.finish()                                             # rank 0: wait for every rank's flag (fused) or the NCCL reduce
        e1.record(stream)
        barrier()
        t_win1 = time.monotonic()
        total_ms = e0.elapsed_time(e1)
        kernel_ms = sum(a.elapsed_time(b) for a, b in kev) / max(1, steps)
        t = torch.tensor([total_ms, kernel_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]) / max(1, steps), float(t[1]), st, (t_win0, t_win1)

    # ---- device-resident timing ------------------------------------------------------------------------------
    sh = ShardedTracer(flat, device=local_rank, rank=rank, world=world, n_bins=nb, mode=args.reduce)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()                      # nvidia-smi needs ~0.5 s to deliver its first sample: start before warm-up
    ms_per_step, kernel_ms, st, (t_win0, t_win1) = timed_resident(sh, rpe, args.steps, args.warmup, 1000)
    if sampler:
        time.sleep(0.15)
        sampler.stop()
    value = traced_per_step / (ms_per_step * 1e-3)
    lost_total = int(sh.lost.sum().item()) if rank == 0 else 0
    tallied = int(sh.counts.sum().item()) if rank == 0 else 0
    flag_timeouts = sh.wait_errors()
    if args.dump_outputs and rank == 0:      # before anything else traces into sh: it still holds the last timed step
        dump_outputs(args.dump_outputs, sh.counts, sh.lost)

    # the other scaling mode, short (N > 1): weak next to the strong headline, or the reverse
    other_scaling = None
    if world > 1 and not args.no_extras:
        o_mode = "weak" if args.scaling == "strong" else "strong"
        base = float(args.rays) if args.rays else DEFAULT_RAYS[args.workload]
        o_rpe = int(base * (world if o_mode == "weak" else 1)) // N
        o_ms, o_kms, _, _ = timed_resident(sh, o_rpe, min(args.steps, 3), 1, 5000)
        other_scaling = {"scaling": o_mode, "rays_per_step": o_rpe * N * nb, "ms_per_step": o_ms, "kernel_ms": o_kms,
                         "value": o_rpe * N * nb / (o_ms * 1e-3), "steps": min(args.steps, 3)}

    # ---- multi-GPU bit-exactness where the driver sees it: strong-sharded fused / NCCL traces against rank 0's own
    # single-GPU trace of the same arguments (north star: "bit-exact across runs and GPU counts") ---------------------
    bit_exact = None
    if world > 1:
        c_rpe = 2000 if args.workload == "cfg3" else max(1, min(rpe, 2000))
        sh.enqueue(c_rpe, seed=0xB17E, **kw); sh.finish()
        torch.cuda.synchronize(dev)
        res = {}
        if rank == 0:
            fused_c, fused_l = sh.counts.clone(), sh.lost.clone()
        other = ShardedTracer(flat, device=local_rank, rank=rank, world=world, n_bins=nb, mode="nccl" if args.reduce == "fused" else "fused")
        other.enqueue(c_rpe, seed=0xB17E, **kw); other.finish()
        torch.cuda.synchronize(dev)
        if rank == 0:
            single = ShardedTracer(flat, device=local_rank, rank=0, world=1, n_bins=nb, mode="local")
            single.enqueue(c_rpe, seed=0xB17E, **kw); single.finish()
            torch.cuda.synchronize(dev)
            h1 = matrix_hash(single.counts)
            res = {"rays_per_emitter": c_rpe, "seed": 0xB17E, "hash_single_gpu": f"{h1:016x}",
                   f"hash_{sh.mode}": f"{matrix_hash(fused_c):016x}", f"hash_{other.mode}": f"{matrix_hash(other.counts):016x}",
                   "counts_equal": bool(torch.equal(fused_c, single.counts) and torch.equal(other.counts, single.counts)),
                   "lost_equal": bool(torch.equal(fused_l, single.lost) and torch.equal(other.lost, single.lost)),
                   "tallied": int(single.counts.sum().item())}
            res["bit_exact_vs_single_gpu"] = bool(res["counts_equal"] and res["lost_equal"] and
                                                  res["hash_single_gpu"] == res[f"hash_{sh.mode}"] == res[f"hash_{other.mode}"])
            del fused_c, fused_l
            single.close()
        other.close()
        bit_exact = res
        barrier()

    # ---- end-to-end through the C ABI with host buffers ------------------------------------------------------
    mesh_bytes = sum(getattr(flat, n).nbytes for n in (
        "coarse_nv", "coarse_vx", "coarse_vy", "coarse_solid", "fine_off", "cell_nv", "cell_vx", "cell_vy", "cell_mid",
        "cell_volume", "cell_surf_id", "kappa", "sigma_s", "epsilon", "uniform_beta"))
    e2e = e2e_per_rank = None
    if not args.no_e2e:
        # (1) ONE process drives all N GPUs — what the drop-in (julia/RTHXExchange.jl) calls: rthx_create_multi +
        #     rthx_trace_exchange_multi into a page-locked host matrix + rthx_destroy.  Rank 0 runs it, the other ranks wait on
        #     the host (gloo): their GPUs are driven by rank 0's process.
        barrier()
        if rank == 0:
            counts_host = pinned_empty((nb, N, N), np.uint64)
            dev_ms, phases = [], []

            def e2e_step(seed):
                tp = [time.perf_counter()]
                trs = create_multi(flat, list(range(world))) if world > 1 else [rthx.DeviceTracer(flat, device=local_rank)]
                tp.append(time.perf_counter())
                if world > 1:
                    out = trace_multi(trs, rpe, counts_out=counts_host, seed=seed, **kw)
                else:
                    out = trs[0].trace(rpe, counts_out=counts_host, seed=seed, **kw)
                tp.append(time.perf_counter())
                for t in trs:
                    t.close()
                tp.append(time.perf_counter())
                dev_ms.append((out["stats"]["kernel_ms"], out["stats"]["total_ms"]))
                phases.append([1e3 * (b - a) for a, b in zip(tp[:-1], tp[1:])])
                return int(out["lost"].sum())

            for w in range(max(1, min(args.warmup, 2))):
                e2e_step(3000 + w)
            t0 = time.perf_counter()
            for s in range(args.steps):
                lost_e2e = e2e_step(3100 + s)
            dt = time.perf_counter() - t0
            ph = np.mean(np.array(phases[-args.steps:]), axis=0)
            e2e = {"value": traced_per_step * args.steps / dt, "unit": UNIT,
                   "h2d_bytes_per_step": int((mesh_bytes + 4 * nb) * world),
                   "d2h_bytes_per_step": int(8 * nb * N * N + 8 * nb * N * world),
                   "ms_per_step": dt / args.steps * 1e3,
                   "device_ms_per_step": {"kernel": float(np.mean([a for a, _ in dev_ms[-args.steps:]])),
                                          "zero+kernel+d2h": float(np.mean([b for _, b in dev_ms[-args.steps:]]))},
                   "phases_ms": {"create": float(ph[0]), "trace+d2h": float(ph[1]), "destroy": float(ph[2])},
                   "path": ("rthx_create + rthx_trace_exchange (page-locked host count matrix) + rthx_destroy" if world == 1 else
                            f"one process, {world} GPUs: rthx_create_multi + rthx_trace_exchange_multi (every device copies its rows into one "
                            "page-locked host matrix over its own PCIe link) + rthx_destroy"),
                   "check_total": int(counts_host.sum()) + lost_e2e}
            del counts_host
        host_barrier()
        barrier()

        # (2) one process per GPU (N > 1): every rank re-uploads the mesh and copies ITS rows into one page-locked matrix in POSIX
        #     shared memory over its own PCIe link (overlapped with tracing); a barrier makes the matrix complete on rank 0.
        if world > 1:
            from rthx._lib import SharedHostMatrix
            shm_name = f"rthx_bench_{os.environ.get('MASTER_PORT', '0')}"
            ok = torch.ones(1, dtype=torch.int32, device=dev)
            shared_host = None
            if rank == 0:
                try:
                    shared_host = SharedHostMatrix(shm_name, (nb, N, N), create=True)
                    shared_host.array[0, 0, :8] = 0          # touch
                except Exception as ex:                       # e.g. a 64 MB /dev/shm
                    print(f"bench.py: shared host matrix unavailable ({ex}); e2e_per_rank skipped", file=sys.stderr)
                    shared_host = None
                    ok.zero_()
            dist.broadcast(ok, src=0)
            if int(ok.item()) == 1:
                if rank != 0:
                    shared_host = SharedHostMatrix(shm_name, (nb, N, N), create=False)
                pr_phases = []

                def pr_step(seed):
                    tp = [time.perf_counter()]
                    tr = rthx.DeviceTracer(flat, device=local_rank)
                    tp.append(time.perf_counter())
                    tr.trace(rpe, counts_out=shared_host.array, seed=seed, emitter_rank=rank, emitter_world=world, **kw)
                    tp.append(time.perf_counter())
                    dist.barrier(device_ids=[local_rank])
                    tp.append(time.perf_counter())
                    tr.close()
                    tp.append(time.perf_counter())
                    pr_phases.append([1e3 * (b - a) for a, b in zip(tp[:-1], tp[1:])])

                pr_step(3500)
                barrier()
                t0 = time.perf_counter()
                for s in range(args.steps):
                    pr_step(3600 + s)
                barrier()
                dt = time.perf_counter() - t0
                tt = torch.tensor([dt], dtype=torch.float64, device=dev)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                dt = float(tt[0])
                ph = np.mean(np.array(pr_phases[1:]), axis=0)
                e2e_per_rank = {"value": traced_per_step * args.steps / dt, "unit": UNIT, "ms_per_step": dt / args.steps * 1e3,
                                "phases_ms": {"create": float(ph[0]), "trace+own-row d2h": float(ph[1]), "barrier": float(ph[2]), "destroy": float(ph[3])},
                                "path": "per rank: rthx_create + rthx_trace_exchange(own rows -> page-locked shared host matrix); NCCL barrier",
                                "check_total": int(shared_host.array.sum()) if rank == 0 else None}
                dist.barrier(device_ids=[local_rank])
                shared_host.close()

    # ---- the public call: mesh(rays; method=:exchange) with its phases (rank 0 drives every GPU) ---------------------
    public_call = None
    if not args.no_extras and args.mode == "first_interaction" and args.locator == "auto":
        barrier()
        if rank == 0:
          try:                               # rank 0 only, no collectives inside: a failure here must not cost the headline line
            runs = []
            for rep in range(3):
                t0 = time.perf_counter()
                rtm(int(rays_of_job(args, world)), method="exchange", verbose=False, seed=7000 + rep, devices=list(range(world)))
                wall = 1e3 * (time.perf_counter() - t0)
                runs.append(dict(rtm.last_phase_ms, wall=wall))
            best = min(runs[1:], key=lambda r: r["wall"])
            F_raw = rtm.F_raw if not isinstance(rtm.F_raw, list) else rtm.F_raw[0]
            public_call = {"call": f"mesh({int(rays_of_job(args, world))}; method=:exchange, devices={list(range(world))}) -> F_raw (CSC) + F_smooth",
                           "wall_ms": best["wall"], "rays_per_s": traced_per_step / (best["wall"] * 1e-3),
                           "phases_ms": {k: best[k] for k in ("flatten", "create", "trace", "csc_F_raw", "smoothing") if k in best},
                           "first_call_wall_ms": runs[0]["wall"],
                           "F_raw_nnz": int(F_raw.nnz), "F_raw_assembly_le_trace": bool(best.get("csc_F_raw", 0) <= best.get("trace", 0)),
                           "note": "flatten is the Python twin walking the domain objects (the Julia shim's loop over the same structs); best of "
                                   "two calls after one that also pays the page-locked allocations"}
            rtm.F_raw = rtm.F_smooth = None
            for t in getattr(rtm, "_devices", None) or []:
                t.close()
            rtm._devices = rtm._device = None
          except Exception as ex:
            public_call = {"error": f"{type(ex).__name__}: {ex}"}
        host_barrier()
        barrier()

    if rank != 0:
        sh.close()
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- the other named configurations, driver-run (N = 1): device-resident rays/s of each ---------------------------
    other_configs = None
    if world == 1 and not args.no_extras and args.workload == "cfg3" and args.mode == "first_interaction":
      try:
        other_configs = {}
        # ... and the two slower paths of the same kernel family on cfg3 / cfg5: the generic locator (what a mesh without a
        # verifiable lattice takes) and the total-exchange mode (every ray followed to absorption)
        variants = [(n, n, {}) for n in ("cfg1", "cfg2", "cfg4", "cfg5")] + \
                   [("cfg3_generic_locator", "cfg3", {"locator": 1}), ("cfg5_generic_locator", "cfg5", {"locator": 1}),
                    ("cfg3_multi_bounce", "cfg3", {"mode": 1})]
        for key, name, extra in variants:
            _, f2, b2 = build_workload(name)
            n2 = f2.n_elements
            rpe2 = int(min(DEFAULT_RAYS[name], 1e9)) // n2
            s2 = ShardedTracer(f2, device=local_rank, rank=0, world=1, n_bins=len(b2), mode="local")
            kw2 = dict(kw, bins=b2, **extra)
            for w in range(3):
                s2.enqueue(rpe2, seed=10 + w, **kw2)
            torch.cuda.synchronize(dev)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for s in range(5):
                s2.enqueue(rpe2, seed=20 + s, **kw2)
            b.record(stream)
            torch.cuda.synchronize(dev)
            ms = a.elapsed_time(b) / 5
            traced = rpe2 * n2 * len(b2)
            other_configs[key] = {"workload": workload_desc(name), "elements": n2, "bands": len(b2), "rays_per_step": traced,
                                   "ms_per_step": ms, "value": traced / (ms * 1e-3), "steps": 5, "warmup": 3,
                                   "tallied_plus_lost_ok": bool(int(s2.counts.sum().item()) + int(s2.lost.sum().item()) == traced)}
            s2.close()
      except Exception as ex:
        other_configs = {"error": f"{type(ex).__name__}: {ex}"}

    # ---- next-stage kernel: dense reciprocity smoothing of the traced matrix on the device (HBM-bound) -----------
    smoothing = solve = None
    if world == 1 and not args.no_smoothing:
      try:
        try:
            hbm_peak = json.load(open(os.path.join(_ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
            peak_src = "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth of this pool's B200)"
        except Exception:
            hbm_peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
        tr = rthx.DeviceTracer(flat, device=local_rank)
        tr.trace(max(1, rpe // 10), dense=False, seed=4000, **kw)
        w = rthx.get_w(rtm)
        _, ss = tr.smooth(w / w.min(), max_iters=1000, measure_pass=True)
        # grey equilibrium solve on the F_smooth that is still resident on the device (equilibriumGrey2D.jl:148-194)
        from rthx import equilibrium as _eq
        _, _b, coeff, h = _eq._system_vectors(rtm, _eq.populateWorkspace(rtm))
        _, _, sv = tr.solve_grey(coeff, h, measure_pass=True, atol=0.0)
        solve = {"kernel": "matvec_t_partial_kernel (y = F'x on the resident dense F_smooth: one read of F per Krylov step)",
                 "bound": "hbm", "achieved": sv["matvec_gbs"], "peak": hbm_peak, "unit": "GB/s",
                 "frac": sv["matvec_gbs"] / hbm_peak, "bytes_per_pass": sv["matvec_bytes"], "pass_ms": sv["matvec_ms"],
                 "iterations": sv["iterations"], "restarts": sv["restarts"], "matvecs": sv["matvecs"],
                 "converged": sv["converged"], "residual": sv["residual"], "rhs_norm": sv["rhs_norm"],
                 "total_ms": sv["total_ms"], "launches": sv["launches"], "peak_source": peak_src,
                 "traffic": 900086016 + 6328576,
                 "traffic_note": "dram bytes read + written per launch, ncu --set full, profiles/r1g_solve_matvec_metrics.csv"}
        tr.close()
        smoothing = {"kernel": "scale_rows_kernel (one alternating-projection iteration: X *= (u_i+u_j)/2 with fused row sums)",
                     "bound": "hbm", "achieved": ss["pass_gbs"], "peak": hbm_peak, "unit": "GB/s",
                     "frac": ss["pass_gbs"] / hbm_peak, "bytes_per_pass": 16 * N * N, "pass_ms": ss["pass_ms"],
                     "iterations": ss["iterations"], "delta_init": ss["delta_init"], "delta": ss["delta"], "converged": ss["converged"],
                     "total_ms": ss["total_ms"], "peak_source": peak_src}
      except Exception as ex:
        smoothing = {"error": f"{type(ex).__name__}: {ex}"}

    # ---- roofline (FP64 pipe) and CPU baseline ---------------------------------------------------------------
    fp64_peak = sh.tracer.measure_fp64_peak()
    # the algorithmic flop count per ray is a property of the workload: the (emitter kind, ending) mix from the oracle's counters
    # on a small sample, at every N
    mix = run_oracle_sample(flat, bins, 2.0e7, seed=7)
    A = flop_per_ray(mix["stats"])
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        sample = min(args.cpu_sample_rays / 5.0, traced_per_step)
        faithful = args.cpu_mode == "faithful"
        run_oracle_sample(flat, bins, sample / 10.0, seed=6, faithful=faithful)
        rs = [run_oracle_sample(flat, bins, sample, seed=7 + k, faithful=faithful) for k in range(3)]
        r = dict(rs[-1], rays_per_s=sum(x["rays"] for x in rs) / sum(x["seconds"] for x in rs),
                 loop_rays_per_s=sum(x["rays"] for x in rs) / sum(x["loop_seconds"] for x in rs))
        other = run_oracle_sample(flat, bins, sample, seed=5, faithful=not faithful)
        cpu = {"value": r["rays_per_s"], "unit": UNIT, "cores": r["stats"]["n_threads"], "kind": "port", "mode": args.cpu_mode,
               "sample": "3 x " + cpu_sample_text(sample, args.cpu_mode, r),
               "other_mode": {"mode": "philox" if faithful else "faithful", "value": other["rays_per_s"], "loop_value": other["loop_rays_per_s"]}}
    kernel_rays_per_s = (traced_per_step / world) / (kernel_ms * 1e-3)
    achieved = kernel_rays_per_s * A / 1e12
    info = sh.tracer.info
    kernel_name = ("trace_exchange_kernel<MULTI> (multi-bounce)" if args.mode != "first_interaction" and info["n_coarse"] > 1 else
                   "trace_exchange_sq_kernel<MULTI> (multi-bounce)" if args.mode != "first_interaction" else
                   "trace_exchange_kernel (generic locator)" if args.locator == "generic" else
                   "trace_exchange_sq_kernel" if info["n_coarse"] == 1 and info["n_affine_faces"] == 1 else
                   "trace_exchange_queue_kernel" if info["n_affine_faces"] + info["n_bilinear_faces"] == info["n_coarse"] else "trace_exchange_kernel")
    hbm_bytes_per_ray = 8.0 * N * N * nb / world / max(1, traced_per_step / world)
    roofline = {"bound": "fp64", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s",
                "frac": achieved / fp64_peak if fp64_peak else None,
                "traffic": NCU_DRAM_BYTES_PER_LAUNCH.get(args.workload, (None, None))[0],
                "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum per launch from the ncu --set full capture "
                                f"{NCU_DRAM_BYTES_PER_LAUNCH.get(args.workload, (None, 'none for this workload'))[1]} (the reductions "
                                "read-modify-write the zeroed 8*N*N-byte count matrix once, independent of the ray count)",
                "kernel": kernel_name, "kernel_ms": kernel_ms, "kernel_rays_per_s": kernel_rays_per_s,
                "flop_per_ray": A, "flop_per_ray_source": "oracle counters (emitter kind x ending mix) on a 2e7-ray sample of this workload",
                "peak_source": "FP64 DFMA-chain micro-benchmark measured in this run (MEASURED_PEAKS.json has no FP64 entry)",
                "hbm": {"algorithmic_bytes_per_ray": hbm_bytes_per_ray,
                        "achieved_gbs": kernel_rays_per_s * hbm_bytes_per_ray / 1e9, "peak_gbs": 6559.4,
                        "note": "count-matrix write-out only; the path is not HBM-bound"}}
    # secondary explanation: the kernel is bound by instruction issue (three half-rate pipes share one issue port per SM
    # sub-partition, DESIGN.md section 4), so state the issue-slot utilisation its measured rate implies
    clocks = sampler.summary(t_win0, t_win1 + 0.1) if sampler else None
    wi = NCU_WARP_INSTR_PER_32_RAYS.get(args.workload)
    if wi and clocks and clocks.get("sm_mhz") and args.mode == "first_interaction" and args.locator == "auto":
        slots = info["sm_count"] * 4 * clocks["sm_mhz"] * 1e6
        roofline["issue"] = {"warp_instr_per_32_rays": wi[0], "source": wi[1], "issue_slots_per_s": slots,
                             "frac": kernel_rays_per_s / 32.0 * wi[0] / slots,
                             "note": "executed warp instructions (ncu) x measured ray rate / (SMs x 4 sub-partitions x SM clock)"}
    n_flag = 0 if sh.mode != "fused" else args.steps * (world * 2 + 2)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": cfg,
        "sharding": {"partition": (f"emitter rows e % {world} == rank; " + (
                         "rows flushed into rank 0's matrix over NVLink peer memory inside the trace kernel (red.sys.add.u64), ranks "
                         "synchronised by device-side step flags in rank 0's memory (no host-launched collective per step)"
                         if sh.mode == "fused" else "one NCCL reduce of the u64 count matrix to rank 0" if sh.mode == "nccl" else "single GPU")),
                     "launch": {k: st[k] for k in ("n_blocks", "block_threads", "row_chunks", "smem_bytes", "hist_in_smem")},
                     "flag_wait_timeouts": flag_timeouts},
        "roofline": roofline, "smoothing": smoothing, "solve": solve, "cpu_baseline": cpu, "e2e": e2e,
        "gpu_launches": args.steps * world + n_flag,
        "launches": {"trace_kernels": args.steps * world, "flag_kernels": n_flag},
        "clocks": clocks,
        "check": {"tallied_last_step": tallied, "lost_last_step": lost_total},
    }
    if e2e_per_rank is not None:
        line["e2e_per_rank"] = e2e_per_rank
    if other_scaling is not None:
        line[other_scaling["scaling"]] = other_scaling
    if bit_exact is not None:
        line["check"].update(bit_exact)
    if public_call is not None:
        line["public_call"] = public_call
    if other_configs is not None:
        line["other_configs"] = other_configs
    print(json.dumps(line))
    sh.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
