"""bench.py's contract: the reference arm (`--impl reference`) prints one JSON line with the keys the driver reads,
runs on rank 0 only under torchrun, and ignores the OMP_NUM_THREADS=1 that torchrun exports to its workers; `--dump-outputs`
writes what the last timed step computed."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra):
    env = dict(os.environ)
    env.update(env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg1", "--steps", "1",
                           "--warmup", "0", "--cpu-sample-rays", "2e6"], capture_output=True, text=True, env=env, timeout=600)


def test_reference_arm_line_and_rank_gating():
    r = _run({"OMP_NUM_THREADS": "1"})
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "exchange_factor_rays_per_sec" and line["unit"] == "rays/s"
    assert line["higher_is_better"] is True and line["value"] > 0 and line["gpu_launches"] == 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] == line["value"]
    n_cores = len(os.sched_getaffinity(0))
    assert line["cpu_baseline"]["cores"] == n_cores                      # not the single thread OMP_NUM_THREADS=1 asks for
    assert line["e2e"] == {"value": line["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["config"]["workload"].startswith("cfg1")
    # under torchrun only rank 0 works and prints
    r1 = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r1.returncode == 0 and r1.stdout.strip() == ""


def test_both_arms_print_the_same_config():
    """The driver compares `config` of this repo's arm and of the reference arm: both come from one function, strong scaling (the
    named ray count split over the GPUs) is the default, and the reference arm's line carries it unchanged."""
    import argparse
    sys.path.insert(0, ROOT)
    import bench
    old = sys.argv
    try:
        sys.argv = ["bench.py", "--workload", "cfg1", "--gpus", "4"]
        args = bench.parse_args()
    finally:
        sys.argv = old
    assert args.scaling == "strong"
    cfg4 = bench.workload_config(args, 165, 1, 4)
    cfg1 = bench.workload_config(args, 165, 1, 1)
    assert cfg4 == cfg1 and cfg4["rays_per_step"] == 999900 and cfg4["rays_per_emitter"] == 6060       # same job at every N
    args.scaling = "weak"
    assert bench.workload_config(args, 165, 1, 4)["rays_per_step"] == 4 * 1_000_000 // 165 * 165
    r = _run({})
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["config"] == cfg1 and line["scaling"] == "strong"
    assert line["cpu_baseline"]["mode"] == "faithful" and line["cpu_baseline"]["other_mode"]["mode"] == "philox"


def test_reference_faithful_mode_is_statistically_the_same_tracer(oracle_mod=None):
    """The timing mode of the CPU arm (per-thread xoshiro256++, Dict-like row tally) traces the same physics as the Philox oracle:
    row sums exact, aggregated wall-to-wall / wall-to-gas fractions equal within Monte Carlo noise."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import rthx
    from oracle import oracle
    flat = rthx.flatten_domain(rthx.meshes.cfg1())
    a = oracle.trace(flat, 4000, seed=1)
    b = oracle.trace(flat, 4000, seed=1, faithful=True)
    oracle.trace(flat, 10, seed=1)                                           # leaves the switch off again
    ns = flat.n_surfaces
    for o in (a, b):
        assert np.all(o["counts"][0].sum(axis=1) + o["lost"][0] == 4000)
    fa = a["counts"][0][:ns, ns:].sum() / a["counts"][0][:ns].sum()
    fb = b["counts"][0][:ns, ns:].sum() / b["counts"][0][:ns].sum()
    assert abs(fa - fb) < 5e-3 and not np.array_equal(a["counts"], b["counts"])


def _bench_module():
    sys.path.insert(0, ROOT)
    import bench
    return bench


def test_steps_must_be_positive_and_dump_needs_the_rthx_path():
    bench = _bench_module()
    old = sys.argv
    try:
        for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"]):
            sys.argv = ["bench.py"] + argv
            with pytest.raises(SystemExit):
                bench.parse_args()
        sys.argv = ["bench.py", "--steps", "3", "--dump-outputs", "d"]
        args = bench.parse_args()
    finally:
        sys.argv = old
    assert args.steps == 3 and args.dump_outputs == "d"


def test_dump_outputs_writes_float64_rows_of_a_fixed_sample(tmp_path, monkeypatch):
    """--dump-outputs: lost whole, the count rows of a seeded emitter sample that depends on the shape only, all rows when they fit."""
    import numpy as np
    import torch
    bench = _bench_module()
    nb, N = 2, 50
    counts = torch.arange(nb * N * N, dtype=torch.int64).reshape(nb, N, N)
    lost = torch.arange(nb * N, dtype=torch.int64).reshape(nb, N)

    def dump(d):
        bench.dump_outputs(str(d), counts, lost)
        return {n: np.load(d / f"{n}.npy") for n in ("counts_rows", "counts_row_ids", "lost")}

    whole = dump(tmp_path / "whole")
    assert all(a.dtype == np.float64 for a in whole.values())
    assert np.array_equal(whole["counts_row_ids"], np.arange(N)) and np.array_equal(whole["counts_rows"], counts.numpy())
    assert np.array_equal(whole["lost"], lost.numpy())
    monkeypatch.setattr(bench, "DUMP_COUNT_BYTES", 7 * 8 * nb * N)
    a, b = dump(tmp_path / "a"), dump(tmp_path / "b")
    ids = a["counts_row_ids"].astype(np.int64)
    assert len(ids) == 7 and np.all(np.diff(ids) > 0) and np.array_equal(a["counts_row_ids"], b["counts_row_ids"])
    assert np.array_equal(a["counts_rows"], counts.numpy()[:, ids]) and np.array_equal(a["lost"], lost.numpy())


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path, rthx_mod, cuda_lib):
    """The dumped tallies are those of the last timed step (seed 1000 + 1000 + steps - 1), identical to a plain trace of that seed."""
    import numpy as np
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg1", "--steps", "2", "--warmup", "1",
                        "--no-extras", "--no-e2e", "--no-smoothing", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    flat = rthx_mod.flatten_domain(rthx_mod.meshes.cfg1())
    want = rthx_mod.DeviceTracer(flat, device=0).trace(line["config"]["rays_per_emitter"], seed=2001)
    ids = np.load(tmp_path / "counts_row_ids.npy").astype(np.int64)
    assert np.array_equal(ids, np.arange(flat.n_elements))
    assert np.array_equal(np.load(tmp_path / "counts_rows.npy"), want["counts"][:, ids].astype(np.float64))
    assert np.array_equal(np.load(tmp_path / "lost.npy"), want["lost"].astype(np.float64))
