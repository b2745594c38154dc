"""Fingerprint of every trace entry point over a fixed matrix of calls, for comparing two builds of the library bit for bit.

    python tools/gpu_trace_equality_probe.py --out run_new.txt
    RTHX_LIBRARY=/path/to/other/librthx.so python tools/gpu_trace_equality_probe.py --out run_other.txt
    diff run_other.txt run_new.txt            # empty: the same results, statistics, launch shapes and error messages

One line per call: the call's name, the rthx_stats fields that do not depend on time (n_blocks, block_threads, row_chunks, smem_bytes,
hist_in_smem, n_launches, rays_traced, rays_lost), the rthx_sparse_stats fields other than reduce_ms, a sha256 of every output array,
and a sha256 of the counts_csr / counts_csc read-outs of every traced bin of the counts the call left resident.  A call the library
refuses prints its message instead.  The matrix:
  meshes     cfg1 (single-quad kernel), cfg5 (queue kernel), cfg5 and cfg1 through the generic locator, a scattering square (MULTI_BOUNCE);
  host       pageable and pinned destinations, RTHX_BATCHES=3, block_threads=128, an explicit row_chunks, a shard, recorded rays;
  rows       a rows trace whose list has several irregular runs (host counts and resident), continued;
  resident   dense trace continued; hashed trace with RTHX_SPARSE_PAIR_CAP forcing row-group splits, continued;
  device     rthx_trace_exchange_device with RTHX_ZERO_ALL, and with RTHX_ZERO_OWN_ROWS on a shard;
  direct     rthx_trace_direct, _fields and _sparse (with the redirection tally), each with and without RTHX_FORCE_GLOBAL_TALLY;
  errors     shapes beyond the launch limits (row_chunks = 2^31 - 1) of a trace, a rows trace and the three direct calls.
"""
import argparse
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import rthx  # noqa: E402
from rthx._abi import RTHX_LOCATOR_GENERIC, RTHX_MULTI_BOUNCE, RTHX_MULTI_BOUNCE_SPECULAR, RTHX_ZERO_ALL, RTHX_ZERO_OWN_ROWS  # noqa: E402
from rthx._lib import pinned_empty  # noqa: E402
from rthx.direct import direct_sources  # noqa: E402

STATS = ("n_blocks", "block_threads", "row_chunks", "smem_bytes", "hist_in_smem", "n_launches", "rays_traced", "rays_lost")
SPARSE = ("pairs", "nnz", "flushes", "pair_capacity", "row_groups", "hash_slots")
KNOBS = ("RTHX_BATCHES", "RTHX_SPARSE_PAIR_CAP", "RTHX_SPARSE_HASH_SLOTS", "RTHX_FORCE_GLOBAL_TALLY", "RTHX_NO_AXIS")


def digest(x):
    a = np.ascontiguousarray(x)
    return f"{a.dtype.str}{list(a.shape)}:{hashlib.sha256(a.tobytes()).hexdigest()[:16]}"


def readouts(tr, n_bins):
    out = {}
    for k in range(n_bins):
        try:
            rp, cols, vals, fv = tr.counts_csr(k, values=True, normalised=True)
            cp, rv, cv, cf = tr.counts_csc(k, values=True, normalised=True, pinned=False)
            out[f"csr{k}"] = [digest(v) for v in (rp, cols, vals, fv)]
            out[f"csc{k}"] = [digest(v) for v in (cp, rv, cv, cf)]
        except rthx.RthxError as e:
            out[f"readout{k}"] = str(e)
    return out


class Probe:
    def __init__(self, f):
        self.f = f

    def call(self, name, fn, env=None, resident=None):
        """Run fn() with the environment knobs `env`; fn returns the output dict of a DeviceTracer call (or of trace_device).  resident:
        (tracer, n_bins) whose resident counts are read out afterwards."""
        saved = {k: os.environ.get(k) for k in KNOBS}
        for k in KNOBS:
            os.environ.pop(k, None)
        os.environ.update(env or {})
        try:
            out = fn()
            rec = {"stats": {k: out["stats"][k] for k in STATS}}
            if "sparse_stats" in out:
                rec["sparse"] = {k: out["sparse_stats"][k] for k in SPARSE}
            for k, v in sorted(out.items()):
                if isinstance(v, np.ndarray):
                    rec[k] = digest(v)
                elif k == "events":
                    rec[k] = v
            if resident is not None:
                rec.update(readouts(*resident))
        except rthx.RthxError as e:
            rec = {"error": str(e)}
        finally:
            for k, v in saved.items():
                os.environ.pop(k, None)
                if v is not None:
                    os.environ[k] = v
        line = f"{name}: {rec}"
        print(line, flush=True)
        self.f.write(line + "\n")


def host_calls(p, label, rtm, rpe, kw):
    tr = rthx.DeviceTracer(rthx.flatten_domain(rtm), device=0)
    N, nb = tr.n_elements, len(kw.get("bins", (0,)))
    base = dict(seed=11, **kw)
    p.call(f"{label}/host_pageable", lambda: tr.trace(rpe, counts_out=np.empty((nb, N, N), np.uint64), **base))
    p.call(f"{label}/host_pinned", lambda: tr.trace(rpe, counts_out=pinned_empty((nb, N, N), np.uint64), **base))
    p.call(f"{label}/host_batches3", lambda: tr.trace(rpe, counts_out=pinned_empty((nb, N, N), np.uint64), **base), env={"RTHX_BATCHES": "3"})
    p.call(f"{label}/host_block128", lambda: tr.trace(rpe, counts_out=np.empty((nb, N, N), np.uint64), block_threads=128, **base))
    p.call(f"{label}/host_row_chunks7", lambda: tr.trace(rpe, counts_out=np.empty((nb, N, N), np.uint64), row_chunks=7, **base))
    p.call(f"{label}/host_shard_1_of_3_recorded", lambda: tr.trace(rpe, emitter_rank=1, emitter_world=3, rec_ids=[1, 4, N - 2], **base))
    p.call(f"{label}/resident", lambda: tr.trace(rpe, dense=False, **base), resident=(tr, nb))
    p.call(f"{label}/resident_continue", lambda: tr.trace_continue(rpe // 2), resident=(tr, nb))
    # several irregular runs: a stride-3 run, single rows, a contiguous run and the last row
    rows = sorted(set(range(0, min(N, 13), 3)) | {N // 3, N // 3 + 5} | set(range(N // 2, N // 2 + 7)) | {N - 1})
    p.call(f"{label}/rows_host", lambda: tr.trace_rows(rows, rpe, rec_ids=[rows[1]], **base))
    p.call(f"{label}/rows_resident", lambda: tr.trace_rows(rows, rpe, dense=False, **base), resident=(tr, nb))
    p.call(f"{label}/rows_continue", lambda: tr.trace_continue(rpe // 2), resident=(tr, nb))
    p.call(f"{label}/rows_row_chunks_5", lambda: tr.trace_rows(rows, rpe, row_chunks=5, **base))
    p.call(f"{label}/error_row_chunks", lambda: tr.trace(rpe, dense=False, row_chunks=2 ** 31 - 1, **base))
    p.call(f"{label}/error_rows_row_chunks", lambda: tr.trace_rows(rows, rpe, dense=False, row_chunks=2 ** 31 - 1, **base))
    if kw.get("mode", 0) == 0:                                 # the hashed tally is FIRST_INTERACTION only
        cap = {"RTHX_SPARSE_PAIR_CAP": str(max(4 * N, 3 * rpe))}
        p.call(f"{label}/sparse_split", lambda: tr.trace_sparse(rpe, **base), env=cap, resident=(tr, nb))
        p.call(f"{label}/sparse_continue", lambda: tr.trace_continue(rpe // 2), env=cap, resident=(tr, nb))
        p.call(f"{label}/sparse_shard_recorded", lambda: tr.trace_sparse(rpe, emitter_rank=1, emitter_world=2, rec_ids=[3], **base),
               resident=(tr, nb))
    device_calls(p, label, tr, rpe, nb, base)
    tr.close()


def device_calls(p, label, tr, rpe, nb, base):
    import torch
    dev = torch.device("cuda", 0)
    N = tr.n_elements
    counts = torch.full((nb, N, N), 7, dtype=torch.int64, device=dev)
    lost = torch.full((nb, N), 7, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def run(zero, **kw):
        st = tr.trace_device(rpe, counts.data_ptr(), lost.data_ptr(), stream=stream, zero_first=zero, **base, **kw)
        torch.cuda.synchronize(dev)
        return dict(stats=st, counts=counts.cpu().numpy().view(np.uint64), lost=lost.cpu().numpy().view(np.uint64))

    p.call(f"{label}/device_zero_all", lambda: run(RTHX_ZERO_ALL))
    p.call(f"{label}/device_zero_own_rows_shard_2_of_3", lambda: run(RTHX_ZERO_OWN_ROWS, emitter_rank=2, emitter_world=3))


def direct_calls(p, label, rtm, bundles, kw):
    flat = rthx.flatten_domain(rtm)
    _, known_T, _, src, rays, w = direct_sources(rtm, bundles)
    reemit = np.zeros(flat.n_elements, np.uint8)
    reemit[:len(known_T)] = ~known_T
    tr = rthx.DeviceTracer(flat, device=0)
    for tally, env in (("", {}), ("_global_tally", {"RTHX_FORCE_GLOBAL_TALLY": "1"})):
        for call, extra, blocks in (("direct", {}, 1), ("direct_fields", dict(redirected=True), 2),
                                    ("direct_sparse", dict(redirected=True, sparse=True), 2)):
            p.call(f"{label}/{call}{tally}", lambda: tr.trace_direct(src, rays, reemit, w, seed=5, **extra, **kw), env=env, resident=(tr, blocks))
    p.call(f"{label}/direct_row_chunks_3_block128", lambda: tr.trace_direct(src, rays, reemit, w, seed=6, row_chunks=3, block_threads=128, **kw),
           resident=(tr, 1))
    for call, extra in (("direct", {}), ("direct_fields", dict(redirected=True)), ("direct_sparse", dict(redirected=True, sparse=True))):
        p.call(f"{label}/error_{call}_row_chunks", lambda: tr.trace_direct(src, rays, reemit, w, seed=5, row_chunks=2 ** 31 - 1, **extra, **kw))
    tr.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    m = rthx.meshes
    scatter = dict(kappa=0.6, sigma_s=0.9, epsilon=(0.3, 0.6, 0.9, 0.5))
    heated = m.square_domain(9, **scatter)
    heated.fine_mesh[0][8].T_in_w[1], heated.fine_mesh[0][8].q_in_w[1] = -1.0, 2.0e4     # a heated wall of known q
    with open(a.out, "w") as f:
        p = Probe(f)
        print(f"library: {os.path.basename(rthx.library_path())}", flush=True)
        host_calls(p, "cfg1", m.cfg1(), 20_000, {})
        host_calls(p, "cfg1_generic", m.cfg1(), 5_000, dict(locator=RTHX_LOCATOR_GENERIC))
        host_calls(p, "cfg5", m.cfg5(), 3_000, {})
        host_calls(p, "cfg5_generic", m.cfg5(), 1_000, dict(locator=RTHX_LOCATOR_GENERIC))
        host_calls(p, "square9_multi_bounce", m.square_domain(9, **scatter), 20_000, dict(mode=RTHX_MULTI_BOUNCE))
        host_calls(p, "cfg4_bins_2_0", m.cfg4(Ndim=13, n_bins=3), 10_000, dict(bins=[2, 0]))
        direct_calls(p, "cfg1", m.cfg1(), 400_000, {})
        direct_calls(p, "square9_specular", heated, 400_000, dict(specular=True))
        direct_calls(p, "cfg5", m.cfg5(), 400_000, {})


if __name__ == "__main__":
    main()
