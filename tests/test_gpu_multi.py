"""Two-process / two-GPU tests of the sharded paths (needs two or more B200s; skipped with one).
Fused peer-memory flush over NVLink vs NCCL reduce vs a single-GPU trace: all bit-identical."""
import os
import socket
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import rthx
    from rthx.dist import ShardedTracer
    flat = rthx.flatten_domain(rthx.meshes.cfg4(Ndim=15, n_bins=3))
    bins = [0, 1, 2]
    for mode in ("fused", "nccl"):
        sh = ShardedTracer(flat, device=rank, rank=rank, world=world, n_bins=3, mode=mode)
        for rep in range(2):                                   # second pass checks the own-row zeroing
            sh.trace(4000, seed=21, bins=bins)
        torch.cuda.synchronize()
        if rank == 0:
            np.save(os.path.join(out_dir, f"{mode}_counts.npy"), sh.counts.cpu().numpy().view(np.uint64))
            np.save(os.path.join(out_dir, f"{mode}_lost.npy"), sh.lost.cpu().numpy().view(np.uint64))
        sh.close()
    # host-output sharding: every rank copies its own rows into one page-locked matrix in POSIX shared memory
    from rthx._lib import SharedHostMatrix
    N = flat.n_elements
    name = f"rthx_test_{port}"
    m = SharedHostMatrix(name, (3, N, N), create=True) if rank == 0 else None
    dist.barrier()
    if rank != 0:
        m = SharedHostMatrix(name, (3, N, N), create=False)
    if rank == 0:
        m.array[:] = 7                                            # stale contents must be overwritten row by row
    dist.barrier()
    tr = rthx.DeviceTracer(flat, device=rank)
    tr.trace(4000, counts_out=m.array, seed=21, bins=bins, emitter_rank=rank, emitter_world=world)
    dist.barrier()
    if rank == 0:
        np.save(os.path.join(out_dir, "hostshared_counts.npy"), np.array(m.array))
    dist.barrier()
    m.close()
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_fused_peer_flush_equals_nccl_reduce_equals_single_gpu(tmp_path, rthx_mod, cuda_lib):
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    flat = rthx_mod.flatten_domain(rthx_mod.meshes.cfg4(Ndim=15, n_bins=3))
    one = rthx_mod.DeviceTracer(flat, device=0).trace(4000, seed=21, bins=[0, 1, 2])
    for mode in ("fused", "nccl"):
        c = np.load(tmp_path / f"{mode}_counts.npy")
        l = np.load(tmp_path / f"{mode}_lost.npy")
        assert np.array_equal(c, one["counts"]), mode
        assert np.array_equal(l, one["lost"]), mode
    assert np.array_equal(np.load(tmp_path / "hostshared_counts.npy"), one["counts"])
