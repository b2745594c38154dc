"""Round-2 rows: CSC read-out + chi on the device, rthx_create_multi / single-process multi-GPU trace (host rows and
device-0 gather), argument guards, the lazily built generic-locator tables, AP's stopping rule and the `devices` keyword."""
import warnings

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu


def _n_gpus():
    from rthx._lib import device_count
    return device_count()


def test_csc_equals_dense_and_stats(rthx_mod, cuda_lib):
    rtm = rthx_mod.meshes.cfg4(Ndim=9, n_bins=3)
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    N, ns = tr.n_elements, flat.n_surfaces
    dense = tr.trace(3000, seed=51, bins=[0, 1, 2])
    tr.trace(3000, seed=51, bins=[0, 1, 2], dense=False)
    for b in (1, 0, 2):
        c = dense["counts"][b]
        nnz, chi = tr.counts_stats(b)
        assert nnz == int((c != 0).sum())
        F = c / np.maximum(c.sum(axis=1, keepdims=True), 1)
        chi_ref = (F[:ns, ns:].sum() + F[ns:, :ns].sum()) / N               # cross_coupling_chi, smoothExchangeFactors.jl:212-241
        assert abs(chi - chi_ref) < 1e-12
        for index64, base in ((False, 0), (True, 1)):
            colptr, rowval, vals, fv = tr.counts_csc(b, values=True, normalised=True, index64=index64, index_base=base)
            assert rowval.dtype == (np.int64 if index64 else np.int32) and colptr[0] == base and colptr[-1] == nnz + base
            m = sp.csc_matrix((vals, rowval - base, colptr - base), shape=(N, N))
            assert np.array_equal(m.toarray(), c)
            for j in (0, ns, N - 1):                                          # rows ascend within a column
                seg = rowval[colptr[j] - base:colptr[j + 1] - base]
                assert np.all(np.diff(seg) > 0)
            Fm = sp.csc_matrix((fv, rowval - base, colptr - base), shape=(N, N)).toarray()
            assert np.allclose(Fm, F, rtol=0, atol=1e-15)
    # the CSR view of the same residency still agrees
    row_ptr, cols, vals, _ = tr.counts_csr(2)
    assert np.array_equal(sp.csr_matrix((vals, cols, row_ptr), shape=(N, N)).toarray(), dense["counts"][2])


def test_csc_into_pageable_arrays_over_staging(rthx_mod, cuda_lib):
    """A pageable destination larger than one staging piece (32 MB) goes through the pinned double buffer."""
    flat = rthx_mod.flatten_domain(rthx_mod.meshes.square_domain(41, kappa=0.3))
    tr = rthx_mod.DeviceTracer(flat, device=0)
    N = tr.n_elements
    ref = tr.trace(20000, seed=5)["counts"][0]
    tr.trace(20000, seed=5, dense=False)
    a = tr.counts_csc(0, values=True, index64=True, pinned=True)
    b = tr.counts_csc(0, values=True, index64=True, pinned=False)
    assert a[1].nbytes > (32 << 20) // 4                                       # big enough to matter, and ...
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    assert np.array_equal(sp.csc_matrix((b[2], b[1], b[0]), shape=(N, N)).toarray(), ref)


def test_multi_entry_point_on_one_device_and_state_reset(rthx_mod, cuda_lib):
    """rthx_create_multi + rthx_trace_exchange_multi with n = 1 (what the Julia shim calls with DEVICES = [0]), host rows and
    resident gather; a multi trace voids the resident view of an earlier single trace (ADVICE r1: stale csr state)."""
    from rthx._lib import create_multi, trace_multi, RthxError
    flat = rthx_mod.flatten_domain(rthx_mod.meshes.cfg5())
    (tr,) = create_multi(flat, [0])
    one = tr.trace(2000, seed=9)
    assert tr.counts_stats(0)[0] == int((one["counts"][0] != 0).sum())
    host = trace_multi([tr], 2000, seed=9)
    assert np.array_equal(host["counts"], one["counts"]) and np.array_equal(host["lost"], one["lost"])
    with pytest.raises(RthxError):                                              # compact rows are no N x N matrix: view is void
        tr.counts_stats(0)
    res = trace_multi([tr], 2000, seed=9, dense=False)
    assert res["counts"] is None and np.array_equal(res["lost"], one["lost"])
    colptr, rowval, vals, _ = tr.counts_csc(0, values=True)
    N = tr.n_elements
    assert np.array_equal(sp.csc_matrix((vals, rowval, colptr), shape=(N, N)).toarray(), one["counts"][0])


def test_argument_guards(rthx_mod, cuda_lib):
    from rthx._lib import RthxError
    flat = rthx_mod.flatten_domain(rthx_mod.meshes.cfg1())
    tr = rthx_mod.DeviceTracer(flat, device=0)
    with pytest.raises(RthxError, match="too many bins"):
        tr.trace(10, bins=[0] * 21)                                             # limit 4 * n_bands + 16 = 20
    assert tr.trace(10, bins=[0] * 20)["counts"].shape[0] == 20
    with pytest.raises(RthxError, match="out of range"):
        tr.trace(2 ** 33, row_chunks=1, dense=False)                            # 2^33 rays in one block: u32 counters would wrap
    with pytest.raises(RthxError, match="out of range"):
        tr.trace(10, row_chunks=2 ** 31 - 1, dense=False)                       # rows * chunks beyond the grid limit


def test_generic_tables_are_built_on_first_use(rthx_mod, oracle_mod, cuda_lib):
    """The analytic paths never build the reference-faithful locator tables; the first RTHX_LOCATOR_GENERIC trace does, and
    later analytic traces on the same handle are unaffected."""
    flat = rthx_mod.flatten_domain(rthx_mod.meshes.cfg5())
    tr = rthx_mod.DeviceTracer(flat, device=0)
    a0 = tr.trace(1500, seed=3)
    g = tr.trace(1500, seed=3, locator=1)
    a1 = tr.trace(1500, seed=3)
    ref = oracle_mod.trace(flat, 1500, seed=3)
    assert np.array_equal(a0["counts"], a1["counts"])
    nd = int(np.abs(g["counts"].astype(np.int64) - ref["counts"].astype(np.int64)).sum() // 2)
    assert nd <= 2 and abs(int(g["lost"].sum()) - int(ref["lost"].sum())) <= 2      # the exact-parity budget of the reference-faithful locator


def test_ap_stopping_rule_reports_convergence(rthx_mod, cuda_lib):
    """Device AP exits only at the target or on an accepted floor (smoothExchangeFactors.jl:578-590); running out of
    iterations is reported, and the public call warns like the reference's @warn (:605-607)."""
    rtm = rthx_mod.meshes.cfg1()
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    tr.trace(20000, seed=4, dense=False)
    w = rthx_mod.get_w(rtm)
    F, st = tr.smooth(w / w.min(), max_iters=1000)
    assert st["converged"] == 1 and st["delta"] <= 2 * 8 * np.finfo(float).eps
    F3, st3 = tr.smooth(w / w.min(), max_iters=3)
    assert st3["converged"] == 0 and st3["iterations"] == 3 and st3["delta"] > st["delta"]
    with warnings.catch_warnings(record=True) as wlist:
        warnings.simplefilter("always")
        rtm(165 * 20000, method="exchange", verbose=False, seed=4, max_iters=3)
    assert any("max_iters" in str(x.message) for x in wlist)


def test_public_call_phases_and_csc_F_raw(rthx_mod, cuda_lib):
    rtm = rthx_mod.meshes.cfg2()
    F_smooth = rtm(1845 * 3000, method="exchange", verbose=False, seed=8)
    assert sp.isspmatrix_csc(rtm.F_raw) and rtm.F_raw.has_sorted_indices
    assert np.allclose(np.asarray(rtm.F_raw.sum(axis=1)).ravel(), 1.0)
    assert set(rtm.last_phase_ms) >= {"flatten", "create", "trace", "csc_F_raw", "smoothing"}
    # same F_raw as the dense read-out + the reference's composition (parallelRayTracing.jl:144-146 + row_normalize!)
    tr = rthx_mod.DeviceTracer(rthx_mod.flatten_domain(rtm), device=0)
    c = tr.trace(3000, seed=8)["counts"][0]
    assert np.allclose(rtm.F_raw.toarray(), rthx_mod.counts_to_F(c, 3000, verbose_loss=False).toarray(), rtol=0, atol=1e-15)
    assert isinstance(F_smooth, np.ndarray) and np.allclose(F_smooth.sum(axis=1), 1.0, atol=1e-9)


@pytest.mark.skipif("_n_gpus() < 2", reason="needs two GPUs")
def test_single_process_multi_gpu_is_bit_exact(rthx_mod, cuda_lib):
    """rthx_trace_exchange_multi over every visible device: host rows, device-0 gather, recorder — all equal to one GPU."""
    from rthx._lib import create_multi, trace_multi
    n = _n_gpus()
    for mesh in (rthx_mod.meshes.cfg4(Ndim=15, n_bins=3), rthx_mod.meshes.cfg5()):
        flat = rthx_mod.flatten_domain(mesh)
        bins = list(range(flat.n_bands))
        one = rthx_mod.DeviceTracer(flat, device=0).trace(4000, seed=21, bins=bins, rec_ids=[3, 40, 41])
        trs = create_multi(flat, list(range(n)))
        N = trs[0].n_elements
        host = trace_multi(trs, 4000, seed=21, bins=bins, rec_ids=[3, 40, 41])
        assert np.array_equal(host["counts"], one["counts"]) and np.array_equal(host["lost"], one["lost"])
        assert np.array_equal(host["origins"], one["origins"]) and np.array_equal(host["endpoints"], one["endpoints"])
        pageable = np.full((len(bins), N, N), 7, np.uint64)                      # stale contents, staged copy path
        trace_multi(trs, 4000, seed=21, bins=bins, counts_out=pageable)
        assert np.array_equal(pageable, one["counts"])
        for rep in range(2):                                                     # the second pass checks the zeroing
            res = trace_multi(trs, 4000, seed=21, bins=bins, dense=False)
        assert np.array_equal(res["lost"], one["lost"])
        for b in bins:
            colptr, rowval, vals, _ = trs[0].counts_csc(b, values=True)
            assert np.array_equal(sp.csc_matrix((vals, rowval, colptr), shape=(N, N)).toarray(), one["counts"][b])
        for t in trs:
            t.close()


@pytest.mark.skipif("_n_gpus() < 2", reason="needs two GPUs")
def test_public_call_devices_keyword(rthx_mod, cuda_lib):
    n = _n_gpus()
    a = rthx_mod.meshes.cfg2()
    b = rthx_mod.meshes.cfg2()
    rec_a, rec_b = rthx_mod.RayRecorder([10, 20]), rthx_mod.RayRecorder([10, 20])
    Fa = a(1845 * 2000, method="exchange", verbose=False, seed=77, devices=[0], rec=rec_a)
    Fb = b(1845 * 2000, method="exchange", verbose=False, seed=77, devices=list(range(n)), rec=rec_b)
    assert (a.F_raw != b.F_raw).nnz == 0
    assert np.array_equal(Fa, Fb)
    oa, ea = rthx_mod.collect_rays(rec_a)
    ob, eb = rthx_mod.collect_rays(rec_b)
    assert np.array_equal(oa, ob) and np.array_equal(ea, eb)


@pytest.mark.parametrize("row_chunks", [1, 0, 5])
def test_row_handover_flush_on_one_gpu(rthx_mod, cuda_lib, monkeypatch, row_chunks):
    """The flush used for matrices in peer memory — chunks add up in a local staging row, the last chunk hands the finished row
    over with plain stores (row_chunks == 1: written out directly) — exercised on one GPU through RTHX_DEST_PEER (what a rank says
    about a CUDA-IPC mapping of rank 0's matrix), two interleaved "ranks" filling one matrix with stale contents.  Bit-identical to
    the plain trace."""
    import torch
    from rthx._abi import RTHX_ZERO_OWN_ROWS, RTHX_DEST_PEER
    flat = rthx_mod.flatten_domain(rthx_mod.meshes.cfg4(Ndim=13, n_bins=2))
    tr = rthx_mod.DeviceTracer(flat, device=0)
    N = tr.n_elements
    ref = tr.trace(30000, seed=31, bins=[1, 0])
    dev = torch.device("cuda", 0)
    counts = torch.full((2, N, N), 7, dtype=torch.int64, device=dev)
    lost = torch.full((2, N), 7, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    for rank in (1, 0):
        st = tr.trace_device(30000, counts.data_ptr(), lost.data_ptr(), stream=stream, zero_first=RTHX_ZERO_OWN_ROWS | RTHX_DEST_PEER, seed=31, bins=[1, 0],
                             emitter_rank=rank, emitter_world=2, row_chunks=row_chunks)
    torch.cuda.synchronize(dev)
    if row_chunks:
        assert st["row_chunks"] == row_chunks
    assert np.array_equal(counts.cpu().numpy().view(np.uint64), ref["counts"])
    assert np.array_equal(lost.cpu().numpy().view(np.uint64), ref["lost"])


def test_row_tiles_equal_the_untiled_trace(rthx_mod, cuda_lib):
    """trace_row_tiles: the emitter rows traced in interleaved tiles, each read out as CSR from the device and merged — the same
    F_raw as one trace (bit-identical counts), for a multi-band launch."""
    from rthx._lib import trace_row_tiles
    flat = rthx_mod.flatten_domain(rthx_mod.meshes.cfg4(Ndim=9, n_bins=3))
    tr = rthx_mod.DeviceTracer(flat, device=0)
    N = tr.n_elements
    ref = tr.trace(4000, seed=71, bins=[2, 0])
    tiled = trace_row_tiles(tr, 4000, 5, seed=71, bins=[2, 0])
    assert np.array_equal(tiled["lost"], ref["lost"])
    for k in range(2):
        row_ptr, cols, vals = tiled["csr"][k]
        F = sp.csr_matrix((vals, cols, row_ptr), shape=(N, N)).toarray()
        c = ref["counts"][k].astype(np.float64)
        assert np.allclose(F, c / np.maximum(c.sum(axis=1, keepdims=True), 1), rtol=0, atol=1e-15)
        tr.trace(4000, seed=71, bins=[2, 0], dense=False)
        assert abs(tiled["chi"][k] - tr.counts_stats(k)[1]) < 1e-12


def test_public_call_beyond_the_shared_memory_histogram_in_row_tiles(rthx_mod, cuda_lib):
    """N = 68 640 elements (260 x 260): the row histogram no longer fits in shared memory (global tally path) and the dense
    matrix would be 37.7 GB; the public call traces it in row tiles and returns a sparse F_raw whose rows sum to one."""
    rtm = rthx_mod.meshes.square_domain(260, kappa=40.0)
    N = rtm.num_elements
    assert N == 4 * 260 + 260 * 260
    rtm(N * 64, method="exchange", verbose=False, seed=5, smooth=False, row_tiles=4)
    F = rtm.F_raw
    assert sp.issparse(F) and F.shape == (N, N) and F.nnz < 64 * N
    assert np.allclose(np.asarray(F.sum(axis=1)).ravel(), 1.0)
    assert rtm.last_trace_stats["hist_in_smem"] == 0 and rtm.last_phase_ms["row_tiles"] == 4


def test_step_flags_signal_wait_and_timeout(rthx_mod, cuda_lib):
    """rthx_flag_signal / rthx_flag_wait: a wait behind its signal passes, a wait for a value nobody writes gives up after its
    timeout and raises the error counter instead of hanging the device."""
    import ctypes as C
    import torch
    dev = torch.device("cuda", 0)
    flags = torch.zeros(8, dtype=torch.int64, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    base = flags.data_ptr()
    assert cuda_lib.rthx_flag_signal(C.c_void_p(base), 5, C.c_void_p(st)) == 0
    assert cuda_lib.rthx_flag_signal(C.c_void_p(base + 8), 7, C.c_void_p(st)) == 0
    assert cuda_lib.rthx_flag_wait(C.c_void_p(base), 2, 5, 1.0, C.c_void_p(base + 56), C.c_void_p(st)) == 0
    torch.cuda.synchronize(dev)
    assert flags.tolist()[:2] == [5, 7] and flags[7].item() == 0
    assert cuda_lib.rthx_flag_wait(C.c_void_p(base), 2, 6, 0.05, C.c_void_p(base + 56), C.c_void_p(st)) == 0   # flags[0] = 5 < 6: times out
    torch.cuda.synchronize(dev)
    assert flags[7].item() == 1


def test_device_count_and_pinned_arrays(rthx_mod, cuda_lib):
    from rthx._lib import device_count, pinned_empty, release_pinned
    import torch
    assert device_count() == torch.cuda.device_count() >= 1
    a = pinned_empty((1000, 300), np.float64)
    a[:] = 3.0
    assert a.shape == (1000, 300) and a.flags["C_CONTIGUOUS"] and float(a.sum()) == 9e5
    addr = a.ctypes.data
    del a
    b = pinned_empty(1000 * 300, np.float64)              # the freed buffer comes back from the pool
    assert b.ctypes.data == addr
    del b
    release_pinned()


@pytest.mark.skipif("_n_gpus() < 2", reason="needs two GPUs")
def test_multi_link_result_copies_equal_single_link(rthx_mod, cuda_lib):
    """rthx_set_copy_helpers: the CSC arrays and F_smooth (> 64 MB each here) leave device 0 in slices over every device's PCIe link
    (NVLink hop + that device's D2H); bit-identical to the single-link copies, flat arrays and pitched rows alike."""
    from rthx._lib import create_multi, trace_multi
    n = _n_gpus()
    rtm = rthx_mod.meshes.square_domain(75, kappa=0.3)
    flat = rthx_mod.flatten_domain(rtm)
    trs = create_multi(flat, list(range(n)))
    tr = trs[0]
    N = tr.n_elements
    trace_multi(trs, 40000, dense=False, seed=3)
    w = rthx_mod.get_w(rtm)
    a = tr.counts_csc(0, values=True, index64=True)
    Fa, _ = tr.smooth(w / w.min(), max_iters=40)
    assert a[1].nbytes >= (64 << 20) and Fa.nbytes >= (64 << 20)
    tr.set_copy_helpers(trs[1:])
    b = tr.counts_csc(0, values=True, index64=True)
    Fb, _ = tr.smooth(w / w.min(), max_iters=40)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    assert np.array_equal(Fa, Fb)
    tr.set_copy_helpers([])
    for t in trs:
        t.close()


@pytest.mark.parametrize("mesh", ["cfg5", "two_quads", "circle_small"])
def test_generic_locator_on_the_ray_queue_equals_lock_step(rthx_mod, oracle_mod, cuda_lib, monkeypatch, mesh):
    """Multi-face meshes under RTHX_LOCATOR_GENERIC run in the queue kernel's generic variant (bucket grid + crossing number at
    every crossing, per-step cell lookup for cell-wise beta, wall lookup from the polygon record).  Same integers as the lock-step
    generic kernel (RTHX_NO_QUEUE_GENERIC=1), as its 80-register build, as a coarser bucket grid, and — within the exact-parity
    budget of the reference-faithful locator — as the CPU oracle."""
    m = rthx_mod.meshes
    rtm = {"cfg5": m.cfg5, "two_quads": lambda: m.two_quads_domain(skew=0.25),           # cell-wise beta, a bilinear face
           "circle_small": lambda: m.circle_domain(N_seg=7, Ndim=4)}[mesh]()
    flat = rthx_mod.flatten_domain(rtm)
    rpe = 3000
    out = {}
    for tag, env in (("queue", {}), ("lockstep", {"RTHX_NO_QUEUE_GENERIC": "1"}), ("queue80", {"RTHX_GENERIC_MINB": "3"}),
                     ("coarse_grid", {"RTHX_GRID_FINE": "2"})):
        for k in ("RTHX_NO_QUEUE_GENERIC", "RTHX_GENERIC_MINB", "RTHX_GRID_FINE"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        tr = rthx_mod.DeviceTracer(flat, device=0)       # (the grid knob is read when the tables are built)
        out[tag] = tr.trace(rpe, seed=17, locator=1, rec_ids=[1, 3])
        tr.close()
    ref = oracle_mod.trace(flat, rpe, seed=17, rec_ids=[1, 3])
    total = rpe * flat.n_elements
    for tag in ("lockstep", "queue80", "coarse_grid"):
        # the same locator arithmetic on every path: identical integers except for points within rounding of a bucket-grid decision
        nd = int(np.abs(out["queue"]["counts"].astype(np.int64) - out[tag]["counts"].astype(np.int64)).sum() // 2)
        assert nd <= max(2, total // 500_000), (tag, nd)
    assert out["queue"]["counts"].sum() + out["queue"]["lost"].sum() == total
    nd = int(np.abs(out["queue"]["counts"].astype(np.int64) - ref["counts"].astype(np.int64)).sum() // 2)
    assert nd <= max(2, total // 500_000), nd
    assert abs(int(out["queue"]["lost"].sum()) - int(ref["lost"].sum())) <= 2
    assert np.allclose(out["queue"]["origins"], ref["origins"], atol=1e-12)


def test_generic_tables_come_from_the_process_cache(rthx_mod, cuda_lib):
    """The generic tables of a mesh are built once per process: a second handle on the same geometry (callers re-create handles
    for every trace) and a handle created after rthx_release_cached() give the same integers as the first; another mesh of the
    same size does not hit the first one's entry."""
    from rthx import _lib
    m = rthx_mod.meshes
    flat = rthx_mod.flatten_domain(m.two_quads_domain(skew=0.25))
    other = rthx_mod.flatten_domain(m.two_quads_domain(skew=0.15))       # same topology and sizes, different vertices
    outs = []
    for i in range(2):
        tr = rthx_mod.DeviceTracer(flat, device=0)
        outs.append(tr.trace(2000, seed=9, locator=1))
        tr.close()
    tr = rthx_mod.DeviceTracer(other, device=0)
    o_other = tr.trace(2000, seed=9, locator=1)
    tr.close()
    _lib.load_library().rthx_release_cached()
    tr = rthx_mod.DeviceTracer(flat, device=0)
    outs.append(tr.trace(2000, seed=9, locator=1))
    a_other = tr.trace(2000, seed=9)            # analytic locator on the same handle
    tr.close()
    assert np.array_equal(outs[0]["counts"], outs[1]["counts"]) and np.array_equal(outs[0]["counts"], outs[2]["counts"])
    assert not np.array_equal(outs[0]["counts"], o_other["counts"])
    tr = rthx_mod.DeviceTracer(other, device=0)
    a = tr.trace(2000, seed=9)
    tr.close()
    nd = int(np.abs(a["counts"].astype(np.int64) - o_other["counts"].astype(np.int64)).sum() // 2)
    assert nd <= 2, nd                          # the other mesh was located with ITS tables (generic == analytic within the budget)
    assert a_other["counts"].sum() > 0
