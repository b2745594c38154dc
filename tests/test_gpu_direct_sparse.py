"""method=:direct on the hashed row tally (rthx_trace_direct_sparse, DeviceTracer.trace_direct(sparse=True), the route directRayTracing
takes when the dense counts do not fit): bit-identity with the dense route in every result and read-out, also with forced small tables
and pair buffers and for any launch shape; the public call on both routes; the isothermal enclosure at N = 161 600, where the dense
counts would need 209 GB; and the rejections."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_direct import _cases, _reemit

pytestmark = pytest.mark.gpu

NAMES = ["cfg1", "square9_diffuse", "square9_specular", "circle", "two_quads_variable_beta", "square9_generic"]


def _setup(rthx_mod, case, rays_tot=120_000):
    from rthx.direct import direct_sources
    name, rtm, kw, _ = _cases()[case]
    flat = rthx_mod.flatten_domain(rtm)
    ws, known_T, E, src, rays, w = direct_sources(rtm, rays_tot)
    return flat, src, rays, _reemit(rtm, flat, known_T), w, kw


def _readouts(tr, n_bins):
    """Every read-out of the resident counts: CSR, nnz and chi, CSC with both index widths and bases, per bin."""
    out = []
    for b in range(n_bins):
        out.append(tr.counts_csr(bin=b, values=True, normalised=True))
        out.append(tr.counts_stats(b))
        for i64 in (False, True):
            for base in (0, 1):
                out.append(tr.counts_csc(bin=b, values=True, normalised=True, index64=i64, index_base=base, pinned=False))
    return out


def _same(a, b, what=""):
    if isinstance(a, (tuple, list)):
        assert len(a) == len(b), what
        for i, (x, y) in enumerate(zip(a, b)):
            _same(x, y, f"{what}[{i}]")
    elif isinstance(a, np.ndarray):
        assert a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8)), what
    elif isinstance(a, float):
        assert np.float64(a).tobytes() == np.float64(b).tobytes(), (what, a, b)
    else:
        assert a == b, (what, a, b)


def _trace(tr, src, rays, reemit, w, redirected, sparse, **kw):
    out = tr.trace_direct(src, rays, reemit, w, redirected=redirected, sparse=sparse, **kw)
    res = dict(absorbed=out["absorbed"], lost=out["lost"], events=out["events"], readouts=_readouts(tr, 2 if redirected else 1))
    if redirected:
        res["redirected"] = out["redirected"]
    return res, out


def _assert_same(got, ref, what):
    assert got.keys() == ref.keys()
    for k in ref:
        _same(got[k], ref[k], f"{what}: {k}")


@pytest.mark.parametrize("redirected", [False, True], ids=["plain", "redirected"])
@pytest.mark.parametrize("case", range(6), ids=NAMES)
def test_hashed_route_is_the_dense_route_bit_for_bit(rthx_mod, cuda_lib, case, redirected):
    flat, src, rays, reemit, w, kw = _setup(rthx_mod, case)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    ref, _ = _trace(tr, src, rays, reemit, w, redirected, False, seed=21, **kw)
    got, out = _trace(tr, src, rays, reemit, w, redirected, True, seed=21, **kw)
    _assert_same(got, ref, NAMES[case])
    assert out["sparse_stats"]["row_groups"] >= 1 and out["sparse_stats"]["nnz"] > 0
    assert out["stats"]["rays_traced"] == rays.sum()


def test_a_table_smaller_than_a_row_spills_and_keeps_the_totals(rthx_mod, cuda_lib, monkeypatch):
    """64 slots against source rows of up to 2 N = 330 distinct keys: tallies that find no slot are appended as pairs of their own."""
    flat, src, rays, reemit, w, kw = _setup(rthx_mod, 0)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    ref, _ = _trace(tr, src, rays, reemit, w, True, False, seed=5)
    monkeypatch.setenv("RTHX_SPARSE_HASH_SLOTS", "64")
    got, out = _trace(tr, src, rays, reemit, w, True, True, seed=5)
    _assert_same(got, ref, "64 slots")
    sst = out["sparse_stats"]
    assert sst["hash_slots"] == 64
    assert sst["pairs"] > sst["flushes"] * 64                     # more pairs than the flushed tables could hold: the insert spilled


def test_a_small_pair_buffer_splits_the_rows_and_counts_each_bundle_once(rthx_mod, cuda_lib, monkeypatch):
    flat, src, rays, reemit, w, kw = _setup(rthx_mod, 1)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    ref, _ = _trace(tr, src, rays, reemit, w, True, False, seed=8)
    # one block per source row (row_chunks = 1) holds at most 2 N keys, so a buffer of 2 N + 64 pairs takes every row on its own
    cap = 2 * flat.n_elements + 64
    _, free = _trace(tr, src, rays, reemit, w, True, True, seed=8, row_chunks=1)
    assert free["sparse_stats"]["pairs"] > 3 * cap
    monkeypatch.setenv("RTHX_SPARSE_PAIR_CAP", str(cap))
    got, out = _trace(tr, src, rays, reemit, w, True, True, seed=8, row_chunks=1)
    _assert_same(got, ref, "small pair buffer")
    assert out["sparse_stats"]["row_groups"] >= 4 and out["sparse_stats"]["pair_capacity"] == cap


@pytest.mark.parametrize("block_threads,row_chunks", [(256, 0), (128, 0), (256, 1), (128, 1)])
def test_results_do_not_depend_on_the_launch_shape(rthx_mod, cuda_lib, block_threads, row_chunks):
    flat, src, rays, reemit, w, kw = _setup(rthx_mod, 1)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    ref, _ = _trace(tr, src, rays, reemit, w, True, False, seed=9)
    got, _ = _trace(tr, src, rays, reemit, w, True, True, seed=9, block_threads=block_threads, row_chunks=row_chunks)
    _assert_same(got, ref, f"{block_threads} threads, row_chunks {row_chunks}")


def _fields(rtm):
    cells = rtm.fine_mesh[0]
    gas = np.array([(c.T_g, c.e_g, c.g_a_g, c.q_g, c.j_g, c.r_g, c.g_g, c.i_g) for c in cells])
    wall = np.array([(c.T_w[w], c.e_w[w], c.g_a_w[w], c.q_w[w], c.j_w[w], c.r_w[w], c.g_w[w], c.i_w[w])
                     for (cc, f, w1), s in sorted(rtm.surface_mapping.items(), key=lambda t: t[1])
                     for c in [rtm.fine_mesh[cc - 1][f - 1]] for w in [w1 - 1]])
    return gas, wall, rtm.energy_error


def _square9(rthx_mod):
    rtm = rthx_mod.meshes.square_domain(9, kappa=0.6, sigma_s=0.9, epsilon=(0.3, 0.6, 0.9, 0.5))
    rtm.fine_mesh[0][8].T_in_w[1], rtm.fine_mesh[0][8].q_in_w[1] = -1.0, 2.0e4
    return rtm


def test_public_call_writes_the_same_fields_on_either_route(rthx_mod, cuda_lib, monkeypatch):
    out = []
    for hashed in (False, True):
        if hashed:
            monkeypatch.setattr(rthx_mod.tracing, "rows_fit_one_device", lambda r, n, b, budget_bytes=48e9: False)
        rtm = _square9(rthx_mod)
        rtm(2_000_000, method="direct", verbose=False, seed=17, all_fields=True)
        assert rtm.last_direct_stats["tally"] == ("sparse" if hashed else "dense")
        out.append((_fields(rtm), rtm.last_direct_stats))
    _same(out[1][0], out[0][0], "fields")
    for k in ("events", "lost", "lost_energy", "redirections"):
        assert out[1][1][k] == out[0][1][k], k


def test_two_devices_on_the_hashed_route_give_the_one_device_fields(rthx_mod, cuda_lib, monkeypatch):
    if rthx_mod._lib.device_count() < 2:
        pytest.skip("needs two GPUs")
    monkeypatch.setattr(rthx_mod.tracing, "rows_fit_one_device", lambda r, n, b, budget_bytes=48e9: False)
    out = []
    for devs in ([0], [0, 1]):
        rtm = _square9(rthx_mod)
        rtm(2_000_000, method="direct", verbose=False, seed=17, devices=devs, all_fields=True)
        assert rtm.last_direct_stats["devices"] == len(devs) and rtm.last_direct_stats["tally"] == "sparse"
        out.append(_fields(rtm))
    _same(out[1], out[0], "fields")


def test_isothermal_enclosure_where_the_dense_counts_do_not_fit(rthx_mod, cuda_lib, record_property):
    """square_domain(400, kappa = 40): black walls and every gas cell at 1000 K, so every element is a source (R = N = 161 600) and the
    dense counts would take 8 R N = 209 GB.  The hashed route traces ~1.6e8 bundles on one device; an isothermal black enclosure is in
    equilibrium, so the walls absorb what they emit."""
    import threading
    import time
    import torch
    rtm = rthx_mod.meshes.square_domain(400, kappa=40.0, T_walls=(1000.0,) * 4)
    for c in rtm.fine_mesh[0]:
        c.T_in_g = 1000.0
    cuda_lib.rthx_release_cached()                                # buffers parked by earlier handles are not this call's
    free0 = low = torch.cuda.mem_get_info(0)[0]
    done = False

    def poll():                                                   # the lowest free memory while the call runs
        nonlocal low
        while not done:
            low = min(low, torch.cuda.mem_get_info(0)[0])
            time.sleep(0.001)
    t = threading.Thread(target=poll)
    t.start()
    try:
        rtm(160_000_000, method="direct", verbose=False, seed=6, device=0)
    finally:
        done = True
        t.join()
    st = rtm.last_direct_stats
    held = free0 - min(low, torch.cuda.mem_get_info(0)[0])
    record_property("device_bytes_held", int(held))
    print(f"isothermal 400 x 400: {st}, device memory held by the call at its peak {held / 1e9:.1f} GB")
    assert st["tally"] == "sparse" and st["sources"] == 161_600
    assert not rthx_mod.tracing.rows_fit_one_device(st["sources"], 161_600, 1)
    cells = [rtm.fine_mesh[c - 1][f - 1] for (c, f, w) in rtm.surface_mapping]
    E = sum(rtm.fine_mesh[c - 1][f - 1].e_w[w - 1] for (c, f, w) in rtm.surface_mapping)
    q = sum(rtm.fine_mesh[c - 1][f - 1].q_w[w - 1] for (c, f, w) in rtm.surface_mapping)
    assert len(cells) == 1600
    assert rtm.energy_error == pytest.approx(st["lost_energy"], rel=1e-9, abs=1e-9 * E)
    assert abs(q) <= 0.01 * E


def test_rejections(rthx_mod, cuda_lib, monkeypatch):
    from rthx import RthxError
    rtm = _square9(rthx_mod)
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    N = flat.n_elements
    tr.trace_rows([0, 1, 2], 5000, dense=False, seed=1)
    before = tr.counts_csr()
    src, rays, re_, w = np.array([0, 4]), np.array([100, 100]), np.zeros(N, np.uint8), np.ones(2)
    bad = [(dict(sources=[4, 0]), "strictly ascending"), (dict(sources=[0, N]), "outside"), (dict(rays=[100, 0]), r"rays\[1\] = 0"),
           (dict(w=[1.0, -1.0]), r"bundle_energy\[1\]"), (dict(bins=(0, 0)), "one bin"), (dict(rec_ids=[0]), "recording"),
           (dict(emitter_world=2), "emitter_rank")]
    for change, msg in bad:
        a = dict(sources=src, rays=rays, w=w)
        kw = {k: v for k, v in change.items() if k not in a}
        a.update({k: v for k, v in change.items() if k in a})
        with pytest.raises(RthxError, match=msg):
            tr.trace_direct(a["sources"], a["rays"], re_, a["w"], sparse=True, **kw)
    args, keep = rthx_mod.make_trace_args(0, mode=0)                    # FIRST_INTERACTION through the C ABI
    s32, r64 = np.ascontiguousarray(src, np.int32), np.ascontiguousarray(rays, np.int64)
    out = np.empty(N)
    rc = cuda_lib.rthx_trace_direct_sparse(tr._h, C.byref(args), s32.ctypes.data_as(C.POINTER(C.c_int32)), r64.ctypes.data_as(C.POINTER(C.c_int64)),
                                           2, re_.ctypes.data_as(C.POINTER(C.c_uint8)), w.ctypes.data_as(C.POINTER(C.c_double)),
                                           out.ctypes.data_as(C.POINTER(C.c_double)), None, None, None, None, None)
    assert rc == 1 and "MULTI_BOUNCE" in cuda_lib.rthx_last_error(tr._h).decode()
    assert cuda_lib.rthx_trace_direct_sparse(None, None, None, None, 0, None, None, None, None, None, None, None, None) == 1
    _same(tr.counts_csr(), before, "resident rows after the rejections")
    # one source row that overruns the pair buffer alone: RTHX_ERR_NOMEM naming it, nothing resident — as the exchange route leaves it
    monkeypatch.setenv("RTHX_SPARSE_PAIR_CAP", "1")
    with pytest.raises(RthxError, match=r"\(-?\d+\).*source row 0 \(element 0\) exceed the pair buffer"):
        tr.trace_direct([0, 4], [5000, 5000], re_, w, sparse=True, seed=2)
    with pytest.raises(RthxError, match="no resident counts"):
        tr.counts_csr()
    with pytest.raises(RthxError, match="exceed the pair buffer"):
        tr.trace_sparse(1000, seed=2)
    with pytest.raises(RthxError, match="no resident counts"):
        tr.counts_csr()


def test_continue_and_smoothing_refuse_hashed_direct_counts(rthx_mod, cuda_lib):
    from rthx import RthxError
    flat = rthx_mod.flatten_domain(_square9(rthx_mod))
    tr = rthx_mod.DeviceTracer(flat, device=0)
    N = flat.n_elements
    src = np.arange(N, dtype=np.int32)
    tr.trace_direct(src, np.full(N, 200), np.ones(N, np.uint8), np.ones(N), sparse=True, seed=5)
    assert tr.counts_csr()[0].shape == (N + 1,)
    with pytest.raises(RthxError, match="direct trace"):
        tr.trace_continue(100, seed=5, mode=1)
    with pytest.raises(RthxError, match="direct trace"):
        tr.smooth(np.ones(N), n=N)
    with pytest.raises(RthxError, match="direct trace"):
        tr.smooth_sparse(np.ones(N), n=N)
