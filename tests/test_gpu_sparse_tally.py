"""The hashed row tally (rthx_trace_exchange_sparse, DeviceTracer.trace_sparse): a trace whose counts never exist in dense form.
Every read-out of the resident counts after it must equal, bit for bit, the same read-out after the dense trace of the same
arguments — also when the blocks flush their hash tables many times and the pair buffer overflows into many row groups."""
import ctypes as C
import re
import shutil
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

from rthx._abi import RTHX_LOCATOR_GENERIC, RTHX_MULTI_BOUNCE

# measured on the shipped build (cuobjdump --dump-resource-usage): 72 / 104 registers, no stack frame (no spills)
HASH_BOUNDS = {"trace_exchange_hash_kernel<true>": (72, 0), "trace_exchange_hash_kernel<false>": (104, 0)}


def _trapezoid(kappa_cells=True):
    from rthx import PolyVolume2D, RayTracingDomain2D
    face = PolyVolume2D([(0.0, 0.0), (2.0, 0.0), (1.5, 1.0), (0.5, 1.0)], (True, True, True, True), 1, 0.8, 0.0)
    face.epsilon = [1.0] * 4
    face.T_in_w = [1000.0, 0.0, 0.0, 0.0]
    face.T_in_g = -1.0
    face.q_in_g = 0.0
    rtm = RayTracingDomain2D([face], [(7, 5)])
    if kappa_cells:
        for i, cell in enumerate(rtm.fine_mesh[0]):
            cell.kappa_g = 0.3 + 0.1 * (i % 9)
        rtm.refresh_spectral_flags()
    return rtm


def _case(rthx_mod, name):
    m = rthx_mod.meshes
    return {
        "cfg1": (m.cfg1(), dict(rec_ids=[0, 9, 29])),
        "cfg4_bins_2_0": (m.cfg4(Ndim=9, n_bins=3), dict(bins=[2, 0])),
        "circle": (m.circle_domain(N_seg=16, Ndim=5), {}),
        "two_quads_variable_beta": (m.two_quads_domain(kappa=(0.5, 3.0)), dict(rec_ids=[1, 20])),
        "trapezoid": (_trapezoid(), {}),
        "generic_locator": (m.cfg1(), dict(locator=RTHX_LOCATOR_GENERIC)),
        "sharded": (m.square_domain(15, kappa=1.0), dict(emitter_rank=1, emitter_world=3)),
        "ray_id_offset": (m.cfg1(), dict(ray_id_offset=(1 << 33) + 12345)),
    }[name]


CASES = ["cfg1", "cfg4_bins_2_0", "circle", "two_quads_variable_beta", "trapezoid", "generic_locator", "sharded", "ray_id_offset"]


def _readout(tr, n_bins, sharded):
    """Every read-out of the resident counts, per traced bin."""
    out = []
    for k in range(n_bins):
        nnz, chi = tr.counts_stats(k)
        rp, cols, vals, fv = tr.counts_csr(k, values=True, normalised=True)
        r = dict(nnz=nnz, chi=chi, csr=(rp.copy(), cols.copy(), vals.copy(), fv.copy()))
        if not sharded:
            cp, rv, cv, cf = tr.counts_csc(k, values=True, normalised=True, pinned=False)
            cp1, rv1, _, _ = tr.counts_csc(k, values=False, normalised=False, index64=True, index_base=1, pinned=False)
            r["csc"] = (cp.copy(), rv.copy(), cv.copy(), cf.copy(), cp1.copy(), rv1.copy())
        out.append(r)
    return out


def _assert_same(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x["nnz"] == y["nnz"]
        assert abs(x["chi"] - y["chi"]) <= 1e-12
        for u, v in zip(x["csr"], y["csr"]):
            assert u.dtype == v.dtype and np.array_equal(u, v)
        assert ("csc" in x) == ("csc" in y)
        for u, v in zip(x.get("csc", ()), y.get("csc", ())):
            assert u.dtype == v.dtype and np.array_equal(u, v)


def _dense_and_sparse(rthx_mod, monkeypatch, name, rpe=2000, seed=91):
    rtm, kw = _case(rthx_mod, name)
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    nb = len(kw.get("bins", (0,)))
    sharded = kw.get("emitter_world", 1) > 1
    d = tr.trace(rpe, seed=seed, dense=False, **kw)
    rd = _readout(tr, nb, sharded)
    s = tr.trace_sparse(rpe, seed=seed, **kw)
    rs = _readout(tr, nb, sharded)
    assert np.array_equal(d["lost"], s["lost"])
    assert d["stats"]["rays_traced"] == s["stats"]["rays_traced"] and d["stats"]["rays_lost"] == s["stats"]["rays_lost"]
    _assert_same(rd, rs)
    assert s["sparse_stats"]["nnz"] == sum(r["nnz"] for r in rs)
    if "rec_ids" in kw:
        # The hashed tally runs the ray loop of the global-atomic kernel: its recorder points are those of that kernel bit for bit.
        # The default dense kernels of these meshes (single-quad, ray-queue) reach the same tallies with differently rounded
        # intermediate positions.
        monkeypatch.setenv("RTHX_FORCE_GLOBAL_TALLY", "1")
        g = tr.trace(rpe, seed=seed, dense=False, **kw)
        monkeypatch.delenv("RTHX_FORCE_GLOBAL_TALLY")
        assert len(s["origins"]) > 0 and s["origins"].shape == d["origins"].shape
        assert np.array_equal(g["origins"], s["origins"]) and np.array_equal(g["endpoints"], s["endpoints"])
        assert np.allclose(d["origins"], s["origins"], rtol=0, atol=1e-12) and np.allclose(d["endpoints"], s["endpoints"], rtol=0, atol=1e-9)
    return d, s, rs


# ---- CPU ------------------------------------------------------------------------------------------------------------------

def test_symbol_exported_and_fails_without_a_device(cuda_lib, rthx_mod):
    import torch
    assert cuda_lib.rthx_trace_exchange_sparse is not None
    assert cuda_lib.rthx_trace_exchange_sparse(None, None, None, None, None, None) == 1       # RTHX_ERR_ARG: no handle
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    flat = rthx_mod.flatten_domain(rthx_mod.meshes.square_domain(3))
    h = C.c_void_p()
    assert cuda_lib.rthx_create(C.byref(h), C.byref(flat.c), 0) == 2                        # RTHX_ERR_CUDA: no handle, no trace
    with pytest.raises(rthx_mod.RthxError, match="no CUDA device|CPU fallback"):
        rthx_mod.DeviceTracer(flat, device=0).trace_sparse(10)


@pytest.mark.skipif(shutil.which("cuobjdump") is None or shutil.which("c++filt") is None, reason="needs cuobjdump and c++filt")
def test_hash_kernels_keep_their_registers_and_stack_frames(cuda_lib, rthx_mod):
    so = rthx_mod.build_library()
    out = subprocess.run(["cuobjdump", "--dump-resource-usage", so], capture_output=True, text=True, check=True).stdout
    names = re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", out)
    dem = subprocess.run(["c++filt"], input="\n".join(n for n, _, _ in names), capture_output=True, text=True, check=True).stdout.splitlines()
    usage = {d: (int(r), int(s)) for d, (_, r, s) in zip(dem, names)}
    for prefix, (regs, stack) in HASH_BOUNDS.items():
        hits = [(k, v) for k, v in usage.items() if k.startswith("void rthx::" + prefix)]
        assert len(hits) == 1, (prefix, [k for k, _ in hits])
        name, (r, s) = hits[0]
        assert r <= regs, f"{name}: {r} registers (bound {regs})"
        assert s <= stack, f"{name}: stack frame {s} bytes (bound {stack}): ptxas spills"


# ---- GPU: exact comparisons against the dense trace -------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_matches_the_dense_trace(rthx_mod, cuda_lib, monkeypatch, name):
    _, s, _ = _dense_and_sparse(rthx_mod, monkeypatch, name)
    assert s["sparse_stats"]["row_groups"] == 1


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_matches_the_dense_trace_with_forced_flushes_and_row_groups(rthx_mod, cuda_lib, monkeypatch, name):
    monkeypatch.setenv("RTHX_SPARSE_HASH_SLOTS", "512")     # 256 threads: the table is flushed before every round that follows an insert
    monkeypatch.setenv("RTHX_SPARSE_PAIR_CAP", "9000")      # one emitter row (<= 2 bins x 2000 rays) fits, the whole mesh does not
    _, s, _ = _dense_and_sparse(rthx_mod, monkeypatch, name)
    ss = s["sparse_stats"]
    assert ss["hash_slots"] == 512 and ss["pair_capacity"] == 9000
    assert ss["row_groups"] >= 2, ss
    assert ss["flushes"] >= 4 * s["stats"]["n_blocks"], ss   # 2000 rays a block: 8 rounds, each flushing
    assert ss["pairs"] > ss["nnz"]


@pytest.mark.gpu
def test_row_too_large_for_the_pair_buffer_is_an_error(rthx_mod, cuda_lib, monkeypatch):
    monkeypatch.setenv("RTHX_SPARSE_PAIR_CAP", "4")
    tr = rthx_mod.DeviceTracer(rthx_mod.flatten_domain(rthx_mod.meshes.cfg1()), device=0)
    with pytest.raises(rthx_mod.RthxError, match=r"\(3\).*pair buffer"):
        tr.trace_sparse(2000, seed=3)
    with pytest.raises(rthx_mod.RthxError, match="no resident counts"):
        tr.counts_stats(0)                                  # nothing half-finished is left resident


@pytest.mark.gpu
def test_sparse_smoothing_from_the_sparse_form(rthx_mod, cuda_lib):
    rtm = rthx_mod.meshes.square_domain(15, kappa=40.0)
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    ns = flat.n_surfaces
    w = rthx_mod.get_w(rtm)
    wn, wc = w / w.min(), w[:ns] / w[:ns].min()
    tr.trace(2000, seed=67, dense=False)
    Fa, sa = tr.smooth_sparse(wn)
    Fa = Fa.copy()
    Fc, sc = tr.smooth_sparse(wc, n=ns)                     # surfaces-only crop: row totals over the crop
    Fc = Fc.copy()
    tr.trace_sparse(2000, seed=67)
    Fb, sb = tr.smooth_sparse(wn)
    Fd, sd = tr.smooth_sparse(wc, n=ns)
    for A, B, x, y in ((Fa, Fb, sa, sb), (Fc, Fd, sc, sd)):
        assert np.array_equal(A.indptr, B.indptr) and np.array_equal(A.indices, B.indices) and np.array_equal(A.data, B.data)
        assert x["iterations"] == y["iterations"] and x["delta"] == y["delta"]


@pytest.mark.gpu
def test_handle_state(rthx_mod, cuda_lib):
    rtm = rthx_mod.meshes.square_domain(9, kappa=1.0)
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    w = rthx_mod.get_w(rtm)
    wn = w / w.min()
    tr.trace(1000, seed=5, dense=False)
    dense = _readout(tr, 1, False)
    Fs_dense, _ = tr.smooth(wn)
    tr.trace_sparse(1000, seed=6)
    with pytest.raises(rthx_mod.RthxError, match=r"\(1\).*sparse form"):
        tr.smooth(wn)                                       # never the stale dense counts of the first trace
    with pytest.raises(rthx_mod.RthxError, match=r"\(1\).*sparse form"):
        tr.smooth(wn, k_dykstra=1)
    assert not np.array_equal(_readout(tr, 1, False)[0]["csr"][2], dense[0]["csr"][2])
    tr.trace(1000, seed=5, dense=False)                     # a dense trace discards the sparse form
    _assert_same(_readout(tr, 1, False), dense)
    Fs2, _ = tr.smooth(wn)
    assert np.array_equal(Fs_dense, Fs2)


@pytest.mark.gpu
def test_multi_bounce_is_rejected(rthx_mod, cuda_lib):
    tr = rthx_mod.DeviceTracer(rthx_mod.flatten_domain(rthx_mod.meshes.cfg1()), device=0)
    with pytest.raises(rthx_mod.RthxError, match=r"\(1\).*FIRST_INTERACTION"):
        tr.trace_sparse(100, seed=1, mode=RTHX_MULTI_BOUNCE)
    with pytest.raises(rthx_mod.RthxError, match=r"\(1\)"):
        tr.trace_sparse(100, seed=1, mode=RTHX_MULTI_BOUNCE + 1)


@pytest.mark.gpu
def test_68640_elements_match_row_tiles(rthx_mod, cuda_lib):
    from rthx._lib import trace_row_tiles
    rtm = rthx_mod.meshes.square_domain(260, kappa=40.0)
    flat = rthx_mod.flatten_domain(rtm)
    N = flat.n_elements
    assert N == 68640
    tr = rthx_mod.DeviceTracer(flat, device=0)
    ref = trace_row_tiles(tr, 16, 4, seed=71)
    s = tr.trace_sparse(16, seed=71)
    rp, cols, vals, fv = tr.counts_csr(0, values=True, normalised=True)
    row_ptr, cols_t, fv_t = ref["csr"][0]
    assert np.array_equal(rp, row_ptr) and np.array_equal(cols, cols_t) and np.array_equal(fv, fv_t)
    assert np.array_equal(s["lost"], ref["lost"])
    assert int(vals.sum()) + int(s["lost"].sum()) == 16 * N
    assert abs(tr.counts_stats(0)[1] - ref["chi"][0]) <= 1e-12


def _ulps(a, b):
    return np.abs(a.view(np.int64) - b.view(np.int64))


@pytest.mark.gpu
def test_public_call_traces_161600_elements_on_one_gpu(rthx_mod, cuda_lib):
    rtm = rthx_mod.meshes.square_domain(400, kappa=40.0)
    N = rtm.num_elements
    assert N == 161600
    rtm(N * 16, method="exchange", verbose=False, seed=73, devices=[0])
    assert rtm.last_trace_stats["tally"] == "sparse" and "row_tiles" not in rtm.last_trace_stats
    assert rtm.last_smooth_stats["path"] == "device_sparse"
    F = rtm.F_raw.tocsc()
    Fs = rtm.F_smooth
    assert sp.issparse(Fs) and Fs.shape == (N, N)
    rtm(N * 16, method="exchange", verbose=False, seed=73, devices=[0], row_tiles=5)
    assert rtm.last_trace_stats["row_tiles"] == 5
    T = rtm.F_raw.tocsc()
    T.sort_indices()
    assert np.array_equal(F.indptr, T.indptr) and np.array_equal(F.indices, T.indices)
    assert _ulps(F.data, T.data).max() <= 1                 # count / total against count * (1 / total)
    rs = np.asarray(F.sum(axis=1)).ravel()
    assert np.abs(rs[rs > 0] - 1.0).max() <= 1e-12


@pytest.mark.gpu
def test_two_gpus_give_the_f_raw_of_one(rthx_mod, cuda_lib):
    from rthx._lib import device_count
    if device_count() < 2:
        pytest.skip("needs two or more GPUs")
    rtm = rthx_mod.meshes.square_domain(400, kappa=40.0)
    N = rtm.num_elements
    rtm(N * 16, method="exchange", verbose=False, seed=79, devices=[0], smooth=False)
    F1 = rtm.F_raw.tocsc()
    rtm(N * 16, method="exchange", verbose=False, seed=79, devices=[0, 1], smooth=False)
    assert rtm.last_trace_stats["tally"] == "sparse" and rtm.last_trace_stats["devices"] == 2
    F2 = rtm.F_raw.tocsc()
    F2.sort_indices()
    assert np.array_equal(F1.indptr, F2.indptr) and np.array_equal(F1.indices, F2.indices) and np.array_equal(F1.data, F2.data)
