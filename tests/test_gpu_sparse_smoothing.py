"""Sparse reciprocity smoothing on the device (rthx_smooth_sparse: AP on the union pattern of F and F') against the numpy
restatement of the reference's alternating projection, through the C ABI, DeviceTracer.smooth_sparse and the public call."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu


def _csc_from_device(tr, bin=0):
    colptr, rowval, _, fv = tr.counts_csc(bin, values=False, normalised=True)
    N = tr.n_elements
    return sp.csc_matrix((fv.copy(), rowval.copy(), colptr.copy()), shape=(N, N))


def _same(A, B):
    return (np.array_equal(A.indptr, B.indptr) and np.array_equal(A.indices, B.indices)
            and np.array_equal(A.data, B.data))


def _same_pattern(A, B):
    A, B = A.tocsc(), B.tocsc()
    A.sort_indices(); B.sort_indices()
    return np.array_equal(A.indptr, B.indptr) and np.array_equal(A.indices, B.indices)


def _max_abs_diff(A, B):
    d = (A - B).tocsc()
    return float(np.abs(d.data).max()) if d.nnz else 0.0


def _checks(Fs, w, rows_atol=1e-12, rows=None):
    rs = np.asarray(Fs.sum(axis=1)).ravel()
    rows = np.arange(Fs.shape[0]) if rows is None else rows
    assert np.abs(rs[rows] - 1.0).max() <= rows_atol
    WF = (sp.diags(w) @ Fs).tocsr()
    assert _max_abs_diff(WF, WF.T) <= 1e-12 * np.abs(WF.data).max()
    assert Fs.data.min() >= 0.0


def _traced(rthx_mod, rtm, rpe, seed):
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    out = tr.trace(rpe, seed=seed, dense=False)
    w = rthx_mod.get_w(rtm)
    return tr, out, w / w.min(), flat.n_surfaces


@pytest.mark.parametrize("mesh", ["square15_kappa40", "diffusion_slab31"])
def test_matches_numpy_from_both_sources(rthx_mod, cuda_lib, mesh):
    rtm = (rthx_mod.meshes.square_domain(15, kappa=40.0) if mesh == "square15_kappa40"
           else rthx_mod.meshes.diffusion_slab_domain(31))
    tr, _, wn, ns = _traced(rthx_mod, rtm, 2000, 61)
    F_raw = _csc_from_device(tr)
    n = tr.n_elements
    assert F_raw.nnz / float(n * n) <= 0.25
    Fa, sa = tr.smooth_sparse(wn)                       # from the counts still resident on the device
    Fb, sb = tr.smooth_sparse(wn, F=F_raw)              # from the host CSC of the same F_raw
    Fa2, _ = tr.smooth_sparse(wn)
    assert Fa.has_sorted_indices and isinstance(Fa, sp.csc_matrix)
    assert _same(Fa, Fb) and _same(Fa, Fa2)
    assert sa["iterations"] == sb["iterations"] and sa["converged"] == 1
    assert sa["dykstra_rounds"] == 0 and sa["delta"] <= sa["delta_init"]
    ref = rthx_mod.smoothing.AP(F_raw, wn, ns, max_iters=sa["iterations"])
    assert _same_pattern(Fa, ref)
    assert _max_abs_diff(Fa, ref) < 1e-10
    _checks(Fa, wn)


def test_crop_keeps_empty_rows_empty(rthx_mod, cuda_lib):
    """n = Ns on an optically thick mesh: most walls exchange nothing with other walls, so their rows and columns of the
    surface block are empty — and stay empty.  Row totals are taken over the crop.  The walls that do exchange form short
    chains near the corners (i - j - k with equal weights), for which no reciprocal matrix with unit row sums exists: AP runs
    to max_iters here, in step with numpy."""
    rtm = rthx_mod.meshes.square_domain(15, kappa=40.0)
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    out = tr.trace(2000, seed=62)                        # host counts too; they stay resident as well
    ns = flat.n_surfaces
    w = rthx_mod.get_w(rtm)[:ns]
    wn = w / w.min()
    c = out["counts"][0][:ns, :ns].astype(np.float64)
    rs = c.sum(axis=1, keepdims=True)
    F_crop = sp.csc_matrix(np.divide(c, rs, out=np.zeros_like(c), where=rs > 0))
    Fs, st = tr.smooth_sparse(wn, n=ns, max_iters=200)
    assert Fs.shape == (ns, ns)
    isolated = np.flatnonzero((c.sum(axis=1) == 0) & (c.sum(axis=0) == 0))
    assert 0 < len(isolated) < ns
    assert np.all(np.diff(Fs.tocsr().indptr)[isolated] == 0)
    ref = rthx_mod.smoothing.AP(F_crop, wn, ns, max_iters=st["iterations"])
    assert _same_pattern(Fs, ref) and _max_abs_diff(Fs, ref) < 1e-10
    live = np.setdiff1d(np.arange(ns), isolated)
    assert np.abs(np.asarray(Fs.sum(axis=1)).ravel()[live] - 1.0).max() <= 1e-12
    assert Fs.data.min() >= 0.0


def test_spectral_variable_bands_through_the_public_call(rthx_mod, cuda_lib):
    rtm = rthx_mod.meshes.square_domain(13, kappa=40.0, n_bins=3, kappa_bins=[30.0, 40.0, 60.0])
    N = rtm.num_elements
    rtm(N * 2000, method="exchange", verbose=False, seed=63)
    assert rtm.last_smooth_stats["path"] == "device_sparse"
    assert isinstance(rtm.F_smooth, list) and len(rtm.F_smooth) == 3
    for b in range(3):
        F_raw = rtm.F_raw[b]
        assert F_raw.nnz / float(N * N) <= 0.25
        w = rthx_mod.get_w(rtm, spectral_bin=b + 1)
        ref = rthx_mod.smoothing.smooth_F(F_raw, w, rtm.num_surfaces)
        assert _same_pattern(rtm.F_smooth[b], ref) and _max_abs_diff(rtm.F_smooth[b], ref) < 1e-10
        _checks(rtm.F_smooth[b], w / w.min())


def test_public_call_routes_sparse_F_to_the_device(rthx_mod, cuda_lib):
    rtm = rthx_mod.meshes.diffusion_slab_domain(31)
    rays = (4 * 31 + 31 ** 2) * 1000
    rtm(rays, method="exchange", verbose=False, seed=64)
    assert rtm.last_smooth_stats["path"] == "device_sparse" and rtm.last_smooth_stats["converged"] == 1
    assert sp.issparse(rtm.F_smooth)
    w = rthx_mod.get_w(rtm)
    ref = rthx_mod.smoothing.smooth_F(rtm.F_raw, w, rtm.num_surfaces, k_dykstra=0)
    assert _max_abs_diff(rtm.F_smooth, ref) < 1e-10
    rtm(rays, method="exchange", verbose=False, seed=64, k_dykstra=1)       # sparse Dykstra rounds stay on the host
    assert rtm.last_smooth_stats["path"] == "host"


def test_row_tiles_match_the_untiled_public_call(rthx_mod, cuda_lib):
    """Row tiles smooth the host CSC F_raw (FROM_CSC), one trace smooths the resident counts: same pattern, same F_smooth up to
    the last bits of F_raw (the tiled read-out multiplies by the reciprocal row total, the CSC read-out divides)."""
    rtm = rthx_mod.meshes.square_domain(60, kappa=40.0)
    N = rtm.num_elements
    rtm(N * 200, method="exchange", verbose=False, seed=65, row_tiles=3)
    assert rtm.last_smooth_stats["path"] == "device_sparse"
    F3 = rtm.F_smooth
    rtm(N * 200, method="exchange", verbose=False, seed=65, row_tiles=1)
    assert rtm.last_smooth_stats["path"] == "device_sparse"
    assert _same_pattern(F3, rtm.F_smooth)
    assert _max_abs_diff(F3, rtm.F_smooth) < 1e-12


def test_public_call_smooths_the_68640_element_mesh_in_row_tiles(rthx_mod, cuda_lib):
    rtm = rthx_mod.meshes.square_domain(260, kappa=40.0)
    N = rtm.num_elements
    assert N == 4 * 260 + 260 * 260
    rtm(N * 64, method="exchange", verbose=False, seed=5, row_tiles=4)
    Fs = rtm.F_smooth
    st = rtm.last_smooth_stats
    assert st["path"] == "device_sparse" and st["converged"] == 1
    assert sp.issparse(Fs) and Fs.shape == (N, N) and Fs.nnz < 2 * 64 * N
    assert _same_pattern(Fs, Fs.T)
    w = rthx_mod.get_w(rtm)
    _checks(Fs, w / w.min(), rows_atol=1e-9)
    assert "smoothing" in rtm.last_phase_ms


def test_sparse_smoothing_replaces_the_dense_result_on_the_handle(rthx_mod, cuda_lib):
    rtm = rthx_mod.meshes.square_domain(9, kappa=0.7)
    tr, _, wn, ns = _traced(rthx_mod, rtm, 2000, 66)
    n = tr.n_elements
    coeff, rhs = np.full(n, 0.5), np.ones(n)
    tr.smooth(wn)
    tr.solve_grey(coeff, rhs)                            # the dense F_smooth is resident
    tr.smooth_sparse(wn)
    with pytest.raises(rthx_mod.RthxError):
        tr.solve_grey(coeff, rhs)                        # ... and no longer after a sparse smoothing
    fresh = rthx_mod.DeviceTracer(rthx_mod.flatten_domain(rtm), device=0)
    colptr, rowval, nzval = np.empty(n + 1, np.int64), np.empty(8, np.int32), np.empty(8)
    rc = cuda_lib.rthx_smooth_sparse_csc(fresh._h, 0, 0, colptr.ctypes.data_as(C.POINTER(C.c_int64)),
                                         rowval.ctypes.data_as(C.c_void_p), nzval.ctypes.data_as(C.POINTER(C.c_double)))
    assert rc == 1 and b"no sparse F_smooth" in cuda_lib.rthx_last_error(fresh._h)


def test_sparse_csc_read_out_conventions(rthx_mod, cuda_lib):
    """1-based and 64-bit row indices, as a Julia SparseMatrixCSC{Float64,Int} holds them."""
    rtm = rthx_mod.meshes.square_domain(9, kappa=20.0)
    tr, _, wn, _ = _traced(rthx_mod, rtm, 2000, 67)
    Fs, _ = tr.smooth_sparse(wn)
    n, nnz = Fs.shape[0], Fs.nnz
    colptr, rowval, nzval = np.empty(n + 1, np.int64), np.empty(nnz, np.int64), np.empty(nnz)
    tr._check(cuda_lib.rthx_smooth_sparse_csc(tr._h, 1, 1, colptr.ctypes.data_as(C.POINTER(C.c_int64)),
                                              rowval.ctypes.data_as(C.c_void_p), nzval.ctypes.data_as(C.POINTER(C.c_double))))
    assert np.array_equal(colptr, Fs.indptr.astype(np.int64) + 1)
    assert np.array_equal(rowval, Fs.indices.astype(np.int64) + 1)
    assert np.array_equal(nzval, Fs.data)


@pytest.mark.parametrize("defect", ["colptr0", "decreasing", "row_out_of_range", "unsorted"])
def test_malformed_csc_is_rejected_on_the_host(rthx_mod, cuda_lib, defect):
    rtm = rthx_mod.meshes.square_domain(5, kappa=20.0)
    tr, _, wn, _ = _traced(rthx_mod, rtm, 2000, 68)
    F = _csc_from_device(tr)
    n = F.shape[0]
    colptr, rowval, nzval = F.indptr.astype(np.int64), F.indices.astype(np.int32), F.data.copy()
    j = int(np.flatnonzero(np.diff(colptr) >= 2)[0])                 # a column with at least two entries
    if defect == "colptr0":
        colptr[0] = 1
    elif defect == "decreasing":
        colptr[j + 1] = colptr[j] - 1
    elif defect == "row_out_of_range":
        rowval[colptr[j + 1] - 1] = n
    else:
        a = colptr[j]
        rowval[a], rowval[a + 1] = rowval[a + 1], rowval[a]
    nnz = C.c_int64(-1)
    rc = cuda_lib.rthx_smooth_sparse(tr._h, rthx_mod._abi.RTHX_SMOOTH_FROM_CSC, 0, n, colptr.ctypes.data_as(C.POINTER(C.c_int64)),
                                     rowval.ctypes.data_as(C.POINTER(C.c_int32)), nzval.ctypes.data_as(C.POINTER(C.c_double)),
                                     wn.ctypes.data_as(C.POINTER(C.c_double)), 100, 0.0, 0, C.byref(nnz), None)
    with pytest.raises(rthx_mod.RthxError, match="colptr|rowval"):
        tr._check(rc)
    assert nnz.value == -1


def test_multi_gpu_resident_counts_match_one_device(rthx_mod, cuda_lib):
    from rthx._lib import create_multi, device_count, trace_multi
    if device_count() < 2:
        pytest.skip("needs two or more GPUs")
    rtm = rthx_mod.meshes.square_domain(15, kappa=40.0)
    flat = rthx_mod.flatten_domain(rtm)
    w = rthx_mod.get_w(rtm)
    wn = w / w.min()
    tr = rthx_mod.DeviceTracer(flat, device=0)
    tr.trace(2000, seed=69, dense=False)
    F1, _ = tr.smooth_sparse(wn)
    trs = create_multi(flat, [0, 1])
    trace_multi(trs, 2000, dense=False, seed=69)
    F2, _ = trs[0].smooth_sparse(wn)
    assert _same(F1, F2)
