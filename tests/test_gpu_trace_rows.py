"""Tracing only the emitter rows a caller names (rthx_trace_exchange_rows, DeviceTracer.trace_rows, parallelRayTracing(emitters=...),
and the surfaces-only route of exchangeRayTracing).  Counts are a pure function of (seed, ray id, emitter, band), so every listed row
must equal, bit for bit, the same row of a full trace, and every read-out of the resident rows must equal the read-out of the full
trace restricted to those rows."""

import numpy as np
import pytest
import scipy.sparse as sp

from rthx._abi import RTHX_LOCATOR_GENERIC, RTHX_MULTI_BOUNCE, RTHX_MULTI_BOUNCE_SPECULAR

RAYS = 600


def _trapezoid():
    from rthx import PolyVolume2D, RayTracingDomain2D
    face = PolyVolume2D([(0.0, 0.0), (2.0, 0.0), (1.5, 1.0), (0.5, 1.0)], (True, True, True, True), 1, 0.8, 0.0)
    face.epsilon = [1.0] * 4
    face.T_in_w = [1000.0, 0.0, 0.0, 0.0]
    face.T_in_g = -1.0
    face.q_in_g = 0.0
    rtm = RayTracingDomain2D([face], [(7, 5)])
    for i, cell in enumerate(rtm.fine_mesh[0]):
        cell.kappa_g = 0.3 + 0.1 * (i % 9)
    rtm.refresh_spectral_flags()
    return rtm


def _case(rthx_mod, name):
    """(domain, trace keywords, environment) of each case: every trace-kernel family and the launch / stream variants."""
    m = rthx_mod.meshes
    scatter = dict(kappa=0.6, sigma_s=0.9, epsilon=(0.3, 0.6, 0.9, 0.5))
    return {
        "cfg1": (m.cfg1(), {}, {}),
        "cfg1_block128": (m.cfg1(), dict(block_threads=128), {}),
        "circle": (m.circle_domain(N_seg=16, Ndim=5), {}, {}),
        "trapezoid": (_trapezoid(), {}, {}),
        "generic_locator": (m.cfg1(), dict(locator=RTHX_LOCATOR_GENERIC), {}),
        "two_quads_variable_beta": (m.two_quads_domain(kappa=(0.5, 3.0)), {}, {}),
        "global_tally": (m.cfg1(), {}, {"RTHX_FORCE_GLOBAL_TALLY": "1"}),
        "multi_bounce": (m.square_domain(9, **scatter), dict(mode=RTHX_MULTI_BOUNCE), {}),
        "multi_bounce_specular": (m.square_domain(9, **scatter), dict(mode=RTHX_MULTI_BOUNCE_SPECULAR), {}),
        "cfg4_bins_2_0": (m.cfg4(Ndim=9, n_bins=3), dict(bins=[2, 0]), {}),
        "ray_id_offset": (m.cfg1(), dict(ray_id_offset=2 ** 33 + 12345), {}),
    }[name]


CASES = ["cfg1", "cfg1_block128", "circle", "trapezoid", "generic_locator", "two_quads_variable_beta", "global_tally", "multi_bounce",
         "multi_bounce_specular", "cfg4_bins_2_0", "ray_id_offset"]


def _lists(N, ns):
    """One row, the last row, a non-contiguous list mixing surfaces and volumes, the surface rows [0, Ns), and all rows."""
    mixed = sorted({0, 2, 3, ns - 1, ns, ns + 1, ns + 4, ns + 7, N - 2} & set(range(N)))
    return {"one": [ns // 2], "last": [N - 1], "mixed": mixed, "surfaces": list(range(ns)), "all": list(range(N))}


def _readout(tr, n_bins):
    out = []
    for k in range(n_bins):
        nnz, chi = tr.counts_stats(k)
        rp, cols, vals, fv = tr.counts_csr(k, values=True, normalised=True)
        cp, rv, cv, cf = tr.counts_csc(k, values=True, normalised=True, pinned=False)
        out.append(dict(nnz=nnz, chi=chi, csr=(rp.copy(), cols.copy(), vals.copy(), fv.copy()), csc=(cp.copy(), rv.copy(), cv.copy(), cf.copy())))
    return out


def _expected(full_counts, rows, ns):
    """Read-outs of the full trace restricted to `rows`, per bin, built on the host from the full count matrix: CSR of the listed rows
    (F = count * (1 / row total), as rthx_counts_csr forms it) and CSC of the N x N matrix whose other rows are empty (F = count / row
    total), with nnz and chi over the listed rows."""
    out = []
    N = full_counts.shape[1]
    for c in full_counts:
        sub = c[rows]
        tot = sub.sum(axis=1)
        csr = sp.csr_matrix(sub)
        csr.sort_indices()
        lens = np.diff(csr.indptr)
        inv = np.where(tot > 0, 1.0 / np.maximum(tot, 1).astype(np.float64), 0.0)
        fv = csr.data.astype(np.float64) * np.repeat(inv, lens)
        full = np.zeros_like(c)
        full[rows] = sub
        csc = sp.csc_matrix(full)
        csc.sort_indices()
        row_tot = full.sum(axis=1)
        cf = csc.data.astype(np.float64) / row_tot[csc.indices].astype(np.float64)
        surf = np.arange(N) < ns
        cross = np.array([sub[i][surf != (rows[i] < ns)].sum() for i in range(len(rows))], dtype=np.float64)
        chi = float(sum(cross[i] / tot[i] for i in range(len(rows)) if tot[i])) / N
        out.append(dict(nnz=int(csr.nnz), chi=chi, csr=(csr.indptr.astype(np.int64), csr.indices.astype(np.int32), csr.data.astype(np.uint64), fv),
                        csc=(csc.indptr.astype(np.int64), csc.indices.astype(np.int32), csc.data.astype(np.uint64), cf)))
    return out


def _assert_same(got, ref):
    assert len(got) == len(ref)
    for x, y in zip(got, ref):
        assert x["nnz"] == y["nnz"]
        assert x["chi"] == pytest.approx(y["chi"], rel=1e-12, abs=1e-15)
        for u, v in zip(x["csr"] + x["csc"], y["csr"] + y["csc"]):
            assert np.array_equal(u, v)


# ---- CPU ------------------------------------------------------------------------------------------------------------------

def test_symbol_exported_and_checks_its_handle(cuda_lib, rthx_mod):
    assert cuda_lib.rthx_trace_exchange_rows is not None
    assert cuda_lib.rthx_trace_exchange_rows(None, None, None, 0, None, None, None, None) == 1       # RTHX_ERR_ARG: no handle


def test_merge_row_tiles_places_listed_rows(rthx_mod):
    from rthx._lib import merge_row_tiles
    N = 7
    tiles = [[(np.array([0, 2, 3]), np.array([1, 4, 0], np.int32), np.array([0.5, 0.5, 1.0]))],
             [(np.array([0, 1]), np.array([6], np.int32), np.array([1.0]))]]
    (rp, cols, vals), = merge_row_tiles(tiles, N, 1, tile_rows=[np.array([1, 5]), np.array([3])])
    dense = sp.csr_matrix((vals, cols, rp), shape=(N, N)).toarray()
    ref = np.zeros((N, N))
    ref[1, 1] = ref[1, 4] = 0.5
    ref[5, 0] = 1.0
    ref[3, 6] = 1.0
    assert np.array_equal(dense, ref)


# ---- GPU: the C ABI through DeviceTracer -----------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_rows_equal_the_rows_of_a_full_trace(rthx_mod, cuda_lib, monkeypatch, name):
    rtm, kw, env = _case(rthx_mod, name)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    N, ns = tr.n_elements, tr.info["n_surfaces"]
    nb = len(kw.get("bins", (0,)))
    full = tr.trace(RAYS, seed=23, **kw)
    for label, rows in _lists(N, ns).items():
        dense = tr.trace_rows(rows, RAYS, seed=23, **kw)
        assert dense["counts"].shape == (nb, len(rows), N)
        assert np.array_equal(dense["counts"], full["counts"][:, rows]), label
        lost = np.zeros_like(full["lost"])
        lost[:, rows] = full["lost"][:, rows]
        assert np.array_equal(dense["lost"], lost), label
        assert dense["stats"]["rays_traced"] == RAYS * len(rows) * nb
        res = tr.trace_rows(rows, RAYS, seed=23, dense=False, **kw)
        assert np.array_equal(res["lost"], lost) and res["counts"] is None
        _assert_same(_readout(tr, nb), _expected(full["counts"], np.asarray(rows), ns))
        if label == "all":
            tr.trace(RAYS, seed=23, dense=False, **kw)
            ref = _readout(tr, nb)
            tr.trace_rows(rows, RAYS, seed=23, dense=False, **kw)
            got = _readout(tr, nb)
            for x, y in zip(got, ref):        # all rows: the same arrays as a full trace, chi included, bit for bit
                assert x["nnz"] == y["nnz"] and x["chi"] == y["chi"]
                for u, v in zip(x["csr"] + x["csc"], y["csr"] + y["csc"]):
                    assert u.dtype == v.dtype and np.array_equal(u, v)


@pytest.mark.gpu
def test_recorder_points_are_those_of_a_full_trace(rthx_mod, cuda_lib):
    rtm = rthx_mod.meshes.cfg1()
    tr = rthx_mod.DeviceTracer(rthx_mod.flatten_domain(rtm), device=0)
    N, ns = tr.n_elements, tr.info["n_surfaces"]
    rec = [3, ns + 5]
    full = tr.trace(RAYS, seed=9, rec_ids=rec)
    got = tr.trace_rows([1, 3, ns + 2, ns + 5, N - 1], RAYS, seed=9, rec_ids=rec)
    assert got["origins"].shape == full["origins"].shape and len(got["origins"]) > 0
    assert np.array_equal(got["origins"], full["origins"]) and np.array_equal(got["endpoints"], full["endpoints"])


@pytest.mark.gpu
def test_rejections_leave_the_resident_counts(rthx_mod, cuda_lib):
    rtm = rthx_mod.meshes.cfg1()
    tr = rthx_mod.DeviceTracer(rthx_mod.flatten_domain(rtm), device=0)
    N = tr.n_elements
    tr.trace_rows([0, 4, 9, N - 1], RAYS, seed=3, dense=False)
    before = _readout(tr, 1)
    bad = [
        (dict(emitters=[4, 2]), "strictly ascending"),
        (dict(emitters=[2, 2]), "strictly ascending"),
        (dict(emitters=[0, N]), "outside"),
        (dict(emitters=[-1, 3]), "outside"),
        (dict(emitters=[]), "empty"),
        (dict(emitters=[1, 2], emitter_rank=1, emitter_world=2), "emitter_rank"),
        (dict(emitters=[1, 2], rec_ids=[3]), "rec_ids"),
    ]
    for kw, match in bad:
        rows = kw.pop("emitters")
        with pytest.raises(rthx_mod.RthxError, match=match):
            tr.trace_rows(rows, RAYS, seed=3, dense=False, **kw)
        after = _readout(tr, 1)
        for x, y in zip(after, before):
            assert x["nnz"] == y["nnz"] and x["chi"] == y["chi"]
            for u, v in zip(x["csr"] + x["csc"], y["csr"] + y["csc"]):
                assert np.array_equal(u, v)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["ap", "dkap1", "sparse"])
def test_smoothing_of_the_surface_rows_equals_that_after_a_full_trace(rthx_mod, cuda_lib, mode):
    rtm = rthx_mod.meshes.square_domain(8, kappa=0.0)
    tr = rthx_mod.DeviceTracer(rthx_mod.flatten_domain(rtm), device=0)
    ns = tr.info["n_surfaces"]
    w = np.ones(ns)

    def smoothed():
        if mode == "sparse":
            F, st = tr.smooth_sparse(w, n=ns, max_iters=200)
            F = F.tocsc(); F.sort_indices()
            return (F.indptr.copy(), F.indices.copy(), F.data.copy()), st["iterations"]
        F, st = tr.smooth(w, n=ns, max_iters=200, k_dykstra=1 if mode == "dkap1" else 0)
        return (F.copy(),), st["iterations"]

    tr.trace(2000, seed=11, dense=False)
    ref = smoothed()
    tr.trace_rows(np.arange(ns), 2000, seed=11, dense=False)
    got = smoothed()
    assert got[1] == ref[1]
    for u, v in zip(got[0], ref[0]):
        assert np.array_equal(u, v)
    tr.trace_rows(np.r_[np.arange(ns - 1), ns + 3], 2000, seed=11, dense=False)     # row ns - 1 of the crop is missing
    with pytest.raises(rthx_mod.RthxError, match=f"row {ns - 1} of the crop"):
        smoothed()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cfg1", "multi_bounce"])
def test_continuations_of_a_rows_trace_equal_one_rows_trace(rthx_mod, cuda_lib, monkeypatch, name):
    rtm, kw, env = _case(rthx_mod, name)
    tr = rthx_mod.DeviceTracer(rthx_mod.flatten_domain(rtm), device=0)
    N, ns = tr.n_elements, tr.info["n_surfaces"]
    rows = _lists(N, ns)["mixed"]
    tr.trace_rows(rows, 700, seed=41, dense=False, **kw)
    tr.trace_continue(500, row_chunks=1)
    third = tr.trace_continue(900)
    cont = _readout(tr, 1)
    single = tr.trace_rows(rows, 2100, seed=41, dense=False, **kw)
    ref = _readout(tr, 1)
    assert np.array_equal(third["lost"], single["lost"])
    for x, y in zip(cont, ref):
        assert x["nnz"] == y["nnz"] and x["chi"] == y["chi"]
        for u, v in zip(x["csr"] + x["csc"], y["csr"] + y["csc"]):
            assert np.array_equal(u, v)


# ---- GPU: the public call -----------------------------------------------------------------------------------------------

def _same_sparse(x, y):
    x, y = sp.csc_matrix(x), sp.csc_matrix(y)
    x.sort_indices(); y.sort_indices()
    return np.array_equal(x.indptr, y.indptr) and np.array_equal(x.indices, y.indices) and np.array_equal(x.data, y.data)


def _same(x, y):
    return _same_sparse(x, y) if sp.issparse(x) or sp.issparse(y) else np.array_equal(x, y)


def _domains(rthx_mod):
    circle = rthx_mod.meshes.circle_domain(N_seg=16, Ndim=5, kappa=0.0)
    return {"square": rthx_mod.meshes.square_domain(8, kappa=0.0), "circle": circle}


def _two_handles_on_device_0(rthx_mod):
    def tracers_for(rtm, devices):
        flat = rthx_mod.flatten_domain(rtm)
        for old in getattr(rtm, "_devices", None) or []:
            old.close()
        trs = [rthx_mod.DeviceTracer(flat, device=0), rthx_mod.DeviceTracer(flat, device=0)]
        rtm._devices, rtm._device, rtm.last_phase_ms = trs, trs[0], {}
        return trs
    return tracers_for


def _public(rthx_mod, rtm, rays, rec_ids=None, **kw):
    rec = rthx_mod.RayRecorder(rec_ids, 1) if rec_ids else None
    rtm(rays, method="exchange", verbose=False, rec=rec, **kw)
    out = dict(F_raw=rtm.F_raw, F_smooth=rtm.F_smooth, rows=rtm.last_trace_stats["rows"], devices=rtm.last_trace_stats.get("devices"),
               path=rtm.last_smooth_stats["path"])
    if rec is not None:
        out["origins"], out["endpoints"] = np.concatenate(rec.origins, axis=0), np.concatenate(rec.endpoints, axis=0)
    return out


def _same_result(a, b):
    assert _same(a["F_raw"], b["F_raw"]) and _same(a["F_smooth"], b["F_smooth"]) and a["path"] == b["path"]
    if "origins" in a or "origins" in b:
        assert len(a["origins"]) > 0
        assert np.array_equal(a["origins"], b["origins"]) and np.array_equal(a["endpoints"], b["endpoints"])


@pytest.mark.gpu
@pytest.mark.parametrize("dom", ["square", "circle"])
def test_public_surface_rows_equal_the_full_route(rthx_mod, cuda_lib, monkeypatch, dom):
    from rthx import tracing
    rtm = _domains(rthx_mod)[dom]
    assert rtm.surfaces_only
    N, ns = rtm.num_elements, rtm.num_surfaces
    rec = [2, 3, ns]                                           # 1-based surface ids
    ref = _public(rthx_mod, rtm, 300 * N, rec, seed=77, devices=[0], trace_volume_rows=True)
    got = _public(rthx_mod, rtm, 300 * N, rec, seed=77, devices=[0])
    assert ref["rows"] == N and got["rows"] == ns
    _same_result(got, ref)
    # refine continues the rows trace: equal to one call with all the rays
    rtm(200 * N, method="exchange", verbose=False, refine=True)
    refined = dict(F_raw=rtm.F_raw, F_smooth=rtm.F_smooth, path=rtm.last_smooth_stats["path"])
    full = _public(rthx_mod, rtm, 500 * N, rec, seed=77, devices=[0], trace_volume_rows=True)
    _same_result(refined, {k: full[k] for k in refined})
    # two handles: the surface rows fit one device, so they are traced and smoothed on the first one; F_raw, F_smooth, the smoothing path
    # and the recorder points are those of the full route (whose multi-device gather leaves the counts of a single-device trace on it)
    monkeypatch.setattr(tracing, "_tracers_for", _two_handles_on_device_0(rthx_mod))
    two = _public(rthx_mod, rtm, 500 * N, rec, seed=77, devices=[0])
    assert two["rows"] == ns and two["devices"] is None
    _same_result(two, full)


@pytest.mark.gpu
def test_rows_beyond_one_device_are_split_over_the_devices(rthx_mod, cuda_lib, monkeypatch):
    from rthx import tracing
    rtm = rthx_mod.meshes.cfg1()
    N, ns = rtm.num_elements, rtm.num_surfaces
    rows = np.array(_lists(N, ns)["mixed"], dtype=np.int32)

    def run():
        rec = rthx_mod.RayRecorder([int(rows[1]) + 1, int(rows[-2]) + 1], 1)
        F, _ = tracing.parallelRayTracing(rtm, 300 * N, None, False, rec=rec, seed=8, devices=[0], emitters=rows)
        return F, dict(rtm.last_trace_stats), np.concatenate(rec.origins, axis=0), np.concatenate(rec.endpoints, axis=0), rtm.last_lost.copy()

    ref = run()
    monkeypatch.setattr(tracing, "rows_fit_one_device", lambda *a, **k: False)
    # the surfaces-only default route does not split its rows: when they do not fit one device it takes the full route, as before
    sq = rthx_mod.meshes.square_domain(8, kappa=0.0)
    _public(rthx_mod, sq, 100 * sq.num_elements, seed=8, devices=[0])
    assert sq.last_trace_stats["rows"] == sq.num_elements
    # an explicit list beyond one device: each of two handles traces a contiguous block, merged bit for bit, recorder in element order
    monkeypatch.setattr(tracing, "_tracers_for", _two_handles_on_device_0(rthx_mod))
    got = run()
    assert got[1]["devices"] == 2 and "devices" not in ref[1] and got[1]["rows"] == ref[1]["rows"] == len(rows)
    assert _same(got[0], ref[0])
    assert len(ref[2]) > 0
    for u, v in zip(got[2:], ref[2:]):
        assert np.array_equal(u, v)


@pytest.mark.gpu
def test_public_recorder_takes_the_route_its_ids_allow(rthx_mod, cuda_lib):
    from rthx import RayRecorder
    rtm = _domains(rthx_mod)["square"]
    N, ns = rtm.num_elements, rtm.num_surfaces
    out = {}
    for label, ids, extra in (("surface", [2, 5], {}), ("surface_full", [2, 5], dict(trace_volume_rows=True)), ("volume", [2, ns + 3], {})):
        rec = RayRecorder(ids, 1)
        rtm(200 * N, method="exchange", verbose=False, seed=5, devices=[0], rec=rec, **extra)
        out[label] = (rtm.last_trace_stats["rows"], np.concatenate(rec.origins, axis=0), np.concatenate(rec.endpoints, axis=0), rtm.F_raw)
    assert out["surface"][0] == ns and out["surface_full"][0] == N and out["volume"][0] == N
    assert len(out["surface"][1]) > 0
    assert np.array_equal(out["surface"][1], out["surface_full"][1]) and np.array_equal(out["surface"][2], out["surface_full"][2])
    assert _same(out["surface"][3], out["surface_full"][3])
