"""Continuing a trace on the device (rthx_trace_exchange_continue, DeviceTracer.trace_continue, rtm(...; refine=True)).  The resident
counts are always those of ONE trace of a contiguous ray-id range with one seed, so k continuations must give, bit for bit, every
read-out that a single trace of the whole range gives — in the dense and in the hashed form, also when the continuation itself splits
into many row groups before it is merged."""

import numpy as np
import pytest
import scipy.sparse as sp

from rthx._abi import RTHX_LOCATOR_GENERIC, RTHX_MULTI_BOUNCE, RTHX_MULTI_BOUNCE_SPECULAR

R1, R2, R3 = 700, 500, 900           # rays per emitter of the trace and of its two continuations


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
    """(domain, trace keywords, environment) of each case."""
    m = rthx_mod.meshes
    scatter = dict(kappa=0.6, sigma_s=0.9, epsilon=(0.3, 0.6, 0.9, 0.5))
    return {
        "cfg1": (m.cfg1(), {}, {}),
        "circle": (m.circle_domain(N_seg=16, Ndim=5), {}, {}),
        "two_quads_variable_beta": (m.two_quads_domain(kappa=(0.5, 3.0)), {}, {}),
        "trapezoid": (_trapezoid(), {}, {}),
        "generic_locator": (m.cfg1(), dict(locator=RTHX_LOCATOR_GENERIC), {}),
        "cfg4_bins_2_0": (m.cfg4(Ndim=9, n_bins=3), dict(bins=[2, 0]), {}),
        "sharded": (m.square_domain(15, kappa=1.0), dict(emitter_rank=1, emitter_world=3), {}),
        "global_tally": (m.cfg1(), {}, {"RTHX_FORCE_GLOBAL_TALLY": "1"}),
        "multi_bounce": (m.square_domain(9, **scatter), dict(mode=RTHX_MULTI_BOUNCE), {}),
        "multi_bounce_specular": (m.square_domain(9, **scatter), dict(mode=RTHX_MULTI_BOUNCE_SPECULAR), {}),
    }[name]


DENSE_CASES = ["cfg1", "circle", "two_quads_variable_beta", "trapezoid", "generic_locator", "cfg4_bins_2_0", "sharded", "global_tally",
               "multi_bounce", "multi_bounce_specular"]
HASHED_CASES = [c for c in DENSE_CASES if not c.startswith("multi_bounce")]


def _readout(tr, n_bins, sharded):
    """Every read-out of the resident counts, per traced bin."""
    out = []
    for k in range(n_bins):
        nnz, chi = tr.counts_stats(k)
        rp, cols, vals, fv = tr.counts_csr(k, values=True, normalised=True)
        r = dict(nnz=nnz, chi=chi, csr=(rp.copy(), cols.copy(), vals.copy(), fv.copy()))
        if not sharded:
            cp, rv, cv, cf = tr.counts_csc(k, values=True, normalised=True, pinned=False)
            r["csc"] = (cp.copy(), rv.copy(), cv.copy(), cf.copy())
        out.append(r)
    return out


def _assert_same(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x["nnz"] == y["nnz"] and x["chi"] == y["chi"]
        assert ("csc" in x) == ("csc" in y)
        for u, v in zip(x["csr"] + x.get("csc", ()), y["csr"] + y.get("csc", ())):
            assert u.dtype == v.dtype and np.array_equal(u, v)


def _continued_and_single(rthx_mod, monkeypatch, name, hashed, seed=41, rays=(R1, R2, R3)):
    """Readouts after trace(R1) -> continue(R2) -> continue(R3) and after one trace of R1 + R2 + R3 rays."""
    R1, R2, R3 = rays
    rtm, kw, env = _case(rthx_mod, name)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    tr = rthx_mod.DeviceTracer(rthx_mod.flatten_domain(rtm), device=0)
    nb = len(kw.get("bins", (0,)))
    sharded = kw.get("emitter_world", 1) > 1
    first = tr.trace_sparse(R1, seed=seed, **kw) if hashed else tr.trace(R1, seed=seed, dense=False, **kw)
    second = tr.trace_continue(R2, row_chunks=1)               # counts do not depend on the launch shape
    third = tr.trace_continue(R3)
    cont = _readout(tr, nb, sharded)
    single = tr.trace(R1 + R2 + R3, seed=seed, dense=False, **kw)
    ref = _readout(tr, nb, sharded)
    _assert_same(cont, ref)
    assert np.array_equal(third["lost"], single["lost"])
    assert third["stats"]["rays_lost"] == single["stats"]["rays_lost"]
    assert third["stats"]["rays_traced"] * (R1 + R2 + R3) == single["stats"]["rays_traced"] * R3
    assert np.all(first["lost"] <= second["lost"]) and np.all(second["lost"] <= third["lost"])
    return first, second, third, cont


# ---- CPU ------------------------------------------------------------------------------------------------------------------

def test_symbol_exported_and_checks_its_handle(cuda_lib, rthx_mod):
    assert cuda_lib.rthx_trace_exchange_continue is not None
    assert cuda_lib.rthx_trace_exchange_continue(None, None, None, None, None, None) == 1       # RTHX_ERR_ARG: no handle


def _fake_previous_call(rtm, rthx_mod, **state):
    """The state a previous public call leaves behind, without a device: handles that only carry their flattened mesh."""
    class _Handle:
        def __init__(self, flat):
            self.flat = flat

        def close(self):
            pass

    rtm._devices = [_Handle(rthx_mod.flatten_domain(rtm))]
    rtm._device = rtm._devices[0]
    base = dict(seed=5, devices=[0], locator=0, row_tiles=None, nudge=rthx_mod._lib.DEFAULT_NUDGE, n_tiles=1, dense_multi=False,
                rays_per_emitter_total=100)
    rtm._trace_state = dict(base, **state)


@pytest.mark.parametrize("case, match", [
    ("no_previous_call", "no previous exchange trace"),
    ("row_tiles", "explicit row_tiles"),
    ("dense_multi", "several devices"),
    ("mesh_changed", "flattened mesh differs"),
    ("seed", "seed=6 differs"),
    ("devices", "devices=\\[1\\] differs"),
    ("device", "devices=\\[1\\] differs"),
    ("locator", "locator=1 differs"),
    ("row_tiles_given", "row_tiles=2 differs"),
    ("nudge", "nudge=0.001 differs"),
])
def test_refine_rejections_without_a_device(rthx_mod, case, match):
    rtm = rthx_mod.meshes.cfg1()
    N = rtm.num_elements
    if case != "no_previous_call":
        _fake_previous_call(rtm, rthx_mod, **({"row_tiles": 3, "n_tiles": 3} if case == "row_tiles" else
                                               {"dense_multi": True, "devices": [0, 1]} if case == "dense_multi" else {}))
    if case == "mesh_changed":
        rtm.fine_mesh[0][3].kappa_g = 7.0
    kw = {"seed": dict(seed=6), "devices": dict(devices=[1]), "device": dict(device=1), "locator": dict(locator=RTHX_LOCATOR_GENERIC),
          "row_tiles_given": dict(row_tiles=2), "nudge": dict(nudge=1e-3)}.get(case, {})
    with pytest.raises(ValueError, match=match):
        rtm(N * 10, method="exchange", verbose=False, refine=True, **kw)


# ---- GPU: continuations against one trace of the whole range --------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", DENSE_CASES)
def test_dense_continuations_equal_one_trace(rthx_mod, cuda_lib, monkeypatch, name):
    _, second, third, _ = _continued_and_single(rthx_mod, monkeypatch, name, hashed=False)
    assert "sparse_stats" not in second and "sparse_stats" not in third


@pytest.mark.gpu
@pytest.mark.parametrize("name", HASHED_CASES)
def test_hashed_continuations_equal_one_trace(rthx_mod, cuda_lib, monkeypatch, name):
    _, second, third, cont = _continued_and_single(rthx_mod, monkeypatch, name, hashed=True)
    assert third["sparse_stats"]["nnz"] == sum(r["nnz"] for r in cont)
    assert third["sparse_stats"]["row_groups"] == 1 and third["sparse_stats"]["reduce_ms"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", HASHED_CASES)
def test_hashed_continuations_with_forced_flushes_and_row_groups(rthx_mod, cuda_lib, monkeypatch, name):
    monkeypatch.setenv("RTHX_SPARSE_HASH_SLOTS", "512")     # the table is flushed before every round that follows an insert
    monkeypatch.setenv("RTHX_SPARSE_PAIR_CAP", "9000")      # one emitter row (<= 2 bins x 2100 rays) fits, the whole mesh does not
    _, second, third, cont = _continued_and_single(rthx_mod, monkeypatch, name, hashed=True, rays=(1900, 2000, 2100))
    for out in (second, third):
        ss = out["sparse_stats"]
        assert ss["hash_slots"] == 512 and ss["pair_capacity"] == 9000
        assert ss["row_groups"] >= 2 and ss["pairs"] > 0, ss
    assert third["sparse_stats"]["nnz"] == sum(r["nnz"] for r in cont)


@pytest.mark.gpu
@pytest.mark.parametrize("hashed", [False, True])
def test_smoothing_after_continuations(rthx_mod, cuda_lib, hashed):
    rtm = rthx_mod.meshes.square_domain(15, kappa=40.0)
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    ns = flat.n_surfaces
    w = rthx_mod.get_w(rtm)
    wn, wc = w / w.min(), w[:ns] / w[:ns].min()

    def smoothed():
        out = []
        for ww, n in ((wn, None), (wc, ns)):                 # whole matrix and surfaces-only crop
            F, st = tr.smooth_sparse(ww, n=n)
            out.append((F.indptr.copy(), F.indices.copy(), F.data.copy(), st["iterations"], st["delta"]))
        if not hashed:
            for k in (0, 1):
                F, st = tr.smooth(wn, k_dykstra=k)
                out.append((F.copy(), st["iterations"], st["delta"]))
        return out

    (tr.trace_sparse(R1, seed=67) if hashed else tr.trace(R1, seed=67, dense=False))
    tr.trace_continue(R2)
    a = smoothed()
    tr.trace(R1 + R2, seed=67, dense=False)
    b = smoothed()
    for x, y in zip(a, b):
        for u, v in zip(x, y):
            assert np.array_equal(u, v)


@pytest.mark.gpu
@pytest.mark.parametrize("hashed", [False, True])
def test_recorder_points_are_those_of_a_trace_with_the_offset(rthx_mod, cuda_lib, monkeypatch, hashed):
    monkeypatch.setenv("RTHX_FORCE_GLOBAL_TALLY", "1")      # the dense trace runs the hashed tally's ray loop: the same points
    rtm = rthx_mod.meshes.two_quads_domain(kappa=(0.5, 3.0))
    tr = rthx_mod.DeviceTracer(rthx_mod.flatten_domain(rtm), device=0)
    rec = dict(rec_ids=[1, 20])
    (tr.trace_sparse(R1, seed=13) if hashed else tr.trace(R1, seed=13, dense=False))
    c = tr.trace_continue(R2, **rec)
    p = tr.trace(R2, seed=13, dense=False, ray_id_offset=R1, **rec)
    assert len(c["origins"]) > 0 and c["origins"].shape == p["origins"].shape
    assert np.array_equal(c["origins"], p["origins"]) and np.array_equal(c["endpoints"], p["endpoints"])


# ---- GPU: rejections ----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("hashed", [False, True])
def test_rejections_leave_the_resident_counts(rthx_mod, cuda_lib, hashed):
    Err = rthx_mod.RthxError
    rtm = rthx_mod.meshes.cfg4(Ndim=9, n_bins=3)
    tr = rthx_mod.DeviceTracer(rthx_mod.flatten_domain(rtm), device=0)
    with pytest.raises(Err, match=r"\(1\).*no resident counts"):
        tr.trace_continue(R1, seed=3, bins=[2, 0])
    tr.trace(R1, seed=3, bins=[2, 0])                        # host output
    with pytest.raises(Err, match=r"\(1\).*host-output"):
        tr.trace_continue(R2)
    kw = dict(seed=3, bins=[2, 0], emitter_rank=1, emitter_world=2)
    (tr.trace_sparse(R1, **kw) if hashed else tr.trace(R1, dense=False, **kw))
    before = _readout(tr, 2, True)
    for bad, match in ((dict(seed=4), "seed"), (dict(nudge=1e-3), "nudge"), (dict(mode=RTHX_MULTI_BOUNCE), "mode"),
                       (dict(locator=RTHX_LOCATOR_GENERIC), "locator"), (dict(bins=[0, 2]), "bins"), (dict(bins=[2]), "bins"),
                       (dict(emitter_rank=0), "shard"), (dict(emitter_world=3), "shard"),
                       (dict(ray_id_offset=R1 + 1), r"ray_id_offset 701 does not continue .*\[0, 700\)"), (dict(ray_id_offset=0), "ray_id_offset")):
        with pytest.raises(Err, match=r"\(1\).*" + match):
            tr.trace_continue(R2, **bad)
        _assert_same(_readout(tr, 2, True), before)
    tr.trace_continue(R2)                                    # the range is still [0, R1)
    cont = _readout(tr, 2, True)
    tr.trace(R1 + R2, dense=False, **kw)
    _assert_same(cont, _readout(tr, 2, True))


@pytest.mark.gpu
def test_failed_hashed_continuation_keeps_the_resident_set(rthx_mod, cuda_lib, monkeypatch):
    tr = rthx_mod.DeviceTracer(rthx_mod.flatten_domain(rthx_mod.meshes.cfg1()), device=0)
    first = tr.trace_sparse(R1, seed=29)
    before = _readout(tr, 1, False)
    monkeypatch.setenv("RTHX_SPARSE_PAIR_CAP", "4")         # one emitter row overruns the pair buffer: RTHX_ERR_NOMEM before the merge
    with pytest.raises(rthx_mod.RthxError, match=r"\(3\).*pair buffer"):
        tr.trace_continue(R2)
    monkeypatch.delenv("RTHX_SPARSE_PAIR_CAP")
    _assert_same(_readout(tr, 1, False), before)
    cont = tr.trace_continue(R2)                             # the range is still [0, R1), its lost counters too
    ro = _readout(tr, 1, False)
    single = tr.trace(R1 + R2, seed=29, dense=False)
    _assert_same(ro, _readout(tr, 1, False))
    assert np.array_equal(cont["lost"], single["lost"]) and np.all(first["lost"] <= cont["lost"])


@pytest.mark.gpu
def test_continuing_a_multi_device_gather_is_rejected(rthx_mod, cuda_lib):
    from rthx._lib import create_multi, device_count, trace_multi
    if device_count() < 2:
        pytest.skip("needs two or more GPUs")
    trs = create_multi(rthx_mod.flatten_domain(rthx_mod.meshes.cfg1()), [0, 1])
    trace_multi(trs, R1, dense=False, seed=8)
    before = _readout(trs[0], 1, False)
    with pytest.raises(rthx_mod.RthxError, match=r"\(1\).*several devices"):
        trs[0].trace_continue(R2)
    _assert_same(_readout(trs[0], 1, False), before)


# ---- GPU: the public call -----------------------------------------------------------------------------------------------

def _public(rtm, N, monkeypatch, tiles, capsys, **kw):
    """F_raw / F_smooth of rtm(a N, seed) + rtm(b N, refine=True) and of rtm((a + b) N, seed)."""
    from rthx import tracing
    if tiles:
        monkeypatch.setattr(tracing, "auto_row_tiles", lambda n, nb, budget_bytes=48e9: tiles)
    a, b, seed = 600, 900, 97
    rtm(a * N, method="exchange", verbose=False, seed=seed, **kw)
    rtm(b * N, method="exchange", verbose=False, refine=True)
    assert f"Maximum ray tracing ray loss per emitter: {int(rtm.last_lost.max())}/{a + b}" in capsys.readouterr().out
    got = (rtm.F_raw, rtm.F_smooth, dict(rtm.last_trace_stats), rtm.last_smooth_stats["path"], rtm.last_lost.copy())
    rtm(a * N + b * N, method="exchange", verbose=False, seed=seed, **kw)
    ref = (rtm.F_raw, rtm.F_smooth, dict(rtm.last_trace_stats), rtm.last_smooth_stats["path"], rtm.last_lost.copy())
    assert got[2]["rays_per_emitter_total"] == ref[2]["rays_per_emitter_total"] == a + b
    assert got[2].get("tally") == ref[2].get("tally") and got[3] == ref[3]
    assert np.array_equal(got[4], ref[4])
    for x, y in ((got[0], ref[0]), (got[1], ref[1])):
        if sp.issparse(x):
            x, y = x.tocsc(), y.tocsc()
            x.sort_indices(); y.sort_indices()
            assert np.array_equal(x.indptr, y.indptr) and np.array_equal(x.indices, y.indices) and np.array_equal(x.data, y.data)
        else:
            assert np.array_equal(x, y)
    return got[2], got[3]


@pytest.mark.gpu
def test_public_refine_dense_branch(rthx_mod, cuda_lib, monkeypatch, capsys):
    rtm = rthx_mod.meshes.cfg1()
    stats, path = _public(rtm, rtm.num_elements, monkeypatch, None, capsys, devices=[0])
    assert path == "device_dense" and "tally" not in stats


@pytest.mark.gpu
def test_public_refine_sparse_branch(rthx_mod, cuda_lib, monkeypatch, capsys):
    rtm = rthx_mod.meshes.square_domain(15, kappa=40.0)
    stats, path = _public(rtm, rtm.num_elements, monkeypatch, None, capsys, devices=[0])
    assert path == "device_sparse" and "tally" not in stats


@pytest.mark.gpu
def test_public_refine_hashed_tally(rthx_mod, cuda_lib, monkeypatch, capsys):
    rtm = rthx_mod.meshes.square_domain(15, kappa=40.0)
    stats, path = _public(rtm, rtm.num_elements, monkeypatch, 2, capsys, devices=[0])
    assert stats["tally"] == "sparse" and path == "device_sparse"


@pytest.mark.gpu
def test_public_refine_hashed_tally_on_two_devices(rthx_mod, cuda_lib, monkeypatch, capsys):
    from rthx._lib import device_count
    if device_count() < 2:
        pytest.skip("needs two or more GPUs")
    rtm = rthx_mod.meshes.square_domain(15, kappa=40.0)
    stats, path = _public(rtm, rtm.num_elements, monkeypatch, 2, capsys, devices=[0, 1])
    assert stats["tally"] == "sparse" and stats["devices"] == 2


@pytest.mark.gpu
def test_public_refine_rejections_after_real_calls(rthx_mod, cuda_lib):
    rtm = rthx_mod.meshes.cfg1()
    N = rtm.num_elements
    rtm(N * 100, method="exchange", verbose=False, seed=5, devices=[0], row_tiles=2)
    with pytest.raises(ValueError, match="explicit row_tiles"):
        rtm(N * 100, method="exchange", verbose=False, refine=True)
    rtm(N * 100, method="exchange", verbose=False, seed=5, devices=[0])
    with pytest.raises(ValueError, match="seed=6 differs"):
        rtm(N * 100, method="exchange", verbose=False, refine=True, seed=6)
    rtm.fine_mesh[0][3].kappa_g = 7.0
    with pytest.raises(ValueError, match="flattened mesh differs"):
        rtm(N * 100, method="exchange", verbose=False, refine=True)
