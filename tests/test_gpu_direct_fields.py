"""method=:direct with the redirection tally on the device (rthx_trace_direct_fields, DeviceTracer.trace_direct(redirected=True),
rtm(...; method=:direct, all_fields=True)): parity of the redirection counts with the CPU oracle, identity with the plain trace, the
exact sums, launch-shape independence, agreement of j / g / r with :exchange + solveEquilibrium, determinism and the C ABI."""
import ctypes as C

import numpy as np
import pytest

import direct_fields_oracle
from helpers import n_differing_rays
from test_gpu_direct import _cases, _square9

pytestmark = pytest.mark.gpu

CASE_IDS = ["cfg1", "square9_diffuse", "square9_specular", "circle", "two_quads_variable_beta", "square9_generic"]
REFLECTING = {"square9_diffuse", "square9_specular", "square9_generic"}   # the others have black walls and no scattering: nothing redirects


def _dense(tr, R, bin=0):
    row_ptr, cols, vals, _ = tr.counts_csr(bin=bin, values=True, normalised=False)
    out = np.zeros((R, tr.n_elements), np.uint64)
    for y in range(R):
        out[y, cols[row_ptr[y]:row_ptr[y + 1]]] = vals[row_ptr[y]:row_ptr[y + 1]]
    return out


def _fixed_order(w, counts):
    out = np.zeros(counts.shape[1])
    for y in range(counts.shape[0]):
        out = out + w[y] * counts[y].astype(np.float64)
    return out


def _setup(rthx_mod, rtm, rays_tot):
    from rthx.direct import direct_sources
    flat = rthx_mod.flatten_domain(rtm)
    ws, known_T, E, src, rays, w = direct_sources(rtm, rays_tot)
    reemit = np.zeros(flat.n_elements, np.uint8)
    reemit[:len(known_T)] = ~known_T
    return flat, src, rays, w, reemit


@pytest.mark.parametrize("case", range(6), ids=CASE_IDS)
def test_redirection_counts_match_the_oracle(rthx_mod, cuda_lib, case):
    """Block 1 against rthx_oracle_trace_direct_fields.  A bundle whose outcome flips on a last-ulp difference moves its absorption and
    its redirection tallies alike, so the redirection budget is the differing-ray budget of test_gpu_direct.py times the tallies a
    bundle carries (segments per bundle, rounded up)."""
    name, rtm, kw, budget = _cases()[case]
    flat, src, rays, w, reemit = _setup(rthx_mod, rtm, 120_000)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    got = tr.trace_direct(src, rays, reemit, w, seed=21, redirected=True, **kw)
    ref = direct_fields_oracle.trace_direct_fields(flat, src, rays, reemit, seed=21, specular=kw.get("specular", False))
    R = len(src)
    c0, c1 = _dense(tr, R, 0), _dense(tr, R, 1)
    rays_budget = max(2, int(budget * int(ref["counts"].sum())))
    per_bundle = -(-ref["segments"] // int(rays.sum()))
    nd0, nd1 = n_differing_rays(c0, ref["counts"]), n_differing_rays(c1, ref["redirected"])
    total1 = int(ref["redirected"].sum())
    assert (total1 > 0) == (name in REFLECTING)
    assert nd0 <= rays_budget, f"{name}: {nd0} absorption tallies differ from the oracle"
    assert nd1 <= rays_budget * per_bundle, f"{name}: {nd1} of {total1} redirection tallies differ from the oracle"
    assert abs(got["events"] - ref["segments"]) <= rays_budget * per_bundle


@pytest.mark.parametrize("case", [1, 2, 3, 5], ids=[CASE_IDS[i] for i in (1, 2, 3, 5)])
def test_fields_trace_keeps_the_plain_trace(rthx_mod, cuda_lib, case):
    """Same arguments with and without the tally: identical absorption counts, absorbed, lost and events; exact sums and the segment
    identity on the fields trace."""
    name, rtm, kw, budget = _cases()[case]
    flat, src, rays, w, reemit = _setup(rthx_mod, rtm, 200_000)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    R = len(src)
    plain = tr.trace_direct(src, rays, reemit, w, seed=5, **kw)
    c_plain = _dense(tr, R, 0)
    fields = tr.trace_direct(src, rays, reemit, w, seed=5, redirected=True, **kw)
    c0, c1 = _dense(tr, R, 0), _dense(tr, R, 1)
    assert np.array_equal(c0, c_plain)
    assert np.array_equal(fields["absorbed"], plain["absorbed"])
    assert np.array_equal(fields["lost"], plain["lost"])
    assert fields["events"] == plain["events"]
    assert np.array_equal(fields["redirected"], _fixed_order(w, c1))
    assert fields["events"] == int(c0.sum()) + int(c1.sum()) + int(fields["lost"].sum())
    assert (c1.sum() > 0) == (name in REFLECTING)


def test_redirection_counts_do_not_depend_on_the_launch_shape(rthx_mod, cuda_lib, monkeypatch):
    rtm = _square9()
    rtm.fine_mesh[0][8].T_in_w[1] = -1.0
    flat, src, rays, w, reemit = _setup(rthx_mod, rtm, 400_000)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    R = len(src)
    ref = tr.trace_direct(src, rays, reemit, w, seed=33, redirected=True)
    c_ref = (_dense(tr, R, 0), _dense(tr, R, 1))
    shapes = [dict(block_threads=128), dict(block_threads=256, row_chunks=3), dict(row_chunks=7), dict(global_tally=True),
              dict(global_tally=True, block_threads=128, row_chunks=5)]
    for shape in shapes:
        kw = dict(shape)
        if kw.pop("global_tally", False):
            monkeypatch.setenv("RTHX_FORCE_GLOBAL_TALLY", "1")
        else:
            monkeypatch.delenv("RTHX_FORCE_GLOBAL_TALLY", raising=False)
        got = tr.trace_direct(src, rays, reemit, w, seed=33, redirected=True, **kw)
        assert np.array_equal(_dense(tr, R, 0), c_ref[0]), shape
        assert np.array_equal(_dense(tr, R, 1), c_ref[1]), shape
        for k in ("absorbed", "redirected", "lost"):
            assert np.array_equal(got[k], ref[k]), (shape, k)
        assert got["events"] == ref["events"], shape


def _walls(rtm, name):
    return np.array([getattr(rtm.fine_mesh[c - 1][f - 1], name)[w - 1] for (c, f, w), s in sorted(rtm.surface_mapping.items(), key=lambda t: t[1])])


def _gas(rtm, name):
    return np.array([getattr(c, name) for c in rtm.fine_mesh[0]])


def test_j_g_r_agree_with_exchange_and_the_grey_solve(rthx_mod, cuda_lib):
    """The reflecting, scattering 9 x 9 square: per-element j, g and r within 5 % of each field's maximum (walls and gas)."""
    ex = _square9()
    ex(20_000_000, method="exchange", verbose=False, seed=1)
    rthx_mod.solveEquilibrium(ex, ex.F_smooth, verbose=False)
    di = _square9()
    di(20_000_000, method="direct", verbose=False, seed=2, all_fields=True)
    for get, names in ((_walls, ("j_w", "g_w", "r_w")), (_gas, ("j_g", "g_g", "r_g"))):
        for name in names:
            a, b = get(ex, name), get(di, name)
            assert np.abs(b - a).max() < 0.05 * np.abs(a).max(), (name, np.abs(b - a).max(), np.abs(a).max())
    assert di.last_direct_stats["redirections"] > 0


def test_pure_scatterer_irradiation_agrees_with_exchange(rthx_mod, cuda_lib):
    """kappa = 0, sigma_s > 0, one hot black wall: the gas absorbs nothing (Abs = 0), its irradiation g is all redirected power."""
    def dom():
        return rthx_mod.meshes.square_domain(9, kappa=0.0, sigma_s=1.0, T_walls=(1000.0, 0.0, 0.0, 0.0))
    ex = dom()
    ex(20_000_000, method="exchange", verbose=False, seed=1)
    rthx_mod.solveEquilibrium(ex, ex.F_smooth, verbose=False)
    di = dom()
    di(20_000_000, method="direct", verbose=False, seed=2, all_fields=True)
    assert np.all(_gas(di, "g_a_g") == 0.0)
    a, b = _gas(ex, "g_g"), _gas(di, "g_g")
    assert a.max() > 0
    assert np.abs(b - a).max() < 0.05 * np.abs(a).max(), (np.abs(b - a).max(), a.max())
    assert np.array_equal(_gas(di, "g_g"), _gas(di, "r_g"))


def test_black_walls_without_scattering_redirect_nothing(rthx_mod, cuda_lib):
    rtm = rthx_mod.meshes.square_domain(9, kappa=0.6)
    rtm(2_000_000, method="direct", verbose=False, seed=3, all_fields=True)
    for get, (r, j, e, g, a) in ((_walls, ("r_w", "j_w", "e_w", "g_w", "g_a_w")), (_gas, ("r_g", "j_g", "e_g", "g_g", "g_a_g"))):
        assert np.all(get(rtm, r) == 0.0)
        assert np.array_equal(get(rtm, j), get(rtm, e)) and np.array_equal(get(rtm, g), get(rtm, a))
    assert rtm.last_direct_stats["redirections"] == 0


FIELDS = ("T_w", "e_w", "g_a_w", "q_w", "j_w", "r_w", "g_w", "i_w", "T_g", "e_g", "g_a_g", "q_g", "j_g", "r_g", "g_g", "i_g")


def _all_fields(rtm):
    return [np.array([getattr(c, f) for c in rtm.fine_mesh[0]]) for f in FIELDS] + [rtm.energy_error]


def test_same_seed_same_fields_across_calls_and_block_shapes(rthx_mod, cuda_lib):
    out = []
    for bt in (256, 256, 128):
        rtm = _square9()
        rtm.fine_mesh[0][8].T_in_w[1] = -1.0
        rtm(2_000_000, method="direct", verbose=False, seed=17, block_threads=bt, all_fields=True)
        out.append(_all_fields(rtm))
    for o in out[1:]:
        for a, b in zip(o, out[0]):
            assert np.array_equal(a, b)


def test_two_devices_give_the_one_device_fields(rthx_mod, cuda_lib):
    if rthx_mod._lib.device_count() < 2:
        pytest.skip("needs two GPUs")
    out = []
    for devs in ([0], [0, 1]):
        rtm = _square9()
        rtm(2_000_000, method="direct", verbose=False, seed=17, devices=devs, all_fields=True)
        assert rtm.last_direct_stats["devices"] == len(devs)
        out.append(_all_fields(rtm) + [rtm.last_direct_stats["redirections"]])
    for a, b in zip(out[0], out[1]):
        assert np.array_equal(a, b)


def _call_fields(cuda_lib, tr, args, src, rays, re_, w, red=True):
    s32, r64 = np.ascontiguousarray(src, np.int32), np.ascontiguousarray(rays, np.int64)
    w64 = np.ascontiguousarray(w, np.float64)
    N = tr.n_elements
    absorbed, redirected = np.empty(N), np.empty(N)
    return cuda_lib.rthx_trace_direct_fields(tr._h, C.byref(args), s32.ctypes.data_as(C.POINTER(C.c_int32)), r64.ctypes.data_as(C.POINTER(C.c_int64)),
                                             len(s32), re_.ctypes.data_as(C.POINTER(C.c_uint8)), w64.ctypes.data_as(C.POINTER(C.c_double)),
                                             absorbed.ctypes.data_as(C.POINTER(C.c_double)),
                                             redirected.ctypes.data_as(C.POINTER(C.c_double)) if red else None, None, None, None)


def test_c_abi_argument_errors_leave_the_resident_counts(rthx_mod, cuda_lib):
    from rthx import RthxError
    rtm = _square9()
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    N = flat.n_elements
    tr.trace_rows([0, 1, 2], 5000, dense=False, seed=1)
    before = tr.counts_csr()
    src, rays, re_, w = np.array([0, 4]), np.array([100, 100]), np.zeros(N, np.uint8), np.ones(2)
    args, keep = rthx_mod.make_trace_args(0, mode=1)
    assert _call_fields(cuda_lib, tr, args, src, rays, re_, w, red=False) == 1
    assert "redirected_out" in cuda_lib.rthx_last_error(tr._h).decode()
    args, keep = rthx_mod.make_trace_args(0, mode=0)
    assert _call_fields(cuda_lib, tr, args, src, rays, re_, w) == 1
    assert "MULTI_BOUNCE" in cuda_lib.rthx_last_error(tr._h).decode()
    bad = [(dict(sources=[4, 0]), "strictly ascending"), (dict(sources=[0, N]), "outside"), (dict(rays=[100, 0]), r"rays\[1\] = 0"),
           (dict(w=[1.0, -1.0]), r"bundle_energy\[1\]"), (dict(bins=(0, 0)), "one bin"), (dict(rec_ids=[0]), "recording"),
           (dict(emitter_world=2), "emitter_rank")]
    for change, msg in bad:
        a = dict(sources=src, rays=rays, w=w)
        kw = {k: v for k, v in change.items() if k not in a}
        a.update({k: v for k, v in change.items() if k in a})
        with pytest.raises(RthxError, match="trace_direct_fields: .*" + msg):
            tr.trace_direct(a["sources"], a["rays"], re_, a["w"], redirected=True, **kw)
        after = tr.counts_csr()
        for x, y in zip(before, after):
            assert np.array_equal(x, y)


def test_redirection_bin_only_after_a_fields_trace(rthx_mod, cuda_lib):
    from rthx import RthxError
    rtm = _square9()
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    N = flat.n_elements
    src = np.arange(N, dtype=np.int32)
    tr.trace_direct(src, np.full(N, 200), np.ones(N, np.uint8), np.ones(N), seed=5)
    with pytest.raises(RthxError, match="no resident counts for that bin"):
        tr.counts_csr(bin=1)
    out = tr.trace_direct(src, np.full(N, 200), np.ones(N, np.uint8), np.ones(N), seed=5, redirected=True)
    row_ptr, cols, vals, _ = tr.counts_csr(bin=1, values=True, normalised=False)
    assert row_ptr.shape == (N + 1,) and int(vals.sum()) > 0
    assert tr.counts_stats(bin=1)[0] == len(cols)
    colptr, rowval, cvals, _ = tr.counts_csc(bin=1, values=True, normalised=False)
    assert int(cvals.sum()) == int(vals.sum())
    assert np.array_equal(out["redirected"], _fixed_order(np.ones(N), _dense(tr, N, 1)))
    with pytest.raises(RthxError, match="no resident counts for that bin"):
        tr.counts_csr(bin=2)
    with pytest.raises(RthxError, match="direct trace"):
        tr.trace_continue(100, seed=5, mode=1)
    with pytest.raises(RthxError, match="direct trace"):
        tr.smooth(np.ones(N), n=N)
    with pytest.raises(RthxError, match="direct trace"):
        tr.smooth_sparse(np.ones(N), n=N)


def test_counts_that_cannot_fit_are_refused_before_anything_resident_changes(rthx_mod, cuda_lib):
    """square_domain(400), every element a source: the two count blocks would take 16 N^2 bytes (about 418 GB)."""
    from rthx import RthxError
    rtm = rthx_mod.meshes.square_domain(400, kappa=40.0)
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    N = flat.n_elements
    tr.trace_rows([0, 1, 2], 50, dense=False, seed=1)
    before = tr.counts_csr()
    with pytest.raises(RthxError, match=r"\(3\).*trace_direct_fields: .*" + str(16 * N * N) + " bytes.*do not fit in device memory"):
        tr.trace_direct(np.arange(N, dtype=np.int32), np.ones(N, np.int64), np.ones(N, np.uint8), np.ones(N), seed=2, redirected=True)
    after = tr.counts_csr()
    for x, y in zip(before, after):
        assert np.array_equal(x, y)
