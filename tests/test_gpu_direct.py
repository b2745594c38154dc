"""method=:direct on the device (rthx_trace_direct, DeviceTracer.trace_direct, rtm(...; method=:direct)): ray-for-ray parity with the
CPU oracle's re-emission, the reduction to MULTI_BOUNCE, the Crosbie & Schrenker table, agreement with :exchange + solveEquilibrium,
energy bookkeeping, determinism and the rejections that need a device.

The oracle and the device draw the same Philox words; a ray's outcome can differ only where a last-ulp difference of libm / FMA flips a
boundary decision, so the bar is that of test_gpu_parity.py (differing outcomes <= max(2, 2e-6 of the tallies), 2e-4 with the analytic
locator on multi-face meshes)."""
import ctypes as C

import numpy as np
import pytest

import direct_oracle

from helpers import n_differing_rays

pytestmark = pytest.mark.gpu

GENERIC = 1


def _dense(tr, R):
    row_ptr, cols, vals, _ = tr.counts_csr(values=True, normalised=False)
    out = np.zeros((R, tr.n_elements), np.uint64)
    for y in range(R):
        out[y, cols[row_ptr[y]:row_ptr[y + 1]]] = vals[row_ptr[y]:row_ptr[y + 1]]
    return out


def _reemit(rtm, flat, known_T):
    r = np.zeros(flat.n_elements, np.uint8)
    r[:len(known_T)] = ~known_T
    return r


def _square9():
    import rthx
    rtm = rthx.meshes.square_domain(9, kappa=0.6, sigma_s=0.9, epsilon=(0.3, 0.6, 0.9, 0.5))
    return rtm


def _cases():
    import rthx
    cfg1 = rthx.meshes.cfg1()
    cfg1.fine_mesh[0][10].T_in_w[1] = -1.0                          # right wall cell of the bottom row: known q = 0 (adiabatic)
    sq = _square9()
    sq.fine_mesh[0][8].T_in_w[1], sq.fine_mesh[0][8].q_in_w[1] = -1.0, 2.0e4       # a heated wall of known q
    circ = rthx.meshes.circle_domain(16, 5)
    circ.fine_mesh[15][-1].T_in_w[1] = -1.0
    quads = rthx.meshes.two_quads_domain(kappa=(0.5, 3.0))
    for c in quads.fine_mesh[1]:
        c.T_in_w = [-1.0 if c.solidWalls[w] else t for w, t in enumerate(c.T_in_w)]   # the right face's walls re-emit
    return [("cfg1", cfg1, {}, 2e-6), ("square9_diffuse", sq, {}, 2e-6), ("square9_specular", sq, dict(specular=True), 2e-6),
            ("circle", circ, {}, 2e-4), ("two_quads_variable_beta", quads, {}, 2e-4), ("square9_generic", sq, dict(locator=GENERIC), 2e-6)]


@pytest.mark.parametrize("case", range(6), ids=["cfg1", "square9_diffuse", "square9_specular", "circle", "two_quads_variable_beta",
                                                "square9_generic"])
def test_counts_match_the_oracle(rthx_mod, oracle_mod, cuda_lib, case):
    from rthx.direct import direct_sources
    name, rtm, kw, budget = _cases()[case]
    flat = rthx_mod.flatten_domain(rtm)
    ws, known_T, E, src, rays, w = direct_sources(rtm, 120_000)
    assert known_T.any() and not known_T.all()
    reemit = _reemit(rtm, flat, known_T)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    got = tr.trace_direct(src, rays, reemit, w, seed=21, **kw)
    ref = direct_oracle.trace_direct(flat, src, rays, reemit, seed=21, specular=kw.get("specular", False))
    counts = _dense(tr, len(src))
    total = int(ref["counts"].sum())
    nd = n_differing_rays(counts, ref["counts"])
    assert nd <= max(2, int(budget * total)), f"{name}: {nd} of {total} tallies differ from the oracle"
    assert np.abs(got["lost"].astype(np.int64) - ref["lost"].astype(np.int64)).sum() <= max(2, int(budget * total))
    # Abs is the fixed-order sum of the counts read out
    Abs = np.zeros(flat.n_elements)
    for y in range(len(src)):
        Abs = Abs + w[y] * counts[y].astype(np.float64)
    assert np.array_equal(got["absorbed"], Abs)
    assert got["stats"]["rays_traced"] == rays.sum() and got["events"] >= rays.sum()


@pytest.mark.parametrize("specular", [False, True])
def test_without_reemission_the_counts_are_the_multi_bounce_rows(rthx_mod, cuda_lib, specular):
    rtm = _square9()
    for c in rtm.fine_mesh[0]:
        c.T_in_g = 500.0                                              # every element at a known temperature
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    src = np.array([0, 5, 12, 35, 36, 50, 80, 100, 116], np.int32)
    rays = np.full(len(src), 30_000, np.int64)
    got = tr.trace_direct(src, rays, np.zeros(flat.n_elements, np.uint8), np.ones(len(src)), specular=specular, seed=77)
    counts = _dense(tr, len(src))
    ref = tr.trace_rows(src, 30_000, seed=77, mode=2 if specular else 1)
    assert np.array_equal(counts, ref["counts"][0])
    assert np.array_equal(got["lost"][src], ref["lost"][0][src])


def test_crosbie_schrenker_centre_line(rthx_mod, cuda_lib):
    """11 x 11, kappa = 1, black walls, bottom at 1000 K, gas of zero net emission, 1e7 bundles: S(tau) on the centre line against the
    table with the reference's norm-relative rtol = 0.05 (test_2d_grey.jl:216), no F, no smoothing, no solve."""
    from oracle import grey_solver as gs
    rtm = rthx_mod.meshes.cfg1()
    rtm(10_000_000, method="direct", verbose=False, seed=4)
    S = gs.centerline_source_function(rtm, 11, 1000.0)
    A = gs.analytical_centerline(11)
    assert np.linalg.norm(S - A) <= 0.05 * max(np.linalg.norm(S), np.linalg.norm(A))
    assert rtm.last_direct_stats["bundles"] == pytest.approx(1e7, rel=1e-4)


def test_direct_agrees_with_exchange_and_the_grey_solve(rthx_mod, cuda_lib):
    """test_2d_spectral.jl:263-283's comparison on the reflecting, scattering 9 x 9 square: per-cell |dT/T| < 5 %, and the fluxes of
    the known-temperature walls."""
    def walls(rtm):
        return np.array([rtm.fine_mesh[c - 1][f - 1].q_w[w - 1] for (c, f, w), s in sorted(rtm.surface_mapping.items(), key=lambda t: t[1])])
    ex = _square9()
    ex(20_000_000, method="exchange", verbose=False, seed=1)
    rthx_mod.solveEquilibrium(ex, ex.F_smooth, verbose=False)
    di = _square9()
    di(20_000_000, method="direct", verbose=False, seed=2)
    Te = np.array([c.T_g for c in ex.fine_mesh[0]])
    Td = np.array([c.T_g for c in di.fine_mesh[0]])
    assert np.abs(Td / Te - 1.0).max() < 0.05
    qe, qd = walls(ex), walls(di)
    assert np.abs(qd - qe).max() < 0.05 * np.abs(qe).max()


def test_isothermal_cavity_and_energy(rthx_mod, cuda_lib):
    rtm = rthx_mod.meshes.square_domain(11, kappa=1.0, T_walls=(1000.0, 1000.0, 1000.0, 1000.0))
    rtm(10_000_000, method="direct", verbose=False, seed=3)
    T = np.array([c.T_g for c in rtm.fine_mesh[0]])
    assert np.abs(T / 1000.0 - 1.0).max() < 0.02
    st = rtm.last_direct_stats
    E = sum(rtm.fine_mesh[c - 1][f - 1].e_w[w - 1] for (c, f, w) in rtm.surface_mapping)
    Abs_T = sum(rtm.fine_mesh[c - 1][f - 1].g_a_w[w - 1] for (c, f, w) in rtm.surface_mapping)
    assert rtm.energy_error == pytest.approx(st["lost_energy"], rel=1e-12, abs=1e-12 * E)
    assert Abs_T + st["lost_energy"] == pytest.approx(E, rel=1e-12)


def _fields(rtm):
    return (np.array([c.T_g for c in rtm.fine_mesh[0]]), np.array([c.q_g for c in rtm.fine_mesh[0]]),
            np.array([c.T_w for c in rtm.fine_mesh[0]]), np.array([c.q_w for c in rtm.fine_mesh[0]]), rtm.energy_error)


def test_same_seed_same_fields_across_calls_and_block_shapes(rthx_mod, cuda_lib):
    out = []
    for bt in (256, 256, 128):
        rtm = _square9()
        rtm.fine_mesh[0][8].T_in_w[1] = -1.0
        rtm(2_000_000, method="direct", verbose=False, seed=17, block_threads=bt)
        out.append(_fields(rtm))
    for o in out[1:]:
        for a, b in zip(o, out[0]):
            assert np.array_equal(a, b)


def test_two_devices_give_the_one_device_fields(rthx_mod, cuda_lib):
    if rthx_mod._lib.device_count() < 2:
        pytest.skip("needs two GPUs")
    out = []
    for devs in ([0], [0, 1]):
        rtm = _square9()
        rtm(2_000_000, method="direct", verbose=False, seed=17, devices=devs)
        assert rtm.last_direct_stats["devices"] == len(devs)
        out.append(_fields(rtm))
    for a, b in zip(out[0], out[1]):
        assert np.array_equal(a, b)


def test_c_abi_argument_errors_leave_the_resident_counts(rthx_mod, cuda_lib):
    from rthx import RthxError
    rtm = _square9()
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    N = flat.n_elements
    tr.trace_rows([0, 1, 2], 5000, dense=False, seed=1)
    before = tr.counts_csr()
    src, rays, re_, w = np.array([0, 4]), np.array([100, 100]), np.zeros(N, np.uint8), np.ones(2)
    bad = [(dict(sources=[4, 0]), "strictly ascending"), (dict(sources=[0, N]), "outside"), (dict(rays=[100, 0]), r"rays\[1\] = 0"),
           (dict(w=[1.0, -1.0]), r"bundle_energy\[1\]"), (dict(mode=0), "MULTI_BOUNCE"), (dict(bins=(0, 0)), "one bin"),
           (dict(rec_ids=[0]), "recording"), (dict(emitter_world=2), "emitter_rank")]
    for change, msg in bad:
        a = dict(sources=src, rays=rays, w=w)
        kw = {k: v for k, v in change.items() if k not in a}
        a.update({k: v for k, v in change.items() if k in a})
        if "mode" in kw:
            args, keep = rthx_mod.make_trace_args(0, mode=kw["mode"])
            s32, r64 = np.ascontiguousarray(a["sources"], np.int32), np.ascontiguousarray(a["rays"], np.int64)
            out = np.empty(N)
            rc = cuda_lib.rthx_trace_direct(tr._h, C.byref(args), s32.ctypes.data_as(C.POINTER(C.c_int32)), r64.ctypes.data_as(C.POINTER(C.c_int64)),
                                            2, re_.ctypes.data_as(C.POINTER(C.c_uint8)), np.asarray(w).ctypes.data_as(C.POINTER(C.c_double)),
                                            out.ctypes.data_as(C.POINTER(C.c_double)), None, None, None)
            assert rc == 1 and msg in cuda_lib.rthx_last_error(tr._h).decode()
            continue
        with pytest.raises(RthxError, match=msg):
            tr.trace_direct(a["sources"], a["rays"], re_, a["w"], **kw)
    after = tr.counts_csr()
    for x, y in zip(before, after):
        assert np.array_equal(x, y)


def test_continue_and_smoothing_refuse_direct_counts(rthx_mod, cuda_lib):
    from rthx import RthxError
    rtm = _square9()
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    N = flat.n_elements
    src = np.arange(N, dtype=np.int32)
    tr.trace_direct(src, np.full(N, 200), np.ones(N, np.uint8), np.ones(N), seed=5)
    assert tr.counts_csr()[0].shape == (N + 1,)
    with pytest.raises(RthxError, match="direct trace"):
        tr.trace_continue(100, seed=5, mode=1)
    with pytest.raises(RthxError, match="direct trace"):
        tr.smooth(np.ones(N), n=N)
    with pytest.raises(RthxError, match="direct trace"):
        tr.smooth_sparse(np.ones(N), n=N)
