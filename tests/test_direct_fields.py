"""method=:direct with the redirection tally, without a GPU: the CPU oracle's fields trace (rthx_oracle_trace_direct_fields) against
its plain trace, the segment identity, the expected ratio of redirections to absorptions, and the j / r / g / i write-back of
directRayTracing(all_fields=True) driven by a stand-in tracer with the device's interface."""
import numpy as np
import pytest

import direct_fields_oracle
import direct_oracle

SIGMA = 5.670374419e-8


def _fixed_order(w, counts):
    """sum_y w[y] counts[y] in ascending y, every product and sum rounded on its own (direct_absorbed_kernel)."""
    out = np.zeros(counts.shape[1])
    for y in range(counts.shape[0]):
        out = out + w[y] * counts[y].astype(np.float64)
    return out


class FieldsOracleTracer:
    """DeviceTracer.trace_direct(redirected=...) / counts_csr(bin=...) computed by the CPU oracle's fields trace."""

    def __init__(self, flat):
        self.flat, self.n_elements = flat, flat.n_elements
        self.blocks = ()

    def trace_direct(self, sources, rays, reemit, w, specular=False, redirected=False, seed=0, nudge=None, locator=0, block_threads=0):
        d = direct_fields_oracle.trace_direct_fields(self.flat, sources, rays, reemit, seed=seed, nudge=nudge, specular=specular)
        self.blocks = (d["counts"], d["redirected"]) if redirected else (d["counts"],)
        out = dict(absorbed=_fixed_order(w, d["counts"]), lost=d["lost"], events=d["segments"], stats=dict(kernel_ms=0.0))
        if redirected:
            out["redirected"] = _fixed_order(w, d["redirected"])
        return out

    def counts_csr(self, bin=0, values=True, normalised=False):
        import scipy.sparse as sp
        if bin >= len(self.blocks):
            raise RuntimeError("counts: no resident counts for that bin")
        c = sp.csr_matrix(self.blocks[bin])
        return c.indptr.astype(np.int64), c.indices.astype(np.int32), c.data.astype(np.uint64), None


@pytest.fixture
def on_fields_oracle(monkeypatch, rthx_mod):
    """Route directRayTracing's device handles to FieldsOracleTracer (one per requested device)."""
    def tracers_for(rtm, devices):
        flat = rthx_mod.flatten_domain(rtm)
        trs = [FieldsOracleTracer(flat) for _ in devices]
        rtm._devices, rtm._device = trs, trs[0]
        return trs
    monkeypatch.setattr(rthx_mod.tracing, "_tracers_for", tracers_for)


def _reflecting_square(rthx_mod):
    rtm = rthx_mod.meshes.square_domain(7, kappa=0.5, sigma_s=0.5, epsilon=(1.0, 0.6, 0.3, 0.6))
    rtm.fine_mesh[0][3].T_in_w[0] = -1.0                          # a bottom wall of known q = 0: re-emits
    return rtm


def _sources(rthx_mod, rtm, rays_tot):
    from rthx.direct import direct_sources
    flat = rthx_mod.flatten_domain(rtm)
    ws, known_T, E, src, rays, w = direct_sources(rtm, rays_tot)
    reemit = np.zeros(flat.n_elements, np.uint8)
    reemit[:len(known_T)] = ~known_T
    return flat, ws, src, rays, w, reemit


@pytest.mark.parametrize("specular", [False, True])
def test_fields_oracle_keeps_the_plain_counts(rthx_mod, specular):
    """The redirection tally draws nothing: absorption counts and lost are those of the plain trace, bit for bit."""
    rtm = _reflecting_square(rthx_mod)
    flat, ws, src, rays, w, reemit = _sources(rthx_mod, rtm, 40_000)
    assert reemit.any()
    plain = direct_oracle.trace_direct(flat, src, rays, reemit, seed=13, specular=specular)
    fields = direct_fields_oracle.trace_direct_fields(flat, src, rays, reemit, seed=13, specular=specular)
    assert np.array_equal(fields["counts"], plain["counts"])
    assert np.array_equal(fields["lost"], plain["lost"])
    assert fields["redirected"].sum() > 0


def test_black_walls_without_scattering_redirect_nothing(rthx_mod):
    rtm = rthx_mod.meshes.square_domain(6, kappa=0.8, T_walls=(1000.0, 400.0, 0.0, 0.0))
    flat, ws, src, rays, w, reemit = _sources(rthx_mod, rtm, 30_000)
    d = direct_fields_oracle.trace_direct_fields(flat, src, rays, reemit, seed=2)
    assert not d["redirected"].any()
    assert d["counts"].sum() > 0


@pytest.mark.parametrize("specular", [False, True])
def test_every_segment_ends_in_one_tally_or_loss(rthx_mod, specular):
    rtm = _reflecting_square(rthx_mod)
    flat, ws, src, rays, w, reemit = _sources(rthx_mod, rtm, 40_000)
    d = direct_fields_oracle.trace_direct_fields(flat, src, rays, reemit, seed=4, specular=specular)
    assert d["segments"] == int(d["counts"].sum()) + int(d["redirected"].sum()) + int(d["lost"].sum())
    assert d["segments"] > int(rays.sum())


def test_redirections_follow_the_reflectance_and_albedo(rthx_mod):
    """Every arrival at an element of redirection probability b (1 - eps at a wall, omega in the gas) is redirected with probability b:
    over the elements of equal b, sum(redirections) ~ b / (1 - b) sum(absorptions), within Monte Carlo noise."""
    from rthx.equilibrium import populateWorkspace
    rtm = _reflecting_square(rthx_mod)
    flat, ws, src, rays, w, reemit = _sources(rthx_mod, rtm, 200_000)
    d = direct_fields_oracle.trace_direct_fields(flat, src, rays, reemit, seed=8)
    ws = populateWorkspace(rtm, 1)
    b = np.concatenate([1.0 - ws["epsw"], ws["omega_g"]])
    n = len(b)
    absorbed = d["counts"].sum(axis=0)[:n].astype(np.float64)
    redirected = d["redirected"].sum(axis=0)[:n].astype(np.float64)
    groups = np.unique(np.round(b, 12))
    assert len(groups) >= 3
    for bg in groups:
        sel = np.isclose(b, bg, rtol=0, atol=1e-12)
        A, Rd = absorbed[sel].sum(), redirected[sel].sum()
        if bg == 0.0:
            assert Rd == 0
            continue
        arrivals = A + Rd
        assert arrivals > 1000
        # Rd ~ Binomial(arrivals, b): within 6 standard deviations of b * arrivals
        assert abs(Rd - bg * arrivals) <= 6.0 * np.sqrt(arrivals * bg * (1.0 - bg)), (bg, A, Rd)
        assert Rd / A == pytest.approx(bg / (1.0 - bg), rel=0.1)


def _cell_fields(rtm, names_w, names_g):
    ordered = sorted(rtm.surface_mapping.items(), key=lambda t: t[1])
    wall = np.array([[getattr(rtm.fine_mesh[c - 1][f - 1], a)[wl - 1] for a in names_w] for (c, f, wl), s in ordered])
    vols = sorted(rtm.volume_mapping.items(), key=lambda t: t[1])
    gas = np.array([[getattr(rtm.fine_mesh[c - 1][f - 1], a) for a in names_g] for (c, f), v in vols])
    return wall, gas


BASE_W, BASE_G = ("T_w", "e_w", "g_a_w", "q_w"), ("T_g", "e_g", "g_a_g", "q_g")
FIELDS_W, FIELDS_G = ("j_w", "r_w", "g_w", "i_w"), ("j_g", "r_g", "g_g", "i_g")
SENTINEL = -123.25


def _run(rthx_mod, devices, all_fields, sentinel=False):
    rtm = _reflecting_square(rthx_mod)
    if sentinel:
        for c in rtm.fine_mesh[0]:
            for a in FIELDS_W:
                setattr(c, a, [SENTINEL] * len(getattr(c, a)))
            for a in FIELDS_G:
                setattr(c, a, SENTINEL)
    rtm(60_000, method="direct", verbose=False, seed=9, devices=devices, all_fields=all_fields)
    return rtm


def test_all_fields_writes_the_grey_solve_split(rthx_mod, on_fields_oracle):
    """r = fixed-order power of the redirection counts, g = Abs + r, j = e + r, i_w = j / (pi A), i_g = j / (4 pi V)."""
    import math
    rtm = _run(rthx_mod, [0], True)
    flat, ws, src, rays, w, reemit = _sources(rthx_mod, rtm, 60_000)
    d = direct_fields_oracle.trace_direct_fields(flat, src, rays, reemit, seed=9)
    r = _fixed_order(w, d["redirected"])
    base_w, base_g = _cell_fields(rtm, BASE_W, BASE_G)
    f_w, f_g = _cell_fields(rtm, FIELDS_W, FIELDS_G)
    ns = rtm.num_surfaces
    assert np.array_equal(f_w[:, 1], r[:ns]) and np.array_equal(f_g[:, 1], r[ns:ns + len(f_g)])
    assert np.array_equal(f_w[:, 2], base_w[:, 2] + f_w[:, 1]) and np.array_equal(f_g[:, 2], base_g[:, 2] + f_g[:, 1])
    assert np.array_equal(f_w[:, 0], base_w[:, 1] + f_w[:, 1]) and np.array_equal(f_g[:, 0], base_g[:, 1] + f_g[:, 1])
    ordered = sorted(rtm.surface_mapping.items(), key=lambda t: t[1])
    area = np.array([rtm.fine_mesh[c - 1][f - 1].area[wl - 1] for (c, f, wl), s in ordered])
    assert np.array_equal(f_w[:, 3], np.array([j / (math.pi * a) for j, a in zip(f_w[:, 0], area)]))
    vol = np.array([rtm.fine_mesh[c - 1][f - 1].volume for (c, f), v in sorted(rtm.volume_mapping.items(), key=lambda t: t[1])])
    assert np.array_equal(f_g[:, 3], np.array([j / (4 * math.pi * v) for j, v in zip(f_g[:, 0], vol)]))
    assert (f_w[:, 1] > 0).any() and (f_g[:, 1] > 0).all()
    st = rtm.last_direct_stats
    assert st["redirections"] == int(d["redirected"].sum())
    assert st["events"] == st["redirections"] + int(d["counts"].sum()) + st["lost"]


def test_all_fields_leaves_the_temperature_fields_bit_for_bit(rthx_mod, on_fields_oracle):
    plain, fields = _run(rthx_mod, [0], False), _run(rthx_mod, [0], True)
    a_w, a_g = _cell_fields(plain, BASE_W, BASE_G)
    b_w, b_g = _cell_fields(fields, BASE_W, BASE_G)
    assert np.array_equal(a_w, b_w) and np.array_equal(a_g, b_g)
    assert plain.energy_error == fields.energy_error
    assert "redirections" not in plain.last_direct_stats


def test_without_all_fields_j_r_g_i_are_left_alone(rthx_mod, on_fields_oracle):
    rtm = _run(rthx_mod, [0], False, sentinel=True)
    f_w, f_g = _cell_fields(rtm, FIELDS_W, FIELDS_G)
    assert np.all(f_w == SENTINEL) and np.all(f_g == SENTINEL)
    rtm = _run(rthx_mod, [0], True, sentinel=True)
    f_w, f_g = _cell_fields(rtm, FIELDS_W, FIELDS_G)
    assert not np.any(f_w == SENTINEL) and not np.any(f_g == SENTINEL)


def test_several_devices_give_the_one_device_fields(rthx_mod, on_fields_oracle):
    names_w, names_g = BASE_W + FIELDS_W, BASE_G + FIELDS_G
    ref = _run(rthx_mod, [0], True)
    ref_w, ref_g = _cell_fields(ref, names_w, names_g)
    for devs in ([0, 1], [0, 1, 2]):
        rtm = _run(rthx_mod, devs, True)
        got_w, got_g = _cell_fields(rtm, names_w, names_g)
        assert np.array_equal(got_w, ref_w) and np.array_equal(got_g, ref_g)
        assert rtm.energy_error == ref.energy_error
        assert rtm.last_direct_stats["redirections"] == ref.last_direct_stats["redirections"]
        assert rtm.last_direct_stats["devices"] == len(devs)


def test_c_abi_rejects_a_missing_handle(cuda_lib):
    assert cuda_lib.rthx_trace_direct_fields(None, None, None, None, 0, None, None, None, None, None, None, None) == 1   # RTHX_ERR_ARG
