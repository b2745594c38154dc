"""method=:direct without a GPU: the source allocation, the rejections, the CPU oracle's re-emission, and the write-back of
directRayTracing driven by the oracle in place of the device (a stand-in tracer with the device's interface)."""
import re
import shutil
import subprocess

import numpy as np
import pytest

import direct_oracle

SIGMA = 5.670374419e-8


class OracleTracer:
    """DeviceTracer.trace_direct / counts_csr computed by the CPU oracle (tests/native/direct_oracle.c); Abs summed like direct_absorbed_kernel (ascending rows, every
    product and sum rounded on its own)."""

    def __init__(self, flat):
        self.flat, self.n_elements = flat, flat.n_elements

    def trace_direct(self, sources, rays, reemit, w, specular=False, seed=0, nudge=None, locator=0, block_threads=0):
        d = direct_oracle.trace_direct(self.flat, sources, rays, reemit, seed=seed, nudge=nudge, specular=specular)
        self.counts = d["counts"]
        absorbed = np.zeros(self.n_elements)
        for y in range(len(sources)):
            absorbed = absorbed + w[y] * self.counts[y].astype(np.float64)
        return dict(absorbed=absorbed, lost=d["lost"], events=0, stats=dict(kernel_ms=0.0))

    def counts_csr(self, values=True, normalised=False):
        import scipy.sparse as sp
        c = sp.csr_matrix(self.counts)
        return c.indptr.astype(np.int64), c.indices.astype(np.int32), c.data.astype(np.uint64), None


@pytest.fixture
def on_oracle(monkeypatch, rthx_mod):
    """Route directRayTracing's device handles to OracleTracer (one per requested device)."""
    def tracers_for(rtm, devices):
        flat = rthx_mod.flatten_domain(rtm)
        trs = [OracleTracer(flat) for _ in devices]
        rtm._devices, rtm._device = trs, trs[0]
        return trs
    monkeypatch.setattr(rthx_mod.tracing, "_tracers_for", tracers_for)


def _fields(rtm):
    T = np.array([c.T_g for c in rtm.fine_mesh[0]])
    wall = [(c.T_w[w], c.e_w[w], c.g_a_w[w], c.q_w[w]) for (cc, f, w), s in sorted(rtm.surface_mapping.items(), key=lambda t: t[1])
            for c in [rtm.fine_mesh[cc - 1][f - 1]] for w in [w - 1]]
    return T, np.array(wall)


def test_sources_follow_the_emissive_powers(rthx_mod):
    from rthx.direct import direct_sources
    rtm = rthx_mod.meshes.square_domain(5, kappa=0.5, T_walls=(1000.0, 500.0, 0.0, 0.0))
    cell = rtm.fine_mesh[0][12]
    cell.T_in_g, cell.q_in_g = -1.0, 3.0e4                           # one gas cell with a known net emission
    ws, known_T, E, sources, rays, w = direct_sources(rtm, 100_000)
    ns = rtm.num_surfaces
    assert known_T[:ns].all() and not known_T[ns:].any()
    assert np.allclose(E[:ns], SIGMA * ws["Area"] * ws["Tw"] ** 4)
    assert np.isclose(E[:ns], SIGMA * 0.2 * 1000.0 ** 4).sum() == 5 and np.isclose(E[:ns], SIGMA * 0.2 * 500.0 ** 4).sum() == 5
    assert E[ns + 12] == 3.0e4 and np.count_nonzero(E[ns:]) == 1
    assert list(sources) == list(np.flatnonzero(E > 0))
    assert np.array_equal(rays, np.maximum(1, np.rint(100_000 * E[sources] / E.sum())).astype(np.int64))
    assert np.allclose(w * rays, E[sources], rtol=1e-15)


def test_negative_q_and_no_source_are_rejected(rthx_mod):
    rtm = rthx_mod.meshes.square_domain(4, kappa=0.5)
    rtm.fine_mesh[0][3].q_in_g = -5.0
    with pytest.raises(ValueError, match=r"volume 4 \(element 19\) has q_in = -5.0 < 0"):
        rtm(10_000, method="direct", verbose=False, devices=[0])
    rtm = rthx_mod.meshes.square_domain(4, kappa=0.5, T_walls=(0.0, 0.0, 0.0, 0.0))
    with pytest.raises(ValueError, match="no element has energy to emit"):
        rtm(10_000, method=":direct", verbose=False, devices=[0])


def test_spectral_domains_and_recorders_are_rejected(rthx_mod):
    rtm = rthx_mod.meshes.square_domain(4, n_bins=3, kappa_bins=[1.0, 1.5, 2.0])
    with pytest.raises(NotImplementedError, match="spectral direct solver"):
        rtm(10_000, method="direct", verbose=False)
    rtm = rthx_mod.meshes.square_domain(4)
    with pytest.raises(ValueError, match="does not record rays"):
        rtm(10_000, method="direct", verbose=False, rec=rthx_mod.RayRecorder([1]))


def test_c_abi_rejects_a_missing_handle(cuda_lib):
    assert cuda_lib.rthx_trace_direct(None, None, None, None, 0, None, None, None, None, None, None) == 1      # RTHX_ERR_ARG


@pytest.mark.parametrize("specular", [False, True])
def test_oracle_without_reemission_is_the_multi_bounce_trace(rthx_mod, oracle_mod, specular):
    """No re-emitting element: the direct counts of each source are its MULTI_BOUNCE row, bit for bit (same Philox calls)."""
    rtm = rthx_mod.meshes.square_domain(9, kappa=0.6, sigma_s=0.9, epsilon=(0.3, 0.6, 0.9, 0.5))
    flat = rthx_mod.flatten_domain(rtm)
    src = np.array([0, 3, 17, 36, 50, 80], np.int32)
    d = direct_oracle.trace_direct(flat, src, [700] * len(src), np.zeros(flat.n_elements, np.uint8), seed=11, specular=specular)
    m = oracle_mod.trace(flat, 700, seed=11, mode=2 if specular else 1)
    assert np.array_equal(d["counts"], m["counts"][0][src])
    assert np.array_equal(d["lost"][src], m["lost"][0][src])


def test_oracle_reemission_keeps_every_bundle_until_a_known_temperature_absorbs_it(rthx_mod, oracle_mod):
    """Each bundle is tallied once at a known-T element or lost; absorptions at re-emitting elements come on top."""
    rtm = rthx_mod.meshes.square_domain(7, kappa=1.0, sigma_s=0.5, epsilon=(1.0, 0.5, 0.5, 0.5))
    flat = rthx_mod.flatten_domain(rtm)
    ns = rtm.num_surfaces
    reemit = np.zeros(flat.n_elements, np.uint8)
    reemit[ns:] = 1
    src = np.arange(7, dtype=np.int32)
    d = direct_oracle.trace_direct(flat, src, [2000] * 7, reemit, seed=3)
    final = d["counts"][:, :ns].sum(axis=1) + d["lost"][src]
    assert np.all(final == 2000)
    assert d["counts"][:, ns:].sum() > 14000                      # kappa = 1 gas: most bundles are re-emitted several times


def test_isothermal_cavity_and_energy_balance(rthx_mod, on_oracle):
    """Black walls at 1000 K around a gas of zero net emission: the gas comes to 1000 K; energy_error is the lost energy."""
    rtm = rthx_mod.meshes.square_domain(5, kappa=1.0, T_walls=(1000.0, 1000.0, 1000.0, 1000.0))
    rtm(400_000, method="direct", verbose=False, seed=5, devices=[0])
    T, wall = _fields(rtm)
    assert np.abs(T / 1000.0 - 1.0).max() < 0.03
    st = rtm.last_direct_stats
    assert rtm.energy_error == pytest.approx(st["lost_energy"], rel=1e-12, abs=1e-9 * wall[:, 1].sum())
    # every known-T wall: q = E - Abs; sum over the known-T elements of Abs plus the lost energy is the emitted energy
    assert np.allclose(wall[:, 1] - wall[:, 2], wall[:, 3], rtol=0, atol=1e-9 * wall[:, 1].max())
    assert wall[:, 2].sum() + st["lost_energy"] == pytest.approx(wall[:, 1].sum(), rel=1e-12)
    assert np.all(wall[:, 0] == 1000.0)


def test_several_devices_give_the_one_device_result(rthx_mod, on_oracle):
    """Contiguous source blocks per device, integer counts merged before the one fixed-order sum: identical fields."""
    out = []
    for devs in ([0], [0, 1], [0, 1, 2]):
        rtm = rthx_mod.meshes.square_domain(6, kappa=0.6, sigma_s=0.3, epsilon=(1.0, 0.6, 0.6, 0.6))
        rtm.fine_mesh[0][0].T_in_w[0] = -1.0                      # a bottom wall of known q = 0 that re-emits
        rtm(60_000, method="direct", verbose=False, seed=9, devices=devs)
        out.append(_fields(rtm) + (rtm.energy_error,))
    for o in out[1:]:
        assert np.array_equal(o[0], out[0][0]) and np.array_equal(o[1], out[0][1]) and o[2] == out[0][2]


@pytest.mark.skipif(shutil.which("cuobjdump") is None or shutil.which("c++filt") is None, reason="needs cuobjdump and c++filt")
def test_direct_kernels_keep_every_value_in_registers(cuda_lib, rthx_mod):
    """The four trace_direct_kernel instances (histogram / global tally x analytic / generic locator) have no stack frame, so nothing
    spills to local memory, inside the ray loop or anywhere else, at the 2 resident blocks of 256 threads their bounds ask for."""
    out = subprocess.run(["cuobjdump", "--dump-resource-usage", rthx_mod.build_library()], capture_output=True, text=True, check=True).stdout
    names = re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", out)
    dem = subprocess.run(["c++filt"], input="\n".join(n for n, _, _ in names), capture_output=True, text=True, check=True).stdout.splitlines()
    usage = {d.split("(")[0]: (int(r), int(s)) for d, (_, r, s) in zip(dem, names)}
    direct = {k: v for k, v in usage.items() if "trace_direct_kernel<" in k}
    assert sorted(direct) == sorted(f"void rthx::trace_direct_kernel<{h}, {f}>" for h in ("true", "false") for f in ("true", "false"))
    for name, (regs, stack) in direct.items():
        assert regs <= 128 and stack == 0, (name, regs, stack)
