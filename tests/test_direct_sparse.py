"""method=:direct on the hashed row tally, without a GPU: which route directRayTracing takes for a block of sources (dense counts when
their 8 R N bytes per count block fit the budget of one device, the hashed tally otherwise), and that the write-back does not depend on
the route.  A stand-in tracer with the device's interface (the CPU oracle's fields trace) records the route it was asked for; its
counts are the same on both routes, as the device's are.  The codegen check of the new kernel instances needs only cuobjdump."""
import re
import shutil
import subprocess

import numpy as np
import pytest

from test_direct_fields import FieldsOracleTracer


class RouteTracer(FieldsOracleTracer):
    """FieldsOracleTracer that accepts trace_direct(sparse=...) and records, per call, (sources, sparse, redirected)."""
    calls = []

    def trace_direct(self, sources, rays, reemit, w, sparse=False, redirected=False, **kw):
        RouteTracer.calls.append((len(sources), sparse, redirected))
        out = super().trace_direct(sources, rays, reemit, w, redirected=redirected, **kw)
        if sparse:
            out["sparse_stats"] = dict(pairs=0, nnz=0, flushes=0, row_groups=1)
        return out


@pytest.fixture
def on_route_tracer(monkeypatch, rthx_mod):
    def tracers_for(rtm, devices):
        flat = rthx_mod.flatten_domain(rtm)
        trs = [RouteTracer(flat) for _ in devices]
        rtm._devices, rtm._device = trs, trs[0]
        return trs
    monkeypatch.setattr(rthx_mod.tracing, "_tracers_for", tracers_for)
    RouteTracer.calls = []
    return RouteTracer.calls


def _budget(monkeypatch, rthx_mod, budget):
    """Set the one-device budget of rows_fit_one_device to `budget` bytes (its estimate: 8 bytes per row, column and count block)."""
    monkeypatch.setattr(rthx_mod.tracing, "rows_fit_one_device", lambda r, n, b, budget_bytes=48e9: 8.0 * r * n * b <= budget)


def _domain(rthx_mod):
    rtm = rthx_mod.meshes.square_domain(6, kappa=0.6, sigma_s=0.3, epsilon=(1.0, 0.6, 0.6, 0.6))
    rtm.fine_mesh[0][0].T_in_w[0] = -1.0                          # a bottom wall of known q = 0 that re-emits
    return rtm


def _state(rtm):
    cells = rtm.fine_mesh[0]
    gas = np.array([(c.T_g, c.e_g, c.g_a_g, c.q_g, c.j_g, c.r_g, c.g_g, c.i_g) for c in cells])
    wall = np.array([(c.T_w[w], c.e_w[w], c.g_a_w[w], c.q_w[w], c.j_w[w], c.r_w[w], c.g_w[w], c.i_w[w])
                     for (cc, f, w1), s in sorted(rtm.surface_mapping.items(), key=lambda t: t[1])
                     for c in [rtm.fine_mesh[cc - 1][f - 1]] for w in [w1 - 1]])
    return gas, wall, rtm.energy_error


def _sources(rthx_mod, rays_tot):
    from rthx.direct import direct_sources
    rtm = _domain(rthx_mod)
    *_, src, rays, w = direct_sources(rtm, rays_tot)
    return len(src), rthx_mod.flatten_domain(rtm).n_elements


@pytest.mark.parametrize("all_fields", [False, True])
def test_hashed_exactly_when_the_dense_counts_pass_the_budget(rthx_mod, monkeypatch, on_route_tracer, all_fields):
    R, N = _sources(rthx_mod, 20_000)
    blocks = 2 if all_fields else 1
    need = 8 * R * N * blocks
    for budget, sparse in ((need, False), (need - 1, True), (10 * need, False)):
        _budget(monkeypatch, rthx_mod, budget)
        on_route_tracer.clear()
        rtm = _domain(rthx_mod)
        rtm(20_000, method="direct", verbose=False, seed=3, devices=[0], all_fields=all_fields)
        assert on_route_tracer == [(R, sparse, all_fields)]
        assert rtm.last_direct_stats["tally"] == ("sparse" if sparse else "dense")


def test_all_fields_doubles_the_estimate(rthx_mod, monkeypatch, on_route_tracer):
    R, N = _sources(rthx_mod, 20_000)
    _budget(monkeypatch, rthx_mod, 8 * R * N * 1.5)               # one count block fits, two do not
    for all_fields, sparse in ((False, False), (True, True)):
        on_route_tracer.clear()
        _domain(rthx_mod)(20_000, method="direct", verbose=False, seed=3, devices=[0], all_fields=all_fields)
        assert on_route_tracer == [(R, sparse, all_fields)]


def test_the_route_is_chosen_per_device_block(rthx_mod, monkeypatch, on_route_tracer):
    R, N = _sources(rthx_mod, 20_000)
    blocks = [len(b) for b in np.array_split(np.arange(R), 2)]
    _budget(monkeypatch, rthx_mod, 8 * max(blocks) * N)             # each half fits, the whole list would not
    rtm = _domain(rthx_mod)
    rtm(20_000, method="direct", verbose=False, seed=3, devices=[0, 1])
    assert sorted(on_route_tracer) == sorted((b, False, False) for b in blocks)
    assert rtm.last_direct_stats["tally"] == "dense"
    on_route_tracer.clear()
    _budget(monkeypatch, rthx_mod, 8 * min(blocks) * N - 1)
    rtm = _domain(rthx_mod)
    rtm(20_000, method="direct", verbose=False, seed=3, devices=[0, 1])
    assert sorted(on_route_tracer) == sorted((b, True, False) for b in blocks)
    assert rtm.last_direct_stats["tally"] == "sparse"


@pytest.mark.parametrize("devices", [[0], [0, 1]])
def test_either_route_writes_back_the_same_fields(rthx_mod, monkeypatch, on_route_tracer, devices):
    out = []
    for budget in (48e9, 0.0):
        _budget(monkeypatch, rthx_mod, budget)
        rtm = _domain(rthx_mod)
        rtm(20_000, method="direct", verbose=False, seed=3, devices=devices, all_fields=True)
        out.append(_state(rtm))
    assert {s for _, s, _ in on_route_tracer} == {False, True}
    for a, b in zip(out[0], out[1]):
        assert np.array_equal(a, b)


@pytest.mark.skipif(shutil.which("cuobjdump") is None or shutil.which("c++filt") is None, reason="needs cuobjdump and c++filt")
def test_direct_hash_kernels_keep_every_value_in_registers(cuda_lib, rthx_mod):
    """The two trace_direct_hash_kernel instances (analytic / generic locator) have no stack frame and fit the 128 registers of 2
    resident blocks of 256 threads."""
    out = subprocess.run(["cuobjdump", "--dump-resource-usage", rthx_mod.build_library()], capture_output=True, text=True, check=True).stdout
    names = re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", out)
    dem = subprocess.run(["c++filt"], input="\n".join(n for n, _, _ in names), capture_output=True, text=True, check=True).stdout.splitlines()
    usage = {d.split("(")[0]: (int(r), int(s)) for d, (_, r, s) in zip(dem, names)}
    direct = {k: v for k, v in usage.items() if "trace_direct_hash_kernel<" in k}
    assert sorted(direct) == sorted(f"void rthx::trace_direct_hash_kernel<{f}>" for f in ("true", "false"))
    for name, (regs, stack) in direct.items():
        assert regs <= 128 and stack == 0, (name, regs, stack)
