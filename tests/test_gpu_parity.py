"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same Philox stream.

Because both sides consume identical variates, tallies agree ray for ray except where last-ulp libm/FMA differences
flip a cell-boundary decision (expected <~1e-6 of rays; SURVEY.md App. A.3).  The bar used here: the number of
differing ray outcomes is <= max(2, 2e-6 * rays) for the reference-faithful generic locator and for single-face
meshes, and row sums are exact.  Multi-face meshes with the analytic locator additionally recover the (few) rays
the reference loses on grazing interface crossings (DESIGN.md, 'permitted deviations'); that budget is 2e-4.
"""
import numpy as np
import pytest

from helpers import n_differing_rays, z_statistics

pytestmark = pytest.mark.gpu

GENERIC = 1


def tracer(rthx_mod, cuda_lib, rtm):
    flat = rthx_mod.flatten_domain(rtm)
    return flat, rthx_mod.DeviceTracer(flat, device=0)


def check_exact(got, ref, rpe, budget_frac=2e-6):
    total = int(ref["counts"].sum())
    nd = n_differing_rays(got["counts"], ref["counts"])
    assert np.all(got["counts"].sum(axis=2) + got["lost"] == rpe), "tallied + lost != rays_per_emitter"
    assert nd <= max(2, int(budget_frac * total)), f"{nd} of {total} ray outcomes differ from the oracle"
    return nd


def test_cfg1_readme_example_full(rthx_mod, oracle_mod, cuda_lib):
    """Config 1 at full size: 11x11, 1e6 rays, recorder ids [10,20,30] like the README."""
    flat, tr = tracer(rthx_mod, cuda_lib, rthx_mod.meshes.cfg1())
    assert tr.info["n_affine_faces"] == 1 and tr.info["n_elements"] == 165
    rpe = 1_000_000 // 165
    ref = oracle_mod.trace(flat, rpe, rec_ids=[9, 19, 29])
    for loc in (0, GENERIC):
        got = tr.trace(rpe, rec_ids=[9, 19, 29], locator=loc)
        check_exact(got, ref, rpe)
        assert np.array_equal(got["lost"], ref["lost"])
        assert got["origins"].shape == ref["origins"].shape
        assert np.allclose(got["origins"], ref["origins"], rtol=0, atol=1e-13)
        assert np.allclose(got["endpoints"], ref["endpoints"], rtol=0, atol=1e-9)


def test_cfg2_reflecting_41(rthx_mod, oracle_mod, cuda_lib):
    flat, tr = tracer(rthx_mod, cuda_lib, rthx_mod.meshes.cfg2())
    rpe = 4000
    ref = oracle_mod.trace(flat, rpe, seed=2)
    check_exact(tr.trace(rpe, seed=2), ref, rpe)
    check_exact(tr.trace(rpe, seed=2, locator=GENERIC), ref, rpe)


def test_cfg3_scattering_101_sample(rthx_mod, oracle_mod, cuda_lib):
    """cfg3's full mesh (101 x 101, 10 605 elements), 5.3e7 rays ray for ray against the oracle (the full 1e10 rays would keep the
    CPU oracle busy for minutes; the full size is covered by the property tests below and by the Crosbie & Schrenker test)."""
    flat, tr = tracer(rthx_mod, cuda_lib, rthx_mod.meshes.cfg3())
    rpe = 5000
    ref = oracle_mod.trace(flat, rpe, seed=3)
    check_exact(tr.trace(rpe, seed=3), ref, rpe)


def test_cfg4_spectral_bands_batched(rthx_mod, oracle_mod, cuda_lib):
    """8 bands with per-band uniform beta, all traced in one launch (band = grid dimension)."""
    rtm = rthx_mod.meshes.cfg4(Ndim=21)
    assert rtm.spectral_mode == "spectral_variable"
    flat, tr = tracer(rthx_mod, cuda_lib, rtm)
    bins = list(range(8))
    rpe = 3000
    ref = oracle_mod.trace(flat, rpe, seed=4, bins=bins)
    got = tr.trace(rpe, seed=4, bins=bins)
    check_exact(got, ref, rpe)
    assert not np.array_equal(got["counts"][0], got["counts"][7])     # bands see different beta and streams
    sub = tr.trace(rpe, seed=4, bins=[5, 2])
    assert np.array_equal(sub["counts"][0], got["counts"][5]) and np.array_equal(sub["counts"][1], got["counts"][2])


def test_cfg5_circle_triangles(rthx_mod, oracle_mod, cuda_lib):
    """16 wedges with transparent spokes and triangle sub-meshes; crossings use the neighbour table (AUTO) or the
    reference's nudged point location (GENERIC)."""
    flat, tr = tracer(rthx_mod, cuda_lib, rthx_mod.meshes.cfg5())
    assert tr.info["n_affine_faces"] == 16 and tr.info["n_elements"] == 1232
    rpe = 8000
    ref = oracle_mod.trace(flat, rpe, seed=5)
    gen = tr.trace(rpe, seed=5, locator=GENERIC)
    check_exact(gen, ref, rpe)
    assert np.array_equal(gen["lost"], ref["lost"]) or n_differing_rays(gen["lost"], ref["lost"]) <= 2
    auto = tr.trace(rpe, seed=5)
    nd = check_exact(auto, ref, rpe, budget_frac=2e-4)
    assert auto["lost"].sum() <= ref["lost"].sum()                     # the analytic path never loses more rays


def test_rotated_and_rectangular_lattices(rthx_mod, oracle_mod, cuda_lib):
    import math
    for rtm in (rthx_mod.meshes.square_domain(9, rotation_angle=math.pi / 5),
                rthx_mod.meshes.square_domain(kappa=2.0, size=(3.0, 0.5), Ndiv=(12, 3)),
                rthx_mod.meshes.square_domain(kappa=0.0, Ndiv=(6, 4))):
        flat, tr = tracer(rthx_mod, cuda_lib, rtm)
        assert tr.info["n_affine_faces"] == 1
        ref = oracle_mod.trace(flat, 5000, seed=6)
        check_exact(tr.trace(5000, seed=6), ref, 5000)
        check_exact(tr.trace(5000, seed=6, locator=GENERIC), ref, 5000)


def test_single_division_quirk_loses_rays(rthx_mod, oracle_mod, cuda_lib):
    """meshQuad.jl:145-161: with Nx == 1 wall 2 is never solid, so hits on it are dropped (index -1) and counted."""
    rtm = rthx_mod.meshes.square_domain(kappa=0.1, Ndiv=(1, 2))
    flat, tr = tracer(rthx_mod, cuda_lib, rtm)
    ref = oracle_mod.trace(flat, 20000, seed=7)
    assert ref["lost"].sum() > 1000
    for loc in (0, GENERIC):
        got = tr.trace(20000, seed=7, locator=loc)
        check_exact(got, ref, 20000)
        assert n_differing_rays(got["lost"], ref["lost"]) <= 2


def test_variable_beta_across_faces(rthx_mod, oracle_mod, cuda_lib):
    """traceRayVariable (traceRay.jl:73-147): beta from the fine cell at each coarse entry point."""
    rtm = rthx_mod.meshes.two_quads_domain(kappa=(0.5, 3.0))
    flat, tr = tracer(rthx_mod, cuda_lib, rtm)
    assert tr.info["n_affine_faces"] == 2
    ref = oracle_mod.trace(flat, 20000, seed=8)
    check_exact(tr.trace(20000, seed=8, locator=GENERIC), ref, 20000)
    check_exact(tr.trace(20000, seed=8), ref, 20000, budget_frac=2e-4)


def test_non_parallelogram_quad_is_a_bilinear_lattice(rthx_mod, oracle_mod, cuda_lib):
    """A quadrilateral that is no parallelogram is meshed by meshQuad.jl:116-136 into the bilinear image of a uniform lattice:
    located by the analytic inverse of the bilinear map in the queue kernel (next to an affine neighbour), by grid +
    point-in-polygon under RTHX_LOCATOR_GENERIC and at block_threads=128, which the queue kernel does not take (lock-step
    general kernel)."""
    rtm = rthx_mod.meshes.two_quads_domain(kappa=(1.0, 1.0), skew=0.3)
    flat, tr = tracer(rthx_mod, cuda_lib, rtm)
    assert tr.info["n_affine_faces"] == 1 and tr.info["n_bilinear_faces"] == 1     # the skewed quad is not a parallelogram
    ref = oracle_mod.trace(flat, 20000, seed=9)
    check_exact(tr.trace(20000, seed=9, locator=GENERIC), ref, 20000)
    check_exact(tr.trace(20000, seed=9), ref, 20000, budget_frac=2e-4)
    check_exact(tr.trace(20000, seed=9, block_threads=128), ref, 20000, budget_frac=2e-4)


def test_bilinear_single_faces_trapezoid_and_general_quad(rthx_mod, oracle_mod, cuda_lib):
    """Single-face domains that are no parallelograms — a trapezoid (two parallel edges: the quadratic of the inverse map
    degenerates to a linear equation along one axis) and a general convex quadrilateral — with uniform and with cell-wise
    varying extinction and a recorder: the bilinear locator against the oracle's grid + point-in-polygon search."""
    shapes = {
        "trapezoid": [(0.0, 0.0), (2.0, 0.0), (1.5, 1.0), (0.5, 1.0)],
        "trapezoid-rotated": [(2.0, 0.0), (1.5, 1.0), (0.5, 1.0), (0.0, 0.0)],
        "general": [(0.0, 0.0), (2.0, 0.3), (2.3, 1.6), (-0.2, 1.1)],
    }
    for name, verts in shapes.items():
        for variable in (False, True):
            rtm = _square_from(verts, (7, 5), kappa=0.8)
            if variable:
                for i, cell in enumerate(rtm.fine_mesh[0]):
                    cell.kappa_g = 0.3 + 0.1 * (i % 9)
                rtm.refresh_spectral_flags()
                assert rtm.uniform_across_bin == [-1.0]
            flat, tr = tracer(rthx_mod, cuda_lib, rtm)
            assert tr.info["n_bilinear_faces"] == 1 and tr.info["n_affine_faces"] == 0, name
            rpe = 20000
            ids = [0, 7, flat.n_surfaces + 11]
            ref = oracle_mod.trace(flat, rpe, seed=47, rec_ids=ids)
            got = tr.trace(rpe, seed=47, rec_ids=ids)
            check_exact(got, ref, rpe, budget_frac=2e-5)
            assert got["stats"]["smem_bytes"] > 10000                    # the queue kernel (40 bytes of queue per ray), not the generic one
            check_exact(tr.trace(rpe, seed=47, locator=GENERIC), ref, rpe)
            if got["origins"].shape == ref["origins"].shape:
                assert np.allclose(got["origins"], ref["origins"], rtol=0, atol=1e-13)
                assert np.allclose(got["endpoints"], ref["endpoints"], rtol=0, atol=1e-9)


def test_determinism_across_launch_shapes_and_shards(rthx_mod, cuda_lib):
    flat, tr = tracer(rthx_mod, cuda_lib, rthx_mod.meshes.square_domain(15, kappa=1.0, sigma_s=1.0))
    rpe = 20000
    base = tr.trace(rpe, seed=10)
    for kw in (dict(block_threads=64), dict(block_threads=128, row_chunks=7), dict(row_chunks=1), dict(row_chunks=64)):
        assert np.array_equal(tr.trace(rpe, seed=10, **kw)["counts"], base["counts"])
    parts = sum(tr.trace(rpe, seed=10, emitter_rank=r, emitter_world=3)["counts"] for r in range(3))
    assert np.array_equal(parts, base["counts"])
    a = tr.trace(8000, seed=10)["counts"] + tr.trace(12000, seed=10, ray_id_offset=8000)["counts"]
    assert np.array_equal(a, base["counts"])
    assert not np.array_equal(tr.trace(rpe, seed=11)["counts"], base["counts"])


def test_statistical_parity_independent_streams(rthx_mod, oracle_mod, cuda_lib):
    """SURVEY.md App. D: different seeds on the two sides -> binomial z statistics, multiple-comparison aware."""
    import math
    flat, tr = tracer(rthx_mod, cuda_lib, rthx_mod.meshes.cfg1())
    rpe = 60_000
    got = tr.trace(rpe, seed=111)["counts"][0]
    ref = oracle_mod.trace(flat, rpe, seed=222)["counts"][0]
    zmax, frac3, M = z_statistics(got, ref)
    assert M > 5000
    assert frac3 < 0.004                                               # expected 0.27 %
    assert zmax < math.sqrt(2 * math.log(M)) + 1.5


def test_device_resident_entry_point(rthx_mod, cuda_lib):
    import torch
    flat, tr = tracer(rthx_mod, cuda_lib, rthx_mod.meshes.square_domain(9))
    N = tr.n_elements
    counts = torch.full((1, N, N), 7, dtype=torch.int64, device="cuda:0")
    lost = torch.full((1, N), 7, dtype=torch.int64, device="cuda:0")
    tr.trace_device(5000, counts.data_ptr(), lost.data_ptr(), stream=torch.cuda.current_stream().cuda_stream,
                    zero_first=True, seed=12)
    torch.cuda.synchronize()
    host = tr.trace(5000, seed=12)
    assert np.array_equal(counts.cpu().numpy().astype(np.uint64), host["counts"])
    assert int(lost.sum()) == int(host["lost"].sum())


def test_multi_handle_single_process(rthx_mod, cuda_lib):
    import torch
    from rthx._lib import trace_multi
    rtm = rthx_mod.meshes.cfg1()
    flat = rthx_mod.flatten_domain(rtm)
    n = min(2, torch.cuda.device_count())
    trs = [rthx_mod.DeviceTracer(flat, device=i) for i in range(n)] if n > 1 else \
        [rthx_mod.DeviceTracer(flat, device=0), rthx_mod.DeviceTracer(flat, device=0)]
    one = trs[0].trace(3000, seed=13, rec_ids=[9, 150])
    multi = trace_multi(trs, 3000, seed=13, rec_ids=[9, 150])
    assert np.array_equal(one["counts"], multi["counts"]) and np.array_equal(one["lost"], multi["lost"])
    assert np.array_equal(one["origins"], multi["origins"]) and np.array_equal(one["endpoints"], multi["endpoints"])
    res = trace_multi(trs, 3000, seed=13, dense=False)                      # rows gathered on trs[0]'s device, matrix stays resident
    row_ptr, cols, vals, _ = trs[0].counts_csr(0)
    import scipy.sparse as sp
    assert np.array_equal(sp.csr_matrix((vals, cols, row_ptr), shape=one["counts"][0].shape).toarray(), one["counts"][0])
    assert np.array_equal(res["lost"], one["lost"])


def test_full_size_properties_cfg3(rthx_mod, cuda_lib):
    """BASELINE size (101x101) at 2e9 rays: size-independent properties — exact row sums, reciprocity of the
    aggregated wall/gas blocks, symmetry of the square."""
    rtm = rthx_mod.meshes.cfg3()
    flat, tr = tracer(rthx_mod, cuda_lib, rtm)
    N, ns = tr.n_elements, flat.n_surfaces
    rpe = 2_000_000_000 // N
    out = tr.trace(rpe, seed=14)
    c = out["counts"][0]
    assert np.all(c.sum(axis=1) + out["lost"][0] == rpe)
    assert out["lost"].sum() == 0
    w = rthx_mod.get_w(rtm)
    F = c / float(rpe)
    # block reciprocity: sum_i in S w_i F_i->V  ==  sum_j in V w_j F_j->S  (exact identity, MC noise ~1e-4 relative)
    sv = (w[:ns, None] * F[:ns, ns:]).sum()
    vs = (w[ns:, None] * F[ns:, :ns]).sum()
    assert abs(sv - vs) / sv < 2e-3
    # four-fold symmetry: total wall->wall transport from each of the four sides agrees
    sides = {k: [] for k in (1, 2, 3, 4)}
    for (cc, f, wl), s in rtm.surface_mapping.items():
        sides[wl].append(s - 1)
    tot = [F[sides[k]][:, :ns].sum() for k in (1, 2, 3, 4)]
    assert max(tot) / min(tot) - 1 < 2e-3


def test_public_api_crosbie_schrenker(rthx_mod, cuda_lib):
    """mesh(N_rays; method=:exchange, rec) through the Python mirror, then the grey solve -> C&S table."""
    from oracle import grey_solver as gs
    rtm = rthx_mod.meshes.cfg1()
    rec = rthx_mod.RayRecorder([10, 20, 30])
    F_smooth = rtm(1_000_000, method="exchange", verbose=False, rec=rec, seed=99)
    assert F_smooth is rtm.F_smooth and rtm.F_raw.shape == (165, 165)
    o, e = rthx_mod.collect_rays(rec)
    assert o.shape == e.shape == (3 * 6060, 2)
    res = gs.solve_grey(rtm, rtm.F_smooth)
    S = gs.centerline_source_function(rtm, 11, 1000.0)
    A = gs.analytical_centerline(11)
    assert np.linalg.norm(S - A) <= 0.05 * max(np.linalg.norm(S), np.linalg.norm(A))
    assert abs(res["energy_error"]) < 1e-4


def test_global_tally_fallback_path(rthx_mod, oracle_mod, cuda_lib, monkeypatch):
    """N > ~57 k elements does not fit a u32 row histogram in 227 KB of shared memory: the kernel then tallies with
    direct global atomics.  Forced here on a small mesh (RTHX_FORCE_GLOBAL_TALLY) so the oracle can check it."""
    flat, tr = tracer(rthx_mod, cuda_lib, rthx_mod.meshes.cfg5())
    ref = oracle_mod.trace(flat, 3000, seed=31)
    monkeypatch.setenv("RTHX_FORCE_GLOBAL_TALLY", "1")
    for loc in (0, GENERIC):
        got = tr.trace(3000, seed=31, locator=loc)
        assert got["stats"]["hist_in_smem"] == 0
        check_exact(got, ref, 3000, budget_frac=2e-4)


def test_many_coarse_faces(rthx_mod, oracle_mod, cuda_lib):
    """150 wedges: 38 KB of coarse descriptors still ride in shared memory next to the ray queue (fewer resident blocks);
    600 wedges: more than the 96 KB staging limit, descriptors are read through L1/L2 and the kernel takes the non-FAST variant."""
    for n_wedges, rpe in ((150, 4000), (600, 300)):
        rtm = rthx_mod.meshes.circle_domain(n_wedges, 2, half_hot=False)
        flat, tr = tracer(rthx_mod, cuda_lib, rtm)
        assert tr.info["n_affine_faces"] == n_wedges
        ref = oracle_mod.trace(flat, rpe, seed=32)
        check_exact(tr.trace(rpe, seed=32, locator=GENERIC), ref, rpe)
        auto = tr.trace(rpe, seed=32)
        check_exact(auto, ref, rpe, budget_frac=5e-4)
        assert auto["lost"].sum() <= ref["lost"].sum()
        queue = auto["stats"]["smem_bytes"] > 256 * n_wedges + 10000       # descriptors + ray queue in shared memory
        assert queue == (n_wedges == 150)


def test_open_boundary_loses_rays_like_the_reference(rthx_mod, oracle_mod, cuda_lib):
    """A non-solid coarse edge with no neighbour: the reference's coarse point location fails and the ray is dropped."""
    rtm = rthx_mod.meshes.square_domain(6, kappa=0.3, solid=(True, False, True, True))
    flat, tr = tracer(rthx_mod, cuda_lib, rtm)
    ref = oracle_mod.trace(flat, 10000, seed=33)
    assert ref["lost"].sum() > 10000
    for loc in (0, GENERIC):
        got = tr.trace(10000, seed=33, locator=loc)
        check_exact(got, ref, 10000)
        assert n_differing_rays(got["lost"], ref["lost"]) <= 2


def test_edge_cases_empty_and_extreme_arguments(rthx_mod, oracle_mod, cuda_lib):
    flat, tr = tracer(rthx_mod, cuda_lib, rthx_mod.meshes.square_domain(4))
    N = tr.n_elements
    z = tr.trace(0, seed=1)                                            # no rays at all
    assert z["counts"].shape == (1, N, N) and z["counts"].sum() == 0 and z["lost"].sum() == 0
    one = tr.trace(1, seed=1)                                          # one ray per emitter
    assert np.all(one["counts"].sum(axis=2) + one["lost"] == 1)
    assert np.array_equal(one["counts"], oracle_mod.trace(flat, 1, seed=1)["counts"])
    big = 2 ** 40 + 12345                                              # ray ids beyond 32 bits, all-ones seed
    got = tr.trace(700, seed=2 ** 64 - 1, ray_id_offset=big)
    ref = oracle_mod.trace(flat, 700, seed=2 ** 64 - 1, ray_id_offset=big)
    assert np.array_equal(got["counts"], ref["counts"])
    rep = tr.trace(500, seed=3, bins=[0, 0, 0])                        # the same band three times: identical slabs
    assert np.array_equal(rep["counts"][0], rep["counts"][1]) and np.array_equal(rep["counts"][0], rep["counts"][2])
    with pytest.raises(rthx_mod.RthxError):
        tr.trace(10, bins=[1])                                         # band out of range
    with pytest.raises(rthx_mod.RthxError):
        tr.trace(10, emitter_rank=2, emitter_world=2)
    with pytest.raises(rthx_mod.RthxError):
        tr.trace(10, mode=7)
    more = tr.trace(50, emitter_rank=N + 3, emitter_world=N + 5)       # a shard that owns no emitter
    assert more["counts"].sum() == 0


def test_cellwise_variable_extinction_inside_one_face(rthx_mod, oracle_mod, cuda_lib):
    """User-edited per-cell kappa inside a single coarse face: uniform_across_bin = -1, so traceRayVariable runs and —
    faithful to traceRay.jl:87-103 — takes beta of the fine cell at the entry point for the whole coarse-face visit."""
    rtm = rthx_mod.meshes.square_domain(8, kappa=1.0)
    for f, cell in enumerate(rtm.fine_mesh[0]):
        cell.kappa_g = 0.2 + 0.15 * (f % 7)
    rtm.refresh_spectral_flags()
    assert rtm.uniform_across_bin == [-1.0]
    flat, tr = tracer(rthx_mod, cuda_lib, rtm)
    ref = oracle_mod.trace(flat, 15000, seed=21)
    check_exact(tr.trace(15000, seed=21), ref, 15000)
    check_exact(tr.trace(15000, seed=21, locator=GENERIC), ref, 15000)
    # rows of cells with different kappa really differ in their self-absorption
    c = ref["counts"][0]
    ns = flat.n_surfaces
    self_abs = np.array([c[ns + f, ns + f] for f in range(64)]) / 15000.0
    assert self_abs[6] > 1.5 * self_abs[0]


def test_recorder_on_spectral_bin(rthx_mod, oracle_mod, cuda_lib):
    """RayRecorder(ids; bin): only rays of that band are recorded (parallelRayTracing.jl:108)."""
    rtm = rthx_mod.meshes.cfg4(Ndim=9, n_bins=3)
    flat, tr = tracer(rthx_mod, cuda_lib, rtm)
    got = tr.trace(400, seed=22, bins=[0, 1, 2], rec_ids=[5, 40], rec_bin=1)
    ref = oracle_mod.trace(flat, 400, seed=22, bins=[0, 1, 2], rec_ids=[5, 40], rec_bin=1)
    assert got["origins"].shape == ref["origins"].shape == (800, 2)
    assert np.allclose(got["origins"], ref["origins"], atol=1e-13) and np.allclose(got["endpoints"], ref["endpoints"], atol=1e-9)
    none = tr.trace(400, seed=22, bins=[0, 2], rec_ids=[5, 40], rec_bin=1)   # the recorded band is not traced
    assert none["origins"].shape == (0, 2)


def test_statistical_parity_cfg2_full_size(rthx_mod, oracle_mod, cuda_lib):
    """Config 2 at its BASELINE size (41x41, 1e8 rays) with INDEPENDENT Philox streams on the two sides: the App. D
    statistic over all entries with enough counts (multiple-comparison aware; a literal 'every entry within 3 sigma'
    is unattainable on 3.4e6 entries)."""
    import math
    flat, tr = tracer(rthx_mod, cuda_lib, rthx_mod.meshes.cfg2())
    rpe = 100_000_000 // tr.n_elements
    got = tr.trace(rpe, seed=1001)["counts"][0]
    ref = oracle_mod.trace(flat, rpe, seed=2002)["counts"][0]
    zmax, frac3, M = z_statistics(got, ref)
    assert M > 500_000
    assert frac3 < 0.004 and zmax < math.sqrt(2 * math.log(M)) + 1.5
    # per-row chi-square of the tallies against the pooled distribution: p-values must not pile up near zero
    cg, co = got.astype(np.float64), ref.astype(np.float64)
    pooled = (cg + co) / 2
    keep = pooled >= 20
    chi2 = np.where(keep, (cg - co) ** 2 / np.maximum(cg + co, 1), 0).sum(axis=1)
    dof = keep.sum(axis=1)
    zrow = (chi2 - dof) / np.sqrt(2 * np.maximum(dof, 1))
    assert np.abs(zrow).max() < 6 and abs(zrow.mean()) < 0.2


def test_full_size_cfg3_reproduces_crosbie_schrenker(rthx_mod, cuda_lib):
    """The north-star acceptance at the NAMED configuration: 101x101 grey absorbing+scattering enclosure (kappa =
    sigma_s = 0.5, tau = 1), 1e10 rays through the public call (trace + CSR read-out + device-side smoothing), then the
    grey equilibrium solve -> centre-line S(tau) against the Crosbie & Schrenker (1984) table of test_2d_grey.jl:25-33.
    In radiative equilibrium the scattering albedo drops out, so the table for tau = 1 applies."""
    from oracle import grey_solver as gs
    rtm = rthx_mod.meshes.cfg3()
    rtm(10_000_000_000, method="exchange", verbose=False, seed=0x5EED0001)
    st = rtm.last_trace_stats
    assert st["rays_traced"] == 942951 * 10605 and st["rays_lost"] <= 10
    assert isinstance(rtm.F_smooth, np.ndarray) and rtm.F_smooth.shape == (10605, 10605)      # dense branch, on the device
    assert rtm.last_smooth_stats["delta"] < 1e-14
    res = gs.solve_grey(rtm, rtm.F_smooth)
    S = gs.centerline_source_function(rtm, 101, 1000.0)
    A = gs.analytical_centerline(101)
    rel = np.linalg.norm(S - A) / max(np.linalg.norm(S), np.linalg.norm(A))
    assert rel <= 0.05                                            # the reference's own tolerance (test_2d_grey.jl:216)
    assert rel <= 0.01 and np.abs(S - A).max() < 0.01             # what 1e10 rays on 101x101 actually deliver
    assert abs(res["energy_error"]) < 1e-4


def _square_from(verts, Ndiv, kappa=1.0, n_bins=1, kappa_cells=None):
    from rthx import PolyVolume2D, RayTracingDomain2D
    face = PolyVolume2D(list(verts), (True, True, True, True), n_bins, kappa, 0.0)
    face.epsilon = [1.0] * 4
    face.T_in_w = [1000.0, 0.0, 0.0, 0.0]
    face.T_in_g = -1.0
    face.q_in_g = 0.0
    return RayTracingDomain2D([face], [Ndiv])


def test_sq_axis_aligned_loop_is_bit_identical_to_the_general_loop(rthx_mod, oracle_mod, cuda_lib, monkeypatch):
    """The single-quad kernel drops the four dot products of distToSurface2D / the lattice inverse when the face is an
    axis-aligned rectangle (n0 = (0, +-1), n1 = (+-1, 0)).  Every product it drops is an exact zero, so the tallies must be
    bit-identical to the general loop (RTHX_NO_AXIS=1) — for the usual vertex order and for one starting at the far corner
    (both normals flipped) — and both agree with the oracle.  Vertex orders starting on a vertical edge are not
    axis-specialised and run the general loop."""
    orders = {
        "bottom-left": [(0.0, 0.0), (2.0, 0.0), (2.0, 1.0), (0.0, 1.0)],
        "top-right": [(2.0, 1.0), (0.0, 1.0), (0.0, 0.0), (2.0, 0.0)],
        "bottom-right": [(2.0, 0.0), (2.0, 1.0), (0.0, 1.0), (0.0, 0.0)],
    }
    for name, verts in orders.items():
        rtm = _square_from(verts, (7, 5), kappa=1.3)
        flat, tr = tracer(rthx_mod, cuda_lib, rtm)
        assert tr.info["n_affine_faces"] == 1
        rpe = 20000
        ref = oracle_mod.trace(flat, rpe, seed=41, rec_ids=[3, 40])
        monkeypatch.delenv("RTHX_NO_AXIS", raising=False)
        a = tr.trace(rpe, seed=41, rec_ids=[3, 40])
        monkeypatch.setenv("RTHX_NO_AXIS", "1")
        g = tr.trace(rpe, seed=41, rec_ids=[3, 40])
        monkeypatch.delenv("RTHX_NO_AXIS", raising=False)
        assert np.array_equal(a["counts"], g["counts"]) and np.array_equal(a["lost"], g["lost"]), name
        assert np.array_equal(a["endpoints"], g["endpoints"]), name
        check_exact(a, ref, rpe)
        assert np.allclose(a["origins"], ref["origins"], rtol=0, atol=1e-13)
        assert np.allclose(a["endpoints"], ref["endpoints"], rtol=0, atol=1e-9)


def test_queue_kernel_mixed_quad_and_triangle_faces_with_recorder(rthx_mod, oracle_mod, cuda_lib):
    """Multi-face FAST mesh with BOTH face kinds (a rectangle with a triangular roof across a transparent interface), cell-wise
    different kappa (variable-beta path) and recorded rays: exercises dist_face for parallelograms and triangles, the absorber
    table for quad lattices, mirrored-triangle lattices (quad and diagonal cells) and the recorder slots of the queue kernel."""
    from rthx import PolyVolume2D, RayTracingDomain2D
    for kappas in ((1.0, 1.0), (0.4, 2.5)):
        box = PolyVolume2D([(0.0, 0.0), (2.0, 0.0), (2.0, 1.0), (0.0, 1.0)], (True, True, False, True), 1, kappas[0], 0.0)
        roof = PolyVolume2D([(0.0, 1.0), (2.0, 1.0), (1.0, 2.0)], (False, True, True), 1, kappas[1], 0.0)
        for f, n in ((box, 4), (roof, 3)):
            f.epsilon = [1.0] * n
            f.T_in_w = [0.0] * n
            f.T_in_g = -1.0
            f.q_in_g = 0.0
        rtm = RayTracingDomain2D([box, roof], [(6, 4), (5, 5)])
        flat, tr = tracer(rthx_mod, cuda_lib, rtm)
        assert tr.info["n_affine_faces"] == 2
        rpe = 20000
        ids = [0, 5, flat.n_surfaces + 3, flat.n_elements - 1]
        ref = oracle_mod.trace(flat, rpe, seed=43, rec_ids=ids)
        got = tr.trace(rpe, seed=43, rec_ids=ids)
        check_exact(got, ref, rpe, budget_frac=2e-4)
        check_exact(tr.trace(rpe, seed=43, locator=GENERIC), ref, rpe)
        assert got["origins"].shape == ref["origins"].shape or abs(len(got["origins"]) - len(ref["origins"])) <= 8
        if got["origins"].shape == ref["origins"].shape:
            assert np.allclose(got["origins"], ref["origins"], rtol=0, atol=1e-13)
            assert np.allclose(got["endpoints"], ref["endpoints"], rtol=0, atol=1e-9)


def test_t_junction_interfaces_keep_the_analytic_fine_locator(rthx_mod, oracle_mod, cuda_lib):
    """One tall face next to two stacked faces: the tall face's open edge has no unique neighbour (a T-junction), so the next
    coarse face is found by the reference's own point location after the advance (traceRay.jl:56-65) — in the general variant
    of the queue kernel, which keeps the analytic lattice inverse for every fine-cell lookup."""
    from rthx import PolyVolume2D, RayTracingDomain2D
    left = PolyVolume2D([(0.0, 0.0), (1.0, 0.0), (1.0, 2.0), (0.0, 2.0)], (True, False, True, True), 1, 0.7, 0.0)
    lower = PolyVolume2D([(1.0, 0.0), (2.0, 0.0), (2.0, 1.0), (1.0, 1.0)], (True, True, False, False), 1, 1.4, 0.0)
    upper = PolyVolume2D([(1.0, 1.0), (2.0, 1.0), (2.0, 2.0), (1.0, 2.0)], (False, True, True, False), 1, 0.2, 0.0)
    for f in (left, lower, upper):
        f.epsilon = [1.0] * 4
        f.T_in_w = [0.0] * 4
        f.T_in_g = -1.0
        f.q_in_g = 0.0
    rtm = RayTracingDomain2D([left, lower, upper], [(3, 6), (4, 4), (5, 3)])
    flat, tr = tracer(rthx_mod, cuda_lib, rtm)
    assert tr.info["n_affine_faces"] == 3 and tr.info["n_bilinear_faces"] == 0
    rpe = 20000
    ref = oracle_mod.trace(flat, rpe, seed=53)
    got = tr.trace(rpe, seed=53)
    check_exact(got, ref, rpe, budget_frac=2e-4)
    assert got["stats"]["smem_bytes"] > 10000                            # queue kernel
    check_exact(tr.trace(rpe, seed=53, locator=GENERIC), ref, rpe)
    # rays do cross the T-junction in both directions
    ns = flat.n_surfaces
    n_left = 18
    c = got["counts"][0]
    assert c[ns:ns + n_left, ns + n_left:].sum() > 1000 and c[ns + n_left:, ns:ns + n_left].sum() > 1000


def test_host_output_pipeline_batches_do_not_change_the_result(rthx_mod, cuda_lib, monkeypatch):
    """rthx_trace_exchange cuts the owned rows into row batches (two compute streams + a copy stream; the last four batches are
    a quarter of the others): counts, lost and recorded rays are identical for 1, 7 (even split), 8 and 16 (tapered) batches,
    for a pinned and a pageable host matrix, single bin and several bins, and for a sharded call (rows of one rank only)."""
    import torch
    rtm = rthx_mod.meshes.square_domain(15, kappa=1.0, sigma_s=0.5, n_bins=3, kappa_bins=[0.5, 1.0, 2.0])
    flat, tr = tracer(rthx_mod, cuda_lib, rtm)
    rpe, ids = 3000, [4, 100]
    N = flat.n_elements
    for bins in ([0], [2, 0, 1]):
        monkeypatch.setenv("RTHX_BATCHES", "1")
        base = tr.trace(rpe, seed=61, bins=bins, rec_ids=ids, rec_bin=bins[0])
        for nb in ("7", "8", "16"):
            monkeypatch.setenv("RTHX_BATCHES", nb)
            got = tr.trace(rpe, seed=61, bins=bins, rec_ids=ids, rec_bin=bins[0])
            assert np.array_equal(got["counts"], base["counts"]) and np.array_equal(got["lost"], base["lost"]), (bins, nb)
            assert np.array_equal(got["endpoints"], base["endpoints"])
            pinned = torch.empty((len(bins), N, N), dtype=torch.int64).pin_memory().numpy().view(np.uint64)
            got = tr.trace(rpe, seed=61, bins=bins, counts_out=pinned)
            assert np.array_equal(got["counts"], base["counts"]), (bins, nb, "pinned")
            part = tr.trace(rpe, seed=61, bins=bins, emitter_rank=1, emitter_world=3)
            assert np.array_equal(part["counts"][:, 1::3], base["counts"][:, 1::3]) and part["counts"][:, 0::3].sum() == 0
    monkeypatch.delenv("RTHX_BATCHES")
