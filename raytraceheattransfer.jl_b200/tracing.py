"""Host-side mirror of the reference's exchange-factor driver, with the emitter loop replaced by the CUDA library.

  dispatch_ray_trace         functor, RT2D/Shared2D/multiDispatchRayTrace2D.jl:1-18
  exchangeRayTracing         RT2D/ExchangeFactors2D/exchangeRayTracing.jl:1-74
  parallelRayTracing         RT2D/ExchangeFactors2D/parallelRayTracing.jl:1-62
  computeExchangeFactorsBin  RT2D/ExchangeFactors2D/parallelRayTracing.jl:64-159 (+ row_normalize! :161-169)
  group_uniform_bins         RT2D/ExchangeFactors2D/parallelRayTracing.jl:171-191
  get_w / get_b              HeatTransfer/exchangeFactorSmoothing/smoothExchangeFactors.jl:320-375

(RT2D = src/RayTracing/RayTracing2D.)  All bands that need a trace are batched into ONE device launch; the
per-band `SparseMatrixCSC` of the reference becomes a `scipy.sparse.csc_matrix`.  New optional keywords that
the reference does not have: `seed` (its RNG is unseeded), `device`, `locator`.
"""
from __future__ import annotations

import secrets
from typing import List, Optional, Sequence, Tuple

import numpy as np
import scipy.sparse as sp

from .flatten import flatten_domain
from ._lib import DeviceTracer, DEFAULT_NUDGE
from ._abi import RTHX_LOCATOR_AUTO


def _isapprox(a: float, b: float, atol: float, rtol: float) -> bool:
    return abs(a - b) <= max(atol, rtol * max(abs(a), abs(b)))


def group_uniform_bins(uniform_across_bin: Sequence[float], atol: float = 1e-8, rtol: float = 1e-8):
    """parallelRayTracing.jl:171-191.  Returns (groups, reps, nonuniform) with 1-based bin indices."""
    groups: List[List[int]] = []
    reps: List[float] = []
    nonuniform: List[int] = []
    for i, v in enumerate(uniform_across_bin, start=1):
        if v < -0.1:
            nonuniform.append(i)
            continue
        idx = next((k for k, r in enumerate(reps) if _isapprox(r, v, atol, rtol)), None)
        if idx is None:
            reps.append(v)
            groups.append([i])
        else:
            groups[idx].append(i)
    return groups, reps, nonuniform


def counts_to_F(counts: np.ndarray, rays_per_emitter: int, verbose_loss: bool = True) -> sp.csc_matrix:
    """Integer tallies -> row-normalised sparse F, composing parallelRayTracing.jl:144-146 (value c/rays) with
    row_normalize! (:161-169): F[i,j] = (c_ij/R) / sum_j(c_ij/R); zero tallies are not stored; the loss line
    is printed unconditionally like the reference (:163)."""
    c = sp.csr_matrix(counts)            # drops zeros
    inv_rays = 1.0 / rays_per_emitter if rays_per_emitter else 0.0
    vals = c.data.astype(np.float64) * inv_rays
    F = sp.csr_matrix((vals, c.indices, c.indptr), shape=c.shape)
    rs = np.asarray(F.sum(axis=1)).ravel()
    if verbose_loss:
        max_loss = int(round(rays_per_emitter * float(np.max(np.abs(1.0 - rs))))) if len(rs) else 0
        print(f"Maximum ray tracing ray loss per emitter: {max_loss}/{rays_per_emitter}")
    with np.errstate(divide="ignore", invalid="ignore"):
        F.data /= np.repeat(rs, np.diff(F.indptr))
    return F.tocsc()


def resolve_devices(devices, device: int, rays_total: int) -> List[int]:
    """The `devices` keyword of the functor (new; SURVEY.md section 5): an int, a list of device ids, or None = every visible
    B200 — capped so that each device still traces >= 2e8 rays (about 2 ms of work; below that the fixed per-device cost of a
    multi-GPU trace exceeds what the extra device saves).  `device` is the single-GPU spelling kept from round 1."""
    if devices is None:
        from ._lib import device_count
        n_use = max(1, min(device_count(), int(rays_total // 200_000_000)))
        return [int(device)] if n_use == 1 else list(range(n_use))
    if isinstance(devices, int):
        return [devices]
    devs = [int(d) for d in devices]
    if not devs or len(set(devs)) != len(devs):
        raise ValueError("devices must be a non-empty list of distinct device ids")
    return devs


def _tracers_for(rtm, devices: Sequence[int]):
    """Re-flatten on every call (user code mutates properties between construction and tracing) and create the device
    handles — one per device, from one host-side preparation; the handles of the previous call are dropped."""
    import time
    t0 = time.perf_counter()
    flat = flatten_domain(rtm)
    t1 = time.perf_counter()
    for old in getattr(rtm, "_devices", None) or ([rtm._device] if getattr(rtm, "_device", None) is not None else []):
        old.close()
    if len(devices) == 1:
        trs = [DeviceTracer(flat, device=devices[0])]
    else:
        from ._lib import create_multi
        trs = create_multi(flat, devices)
    rtm._devices = trs
    rtm._device = trs[0]          # the handle that holds the resident counts / F_smooth afterwards
    rtm.last_phase_ms = {"flatten": 1e3 * (t1 - t0), "create": 1e3 * (time.perf_counter() - t1)}
    return trs


def auto_row_tiles(n_elements: int, n_bins: int, budget_bytes: float = 48e9) -> int:
    """Row tiles needed to keep the resident UInt64 counts (8 N^2 bytes per traced bin) within `budget_bytes` of device memory."""
    return max(1, int(np.ceil(8.0 * n_elements * n_elements * n_bins / budget_bytes)))


def _same_flat(a, b) -> bool:
    keys = [k for k in a.__dict__ if k != "c"]
    return keys == [k for k in b.__dict__ if k != "c"] and all(np.array_equal(np.asarray(a.__dict__[k]), np.asarray(b.__dict__[k])) for k in keys)


def _refine_state(rtm, seed, devices, locator, row_tiles, nudge):
    """The state of the previous call that `refine=True` continues; ValueError when it cannot be continued with these keywords."""
    state = getattr(rtm, "_trace_state", None)
    if state is None or not getattr(rtm, "_devices", None):
        raise ValueError("refine=True: there is no previous exchange trace on this domain to refine")
    if state["row_tiles"] is not None:
        raise ValueError("refine=True: the previous call traced explicit row_tiles, whose tile counts are not kept")
    if state["dense_multi"]:
        raise ValueError("refine=True: the previous call gathered dense counts from several devices, which cannot be continued")
    for name, given in (("seed", seed), ("devices", devices), ("locator", locator), ("row_tiles", row_tiles), ("nudge", nudge)):
        if given is not None and given != state[name]:
            raise ValueError(f"refine=True: {name}={given!r} differs from the previous call's {state[name]!r}")
    if not _same_flat(flatten_domain(rtm), rtm._devices[0].flat):
        raise ValueError("refine=True: the domain changed since the previous call (its flattened mesh differs)")
    return state


def computeExchangeFactorsBins(rtm, rays_per_emitter: int, nudge: float, spectral_bins: Sequence[int],
                               verbose: bool, rec, seed: int, device: int = 0,
                               locator: int = RTHX_LOCATOR_AUTO, devices=None, row_tiles: Optional[int] = None,
                               refine: bool = False) -> List[sp.csc_matrix]:
    """Batched form of computeExchangeFactorsBin: traces every requested (1-based) bin in one launch per device.  refine=True adds
    the rays to the counts the previous call left resident (parallelRayTracing checks that it can)."""
    import time
    if refine:
        state = rtm._trace_state
        trs = rtm._devices
        devs = state["devices"]
        rtm.last_phase_ms = {}
    else:
        rtm._trace_state = None
        devs = resolve_devices(devices if devices is not None else [device], device, 0)
        trs = _tracers_for(rtm, devs)
    tr = trs[0]
    rpe_total = rays_per_emitter + (state["rays_per_emitter_total"] if refine else 0)
    rec_ids = [i - 1 for i in rec.ids] if rec is not None else None
    rec_bin = (rec.bin - 1) if rec is not None else 0
    verbose and print(f"  Using CUDA device(s) {devs} for spectral bins {list(spectral_bins)}")
    # The counts stay on the device (with several devices: gathered on the first one over NVLink peer memory inside the trace
    # kernels); only their non-zeros come back, already row-normalised, as the three arrays of the CSC matrix the reference
    # returns (parallelRayTracing.jl:144-158 + row_normalize! :161-169) — no N^2 host traffic, no sparse(I, J, V), no transpose.
    t0 = time.perf_counter()
    kw = dict(seed=seed, bins=[b - 1 for b in spectral_bins], nudge=nudge, rec_ids=rec_ids, rec_bin=rec_bin, locator=locator)
    if refine:
        n_tiles = state["n_tiles"]
    else:
        n_tiles = auto_row_tiles(tr.n_elements, len(spectral_bins)) if row_tiles is None else int(row_tiles)
    new_state = dict(seed=seed, devices=devs, locator=locator, row_tiles=row_tiles, nudge=nudge, n_tiles=n_tiles,
                     dense_multi=n_tiles == 1 and len(trs) > 1, rays_per_emitter_total=rpe_total)
    sparse_multi = row_tiles is None and n_tiles > 1 and len(trs) > 1
    if n_tiles > 1 and (row_tiles is not None or sparse_multi):
        # N >> 57 k elements: the dense count matrix is the limit, not the tally (SURVEY.md section 5).  Several devices: each traces
        # its emitter shard with the hashed row tally and only the non-zeros come back.  An explicit row_tiles: the rows are traced in
        # tiles on one device, keeping only each tile's non-zeros; the recorder is not available there.
        if sparse_multi:
            from ._lib import trace_sparse_multi
            res = trace_sparse_multi(trs, rays_per_emitter, refine=refine, **kw)
            stats = dict(res["stats"], tally="sparse", devices=len(trs), sparse=res["sparse_stats"], rays_per_emitter_total=rpe_total)
            if rec is not None and "origins" in res:
                rec.origins[0] = np.concatenate([rec.origins[0], res["origins"]], axis=0)
                rec.endpoints[0] = np.concatenate([rec.endpoints[0], res["endpoints"]], axis=0)
        else:
            if rec is not None:
                raise ValueError("RayRecorder is not supported together with row tiles")
            from ._lib import trace_row_tiles
            kw.pop("rec_ids"); kw.pop("rec_bin")
            res = trace_row_tiles(tr, rays_per_emitter, n_tiles, **kw)
            stats = dict(res["stats"], row_tiles=n_tiles, rays_per_emitter_total=rpe_total)
        t1 = time.perf_counter()
        rtm._trace_state = new_state
        rtm.last_trace_stats = stats
        rtm.last_lost = res["lost"]
        N = tr.n_elements
        mats = []
        rtm.last_counts_stats = []
        for k in range(len(spectral_bins)):
            row_ptr, cols, vals = res["csr"][k]
            print(f"Maximum ray tracing ray loss per emitter: {int(res['lost'][k].max()) if N else 0}/{rpe_total}")   # unconditional, :163
            rtm.last_counts_stats.append({"nnz": int(row_ptr[-1]), "chi": float(res["chi"][k]), "density": row_ptr[-1] / float(N * N)})
            mats.append(sp.csr_matrix((vals, cols, row_ptr), shape=(N, N)).tocsc())
        rtm.last_phase_ms.update({"trace": 1e3 * (t1 - t0), "csc_F_raw": 1e3 * (time.perf_counter() - t1), "row_tiles": n_tiles})
        return mats
    if n_tiles > 1:
        # one device, dense matrix beyond the budget: the hashed row tally keeps the counts on the device in sparse form
        out = tr.trace_continue(rays_per_emitter, **kw) if refine else tr.trace_sparse(rays_per_emitter, **kw)
        out["stats"] = dict(out["stats"], tally="sparse", sparse=out["sparse_stats"])
    elif len(trs) == 1:
        out = tr.trace_continue(rays_per_emitter, **kw) if refine else tr.trace(rays_per_emitter, dense=False, **kw)
    else:
        from ._lib import trace_multi
        out = trace_multi(trs, rays_per_emitter, dense=False, **kw)
        tr.set_copy_helpers(trs[1:])           # the read-outs below leave through every device's PCIe link
    t1 = time.perf_counter()
    rtm._trace_state = new_state
    rtm.last_trace_stats = dict(out["stats"], rays_per_emitter_total=rpe_total)
    rtm.last_lost = out["lost"]
    if rec is not None and "origins" in out:
        # parallelRayTracing.jl:120-123 push into rec.origins[tid]; any slot works for collect_rays
        rec.origins[0] = np.concatenate([rec.origins[0], out["origins"]], axis=0)
        rec.endpoints[0] = np.concatenate([rec.endpoints[0], out["endpoints"]], axis=0)
    N = tr.n_elements
    mats = []
    rtm.last_counts_stats = []
    for k in range(len(spectral_bins)):
        nnz, chi = tr.counts_stats(k)
        rtm.last_counts_stats.append({"nnz": nnz, "chi": chi, "density": nnz / float(N * N) if N else 0.0})
        colptr, rowval, _, fvals = tr.counts_csc(k, values=False, normalised=True)
        max_loss = int(out["lost"][k].max()) if N else 0
        print(f"Maximum ray tracing ray loss per emitter: {max_loss}/{rpe_total}")   # unconditional, :163
        if nnz < 2 ** 31:
            colptr = colptr.astype(np.int32)          # scipy wants one index type; N + 1 entries, the big array stays as it is
        else:
            rowval = rowval.astype(np.int64)
        F = sp.csc_matrix((fvals, rowval, colptr), shape=(N, N), copy=False)
        F.has_sorted_indices = True                    # rows ascend within each column by construction
        mats.append(F)
    rtm.last_phase_ms.update({"trace": 1e3 * (t1 - t0), "csc_F_raw": 1e3 * (time.perf_counter() - t1)})
    return mats


def computeExchangeFactorsBin(rtm, rays_per_emitter: int, nudge: float, spectral_bin: int, verbose: bool = False,
                              rec=None, seed: int = 0x5EED0001, device: int = 0,
                              locator: int = RTHX_LOCATOR_AUTO, devices=None, row_tiles: Optional[int] = None) -> sp.csc_matrix:
    """computeExchangeFactorsBin(rtm, rays_per_emitter, nudge, spectral_bin, ..., rec) -> sparse F (1-based bin)."""
    return computeExchangeFactorsBins(rtm, rays_per_emitter, nudge, [spectral_bin], verbose, rec, seed, device,
                                      locator, devices, row_tiles)[0]


def parallelRayTracing(rtm, rays_total: int, nudge: Optional[float], verbose: bool, rec=None, seed: Optional[int] = None,
                       device: Optional[int] = None, locator: Optional[int] = None, devices=None, row_tiles: Optional[int] = None,
                       refine: bool = False):
    """parallelRayTracing(rtm, rays_total, nudge, verbose; rec) -> (F_raw, rays_per_emitter).  refine=True (new): add
    rays_total // N rays per emitter to the counts the previous call left on the device(s) — same handles, seed, bins, nudge and
    locator — and return the F_raw of ONE trace of all rays so far, with their number per emitter.  ValueError when there is no
    previous call, it traced explicit row_tiles or gathered dense counts from several devices, the flattened mesh changed, or
    seed / devices / device / locator / row_tiles / nudge are given and differ (`device=d` stands for `devices=[d]`)."""
    num_emitters = rtm.num_elements
    rays_per_emitter = rays_total // num_emitters                        # parallelRayTracing.jl:6
    n_bins = rtm.n_spectral_bins
    if refine:
        given = resolve_devices(devices, 0, rays_total) if devices is not None else ([int(device)] if device is not None else None)
        state = _refine_state(rtm, seed, given, locator, row_tiles, nudge)
        seed, devices, locator, nudge = state["seed"], state["devices"], state["locator"], state["nudge"]
        device = devices[0]
    else:
        if seed is None:
            seed = secrets.randbits(64)   # the reference is unseeded: a fresh stream per call
        if locator is None:
            locator = RTHX_LOCATOR_AUTO
        if nudge is None:
            nudge = DEFAULT_NUDGE
        if device is None:
            device = 0
        devices = resolve_devices(devices, device, rays_total)
    if rtm.spectral_mode == "spectral_variable":
        verbose and print(f"Computing {n_bins} separate F matrices for variable spectral extinction")
        groups, reps, nonuniform = group_uniform_bins(rtm.uniform_across_bin)
        to_trace = list(nonuniform) + [g[0] for g in groups]
        mats = computeExchangeFactorsBins(rtm, rays_per_emitter, nudge, to_trace, verbose, rec, seed, device, locator, devices, row_tiles,
                                          refine)
        rtm._traced_bins = list(to_trace)
        F_raw_vector: List[Optional[sp.csc_matrix]] = [None] * n_bins
        for b, F in zip(to_trace[: len(nonuniform)], mats[: len(nonuniform)]):
            F_raw_vector[b - 1] = F
        for g, F in zip(groups, mats[len(nonuniform):]):
            for j in g:
                F_raw_vector[j - 1] = F                                  # group members alias one matrix (:38-41)
        return F_raw_vector, rtm._trace_state["rays_per_emitter_total"]
    if rtm.spectral_mode != "grey":
        verbose and print(f"Computing single F matrix for uniform spectral extinction ({n_bins} bins)")
    else:
        verbose and print("Computing single F matrix for grey extinction")
    F_raw = computeExchangeFactorsBins(rtm, rays_per_emitter, nudge, [1], verbose, rec, seed, device, locator, devices, row_tiles, refine)[0]
    rtm._traced_bins = [1]
    return F_raw, rtm._trace_state["rays_per_emitter_total"]


def get_w(rtm, spectral_bin: int = 1) -> np.ndarray:
    """Reciprocity weights: wall length for surfaces, max(1e-6, 4*beta*V) for volumes
    (smoothExchangeFactors.jl:320-341)."""
    ns = rtm.num_surfaces
    w = np.zeros(rtm.num_elements)
    for (c, f, wall), s in rtm.surface_mapping.items():
        w[s - 1] = rtm.fine_mesh[c - 1][f - 1].area[wall - 1]
    for (c, f), v in rtm.volume_mapping.items():
        cell = rtm.fine_mesh[c - 1][f - 1]
        w[ns + v - 1] = max(1e-6, 4 * cell.beta(spectral_bin - 1) * cell.volume)
    return w


def get_b(rtm) -> np.ndarray:
    """Reflection-scattering coefficient b: 1-eps for surfaces, sigma_s/(sigma_s+kappa) for volumes, per band
    (smoothExchangeFactors.jl:343-357)."""
    ns = rtm.num_surfaces
    nb = rtm.n_spectral_bins
    b = np.zeros((rtm.num_elements, nb))
    for m in range(nb):
        for (c, f, wall), s in rtm.surface_mapping.items():
            b[s - 1, m] = 1 - rtm.fine_mesh[c - 1][f - 1].eps(wall - 1, m)
        for (c, f), v in rtm.volume_mapping.items():
            cell = rtm.fine_mesh[c - 1][f - 1]
            k = cell.kappa_g[m] if isinstance(cell.kappa_g, list) else cell.kappa_g
            s_ = cell.sigma_s_g[m] if isinstance(cell.sigma_s_g, list) else cell.sigma_s_g
            b[ns + v - 1, m] = s_ / (s_ + k) if (s_ + k) != 0 else 0.0
    return b


def _warn_smoothing(st, max_iters: int):
    import warnings
    if not st["converged"]:          # the reference @warns here (smoothExchangeFactors.jl:605-607)
        warnings.warn(f"AP reached max_iters = {max_iters}. Final delta_R = {st['delta']:.3e}")
    if st["delta"] > max(st["delta_init"], 16 * np.finfo(np.float64).eps):       # :608-610
        warnings.warn("Smoothing increased the distance to the target manifold; use F_raw instead of F_smooth.")


def _smooth_on_device(rtm, k: int, F_raw, w, ns: int, max_iters: int, verbose: bool, k_dykstra=None):
    """smooth_F on the GPU for traced bin number `k` (0-based position in the last launch).  Dense branch (density > 0.25,
    smoothExchangeFactors.jl:432-434): straight from the counts the trace left on the device.  Sparse branch with AP only
    (k_dykstra nothing or 0): AP on the non-zero pattern, from the resident counts (dense, or the hashed tally's of a single-device
    trace), or from the host CSC F_raw after a trace in row tiles or a multi-device hashed-tally trace (only one shard is resident).  Returns None where the host path applies: sparse Dykstra rounds, or a dense
    F traced in row tiles or with the hashed row tally."""
    tr = getattr(rtm, "_device", None)
    n = F_raw.shape[0]
    if tr is None or max_iters <= 0:
        return None
    trace_stats = getattr(rtm, "last_trace_stats", None) or {}
    row_tiled = trace_stats.get("row_tiles", 1) > 1
    sparse_tally = trace_stats.get("tally") == "sparse"
    resident = not row_tiled and not (sparse_tally and trace_stats.get("devices", 1) > 1)   # all rows of F_raw on this device
    wn = w[:n] / np.min(w[:n])
    if F_raw.nnz / float(n * n) <= 0.25:
        if k_dykstra not in (None, 0):
            return None
        verbose and print(f"Matrix size: {n}x{n}; sparse smoothing on the device (AP, {F_raw.nnz} non-zeros)")
        if not resident:
            F_smooth, st = tr.smooth_sparse(wn, F=F_raw, max_iters=max_iters)
        else:
            F_smooth, st = tr.smooth_sparse(wn, n=n, bin=k, max_iters=max_iters)
        st["path"] = "device_sparse"
        rtm.last_smooth_stats = st
        _warn_smoothing(st, max_iters)
        verbose and print(f"AP: {st['iterations']} iterations, delta_R {st['delta_init']:.3e} -> {st['delta']:.3e}, "
                          f"{st['total_ms']:.1f} ms on the device")
        return F_smooth
    if row_tiled or sparse_tally:
        return None                                          # a dense F traced in row tiles or with the hashed tally: no dense counts resident
    if k_dykstra is None:       # smooth_F :441-450: one Dykstra round when surfaces and gas are strongly coupled, else AP only
        stats = getattr(rtm, "last_counts_stats", None)
        if rtm.surfaces_only:
            chi = 0.0                                                  # convex enclosure (:425-426)
        elif stats is not None and k < len(stats):
            chi = stats[k]["chi"]                                      # cross_coupling_chi computed by the device row pass
        else:
            from .smoothing import cross_coupling_chi
            chi = cross_coupling_chi(F_raw, ns)
        k_dykstra = 1 if chi >= 0.4 else 0
    verbose and print(f"Matrix size: {n}x{n}; dense smoothing on the device ({k_dykstra} Dykstra rounds + AP)")
    F_smooth, st = tr.smooth(wn, n=n, bin=k, max_iters=max_iters, k_dykstra=int(k_dykstra))
    st["path"] = "device_dense"
    rtm.last_smooth_stats = st
    _warn_smoothing(st, max_iters)
    # the smoothed matrix also stays on the device: solveEquilibrium reads it there when handed this very array
    from .equilibrium import _sample_of
    tr._resident_F = (F_smooth, _sample_of(F_smooth))
    verbose and print(f"AP: {st['iterations']} iterations, delta_R {st['delta_init']:.3e} -> {st['delta']:.3e}, "
                      f"{st['total_ms']:.1f} ms on the device")
    return F_smooth


def exchangeRayTracing(rtm, rays_tot: int, nudge: Optional[float], max_iters: int, k_dykstra, verbose: bool, rec,
                       seed: Optional[int] = None, device: Optional[int] = None, locator: Optional[int] = None,
                       smooth: bool = True, devices=None, row_tiles: Optional[int] = None, refine: bool = False):
    """exchangeRayTracing!(rtm, rays_tot, nudge, max_iters, k_dykstra, verbose, rec): trace, optional
    surfaces-only crop (:9-11), smooth (:14-70), store rtm.F_raw / rtm.F_smooth (:73-74).  refine=True: see parallelRayTracing."""
    import time
    from .smoothing import smooth_F
    F_raw, rays_per_emitter = parallelRayTracing(rtm, rays_tot, nudge, verbose, rec=rec, seed=seed, device=device,
                                                 locator=locator, devices=devices, row_tiles=row_tiles, refine=refine)
    t0 = time.perf_counter()
    ns = rtm.num_surfaces
    if rtm.surfaces_only and not isinstance(F_raw, list):
        F_raw = F_raw[:ns, :ns]

    def smooth_one(k, F, spectral_bin):
        # the device path for both branches of the reference; the host iteration for what the device does not cover
        w = get_w(rtm, spectral_bin=spectral_bin)
        Fs = _smooth_on_device(rtm, k, F, w, ns, max_iters, verbose, k_dykstra=k_dykstra)
        if Fs is None:
            Fs = smooth_F(F, w, ns, max_iters=max_iters, k_dykstra=k_dykstra, verbose=verbose,
                          smooth_surfaces_only=rtm.surfaces_only)
            rtm.last_smooth_stats = {"path": "host"}
        return Fs

    if not smooth:
        F_smooth = F_raw
    elif rtm.spectral_mode == "spectral_variable":
        # one smoothing per traced bin, with that bin's weights (exchangeRayTracing.jl:14-48); grouped bins alias one matrix
        groups, reps, nonuniform = group_uniform_bins(rtm.uniform_across_bin)
        F_smooth = [None] * rtm.n_spectral_bins
        traced = list(nonuniform) + [g[0] for g in groups]
        done = {b: smooth_one(k, F_raw[b - 1], b) for k, b in enumerate(traced)}
        for b in nonuniform:
            F_smooth[b - 1] = done[b]
        for g in groups:
            for j in g:
                F_smooth[j - 1] = done[g[0]]
    else:
        F_smooth = smooth_one(0, F_raw, 1)
    rtm.F_raw = F_raw
    rtm.F_smooth = F_smooth
    if getattr(rtm, "last_phase_ms", None) is not None:
        rtm.last_phase_ms["smoothing"] = 1e3 * (time.perf_counter() - t0)
    return F_smooth


def dispatch_ray_trace(rtm, rays_tot: int, method: str = "exchange", nudge: Optional[float] = None,
                       k_dykstra=None, max_iters: int = 1000, verbose: bool = True, rec=None, **kw):
    """(rtm)(rays_tot; method, nudge, k_dykstra, max_iters, verbose, rec) — multiDispatchRayTrace2D.jl:1-18.  New keyword
    refine=True (method=:exchange): add rays_tot // N rays per emitter to the previous call's trace and smooth again (parallelRayTracing)."""
    method = method.lstrip(":")
    if method == "exchange":
        return exchangeRayTracing(rtm, rays_tot, nudge, max_iters, k_dykstra, verbose, rec, **kw)
    if method == "direct":
        raise NotImplementedError("method=:direct is outside the scope of this drop-in (exchange path only)")
    raise ValueError(f"Unknown ray tracing method: {method}, must be :exchange or :direct")
