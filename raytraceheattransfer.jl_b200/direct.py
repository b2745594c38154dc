"""method=:direct of the reference's functor for grey domains (DESIGN.md section "method=:direct"): energy bundles are traced from
the elements that have energy to emit until an element of known temperature absorbs them; an element of unknown temperature that
absorbs a bundle emits it again.  The absorbed powers give the temperatures directly — no exchange factors, no smoothing, no solve,
so the result is an independent check of the :exchange route (test/test_2d_spectral.jl:263-283 compares the two).

  directRayTracing   the :direct branch of multiDispatchRayTrace2D.jl:1-18 (RT2D/DirectTracing2D)

The traversal and the event rules are the device kernels' (rthx_trace_direct); this module forms the sources and writes the result
back to the domain.
"""
from __future__ import annotations

import math
from typing import Optional

import numpy as np

from .equilibrium import STEFAN_BOLTZMANN, populateWorkspace
from ._abi import RTHX_LOCATOR_AUTO
from ._lib import DEFAULT_NUDGE


def direct_sources(rtm, rays_tot: int):
    """The bundle sources of a grey domain, elements numbered as on the exchange path (surfaces, then volumes).  Returns (ws, known_T,
    E, sources, rays, bundle_energy): E_i = eps sigma A T^4 (wall) or 4 kappa sigma V T^4 (gas) where T_in >= 0, q_in where T_in < 0;
    source i gets R_i = max(1, round(rays_tot E_i / sum E)) bundles of E_i / R_i each."""
    ws = populateWorkspace(rtm, 1)
    known_T = np.concatenate([~ws["Qw_known"], ~ws["Qg_known"]])
    E_T = np.concatenate([ws["epsw"] * STEFAN_BOLTZMANN * ws["Area"] * ws["Tw"] ** 4,
                          4 * ws["kappa_g"] * STEFAN_BOLTZMANN * ws["Volume"] * ws["Tg"] ** 4])
    q = np.concatenate([ws["qw"], ws["qg"]])
    ns = len(ws["Area"])
    bad = np.flatnonzero(~known_T & (q < 0.0))
    if len(bad):
        i = int(bad[0])
        what = f"surface {i + 1}" if i < ns else f"volume {i - ns + 1}"
        raise ValueError(f"method=:direct: {what} (element {i}) has q_in = {q[i]} < 0; a negative source cannot be carried by energy bundles")
    E = np.where(known_T, E_T, q)
    total = float(E.sum())
    if not total > 0.0:
        raise ValueError("method=:direct: no element has energy to emit (sum of E = 0): give a temperature above 0 K or a q_in > 0")
    sources = np.flatnonzero(E > 0.0).astype(np.int32)
    rays = np.maximum(1, np.rint(float(rays_tot) * E[sources] / total)).astype(np.int64)
    return ws, known_T, E, sources, rays, E[sources] / rays


def _row_sum(row_ptr, cols, vals, rows, w, out):
    """out[k] += w[i] count[y][k] over the CSR rows y of the source indices `rows` (ascending), every product and sum rounded on its own:
    the order and rounding of direct_absorbed_kernel."""
    for y, i in enumerate(rows):
        s = slice(row_ptr[y], row_ptr[y + 1])
        out[cols[s]] = out[cols[s]] + w[i] * vals[s].astype(np.float64)


def _hashed(n_rows: int, N: int, all_fields: bool) -> bool:
    """Whether a device block of n_rows sources takes the hashed row tally (rthx_trace_direct_sparse): its dense counts, 8 R N bytes per
    count block (two with all_fields), would pass the budget of one device that the :exchange route keeps to."""
    from .tracing import rows_fit_one_device
    return not rows_fit_one_device(n_rows, N, 2 if all_fields else 1)


def _route(n_rows: int, N: int, all_fields: bool):
    """trace_direct keywords of a device block of n_rows sources: the redirection tally with all_fields, the hashed tally when the dense
    counts do not fit (_hashed)."""
    out = dict(redirected=True) if all_fields else {}
    if _hashed(n_rows, N, all_fields):
        out["sparse"] = True
    return out


def _absorbed_multi(trs, sources, rays, reemit, w, N: int, specular: bool, kw, all_fields: bool = False):
    """Contiguous blocks of the source rows, one per device; the integer counts of every block are read back and reduced on the host in
    ascending row order with the device reduction's rounding, so the result does not depend on the number of devices.  all_fields: the
    redirection counts (bin 1) are traced, read back and reduced the same way.  Each block takes the dense or the hashed tally on its own
    (_route); both read out the same counts."""
    from concurrent.futures import ThreadPoolExecutor
    blocks = [b for b in np.array_split(np.arange(len(sources)), len(trs)) if len(b)]

    def run(k):
        b = blocks[k]
        out = trs[k].trace_direct(sources[b], rays[b], reemit, w[b], specular=specular, **_route(len(b), N, all_fields), **kw)
        out["csr"] = trs[k].counts_csr(values=True, normalised=False)
        if all_fields:
            out["csr_redirected"] = trs[k].counts_csr(bin=1, values=True, normalised=False)
        return out

    with ThreadPoolExecutor(len(blocks)) as ex:
        outs = list(ex.map(run, range(len(blocks))))
    res = dict(absorbed=np.zeros(N), lost=np.zeros(N, np.uint64), events=0, kernel_ms=0.0,
               tally="sparse" if any(_hashed(len(b), N, all_fields) for b in blocks) else "dense")
    if all_fields:
        res.update(redirected=np.zeros(N), redirections=0)
    for b, out in zip(blocks, outs):
        row_ptr, cols, vals, _ = out["csr"]
        _row_sum(row_ptr, cols, vals, b, w, res["absorbed"])
        if all_fields:
            row_ptr, cols, vals, _ = out["csr_redirected"]
            _row_sum(row_ptr, cols, vals, b, w, res["redirected"])
            res["redirections"] += int(vals.sum())
        res["lost"] += out["lost"]
        res["events"] += out["events"]
        res["kernel_ms"] = max(res["kernel_ms"], out["stats"]["kernel_ms"])
    return res


def directRayTracing(rtm, rays_tot: int, nudge: Optional[float] = None, verbose: bool = True, rec=None, seed: Optional[int] = None,
                     device: Optional[int] = None, devices=None, locator: Optional[int] = None, specular: bool = False,
                     block_threads: int = 0, all_fields: bool = False) -> None:
    """(rtm)(rays_tot; method=:direct): trace about rays_tot energy bundles and write T_w / T_g, e_*, g_a_* (absorbed power) and q_* to
    the domain, and rtm.energy_error = sum(e - Abs), the energy of the bundles that were lost.  Returns None.
      all_fields=True also tallies every scattering and reflection (rthx_trace_direct_fields; twice the device memory of the counts)
      and writes j, r, g and i as equilibriumGrey2D does: r = the power of the bundles redirected by the element, g = Abs + r, j = e + r,
      i_w = j / (pi A), i_g = j / (4 pi V).  T, e, g_a, q and energy_error are bit for bit those of all_fields=False.  With the default
      all_fields=False, j, r, g and i are left untouched.
      Elements of known temperature (T_in >= 0) keep it and get q = E - Abs; elements of known net emission q_in (T_in < 0) re-emit what
      they absorb and get e = Abs + q_in and the temperature of computeTemperaturesVariable (0 where eps A or kappa V is 0).
      specular=True reflects at walls like a mirror (RTHX_MULTI_BOUNCE_SPECULAR); seed, device / devices and locator as for
      method=:exchange.  Several devices trace contiguous blocks of the sources; the result is bit-identical to one device's.
      A device block of R sources whose dense counts (8 R N bytes, 16 R N with all_fields) would pass the 48 GB budget of the :exchange
      route is tallied in the hashed row tally instead (rthx_trace_direct_sparse): every field is bit for bit the same.
    rtm.last_direct_stats: bundles, events, lost bundles, lost energy, kernel ms, devices, tally ("dense" or "sparse"); with all_fields
    the redirections too."""
    import secrets
    from .tracing import _tracers_for, resolve_devices
    if rtm.spectral_mode != "grey":
        raise NotImplementedError("method=:direct on spectral domains needs the reference's spectral direct solver (band fractions of the "
                                  "spectral bins), which this drop-in does not implement; use method=:exchange")
    if rec is not None:
        raise ValueError("method=:direct does not record rays (RayRecorder): record them with method=:exchange")
    say = print if verbose else (lambda *a, **k: None)
    ws, known_T, E, sources, rays, w = direct_sources(rtm, rays_tot)
    ns = len(ws["Area"])
    n = len(known_T)
    devs = resolve_devices(devices, 0 if device is None else int(device), int(rays.sum()))
    trs = _tracers_for(rtm, devs)
    N = trs[0].n_elements
    reemit = np.zeros(N, np.uint8)
    reemit[:n] = ~known_T
    kw = dict(seed=secrets.randbits(63) if seed is None else int(seed), nudge=DEFAULT_NUDGE if nudge is None else float(nudge),
              locator=RTHX_LOCATOR_AUTO if locator is None else int(locator), block_threads=int(block_threads))
    if len(trs) == 1:
        route = _route(len(sources), N, all_fields)
        out = trs[0].trace_direct(sources, rays, reemit, w, specular=specular, **route, **kw)
        res = dict(absorbed=out["absorbed"], lost=out["lost"], events=out["events"], kernel_ms=out["stats"]["kernel_ms"],
                   tally="sparse" if route.get("sparse") else "dense")
        if all_fields:
            res.update(redirected=out["redirected"], redirections=int(trs[0].counts_csr(bin=1, values=True, normalised=False)[2].sum()))
    else:
        res = _absorbed_multi(trs, sources, rays, reemit, w, N, specular, kw, all_fields)
    absorbed, lost, events, kernel_ms = res["absorbed"], res["lost"], res["events"], res["kernel_ms"]
    Abs = absorbed[:n]
    q_in = np.concatenate([ws["qw"], ws["qg"]])
    e = np.where(known_T, E, Abs + q_in)
    T = np.concatenate([ws["Tw"], ws["Tg"]])
    with np.errstate(divide="ignore", invalid="ignore"):
        Tw = np.where((ws["epsw"] > 0.0) & (ws["Area"] > 0.0), (e[:ns] / (ws["epsw"] * STEFAN_BOLTZMANN * ws["Area"])) ** 0.25, 0.0)
        Tg = np.where((ws["kappa_g"] > 0.0) & (ws["Volume"] > 0.0), (e[ns:] / (4 * ws["kappa_g"] * ws["Volume"] * STEFAN_BOLTZMANN)) ** 0.25, 0.0)
    T = np.where(known_T, T, np.nan_to_num(np.concatenate([Tw, Tg]), nan=0.0))
    qnet = e - Abs
    if all_fields:                                      # the receiver-indexed split of equilibriumGrey2D, from the redirection tally
        r = res["redirected"][:n]
        g = Abs + r
        j = e + r
    for (c, f, wl), s in rtm.surface_mapping.items():
        cell = rtm.fine_mesh[c - 1][f - 1]
        i = s - 1
        cell.T_w[wl - 1] = float(T[i]); cell.e_w[wl - 1] = float(e[i]); cell.g_a_w[wl - 1] = float(Abs[i]); cell.q_w[wl - 1] = float(qnet[i])
        if all_fields:
            cell.j_w[wl - 1] = float(j[i]); cell.r_w[wl - 1] = float(r[i]); cell.g_w[wl - 1] = float(g[i])
            cell.i_w[wl - 1] = float(j[i] / (math.pi * cell.area[wl - 1]))
    if not rtm.surfaces_only:
        for (c, f), v in rtm.volume_mapping.items():
            cell = rtm.fine_mesh[c - 1][f - 1]
            i = ns + v - 1
            cell.T_g = float(T[i]); cell.e_g = float(e[i]); cell.g_a_g = float(Abs[i]); cell.q_g = float(qnet[i])
            if all_fields:
                cell.j_g = float(j[i]); cell.r_g = float(r[i]); cell.g_g = float(g[i]); cell.i_g = float(j[i] / (4 * math.pi * cell.volume))
    rtm.energy_error = float(np.sum(e - Abs))
    lost_energy = float(np.sum(w * lost[sources].astype(np.float64)))
    rtm.last_direct_stats = dict(bundles=int(rays.sum()), events=int(events), lost=int(lost.sum()), lost_energy=lost_energy,
                                 kernel_ms=float(kernel_ms), devices=len(trs), sources=len(sources), tally=res["tally"])
    if all_fields:
        rtm.last_direct_stats["redirections"] = res["redirections"]
    say(f"method=:direct: {int(rays.sum())} bundles from {len(sources)} sources, {int(lost.sum())} lost, {events} events, "
        f"{kernel_ms:.2f} ms on {len(trs)} device(s), {res['tally']} tally")
    return None
