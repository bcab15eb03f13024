"""The resynthesis exports driven on the SIMT emulator (tests/emu), host arrays standing in for device
memory: ``render`` is one render call of a table (the export choice of pv._resynth_ex), ``sharded`` the
simulated ranks of a segment-sharded render, and the rest are the helpers the resynthesis tests share.

``sharded`` runs every rank's stages (pvk_resynth_scan, the all_gather of the hand-over records,
pvk_resynth_handover, the Nyquist flags and their all_reduce(MAX), pvk_resynth_import_flags,
pvk_resynth_render) one rank after another on host arrays, the collectives replaced by their
definition."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

import emu_harness as eh                                           # noqa: E402
import render_contract as rc                                       # noqa: E402
from golden_util import case_golden, case_signal, pv_kwargs        # noqa: E402
from pypevoc_b200 import dist as D                                 # noqa: E402


def pack(tid, f, mag, realph):
    """Renumber the partials of an id table in order of first appearance and pack their points
    (pvk_track_pack's layout): (tid int32 [F, K], pk)."""
    F, K = tid.shape
    flat = tid.reshape(-1)
    ids, first = np.unique(flat[flat >= 0], return_index=True)
    order = ids[np.argsort(first)]
    remap = np.full(int(flat.max()) + 2 if flat.size and flat.max() >= 0 else 1, -1, dtype=np.int64)
    remap[order] = np.arange(len(order))
    out = np.where(tid >= 0, remap[np.maximum(tid, 0)], -1).astype(np.int32)
    nt = len(order)
    rows, cols = np.nonzero(out >= 0)
    v = out[rows, cols]
    srt = np.lexsort((rows, v))
    rows, cols, v = rows[srt], cols[srt], v[srt]
    cnt = np.bincount(v, minlength=nt)
    toff = np.zeros(nt + 1, dtype=np.int64)
    toff[1:] = np.cumsum(cnt)
    tstart = np.array([rows[toff[i]] for i in range(nt)], dtype=np.int32)
    pk = dict(tstart=tstart, tlen=cnt.astype(np.int32), toff=toff,
              pf=np.ascontiguousarray(f[rows, cols], dtype=np.float64),
              pmag=np.ascontiguousarray(mag[rows, cols], dtype=np.float64),
              prealph=np.ascontiguousarray(realph[rows, cols], dtype=np.float64))
    return out, pk


def workspace(F, K, nt, nblocks, ws_blocks=None):
    """Render workspace of a table [F, K] with ``nt`` partials for ``nblocks`` output blocks; with
    ``ws_blocks``, room for that many staged blocks only, which forces chunked rendering."""
    L = eh.lib()
    if ws_blocks is None:
        wsb = L.pvk_resynth_workspace_bytes(F, K, nt, max(nblocks, 1))
    else:
        wsb = L.pvk_resynth_workspace_bytes(F, K, nt, 0) + (ws_blocks - 1) * rc.row_ws_bytes(K)
    return np.zeros(max(int(wsb), 8), dtype=np.uint8)


def phase_scratch(pk):
    """The integrated-phase render's block start phases: one double per packed point."""
    return np.full(max(len(pk["pf"]), 1), np.nan)


def max_end(tid):
    """The last row of an id table with a point."""
    return int(np.nonzero((tid >= 0).any(axis=1))[0].max())


def parts(pk):
    """The partials of a pack, as the numpy models take them."""
    o = pk["toff"]
    return [dict(start_idx=int(pk["tstart"][v]), f=pk["pf"][o[v]:o[v + 1]], mag=pk["pmag"][o[v]:o[v + 1]],
                 realph=pk["prealph"][o[v]:o[v + 1]]) for v in range(len(pk["tstart"]))]


def golden_tracked(name):
    """A golden case tracked by the emulated pvk_track and packed by ``pack``:
    (g, sr, nfft, hop_an, tid, pk)."""
    g = case_golden(name)
    _, sr = case_signal(name)
    tr = eh.track(g["f"], g["mag"])
    tid, pk = pack(np.ascontiguousarray(tr["tid"][0]), g["f"], g["mag"], g["realph"])
    return g, sr, pv_kwargs(name)["nfft"], int(g["hop"]), tid, pk


def _ratio(fscale):
    """The ratio arguments of an export and the suffix of its name: a float, or ratio 1 and a curve
    (the ``_curve`` form)."""
    if np.ndim(fscale) == 0:
        return (float(fscale),), ""
    fc = np.ascontiguousarray(fscale, dtype=np.float64)
    return (1.0, eh.ptr(fc), fc.size), "_curve"


def render(tid, pk, sr, hop, nfft, hop_an, edge=1.0, minframes=3, phase_preserve=False, fscale=1.0, pmag=None,
           block0=0, nblocks=-1, nout=None, ws=None, ws_blocks=None, phase_ws=None, reuse_tracks=False, scanned=False):
    """Blocks [block0, block0 + nblocks) (-1: to the end) of a signal of ``nout`` samples (default: the
    synth length up to the pack's last frame), through pvk_resynth_ex, or pvk_resynth_render when
    ``scanned`` (block start phases and Nyquist flags already in ``ws`` / ``phase_ws``).  ``fscale`` is a
    ratio, or a curve of one ratio per row of ``tid`` for the ``_curve`` exports.  ``pmag`` replaces the
    packed magnitudes.  ``ws`` / ``phase_ws`` are workspaces to (re)use across calls; by default fresh
    ones (``ws_blocks``: see workspace), and no phase scratch with ``phase_preserve``.  The output
    starts as NaN, so a sample the render does not write fails."""
    L = eh.lib()
    tid = np.ascontiguousarray(tid, dtype=np.int32)
    F, K = tid.shape
    nt = len(pk["tstart"])
    if nout is None:
        nout, _ = D.P.synth_geometry(int((pk["tstart"] + pk["tlen"] - 1).max()), hop, nfft, hop_an, edge)
    nb = -(-nout // hop) - block0 if nblocks < 0 else nblocks
    out = np.full(min(nb * hop, nout - block0 * hop), np.nan)
    if ws is None:
        ws = workspace(F, K, nt, nb, ws_blocks)
    if phase_ws is None and not phase_preserve:
        phase_ws = phase_scratch(pk)
    ratio, sfx = _ratio(fscale)
    fn = getattr(L, ("pvk_resynth_render" if scanned else "pvk_resynth_ex") + sfx)
    eh.check(fn(eh.ptr(tid), F, K, nt, None, eh.ptr(pk["tstart"]), eh.ptr(pk["tlen"]), eh.ptr(pk["toff"]),
                eh.ptr(pk["pf"]), eh.ptr(pk["pmag"] if pmag is None else pmag), eh.ptr(pk["prealph"]), float(sr),
                int(hop), int(nfft), int(hop_an), float(edge), int(minframes), eh.ptr(out), int(nout), int(block0),
                int(nblocks), eh.ptr(ws), ws.size, int(reuse_tracks), int(phase_preserve), *ratio, eh.ptr(phase_ws),
                0 if phase_ws is None else phase_ws.size, None))
    return out


def plans_for(F, nfft, hop_an, world, edge, minframes):
    nsamp = nfft + (F - 1) * hop_an + 1 if F > 0 else nfft
    plans = D.plan_segments(nsamp, nfft, hop_an, world, edge, minframes)
    assert plans[0]["frames_total"] == F
    return plans


def sharded(tid, f, mag, realph, sr, hop, nfft, hop_an, edge, minframes, fscale, world, plans=None,
            phase_preserve=False, handover=True, global_flags=True, window_rows=True):
    """Every rank's own blocks, rendered from its window rows only, put together: (signal, ranks),
    ``ranks`` the per-rank state (plan, local tables, records, flags) for further checks.  ``fscale``: a
    ratio, or a curve over the global frames of which each rank passes its window's rows [w0, w1) to
    the scan and the render and its own rows [j0, j1) to the Nyquist flags.  ``phase_preserve``: each
    rank renders its blocks with pvk_resynth_ex, without scan or exchange.  ``handover`` /
    ``global_flags`` = False leave the seed / the flag exchange out, and ``window_rows`` = False has a
    rank pass the curve rows from its first own row on instead of its window's (to show that the cases
    exercise them)."""
    L = eh.lib()
    F, K = tid.shape
    if plans is None:
        plans = plans_for(F, nfft, hop_an, world, edge, minframes)
    ntracks = int(tid.max()) + 1 if tid.size else 0
    me = max_end(tid)
    curve = np.ndim(fscale) > 0
    ranks = []
    for p in plans:                                                # stage 1: scan + hand-over record
        w0, w1 = p["w0"], p["w1"]
        tl, pk = pack(tid[w0:w1], f[w0:w1], mag[w0:w1], realph[w0:w1])
        b0, b1, nout = D.render_range(p, plans, me, hop, nfft, hop_an, edge)
        Fl, nt = tl.shape[0], len(pk["tstart"])
        r = dict(plan=p, tid=tl, pk=pk, b=(b0, b1), nout=nout, fscale=fscale, ws=None, pws=None)
        ranks.append(r)
        if curve:
            rows = fscale[w0:w1] if window_rows else np.concatenate([fscale, np.ones(F)])[p["j0"]:p["j0"] + Fl]
            r["fscale"] = np.ascontiguousarray(rows)
        if phase_preserve:
            continue
        r.update(ws=workspace(Fl, K, nt, b1 - b0), pws=phase_scratch(pk), rec=np.full(2 * K, -7, dtype=np.int64),
                 rows=D.handover_rows(p, plans, nfft, hop_an, edge))
        ratio, sfx = _ratio(r["fscale"])
        eh.check(getattr(L, "pvk_resynth_scan" + sfx)(
            eh.ptr(tl), Fl, K, nt, eh.ptr(pk["tstart"]), eh.ptr(pk["tlen"]), eh.ptr(pk["toff"]), eh.ptr(pk["pf"]),
            eh.ptr(pk["prealph"]), float(sr), hop, nfft, hop_an, *ratio, eh.ptr(r["ws"]), r["ws"].size,
            eh.ptr(r["pws"]), r["pws"].size, r["rows"][0], r["rows"][1], eh.ptr(r["rec"]), r["rec"].size, None))
    flags = np.zeros(max(ntracks, 1), dtype=np.uint8)
    if not phase_preserve:
        recs = np.ascontiguousarray(np.concatenate([r["rec"] for r in ranks]))   # the all_gather
        for r in ranks:                                            # stage 2: seed + fix-up, local flags
            p, tl, pk = r["plan"], r["tid"], r["pk"]
            Fl, nt = tl.shape[0], len(pk["tstart"])
            eh.check(L.pvk_resynth_handover(eh.ptr(tl), Fl, K, nt, eh.ptr(pk["tstart"]), eh.ptr(pk["tlen"]),
                                            eh.ptr(pk["toff"]), eh.ptr(r["pws"]), r["pws"].size, eh.ptr(recs),
                                            recs.size, world, p["rank"], r["rows"][0] if handover else -1,
                                            eh.ptr(r["ws"]), r["ws"].size, None))
            fo = np.ascontiguousarray(f[p["j0"]:p["j1"]], dtype=np.float64)
            go = np.ascontiguousarray(tid[p["j0"]:p["j1"]], dtype=np.int32)
            ratio, sfx = _ratio(fscale[p["j0"]:p["j1"]] if curve else fscale)
            mine = np.zeros_like(flags)
            eh.check(getattr(L, "pvk_nyquist_flags" + sfx)(eh.ptr(fo), eh.ptr(go), go.size, float(sr), *ratio,
                                                            *((K,) if curve else ()), eh.ptr(mine), ntracks, None))
            r["flags"] = mine
            flags = np.maximum(flags, mine)                        # the all_reduce(MAX)
    sig = np.zeros(D.P.synth_geometry(me, hop, nfft, hop_an, edge)[0])
    table = np.ascontiguousarray(tid, dtype=np.int32)
    for r in ranks:                                                # stage 3: import flags, render
        p, tl, pk = r["plan"], r["tid"], r["pk"]
        if global_flags and not phase_preserve:
            eh.check(L.pvk_resynth_import_flags(eh.ptr(tl), tl.shape[0], K, len(pk["tstart"]), eh.ptr(pk["tstart"]),
                                                eh.ptr(table), F, p["w0"], eh.ptr(flags), ntracks, eh.ptr(r["ws"]),
                                                r["ws"].size, None))
        b0, b1 = r["b"]
        if b1 <= b0:
            continue
        w0 = p["w0"]
        r["out"] = render(tl, pk, sr, hop, nfft, hop_an, edge, minframes, phase_preserve, r["fscale"], block0=b0 - w0,
                          nblocks=b1 - b0, nout=r["nout"] - w0 * hop, ws=r["ws"], phase_ws=r["pws"],
                          scanned=not phase_preserve)
        sig[b0 * hop:b0 * hop + len(r["out"])] = r["out"]
    return sig, ranks
