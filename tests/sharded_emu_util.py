"""Simulated ranks of a segment-sharded integrated-phase resynthesis on the SIMT emulator: every rank's
stages (pvk_resynth_scan, the all_gather of the hand-over records, pvk_resynth_handover, the Nyquist
flags and their all_reduce(MAX), pvk_resynth_import_flags, pvk_resynth_render) run one rank after
another on host arrays, the collectives replaced by their definition.  Used by
tests/test_sharded_synth_modes_cpu.py."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

import emu_harness as eh                                           # noqa: E402
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


def _ws(F, K, nt, nblocks):
    return np.zeros(max(int(eh.lib().pvk_resynth_workspace_bytes(F, K, nt, max(nblocks, 1))), 8), dtype=np.uint8)


def _pws(pk):
    return np.full(max(len(pk["pf"]), 1), np.nan)


def unsharded(tid, pk, sr, hop, nfft, hop_an, edge, minframes, fscale, max_end):
    """pvk_resynth_ex(phase_preserve=0) over the whole table."""
    L = eh.lib()
    F, K = tid.shape
    nout, _ = D.P.synth_geometry(max_end, hop, nfft, hop_an, edge)
    nb = -(-nout // hop)
    out = np.full(nout, np.nan)
    ws, pws = _ws(F, K, len(pk["tstart"]), nb), _pws(pk)
    eh.check(L.pvk_resynth_ex(eh.ptr(tid), F, K, len(pk["tstart"]), None, eh.ptr(pk["tstart"]), eh.ptr(pk["tlen"]),
                              eh.ptr(pk["toff"]), eh.ptr(pk["pf"]), eh.ptr(pk["pmag"]), eh.ptr(pk["prealph"]), float(sr),
                              hop, nfft, hop_an, float(edge), minframes, eh.ptr(out), nout, 0, nb, eh.ptr(ws), ws.size, 0,
                              0, float(fscale), eh.ptr(pws), pws.size, None))
    return out


def plans_for(F, nfft, hop_an, world, edge, minframes):
    nsamp = nfft + (F - 1) * hop_an + 1 if F > 0 else nfft
    plans = D.plan_segments(nsamp, nfft, hop_an, world, edge, minframes)
    assert plans[0]["frames_total"] == F
    return plans


def sharded(tid, f, mag, realph, sr, hop, nfft, hop_an, edge, minframes, fscale, world, plans=None, handover=True,
            global_flags=True):
    """Every rank's own blocks, rendered from its window rows only, put together: (signal, ranks),
    ``ranks`` the per-rank state (plan, local tables, records, flags) for further checks.
    ``handover`` / ``global_flags`` = False leave the seed / the flag exchange out (to show that the
    cases exercise them)."""
    L = eh.lib()
    F, K = tid.shape
    if plans is None:
        plans = plans_for(F, nfft, hop_an, world, edge, minframes)
    ntracks = int(tid.max()) + 1 if tid.size else 0
    max_end = int(np.nonzero((tid >= 0).any(axis=1))[0].max())
    ranks = []
    for p in plans:                                                # stage 1: scan + hand-over record
        w0, w1 = p["w0"], p["w1"]
        tl, pk = pack(tid[w0:w1], f[w0:w1], mag[w0:w1], realph[w0:w1])
        b0, b1, nout = D.render_range(p, plans, max_end, hop, nfft, hop_an, edge)
        Fl, nt = tl.shape[0], len(pk["tstart"])
        r = dict(plan=p, tid=tl, pk=pk, b=(b0, b1), nout=nout, ws=_ws(Fl, K, nt, b1 - b0), pws=_pws(pk),
                 rec=np.full(2 * K, -7, dtype=np.int64))
        r["rows"] = D.handover_rows(p, plans, nfft, hop_an, edge)
        eh.check(L.pvk_resynth_scan(eh.ptr(tl), Fl, K, nt, eh.ptr(pk["tstart"]), eh.ptr(pk["tlen"]), eh.ptr(pk["toff"]),
                                    eh.ptr(pk["pf"]), eh.ptr(pk["prealph"]), float(sr), hop, nfft, hop_an, float(fscale),
                                    eh.ptr(r["ws"]), r["ws"].size, eh.ptr(r["pws"]), r["pws"].size, r["rows"][0],
                                    r["rows"][1], eh.ptr(r["rec"]), r["rec"].size, None))
        ranks.append(r)
    recs = np.ascontiguousarray(np.concatenate([r["rec"] for r in ranks]))       # the all_gather
    flags = np.zeros(max(ntracks, 1), dtype=np.uint8)
    for r in ranks:                                                # stage 2: seed + fix-up, local flags
        p, tl, pk = r["plan"], r["tid"], r["pk"]
        Fl, nt = tl.shape[0], len(pk["tstart"])
        eh.check(L.pvk_resynth_handover(eh.ptr(tl), Fl, K, nt, eh.ptr(pk["tstart"]), eh.ptr(pk["tlen"]),
                                        eh.ptr(pk["toff"]), eh.ptr(r["pws"]), r["pws"].size, eh.ptr(recs), recs.size,
                                        world, p["rank"], r["rows"][0] if handover else -1, eh.ptr(r["ws"]),
                                        r["ws"].size, None))
        fo = np.ascontiguousarray(f[p["j0"]:p["j1"]], dtype=np.float64)
        go = np.ascontiguousarray(tid[p["j0"]:p["j1"]], dtype=np.int32)
        mine = np.zeros_like(flags)
        eh.check(L.pvk_nyquist_flags(eh.ptr(fo), eh.ptr(go), go.size, float(sr), float(fscale), eh.ptr(mine), ntracks,
                                     None))
        r["flags"] = mine
        flags = np.maximum(flags, mine)                            # the all_reduce(MAX)
    sig = np.zeros(D.P.synth_geometry(max_end, hop, nfft, hop_an, edge)[0])
    table = np.ascontiguousarray(tid, dtype=np.int32)
    for r in ranks:                                                # stage 3: import flags, render
        p, tl, pk = r["plan"], r["tid"], r["pk"]
        Fl, nt = tl.shape[0], len(pk["tstart"])
        if global_flags:
                eh.check(L.pvk_resynth_import_flags(eh.ptr(tl), Fl, K, nt, eh.ptr(pk["tstart"]), eh.ptr(table), F, p["w0"],
                                                eh.ptr(flags), ntracks, eh.ptr(r["ws"]), r["ws"].size, None))
        b0, b1 = r["b"]
        if b1 <= b0:
            continue
        w0 = p["w0"]
        nloc = r["nout"] - w0 * hop
        out = np.full(min((b1 - b0) * hop, nloc - (b0 - w0) * hop), np.nan)
        eh.check(L.pvk_resynth_render(eh.ptr(tl), Fl, K, nt, None, eh.ptr(pk["tstart"]), eh.ptr(pk["tlen"]),
                                      eh.ptr(pk["toff"]), eh.ptr(pk["pf"]), eh.ptr(pk["pmag"]), eh.ptr(pk["prealph"]),
                                      float(sr), hop, nfft, hop_an, float(edge), minframes, eh.ptr(out), nloc, b0 - w0,
                                      b1 - b0, eh.ptr(r["ws"]), r["ws"].size, 0, 0, float(fscale), eh.ptr(r["pws"]),
                                      r["pws"].size, None))
        sig[b0 * hop:b0 * hop + len(out)] = out
        r["out"] = out
    return sig, ranks
