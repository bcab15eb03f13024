"""The time-map stage of the resynthesis (pvk_time_map) driven on the SIMT emulator (tests/emu), host arrays
standing in for device memory, next to the render drivers of tests/resynth_emu.py: ``time_map`` is one call
of the export, ``time_map_pack`` the map followed by the pack of its tables, as pv.time_map_device runs them."""
import numpy as np

import resynth_emu as rem

eh = rem.eh


def time_map(tid, pk, tau, ntracks=None):
    """pvk_time_map: the partials of ``tid`` / ``pk`` read at the fractional frames ``tau``, as tables
    (tid', f', mag', realph') ``[len(tau), K]``.  ``ntracks`` defaults to the pack's partial count.  The
    outputs start as sentinels (-99, NaN), so a slot the kernel does not write fails."""
    L = eh.lib()
    tid = np.ascontiguousarray(tid, dtype=np.int32)
    F, K = tid.shape
    tau = np.ascontiguousarray(tau, dtype=np.float64)
    B = tau.size
    nt = len(pk["tstart"]) if ntracks is None else int(ntracks)
    tid_out = np.full((B, K), -99, dtype=np.int32)
    outs = [np.full((B, K), np.nan) for _ in range(3)]
    arrs = [np.ascontiguousarray(pk[n], dtype=dt) for n, dt in (("tstart", np.int32), ("tlen", np.int32),
                                                                ("toff", np.int64), ("pf", np.float64),
                                                                ("pmag", np.float64), ("prealph", np.float64))]
    eh.check(L.pvk_time_map(eh.ptr(tid), F, K, nt, *(eh.ptr(a) for a in arrs), eh.ptr(tau), B, eh.ptr(tid_out),
                            *(eh.ptr(o) for o in outs), None))
    return (tid_out, *outs)


def time_map_pack(tid, pk, tau, ntracks=None):
    """The time map and the pack of its tables (pvk_track_pack, ids kept: a partial the map skips has
    tlen 0): (tid', pk', max_end'), ``max_end'`` the last output row with a point (-1: none)."""
    nt = len(pk["tstart"]) if ntracks is None else int(ntracks)
    tm, fm, mm, rm = time_map(tid, pk, tau, nt)
    pkm = eh.track_pack(fm, mm, rm, rm, tm, None, nt)
    rows = np.nonzero((tm >= 0).any(axis=1))[0]
    return tm, pkm, int(rows.max()) if rows.size else -1
