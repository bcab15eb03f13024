"""The remap stage of the resynthesis (pvk_time_map, then pvk_track_relink) driven on the SIMT emulator
(tests/emu), host arrays standing in for device memory, beside tests/time_map_emu.py: ``relink`` is one
call of the relink export, ``remap_pack`` the map, the relink, the stats and the pack as pv.remap_device
runs them."""
import numpy as np

import time_map_emu as tme

eh = tme.eh


def relink(tid, pk, tid_map, tau, ntracks=None):
    """pvk_track_relink of the time-mapped id table ``tid_map`` ``[len(tau), K]`` of the source ``tid`` /
    ``pk``: (tid', link', ntracks').  The outputs start as sentinels, so a slot the kernels do not write
    fails."""
    L = eh.lib()
    tid = np.ascontiguousarray(tid, dtype=np.int32)
    F, K = tid.shape
    tau = np.ascontiguousarray(tau, dtype=np.float64)
    tid_map = np.ascontiguousarray(tid_map, dtype=np.int32)
    B = tau.size
    nt = len(pk["tstart"]) if ntracks is None else int(ntracks)
    tid_out = np.full((B, K), -99, dtype=np.int32)
    link = np.full((B, K), -99, dtype=np.int32)
    ntr = np.full(1, -7, dtype=np.int32)
    wsb = int(L.pvk_track_relink_workspace_bytes(F, K, B))
    ws = np.zeros(max(wsb, 8), dtype=np.uint8)
    arrs = [np.ascontiguousarray(pk[n], dtype=dt) for n, dt in (("tstart", np.int32), ("tlen", np.int32),
                                                                ("toff", np.int64))]
    eh.check(L.pvk_track_relink(eh.ptr(tid), F, K, nt, *(eh.ptr(a) for a in arrs), eh.ptr(tid_map), eh.ptr(tau), B,
                                eh.ptr(tid_out), eh.ptr(link), eh.ptr(ntr), eh.ptr(ws), wsb, None))
    return tid_out, link, int(ntr[0])


def remap_pack(tid, pk, tau):
    """The remap as pv.remap_device runs it: (tid', link', pk', stats), ``stats`` = (points, last output
    row with a point, partials) of pvk_track_stats."""
    L = eh.lib()
    tm, fm, mm, rm = tme.time_map(tid, pk, tau)
    tid_r, link, nt = relink(tid, pk, tm, tau)
    B, K = tid_r.shape
    stats = np.full((3, 1), -77, dtype=np.int64)
    ntd = np.array([nt], dtype=np.int32)
    eh.check(L.pvk_track_stats(eh.ptr(tid_r), eh.ptr(ntd), 1, B, K, eh.ptr(stats), None))
    pkr = eh.track_pack(fm, mm, rm, rm, tid_r, None, nt)
    return tid_r, link, pkr, tuple(int(x) for x in stats[:, 0])
