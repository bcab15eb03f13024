"""float64 numpy model of the remap of the partials (DESIGN.md 4.3, "Remap"): the time map of
tests/time_map_oracle.py under a map ``tau`` in ANY order, with every source partial split into its runs of
consecutive output rows and the runs numbered as partials.

Slot ``(b, c)`` holding source partial ``v`` continues the run of ``v`` when ``b > 0`` and output row
``b - 1`` holds ``v``, i.e. ``tstart[v] <= floor(tau[b - 1]) <= end[v]``; otherwise it starts a new run.
Runs are numbered in ascending order of (first output row, source id)."""
import numpy as np

import time_map_oracle as tmo


def relink(tid_map, tau, pk):
    """(link', tid', ntracks') of the time-mapped id table ``tid_map`` ``[B, K]`` (source ids) of the map
    ``tau`` and the source pack ``pk``: link' in pvk_track's encoding (column in row b - 1, -1 = not a
    point, -2 - rank = new run of that rank among the row's new runs by source id) and the run ids."""
    tid_map = np.asarray(tid_map)
    B, K = tid_map.shape
    i = np.floor(np.asarray(tau, dtype=np.float64)).astype(np.int64)
    ts = np.asarray(pk["tstart"], dtype=np.int64)
    end = ts + np.asarray(pk["tlen"], dtype=np.int64) - 1
    present = tid_map >= 0
    v = np.where(present, tid_map, 0)
    ip = np.concatenate([[-1], i[:-1]])[:, None]
    cont = present & (ip >= 0) & (ts[v] <= ip) & (ip <= end[v])
    new = present & ~cont
    link = np.where(present, 0, -1).astype(np.int32)
    tid = np.full((B, K), -1, dtype=np.int32)
    rows, cols = np.nonzero(new)                                   # row-major: rows ascend
    order = np.lexsort((tid_map[rows, cols], rows))                # by (first output row, source id)
    ids = np.empty(len(order), dtype=np.int64)
    ids[order] = np.arange(len(order))
    tid[rows, cols] = ids
    first = np.searchsorted(rows[order], rows[order], side="left")  # id of the first new run of each row
    link[rows[order], cols[order]] = -2 - (np.arange(len(order)) - first)
    colof = np.full(max(int(tid_map.max()) + 1, 1) if tid_map.size else 1, -1, dtype=np.int64)
    for b in range(1, B):
        prev = tid_map[b - 1]
        pc = np.nonzero(prev >= 0)[0]
        colof[prev[pc]] = pc
        cc = np.nonzero(cont[b])[0]
        src = colof[tid_map[b, cc]]
        assert (src >= 0).all()
        link[b, cc] = src
        tid[b, cc] = tid[b - 1, src]
        colof[prev[pc]] = -1
    return link, tid, len(order)


def pack(tid, f, mag, realph, ntracks):
    """pvk_track_pack's layout of the id table ``tid`` (ids kept): tstart, tlen, toff and the packed
    f / mag / realph (ph = realph) of every partial, rows ascending."""
    rows, cols = np.nonzero(tid >= 0)
    v = tid[rows, cols].astype(np.int64)
    srt = np.lexsort((rows, v))
    rows, cols, v = rows[srt], cols[srt], v[srt]
    cnt = np.bincount(v, minlength=ntracks)
    toff = np.zeros(ntracks + 1, dtype=np.int64)
    toff[1:] = np.cumsum(cnt)
    tstart = rows[toff[:-1][cnt > 0]] if ntracks else np.zeros(0, dtype=np.int64)
    assert (cnt > 0).all()                                         # every run holds a point
    for n in range(ntracks):                                       # one slot per row, consecutive rows
        r = rows[toff[n]:toff[n + 1]]
        assert np.array_equal(r, np.arange(r[0], r[0] + len(r)))
    return dict(tstart=tstart.astype(np.int32), tlen=cnt.astype(np.int32), toff=toff,
                pf=f[rows, cols], pmag=mag[rows, cols], prealph=realph[rows, cols])


def remap(tid, pk, tau):
    """The remapped partials of ``tid [F, K]`` / ``pk`` under ``tau``: (tid', link', pk', tables), tables =
    (f', mag', realph') ``[B, K]`` of the time map."""
    tm, f, mag, rp = tmo.time_map(tid, pk, tau)
    link, tid_r, nt = relink(tm, tau, pk)
    return tid_r, link, pack(tid_r, f, mag, rp, nt), (f, mag, rp)


def check_pack(got, ref):
    """Assert that two packs are equal bit for bit (tstart, tlen, toff, pf, pmag, prealph and pph = prealph)."""
    for n in ("tstart", "tlen", "toff", "pf", "pmag", "prealph"):
        g, r = np.asarray(got[n]), np.asarray(ref[n])
        assert g.shape == r.shape, n
        if g.dtype.kind == "f":
            assert np.array_equal(g.view(np.int64), r.view(np.int64)), n
        else:
            assert np.array_equal(g, r), n
    if "pph" in got:
        assert np.array_equal(np.asarray(got["pph"]).view(np.int64), np.asarray(ref["prealph"]).view(np.int64))


def remap_maps(F):
    """The non-monotone maps of a table of ``F >= 12`` rows the tests run, by name: a full reverse, a
    sawtooth loop, a ping-pong, a random-walk scrub with fractional steps, a jump back onto a row where
    some partials persist and some do not, and a single row."""
    rng = np.random.default_rng(F)
    lo, hi = F // 3, (2 * F) // 3
    walk = np.clip(np.cumsum(np.concatenate([[F / 2.0], rng.normal(0.0, 0.9, 3 * F)])), 0.0, F - 1.0)
    return dict(reverse=np.arange(F - 1, -1, -1.0),
                loop=np.concatenate([np.arange(0.0, hi + 1.0), np.tile(np.arange(lo, hi + 1.0), 3),
                                     np.arange(hi + 1.0, F)]),
                pingpong=np.concatenate([np.arange(0.0, hi, 0.75), np.arange(hi, lo, -0.5), np.arange(lo, F - 1.0, 1.25)]),
                scrub=walk,
                jump_back=np.concatenate([np.arange(0.0, F - 2.0), np.arange(F // 2, F, 1.0)]),
                one_row=np.array([F / 2.0 + 0.4]))


def all_maps(F):
    """remap_maps() and every map of time_map_oracle.example_maps()."""
    d = dict(remap_maps(F))
    d.update(("mono_" + k, v) for k, v in tmo.example_maps(F).items())
    return d
