"""float64 numpy model of the time map of the resynthesis (DESIGN.md 4.3, "Time map"): the partials of a
packed table resampled onto the output rows of a non-decreasing map ``tau`` of fractional frames.

Output row ``b`` reads frame row ``i = floor(tau[b])`` at ``u = tau[b] - i``: every slot keeps its partial
id, a point's frequency and magnitude become ``x0 + u * (x1 - x0)`` with ``x0`` / ``x1`` the partial's knots
at rows ``i`` / ``i + 1`` (``x1 = x0`` past its last knot, as ``np.interp``), and its realph is the lower
knot's.  Slots without a point are ``-1`` with zero values."""
import numpy as np


def time_map(tid, pk, tau):
    """(tid', f', mag', realph') ``[len(tau), K]`` of the id table ``tid [F, K]`` and its pack ``pk``
    (tstart / tlen / toff / pf / pmag / prealph) under the map ``tau``."""
    tid = np.asarray(tid)
    tau = np.asarray(tau, dtype=np.float64)
    B, K = len(tau), tid.shape[1]
    i = np.floor(tau).astype(np.int64)
    u = tau - np.floor(tau)
    src = tid[i]                                                   # [B, K]
    present = src >= 0
    v = np.where(present, src, 0).astype(np.int64)
    ts = np.asarray(pk["tstart"], dtype=np.int64)
    tl = np.asarray(pk["tlen"], dtype=np.int64)
    toff = np.asarray(pk["toff"], dtype=np.int64)
    k = i[:, None] - ts[v]
    o = np.where(present, toff[v] + k, 0)
    o1 = np.where(present & (k + 1 < tl[v]), o + 1, o)
    uu = np.broadcast_to(u[:, None], (B, K))
    pf, pmag, pr = (np.asarray(pk[n], dtype=np.float64) for n in ("pf", "pmag", "prealph"))
    if len(pf) == 0:                                               # no points: every slot is empty
        pf = pmag = pr = np.zeros(1)

    def lerp(x):
        x0, x1 = x[o], x[o1]
        return np.where(present, x0 + uu * (x1 - x0), 0.0)
    return (np.where(present, src, -1).astype(np.int32), lerp(pf), lerp(pmag),
            np.where(present, pr[o], 0.0))


def speed_map(speed, F):
    """The map of a per-output-block speed curve (input frames per output block): the running sum of
    ``speed`` from 0, cut where it passes ``F - 1``."""
    tau = np.concatenate([[0.0], np.cumsum(np.asarray(speed, dtype=np.float64))])
    return tau[tau <= F - 1]


def example_maps(F):
    """Every kind of map of a table of ``F >= 8`` rows the tests run, by name: the identity, a freeze,
    a constant fractional rate, jumps over whole rows, a map that starts late and ends early, one that
    ends exactly on the last row, and a single output row."""
    return dict(identity=np.arange(F, dtype=np.float64),
                freeze=np.concatenate([np.arange(0.0, 4.0), np.full(5, 4.0), np.arange(4.0, F)]),
                rate037=np.arange(0.0, F - 1, 0.37),
                jump35=np.arange(0.0, F - 1, 3.5),
                late_early=np.linspace(2.25, F - 3.5, 17),
                to_last=np.linspace(0.0, F - 1, 2 * F - 3),
                one_row=np.array([F / 2.0 + 0.3]))


def check_bits(got, ref):
    """Assert that the tables (tid', f', mag', realph') ``got`` equal ``ref`` bit for bit."""
    for g, r, name in zip(got, ref, ("tid", "f", "mag", "realph")):
        g, r = np.asarray(g), np.asarray(r)
        assert g.shape == r.shape, name
        if g.dtype.kind == "f":
            assert np.array_equal(g.view(np.int64), r.view(np.int64)), name   # -0.0 != 0.0, NaN fails
        else:
            assert np.array_equal(g, r), name
