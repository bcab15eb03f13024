"""float64 numpy model of the formant gains of the resynthesis (DESIGN.md 4.3), the reference of
``pvk_formant_gains`` in the tests.

Row ``j`` of a peak table: its knots are the slots with ``tid >= 0``, sorted by frequency with ties in
column order; ``L_j`` is ``np.interp`` of ``ln(mag)`` over their frequencies (held at the end values
outside).  A point ``(f, m)`` of the row takes ``m * exp(L_j(f * q_j) - L_j(f))``, and exactly ``m``
where ``f * q_j == f``."""
import numpy as np


def row_gains(f, m, q):
    """Gained magnitudes of the points ``(f, m)`` of one row (in column order), ratio ``q``."""
    f = np.asarray(f, dtype=np.float64)
    m = np.asarray(m, dtype=np.float64)
    if f.size == 0:
        return m.copy()
    order = np.argsort(f, kind="stable")
    xs, ys = f[order], np.log(m[order])
    x = f * q
    out = m * np.exp(np.interp(x, xs, ys) - np.interp(f, xs, ys))
    return np.where(x == f, m, out)


def ratio_rows(q, F):
    """``q`` (scalar or one per row) as one float64 per row."""
    q = np.asarray(q, dtype=np.float64)
    return np.full(F, float(q)) if q.ndim == 0 else q


def gained_table(tid, f, mag, q):
    """``[F, K]`` magnitudes with every slot of a partial gained; other slots as given."""
    tid = np.asarray(tid)
    out = np.array(mag, dtype=np.float64, copy=True)
    qr = ratio_rows(q, tid.shape[0])
    for j in range(tid.shape[0]):
        c = np.nonzero(tid[j] >= 0)[0]
        out[j, c] = row_gains(f[j, c], mag[j, c], qr[j])
    return out


def gained_packed(tid, pk, q):
    """The packed magnitudes of ``pk`` (pvk_track_pack's layout: point ``toff[v] + j - tstart[v]``) gained."""
    tid = np.asarray(tid)
    out = np.array(pk["pmag"], dtype=np.float64, copy=True)
    qr = ratio_rows(q, tid.shape[0])
    for j in range(tid.shape[0]):
        c = np.nonzero(tid[j] >= 0)[0]
        v = tid[j, c].astype(np.int64)
        i = pk["toff"][v] + j - pk["tstart"][v].astype(np.int64)
        out[i] = row_gains(pk["pf"][i], pk["pmag"][i], qr[j])
    return out
