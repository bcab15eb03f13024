"""Host side of the B200 phase vocoder: drop-in mirrors of ``pypevoc.PV`` and
``pypevoc.SinSum`` (reference pypevoc/PVAnalysis.py:71-417, 585-756, 797-1111).

Same constructor arguments, method names, attribute names, array shapes and dtypes as the
reference, so code written against ``pypevoc.PVAnalysis.PV`` runs unchanged:

    from pypevoc_b200 import PV
    pv = PV(sig, sr, nfft=2048, hop=512, npks=50); pv.run_pv()
    pv.f, pv.mag, pv.ph, pv.realph, pv.binno     # float64 [nframes, npks], zero padded
    ss = pv.toSinSum(); w = ss.synth(sr, pv.hop)

All arithmetic of the hot path runs in libpvk.so (hand written sm_100a kernels) through the
C ABI of include/pvk.h; torch is used only for device memory, streams and copies.  There is
no CPU fallback: without a CUDA device or without the built extension every compute call
raises.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib

pi2 = 2.0 * np.pi


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _device(device=None):
    if not torch.cuda.is_available():
        raise RuntimeError("pypevoc_b200 needs a CUDA device (B200); there is no CPU fallback")
    if device is None:
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device(device)


_side = {}
TRACE = None     # set to a list to collect (label, cuda event) marks of the streamed pipeline (diagnostics)


def _mark(label, stream):
    if TRACE is not None:
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(stream)
        TRACE.append((label, ev))



def _side_streams(dev):
    """(host->device, device->host) copy streams of a device, created once."""
    st = _side.get(dev.index)
    if st is None:
        st = (torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev))
        _side[dev.index] = st
    return st


def _pinned(hostbuf, key, shape, dtype):
    """Reusable pinned host tensor ``hostbuf[key]`` of at least ``shape`` (first dimension may be
    larger: buffers are kept across calls and only grow)."""
    hb = hostbuf.get(key)
    if (hb is None or hb.dtype != dtype or hb.dim() != len(shape) or tuple(hb.shape[1:]) != tuple(shape[1:])
            or hb.shape[0] < shape[0]):
        hb = torch.empty(shape, dtype=dtype, device="cpu", pin_memory=True)
        hostbuf[key] = hb
    return hb


def _chunk_bounds(n, chunks):
    """Boundaries of ``chunks`` consecutive pieces of ``n`` items for a copy-bound pipeline: a short first
    piece (the kernels start early), a short last one (little is left to do once the last upload has
    landed), the rest in the middle -- weights 1 2 ... 2 1."""
    if chunks <= 2:
        return [(n * i) // chunks for i in range(chunks + 1)]
    w = [1] + [2] * (chunks - 2) + [1]
    tot, acc, out = float(sum(w)), 0, [0]
    for v in w:
        acc += v
        out.append(int(round(n * acc / tot)))
    out[-1] = n
    return out


class Progress(object):
    """Minimal stand-in for pypevoc.ProgressDisplay.Progress (ProgressDisplay.py:58-117):
    the GPU path finishes in one launch, so only completion is reported."""

    def __init__(self, end=100):
        self.end = end
        self.value = 0

    def update(self, value):
        self.value = value


_table_cache = {}


def _analysis_tables(nfft, dev):
    """Twiddle tables of libpvk for (device, nfft), built once by pvk_analyze_init."""
    key = (dev.index, nfft)
    tab = _table_cache.get(key)
    if tab is None:
        L = _lib.lib()
        nbytes = L.pvk_analyze_tables_bytes(nfft)
        if nbytes <= 0:
            raise ValueError("nfft=%r is not supported by the CUDA kernels: it must be a power of two "
                             "in [64, 8192]" % (nfft,))
        tab = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.check(L.pvk_analyze_init(nfft, _ptr(tab), _stream()), "pvk_analyze_init")
        _table_cache[key] = tab
    return tab


def n_frames(nsamp, nfft, hop):
    """Number of iterations of run_pv's ``while curpos < nsamp - nfft`` (PVAnalysis.py:223-225)."""
    span = nsamp - nfft
    return 0 if span <= 0 else -(-span // hop)


def host_tables(sr, nfft, hop, wind=np.hanning):
    """Window / normalisation / per-bin tables, evaluated on the host with the reference's own
    numpy expressions (PVAnalysis.py:97-118) so that the unwrapping constants are bit-identical."""
    win = wind(nfft)
    wsum = sum(win)
    wsum2 = sum(win ** 2)
    wfact = np.sqrt(wsum2 * nfft) / 2.0
    fstep = float(sr) / float(nfft)
    dt = float(hop) / float(sr)
    fbin = np.arange(float(nfft)) * fstep
    dthetabin = pi2 * fbin * dt
    wfbin = np.round(dthetabin / pi2) * pi2
    return dict(win=win, wsum=wsum, wsum2=wsum2, wfact=wfact, fstep=fstep, dt=dt, fbin=fbin, wfbin=wfbin)


def analyze_device(xd, sr, nfft, hop, npks, pkthresh, tb, frame0=0, nframes=None, prev_zero=True,
                   run_frames=0, spectra=False, out=None, refine=False, out_rows=None):
    """Launch pvk_analyze on a device signal.

    ``xd``: float32 CUDA tensor, ``[nsamp]`` or ``[nclips, nsamp]``.  Returns a dict of device
    tensors ``f mag ph realph binno`` (float64 ``[nclips, nframes, npks]``), ``npk`` (int32),
    ``totalmag`` (float64) and optionally ``fx`` (complex64 ``[nclips, nframes, nfft/2]``);
    ``refine=True`` adds ``fine_pos`` / ``fine_val`` (PeakFinder.refine of every emitted peak,
    PeakFinder.py:331-372).  ``out_rows`` (>= nframes; pvk_analyze_batch): the tables get
    ``out_rows`` rows per clip, the rows beyond ``nframes`` are zero guard rows (clip batches that
    go on to tracking / resynthesis as ONE flattened table).  Asynchronous on the current stream.
    """
    L = _lib.lib()
    if xd.dim() == 1:
        xd = xd.unsqueeze(0)
    assert xd.dtype == torch.float32 and xd.is_cuda and xd.stride(1) == 1
    dev = xd.device
    nclips, nsamp = xd.shape
    if nframes is None:
        nframes = max(n_frames(nsamp, nfft, hop) - frame0, 0)
    key = ("dev", dev.index)
    if key not in tb:
        tb[key] = dict(
            win=torch.from_numpy(np.ascontiguousarray((tb["win"] / tb["wfact"]).astype(np.float32))).to(dev),
            fbin=torch.from_numpy(np.ascontiguousarray(tb["fbin"], dtype=np.float64)).to(dev),
            wfbin=torch.from_numpy(np.ascontiguousarray(tb["wfbin"], dtype=np.float64)).to(dev))
    dtb = tb[key]
    tables = _analysis_tables(nfft, dev)
    rows = int(nframes if out_rows is None else out_rows)
    assert rows >= nframes and not (spectra and rows != nframes)
    if out is None:
        out = {}
        for k in ("f", "mag", "ph", "realph", "binno"):
            out[k] = torch.empty((nclips, rows, npks), dtype=torch.float64, device=dev)
        out["npk"] = torch.empty((nclips, rows), dtype=torch.int32, device=dev)
        out["totalmag"] = torch.empty((nclips, rows), dtype=torch.float64, device=dev)
        if rows > nframes:                                    # guard rows: zero (memset-like strided fills)
            for v in out.values():
                v[:, nframes:].zero_()
    spec = torch.empty((nclips, nframes, nfft // 2), dtype=torch.complex64, device=dev) if spectra else None
    if refine and "fine_pos" not in out:
        out["fine_pos"] = torch.empty((nclips, nframes, npks), dtype=torch.float64, device=dev)
        out["fine_val"] = torch.empty((nclips, nframes, npks), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.pvk_analyze_batch(
            _ptr(xd), nclips, xd.stride(0), nsamp, _ptr(dtb["win"]), _ptr(dtb["fbin"]), _ptr(dtb["wfbin"]),
            _ptr(tables), int(nfft), int(hop), int(npks), float(pkthresh), float(tb["dt"]), float(tb["fstep"]),
            int(frame0), int(nframes), 1 if prev_zero else 0, int(run_frames),
            _ptr(out["f"]), _ptr(out["mag"]), _ptr(out["ph"]), _ptr(out["realph"]), _ptr(out["binno"]),
            _ptr(out["npk"]), _ptr(out["totalmag"]), _ptr(spec),
            _ptr(out["fine_pos"]) if refine else None, _ptr(out["fine_val"]) if refine else None,
            rows, _stream()), "pvk_analyze")
    if spectra:
        out["fx"] = spec
    return out


def _device_tables(tb, dev):
    key = ("dev", dev.index)
    if key not in tb:
        tb[key] = dict(
            win=torch.from_numpy(np.ascontiguousarray((tb["win"] / tb["wfact"]).astype(np.float32))).to(dev),
            fbin=torch.from_numpy(np.ascontiguousarray(tb["fbin"], dtype=np.float64)).to(dev),
            wfbin=torch.from_numpy(np.ascontiguousarray(tb["wfbin"], dtype=np.float64)).to(dev))
    return tb[key]


def harmonic_device(xd, sr, nfft, hop, npks, f0d, tb, fmin=30.0, nframes=None, run_frames=0):
    """Launch pvk_harmonic (PVHarmonic.run_pv, PVAnalysis.py:419-538) on a 1-D float32 device
    signal with one float64 device f0 value per frame.  Returns device ``f mag ph``
    (float64 ``[nframes, npks]``), ``residuals`` (float64), ``nharm`` (int32).  Asynchronous."""
    L = _lib.lib()
    assert xd.dtype == torch.float32 and xd.is_cuda and xd.dim() == 1 and xd.is_contiguous()
    dev = xd.device
    nsamp = xd.shape[0]
    if nframes is None:
        nframes = n_frames(nsamp, nfft, hop)
    assert f0d.dtype == torch.float64 and f0d.is_cuda and f0d.is_contiguous() and f0d.numel() >= nframes
    dtb = _device_tables(tb, dev)
    tables = _analysis_tables(nfft, dev)
    out = {k: torch.empty((nframes, npks), dtype=torch.float64, device=dev) for k in ("f", "mag", "ph")}
    out["residuals"] = torch.empty((nframes,), dtype=torch.float64, device=dev)
    out["nharm"] = torch.empty((nframes,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.pvk_harmonic(
            _ptr(xd), nsamp, _ptr(dtb["win"]), _ptr(dtb["fbin"]), _ptr(dtb["wfbin"]), _ptr(tables), int(nfft),
            int(hop), int(npks), float(tb["dt"]), float(sr), float(fmin), _ptr(f0d), int(nframes), int(run_frames),
            _ptr(out["f"]), _ptr(out["mag"]), _ptr(out["ph"]), _ptr(out["residuals"]), _ptr(out["nharm"]),
            _stream()), "pvk_harmonic")
    return out


def frame_stats_device(fd, magd, fmin=50, fmax=10000, thr=0.1):
    """pvk_frame_stats on device tables ``[F, K]``: (fm, fundamental_idx, partial_sum_magnitude)
    = PV.calc_f0 (PVAnalysis.py:371-391) and PV.partial_sum_magnitude (:411-413).  Asynchronous."""
    L = _lib.lib()
    assert fd.dtype == torch.float64 and fd.is_contiguous() and magd.is_contiguous() and fd.dim() == 2
    dev = fd.device
    F, K = fd.shape
    fm = torch.empty((F,), dtype=torch.float64, device=dev)
    idx = torch.empty((F,), dtype=torch.int32, device=dev)
    ps = torch.empty((F,), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.pvk_frame_stats(_ptr(fd), _ptr(magd), F, K, float(fmin), float(fmax), float(thr), _ptr(fm),
                                     _ptr(idx), _ptr(ps), _stream()), "pvk_frame_stats")
    return fm, idx, ps


def harmonic_power_device(fd, magd, f_threshold=0.01):
    """pvk_harmonic_power on device tables ``[F, K]``: (hpower, nharmonics) float64 ``[F, K]`` and
    the int32 out-of-range flag = PV.calc_harmonic_power (PVAnalysis.py:266-297).  Asynchronous."""
    L = _lib.lib()
    assert fd.dtype == torch.float64 and fd.is_contiguous() and magd.is_contiguous() and fd.dim() == 2
    dev = fd.device
    F, K = fd.shape
    hp = torch.empty((F, K), dtype=torch.float64, device=dev)
    nh = torch.empty((F, K), dtype=torch.float64, device=dev)
    rowpow = torch.empty((max(min(F, K), 1),), dtype=torch.float64, device=dev)
    err = torch.zeros((1,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.pvk_harmonic_power(_ptr(fd), _ptr(magd), F, K, float(f_threshold), _ptr(rowpow), _ptr(hp),
                                        _ptr(nh), _ptr(err), _stream()), "pvk_harmonic_power")
    return hp, nh, err


def track_device(fd, magd, maxpitchjmp=0.5):
    """pvk_track on device tables ``[nclips, F, K]`` (or ``[F, K]``); returns device ``tid``,
    ``link`` (int32, same shape) and ``ntracks`` (int32 ``[nclips]``).  Asynchronous."""
    L = _lib.lib()
    squeeze = fd.dim() == 2
    if squeeze:
        fd, magd = fd.unsqueeze(0), magd.unsqueeze(0)
    assert fd.dtype == torch.float64 and fd.is_contiguous() and magd.is_contiguous()
    dev = fd.device
    nclips, F, K = fd.shape
    tid = torch.empty((nclips, F, K), dtype=torch.int32, device=dev)
    link = torch.empty((nclips, F, K), dtype=torch.int32, device=dev)
    ntracks = torch.empty((nclips,), dtype=torch.int32, device=dev)
    wsb = L.pvk_track_workspace_bytes(nclips, F, K)
    ws = torch.empty(max(int(wsb), 8), dtype=torch.uint8, device=dev)
    stats = torch.empty((3, nclips), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.pvk_track(_ptr(fd), _ptr(magd), nclips, F, K, float(maxpitchjmp), _ptr(tid), _ptr(link),
                               _ptr(ntracks), _ptr(ws), int(wsb), _stream()), "pvk_track")
        _lib.check(L.pvk_track_stats(_ptr(tid), _ptr(ntracks), nclips, F, K, _ptr(stats), _stream()),
                   "pvk_track_stats")
    if squeeze:
        tid, link = tid[0], link[0]
    return dict(tid=tid, link=link, ntracks=ntracks, stats=stats)


def track_counts(tr, clip=0):
    """(number of partials, number of points, last frame holding a point) of one clip of a
    track_device() result: ONE 24-byte device->host read-back (synchronises the stream)."""
    s = tr["stats"][:, clip].cpu()
    return int(s[2]), int(s[0]), int(s[1])


def pack_device(fd, magd, phd, realphd, tid, link, ntracks, npts=None):   # link: unused, kept for call sites
    """pvk_track_pack for one clip (``[F, K]`` device tables, ``ntracks`` python int; ``npts`` =
    number of points from track_counts(), counted here when not given)."""
    L = _lib.lib()
    dev = fd.device
    F, K = fd.shape
    if npts is None:
        npts = int((tid >= 0).sum().item()) if F * K else 0
    nt = int(ntracks)
    tstart = torch.empty((max(nt, 1),), dtype=torch.int32, device=dev)
    tlen = torch.empty((max(nt, 1),), dtype=torch.int32, device=dev)
    toff = torch.empty((nt + 1,), dtype=torch.int64, device=dev)
    packed = [torch.empty((max(npts, 1),), dtype=torch.float64, device=dev) for _ in range(4)]
    wsb = int(L.pvk_track_pack_workspace_bytes(nt))
    ws = torch.empty(max(wsb, 8), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.pvk_track_pack(_ptr(fd), _ptr(magd), _ptr(phd), _ptr(realphd), _ptr(tid), F, K, nt,
                                    _ptr(tstart), _ptr(tlen), _ptr(toff), _ptr(packed[0]), _ptr(packed[1]),
                                    _ptr(packed[2]), _ptr(packed[3]), _ptr(ws), wsb, _stream()), "pvk_track_pack")
    return dict(tstart=tstart[:nt], tlen=tlen[:nt], toff=toff, pf=packed[0][:npts], pmag=packed[1][:npts],
                pph=packed[2][:npts], prealph=packed[3][:npts], npts=npts)


PACK_SPEC_CAP = 4 << 20      # most partials a speculative pack is sized for (larger tables are re-packed)


def _pack_speculative(fd, magd, phd, realphd, tr):
    """Launch pvk_track_pack_dev sized by upper bounds (the exact counts still sit on the device):
    returns (capacity, tstart, tlen, toff, packed arrays)."""
    L = _lib.lib()
    dev = fd.device
    F, K = fd.shape
    nt_ub = min(F * K, PACK_SPEC_CAP)
    tstart = torch.empty((nt_ub,), dtype=torch.int32, device=dev)
    tlen = torch.empty((nt_ub,), dtype=torch.int32, device=dev)
    toff = torch.empty((nt_ub + 1,), dtype=torch.int64, device=dev)
    packed = [torch.empty((F * K,), dtype=torch.float64, device=dev) for _ in range(4)]
    wsb = int(L.pvk_track_pack_workspace_bytes(nt_ub))
    ws = torch.empty(max(wsb, 8), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.pvk_track_pack_dev(_ptr(fd), _ptr(magd), _ptr(phd), _ptr(realphd), _ptr(tr["tid"]), F, K, nt_ub,
                                        _ptr(tr["ntracks"]), _ptr(tstart), _ptr(tlen), _ptr(toff), _ptr(packed[0]),
                                        _ptr(packed[1]), _ptr(packed[2]), _ptr(packed[3]), _ptr(ws), wsb, _stream()),
                   "pvk_track_pack")
    return nt_ub, tstart, tlen, toff, packed


def _pack_sliced(raw, nt, npts):
    _, tstart, tlen, toff, packed = raw
    return dict(tstart=tstart[:nt], tlen=tlen[:nt], toff=toff[:nt + 1], pf=packed[0][:npts], pmag=packed[1][:npts],
                pph=packed[2][:npts], prealph=packed[3][:npts], npts=npts)


def track_pack_device(fd, magd, phd, realphd, maxpitchjmp=0.5, after_link=None):
    """pvk_track + pvk_track_pack of one clip with ONE host read-back: the pack is launched with
    upper bounds for the number of partials / points (the exact counts still sit on the device)
    before the host waits for them, so the device does not idle while the host sizes and
    launches it; the few KB of over-allocated index arrays are sliced afterwards.  ``after_link``
    (optional) is called with the track dict right after the link kernels are launched.
    Returns (tr, pk) as track_device() + track_counts() and pack_device() give them."""
    tr = track_device(fd, magd, maxpitchjmp)
    if after_link is not None:
        after_link(tr)
    F, K = fd.shape
    raw = _pack_speculative(fd, magd, phd, realphd, tr) if F * K > 0 else None
    nt, npts, last = track_counts(tr)
    tr["ntracks_dev"] = tr["ntracks"]
    tr["ntracks"], tr["npts"], tr["max_end"] = nt, npts, last
    if raw is not None and 0 < nt <= raw[0]:
        pk = _pack_sliced(raw, nt, npts)
    elif nt == 0:
        pk = None
    else:                                                       # more partials than the speculative cap
        pk = pack_device(fd, magd, phd, realphd, tr["tid"], None, nt, npts=npts)
    return tr, pk


class _DeviceCurve(object):
    """A frequency-ratio curve that synth_mode() has checked, uploaded once per call: ``t`` is a
    float64 CUDA tensor with one ratio per frame row of the table it goes with."""
    __slots__ = ("t",)

    def __init__(self, t):
        self.t = t


def _curve_values(fscale):
    """float64 numpy copy of a ratio curve of any shape, every value finite and > 0."""
    if isinstance(fscale, torch.Tensor):
        if fscale.dtype == torch.bool or fscale.is_complex():
            raise TypeError("an fscale curve must hold real numbers, not %s" % fscale.dtype)
        a = fscale.detach().cpu().numpy()
    else:
        a = np.asarray(fscale)
    if a.dtype.kind not in "iuf":
        raise TypeError("an fscale curve must hold real numbers, not %s" % a.dtype)
    a = np.ascontiguousarray(a, dtype=np.float64)
    if not np.all(np.isfinite(a)) or np.any(a <= 0.0):
        raise ValueError("every value of an fscale curve must be finite and > 0")
    return a


def synth_mode(phase_preserve=True, fscale=1.0, nframes=None):
    """Checked (phase_preserve, fscale) of a resynthesis call.  ``phase_preserve=False`` integrates the
    phase from the frequency track (pitch shift by ``fscale``, time stretch by a synthesis hop other
    than the analysis hop); the phase-preserving model honours the analysed phases and so takes no
    ``fscale`` other than 1.

    ``fscale`` is one ratio for the whole signal, or a curve: a 1-D numpy array, sequence or torch
    tensor of ``nframes`` real ratios, one per analysis frame (row of the frame table), returned as a
    float64 numpy array.  Ratio ``r[b]`` applies to every partial in output block ``b`` (output samples
    ``[b*hop, (b+1)*hop)``, input samples ``[b*hop_an, (b+1)*hop_an)``); the phase stays continuous
    and the frequency steps by ``r[b+1] / r[b]`` between blocks (DESIGN.md 4.3).  To build one from
    time, use the input time of the frame rows, ``r = ratio_of(np.arange(nframes) * hop_an / sr)``
    (not ``PV.t``, which is offset by ``nfft / 2``).  A curve needs ``phase_preserve=False``."""
    if isinstance(fscale, _DeviceCurve):
        if phase_preserve:
            raise ValueError("an fscale curve needs phase_preserve=False")
        if nframes is not None and fscale.t.numel() != nframes:
            raise ValueError("the fscale curve has %d ratios for %d frames" % (fscale.t.numel(), nframes))
        return False, fscale
    if isinstance(fscale, (np.ndarray, torch.Tensor, list, tuple)):
        r = _curve_values(fscale)
        if r.ndim != 1:
            raise ValueError("an fscale curve must be 1-D (one ratio per frame), not of shape %s" % (r.shape,))
        if nframes is not None and len(r) != nframes:
            raise ValueError("the fscale curve has %d ratios for %d frames" % (len(r), nframes))
        if phase_preserve:
            raise ValueError("an fscale curve needs phase_preserve=False: the analysed phases cannot be honoured "
                             "at a scaled frequency")
        return False, r
    if isinstance(fscale, bool) or not isinstance(fscale, (int, float, np.integer, np.floating)):
        raise TypeError("fscale must be a real number, not %s" % type(fscale).__name__)
    fscale = float(fscale)
    if not np.isfinite(fscale) or fscale <= 0.0:
        raise ValueError("fscale=%r must be finite and > 0" % fscale)
    phase_preserve = bool(phase_preserve)
    if phase_preserve and fscale != 1.0:
        raise ValueError("fscale=%r needs phase_preserve=False: the analysed phases cannot be honoured at a "
                         "scaled frequency" % fscale)
    return phase_preserve, fscale


def _on_device(fscale, dev):
    """fscale as the kernels take it: a float, or a checked curve (numpy) uploaded as float64."""
    if isinstance(fscale, np.ndarray):
        return _DeviceCurve(torch.from_numpy(fscale).to(dev))
    return fscale


def _phase_ws(phase_preserve, npts, dev):
    """Scratch of the integrated-phase scan: one double per packed point (None when preserving phase)."""
    if phase_preserve:
        return None
    return torch.empty((max(int(npts), 1),), dtype=torch.float64, device=dev)


def _resynth_ex(L, tid, F, K, nt, nt_dev, tstart, tlen, toff, pf, pmag, prealph, sr, hop, nfft, hop_an, edge, minframes,
                out, nout, block0, nblocks, ws, reuse_tracks, phase_preserve, fscale, phase_ws, scanned=False):
    # scanned: the block start phases and Nyquist flags are in place already (pvk_resynth_render)
    # fscale: a float, or a _DeviceCurve (the _curve exports, ratio 1 + the curve)
    render = scanned and not reuse_tracks
    if isinstance(fscale, _DeviceCurve):
        fn = L.pvk_resynth_render_curve if render else L.pvk_resynth_ex_curve
        ratio = (1.0, _ptr(fscale.t), int(fscale.t.numel()))
    else:
        fn = L.pvk_resynth_render if render else L.pvk_resynth_ex
        ratio = (float(fscale),)
    _lib.check(fn(_ptr(tid), F, K, nt, _ptr(nt_dev), _ptr(tstart), _ptr(tlen), _ptr(toff), _ptr(pf),
                  _ptr(pmag), _ptr(prealph), float(sr), int(hop), int(nfft), int(hop_an), float(edge),
                  int(minframes), _ptr(out), int(nout), int(block0), int(nblocks), _ptr(ws), int(ws.numel()),
                  1 if reuse_tracks else 0, 1 if phase_preserve else 0, *ratio, _ptr(phase_ws),
                  0 if phase_ws is None else int(phase_ws.numel()), _stream()), "pvk_resynth")


def track_pack_resynth_device(fd, magd, phd, realphd, sr, hop, nfft, hop_an, edge=1.0, minframes=3,
                              maxpitchjmp=0.5, after_link=None, after_pack=None, block_range=None, before_sync=None,
                              phase_preserve=True, fscale=1.0):
    """The whole back half of the hot path of one clip -- link, id resolution, pack, resynthesis --
    queued back to back with ONE host read-back at the very end: pack and resynthesis are launched
    sized by upper bounds (capacity of the index arrays, (F + 1) * hop + edge output samples) and
    read the real number of partials on the device (pvk_track_pack_dev / pvk_resynth_dev); the
    host then reads the 24 bytes of counts and slices.  Returns (tr, pk, w): as track_pack_device()
    plus the float64 device signal (None without partials).  ``block_range`` = (block0, nblocks,
    nout): render only these output blocks of a signal of (at most) ``nout`` samples and return them
    uncut (segment-sharded runs: the caller knows its block range without any count and trims once the
    global last frame is known).  ``before_sync`` (optional) is called once everything is queued,
    before the host waits: work launched there runs behind the rendering instead of after the wait.
    ``phase_preserve`` / ``fscale``: see synth_mode() (a curve has one ratio per row of ``fd``)."""
    phase_preserve, fscale = synth_mode(phase_preserve, fscale, nframes=fd.shape[0])
    fscale = _on_device(fscale, fd.device)
    L = _lib.lib()
    F, K = fd.shape
    if F * K == 0:
        tr, pk = track_pack_device(fd, magd, phd, realphd, maxpitchjmp, after_link)
        return tr, pk, None
    tr = track_device(fd, magd, maxpitchjmp)
    if after_link is not None:
        after_link(tr)
    dev = fd.device
    raw = _pack_speculative(fd, magd, phd, realphd, tr)
    if after_pack is not None:
        after_pack(tr)
    nt_ub, tstart, tlen, toff, packed = raw
    if block_range is None:
        nout_ub, _ = synth_geometry(F - 1, hop, nfft, hop_an, edge)
        b0, nb = 0, -(-nout_ub // hop)
    else:
        b0, nb, nout_ub = (int(v) for v in block_range)
    nsamp_out = max(min(nb * hop, nout_ub - b0 * hop), 0)
    out = torch.empty((nsamp_out,), dtype=torch.float64, device=dev)
    if nsamp_out > 0:
        ws = resynth_workspace(F, K, nt_ub, nb, dev, hop=hop)
        pws = _phase_ws(phase_preserve, F * K, dev)
        with torch.cuda.device(dev):
            _resynth_ex(L, tr["tid"], F, K, nt_ub, tr["ntracks"], tstart, tlen, toff, packed[0], packed[1], packed[3], sr,
                        hop, nfft, hop_an, edge, minframes, out, nout_ub, b0, nb, ws, False, phase_preserve, fscale, pws)
    if before_sync is not None:
        before_sync(tr)
    nt, npts, last = track_counts(tr)                           # the hot path's one read-back
    tr["ntracks_dev"] = tr["ntracks"]
    tr["ntracks"], tr["npts"], tr["max_end"] = nt, npts, last
    if nt == 0:
        return tr, None, (None if block_range is None else out.zero_())
    if nt > nt_ub:                                              # more partials than the speculative cap: redo, sized exactly
        pk = pack_device(fd, magd, phd, realphd, tr["tid"], None, nt, npts=npts)
        mode = dict(phase_preserve=phase_preserve, fscale=fscale)
        if block_range is None:
            return tr, pk, resynth_device(tr["tid"], pk, sr, hop, nfft, hop_an, edge=edge, minframes=minframes, max_end=last,
                                          **mode)
        return tr, pk, resynth_device(tr["tid"], pk, sr, hop, nfft, hop_an, edge=edge, minframes=minframes, block0=b0,
                                      nblocks=nb, nout=nout_ub, out=out, **mode)
    if block_range is not None:
        return tr, _pack_sliced(raw, nt, npts), out
    nout, _ = synth_geometry(last, hop, nfft, hop_an, edge)
    return tr, _pack_sliced(raw, nt, npts), out[:nout]


def spans_device(tid, ntracks):
    """pvk_track_spans: first frame / length of every partial of an id table ``[F, K]`` (device)."""
    L = _lib.lib()
    dev = tid.device
    F, K = tid.shape
    nt = int(ntracks)
    tstart = torch.empty((max(nt, 1),), dtype=torch.int32, device=dev)
    tlen = torch.empty((max(nt, 1),), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.pvk_track_spans(_ptr(tid), F, K, nt, _ptr(tstart), _ptr(tlen), _stream()), "pvk_track_spans")
    return tstart[:nt], tlen[:nt]


def synth_geometry(max_end, hop, nfft, hop_an, edge=1.0):
    """Output length of SinSum.synth (PVAnalysis.py:1055-1059,1070) and the edge length."""
    dfr = nfft / hop_an / 2.
    edgsamp = int(edge * hop * dfr)
    return (max_end + 2) * hop + edgsamp, edgsamp


def resynth_device(tid, pk, sr, hop, nfft, hop_an, edge=1.0, minframes=3, max_end=None, block0=0,
                   nblocks=-1, out=None, ws=None, reuse_tracks=False, nout=None, phase_preserve=True, fscale=1.0,
                   phase_ws=None, scanned=False):
    """pvk_resynth_ex for one clip; returns the float64 device signal (asynchronous).  ``ws``: a
    workspace tensor to (re)use; ``reuse_tracks``: ``ws`` (and ``phase_ws``) already hold the per-partial
    masks, fade parameters (and block start phases) of an earlier call with the same tracks and
    synthesis parameters.  ``phase_preserve`` / ``fscale``: see synth_mode(); ``phase_ws``: the
    integrated-phase scratch to (re)use, one float64 per packed point.  ``scanned``: ``ws`` and
    ``phase_ws`` already hold the block start phases and Nyquist flags (dist.py's hand-over), so the
    scan is left out (pvk_resynth_render).  A ``fscale`` curve has one ratio per row of ``tid``."""
    phase_preserve, fscale = synth_mode(phase_preserve, fscale, nframes=tid.shape[0])
    fscale = _on_device(fscale, tid.device)
    if scanned and (phase_preserve or phase_ws is None):
        raise ValueError("scanned=True needs phase_preserve=False and the phase_ws of the scan")
    L = _lib.lib()
    dev = tid.device
    F, K = tid.shape
    if nout is None:
        if max_end is None:
            max_end = int((pk["tstart"] + pk["tlen"] - 1).max().item()) if len(pk["tstart"]) else -1
        nout, _ = synth_geometry(max_end, hop, nfft, hop_an, edge)
    nblk = -(-nout // hop)
    nb = nblk - block0 if nblocks < 0 else nblocks
    if out is None:
        out = torch.empty((max(min(nb * hop, nout - block0 * hop), 0),), dtype=torch.float64, device=dev)
    nt = int(pk["tstart"].shape[0])
    if ws is None:
        ws = resynth_workspace(F, K, nt, nb, dev)
    if phase_ws is None and not phase_preserve:
        if reuse_tracks:
            raise ValueError("reuse_tracks with phase_preserve=False needs the phase_ws of the first call")
        phase_ws = _phase_ws(False, pk["pf"].numel(), dev)
    with torch.cuda.device(dev):
        _resynth_ex(L, tid, F, K, nt, None, pk["tstart"], pk["tlen"], pk["toff"], pk["pf"], pk["pmag"], pk["prealph"], sr,
                    hop, nfft, hop_an, edge, minframes, out, nout, block0, nblocks, ws, reuse_tracks, phase_preserve,
                    fscale, None if phase_preserve else phase_ws, scanned)
    return out


def resynth_workspace(F, K, ntracks, nblocks, dev, hop=None):
    """Scratch of pvk_resynth.  ``hop`` given and a multiple of 128: the tile kernels build the partial
    bodies themselves and need no per-block staging area."""
    if hop is not None and int(hop) % 128 == 0:
        nblocks = 1
    wsb = int(_lib.lib().pvk_resynth_workspace_bytes(int(F), int(K), int(ntracks), max(int(nblocks), 0)))
    return torch.empty(max(wsb, 8), dtype=torch.uint8, device=dev)


# =========================================================================== PV
class PV(object):
    def __init__(self, x, sr, nfft=1024, hop=None, npks=20, pkthresh=0.005, wind=np.hanning,
                 progress=True, device=None):
        '''
        Phase vocoder object (GPU).  Arguments as pypevoc.PV (PVAnalysis.py:72-82):
            * sr   = Sampling rate
            * nfft = Number of points in FFT analysis window (power of two, 64..8192)
            * hop  = Number of points between FFT windows (default nfft/2)
            * npks = Maximum number of peaks at each frame
            * pkthresh = Threshold of peak amplitude relative of maximum
            * wind = window callable evaluated on the host (default np.hanning)
        x may be a sequence, a numpy array or a torch tensor (CPU or CUDA); the kernels work
        on its float32 rounding.  ``device`` selects the GPU (default: current device).
        '''
        self._dev = _device(device if device is not None else (x.device if torch.is_tensor(x) and x.is_cuda else None))
        self._xh_pinned = None
        if torch.is_tensor(x):
            xd = x.detach()
            if xd.dim() != 1:
                raise ValueError("PV expects a 1-D signal")
            if (not xd.is_cuda) and xd.is_pinned() and xd.dtype == torch.float32 and xd.is_contiguous():
                # pinned host signal: uploaded by run_pv (in chunks that overlap the analysis when a
                # ``hostbuf`` is given, in one asynchronous copy otherwise)
                self._xh_pinned = xd
                self._xd_t = None
            else:
                self._xd_t = xd.to(device=self._dev, dtype=torch.float32, non_blocking=True).contiguous()
            self._x_host = None
        else:
            xh = np.array(x)
            if xh.ndim != 1:
                raise ValueError("PV expects a 1-D signal")
            self._x_host = xh
            x32 = np.ascontiguousarray(xh, dtype=np.float32)
            self._xd_t = torch.from_numpy(x32).to(self._dev, non_blocking=False)
        self.nsamp = int((self._xh_pinned if self._xh_pinned is not None else self._xd_t).shape[0])
        self.sr = sr
        self.nfft = nfft
        self.nfft2 = int(nfft / 2)
        if hop is None:
            self.hop = int(self.nfft / 2)
        else:
            self.hop = hop
        if int(self.hop) != self.hop or self.hop < 1:
            raise ValueError("hop must be a positive integer")
        self.hop = int(self.hop)
        if int(npks) < 1 or int(npks) > 1024:
            raise ValueError("npks must be in [1, 1024]")
        self.peakthresh = pkthresh
        self.npeaks = int(npks)
        self.nframes = 0
        if nfft < 64 or nfft > 8192 or (nfft & (nfft - 1)) != 0:
            raise ValueError("nfft=%r is not supported by the CUDA kernels: it must be a power of two "
                             "in [64, 8192]" % (nfft,))

        self._tb = host_tables(sr, nfft, self.hop, wind)
        self.win = self._tb["win"]
        self.wsum = self._tb["wsum"]
        self.wsum2 = self._tb["wsum2"]
        self.wfact = self._tb["wfact"]
        self.fstep = self._tb["fstep"]
        self.dt = self._tb["dt"]
        self.fbin = self._tb["fbin"]
        self.wfbin = self._tb["wfbin"]
        # the reference carries the previous frame here (PVAnalysis.py:121,209); the GPU path
        # keeps it in shared memory, so this stays the initial all-zero spectrum
        self.oldfft = np.zeros(self.nfft2)

        self._host = {"t": [], "f": [], "ph": [], "mag": []}
        self._devout = None
        self._hostbuf = None
        self._d2h_event = None
        self._stats = None
        if progress:
            self.progress = Progress(end=self.nsamp)
        else:
            self.progress = None

    # -- lazily materialised host arrays (float64, the reference's layout) ------------
    @property
    def _xd(self):
        """The float32 device signal (a pinned host input is uploaded on first use)."""
        if self._xd_t is None:
            self._xd_t = self._xh_pinned.to(device=self._dev, non_blocking=True)
        return self._xd_t

    def _get(self, name):
        if name not in self._host:
            if self._devout is None and self._hostbuf is None:
                raise AttributeError(name)
            self._host[name] = self._fetch(name)
        return self._host[name]

    def _fetch(self, name):
        d = self._devout
        if self._hostbuf is not None and name in getattr(self, "_streamed", ()):
            # run_pv(hostbuf=...) already streamed the tables into pinned memory
            if self._d2h_event is not None:
                self._d2h_event.synchronize()
                self._d2h_event = None
            hb = self._hostbuf[name][:self.nframes].numpy()
            if name == "totalmag":
                return [v for v in hb]
            return hb if self.nframes else np.array([])
        if d is None:
            raise AttributeError("%s was not kept by the last (chunked) run_pv" % name)
        if name == "totalmag":
            return [v for v in d["totalmag"][0].cpu().numpy()]
        if name not in d:
            raise AttributeError("%s was not computed by the last run_pv" % name)
        if self.nframes == 0:
            return np.array([])
        return d[name][0].cpu().numpy()

    def _prop(name):  # noqa: N805
        def g(self):
            return self._get(name)

        def s(self, value):
            self._host[name] = value
        return property(g, s)

    f = _prop("f")
    mag = _prop("mag")
    ph = _prop("ph")
    realph = _prop("realph")
    binno = _prop("binno")
    totalmag = _prop("totalmag")
    t = _prop("t")
    fine_pos = _prop("fine_pos")
    fine_val = _prop("fine_val")
    del _prop

    @property
    def x(self):
        if self._x_host is None:
            self._x_host = self._xd.cpu().numpy()
        return self._x_host

    @property
    def device_tables(self):
        """Device tensors of the last run_pv: f mag ph realph binno [nframes, npks] float64,
        npk int32 [nframes], totalmag float64 [nframes]."""
        if self._devout is None:
            raise RuntimeError("run_pv() has not been called")
        return {k: v[0] for k, v in self._devout.items()}

    def fetch_into(self, hostbuf, extra=None):
        """Copy the peak tables of the last run_pv (and any ``extra`` device tensors) into
        reusable pinned host tensors kept in the dict ``hostbuf`` (allocated on first use), with
        asynchronous copies on the current stream; the caller synchronises.  The tables become
        this object's ``f mag ph realph binno totalmag`` attributes (numpy views of the pinned
        buffers, valid until the next fetch_into with the same ``hostbuf``).  Returns the number
        of bytes copied device -> host."""
        src = {k: self._devout[k][0] for k in ("f", "mag", "ph", "realph", "binno", "totalmag")}
        if extra:
            src.update(extra)
        nbytes = 0
        for k, t in src.items():
            hb = hostbuf.get(k)
            if hb is None or hb.shape != t.shape or hb.dtype != t.dtype:
                hb = torch.empty(t.shape, dtype=t.dtype, device="cpu", pin_memory=True)
                hostbuf[k] = hb
            hb.copy_(t, non_blocking=True)
            nbytes += t.numel() * t.element_size()
        for k in ("f", "mag", "ph", "realph", "binno"):
            self._host[k] = hostbuf[k].numpy() if self.nframes else np.array([])
        self._host["totalmag"] = hostbuf["totalmag"].numpy()
        return nbytes

    # -- analysis ----------------------------------------------------------------------
    def run_pv(self, run_frames=0, hostbuf=None, chunks=8, refine=False, device_budget=None, stream_tables=None):
        """STFT + peak picking + instantaneous frequency for every frame (PVAnalysis.py:213-264)
        in one kernel launch.  Results appear as the reference's attributes ``f mag ph realph
        binno`` (float64 ``[nframes, npks]``), ``t``, ``nframes``, ``totalmag`` (list).

        ``hostbuf`` (a dict, reused across calls): stream the tables into pinned host memory
        while the analysis is still running -- the frames are analysed in ``chunks`` launches, the
        upload of a pinned host signal, the kernels and the download of finished rows overlap on
        three streams; the attributes are numpy views of the pinned buffers (valid until the next
        call with the same ``hostbuf``) and synchronise on first access.

        ``stream_tables`` (with ``hostbuf``): names of the tables to stream (default: all of ``f mag ph
        realph binno totalmag``).  The others stay on the device and are downloaded on first access of
        the attribute, so a caller that only reads e.g. ``f mag ph`` moves 3/5 of the bytes.

        ``refine=True`` additionally evaluates ``PeakFinder.refine`` (PeakFinder.py:331-372) for
        every peak: attributes ``fine_pos`` (fractional bin) and ``fine_val`` (interpolated
        |fx|), float64 ``[nframes, npks]``, columns aligned with ``binno``.  The reference's PV
        never refines (PVAnalysis.py:175-178), so this is an opt-in extra.

        ``device_budget`` (bytes; needs a pinned host signal and ``hostbuf``): signals whose samples
        and peak tables exceed a device-memory budget (the reference reads the whole file,
        AudioInterface.py:15-37, and keeps every table on the host).  The frames are analysed in
        frame-aligned chunks sized so that two chunks (signal slice + tables) fit the budget; every
        chunk re-computes the frame before its first one as warm-up (the previous spectrum), results
        stream into the pinned host tables and nothing but the two chunk buffers stays on the device.
        Bit-identical to the one-shot run.  ``toSinSum`` then uploads the host tables."""
        self._hostbuf = None
        self._d2h_event = None
        self._stats = None
        if device_budget is not None:
            if hostbuf is None or self._xh_pinned is None:
                raise ValueError("run_pv(device_budget=...) needs a pinned float32 host signal and hostbuf={}")
            self._run_pv_chunked(hostbuf, int(device_budget), run_frames, refine=refine)
            self._host = {}
            self._host["t"] = (np.arange(self.nframes) * self.hop + self.nfft / 2.0) / self.sr   # :247
            if self.progress:
                self.progress.update(self.nsamp)
            return
        if hostbuf is not None:
            self._run_pv_streamed(hostbuf, int(chunks), run_frames, refine=refine, stream_tables=stream_tables)
        else:
            self._devout = analyze_device(self._xd, self.sr, self.nfft, self.hop, self.npeaks, self.peakthresh,
                                          self._tb, run_frames=run_frames, refine=refine)
        self.nframes = int(self._devout["f"].shape[1])
        self._host = {}
        self._host["t"] = (np.arange(self.nframes) * self.hop + self.nfft / 2.0) / self.sr   # :247
        if self.progress:
            self.progress.update(self.nsamp)

    def _run_pv_streamed(self, hostbuf, chunks, run_frames, frame_lo=0, nframes=None, prev_zero=True, refine=False,
                         stream_tables=None):
        """Rows r = 0 .. F-1 are the frames starting at sample (frame_lo + r)*hop (frame_lo = 1 with
        prev_zero=False: frame 0 of the buffer is only the warm-up of a sharded window)."""
        dev, K = self._dev, self.npeaks
        F = n_frames(self.nsamp, self.nfft, self.hop) - frame_lo if nframes is None else int(nframes)
        cur = torch.cuda.current_stream(dev)
        h2d, d2h = _side_streams(dev)
        names = ("f", "mag", "ph", "realph", "binno")
        with torch.cuda.device(dev):
            out = {k: torch.empty((1, F, K), dtype=torch.float64, device=dev) for k in names}
            out["npk"] = torch.empty((1, F), dtype=torch.int32, device=dev)
            out["totalmag"] = torch.empty((1, F), dtype=torch.float64, device=dev)
            if refine:      # stays on the device, fetched on first access
                out["fine_pos"] = torch.empty((1, F, K), dtype=torch.float64, device=dev)
                out["fine_val"] = torch.empty((1, F, K), dtype=torch.float64, device=dev)
            want = set(names + ("totalmag",)) if stream_tables is None else set(stream_tables)
            if not want <= set(names + ("totalmag",)):
                raise ValueError("stream_tables: unknown table name(s) %r" % sorted(want - set(names + ("totalmag",))))
            snames = tuple(k for k in names if k in want)
            hb = {k: _pinned(hostbuf, k, (F, K), torch.float64) for k in snames}
            if "totalmag" in want:
                hb["totalmag"] = _pinned(hostbuf, "totalmag", (F,), torch.float64)
            upload = self._xd_t is None
            if upload:
                xd = torch.empty((self.nsamp,), dtype=torch.float32, device=dev)
                h2d.wait_stream(cur)          # the buffers may be recycled memory still in use on `cur`
            else:
                xd = self._xd_t
            d2h.wait_stream(cur)
            chunks = max(1, min(chunks, F // 64 if F >= 64 else 1))
            bounds = _chunk_bounds(F, chunks)
            s_done = 0
            _mark("start", cur)
            for i in range(chunks if F else 0):
                j0, j1 = bounds[i], bounds[i + 1]
                if upload:
                    s_end = self.nsamp if i == chunks - 1 else (frame_lo + j1 - 1) * self.hop + self.nfft
                    with torch.cuda.stream(h2d):
                        xd[s_done:s_end].copy_(self._xh_pinned[s_done:s_end], non_blocking=True)
                        ev = torch.cuda.Event()
                        ev.record(h2d)
                        _mark("h2d %d" % i, h2d)
                    cur.wait_event(ev)
                    s_done = s_end
                view = {k: v[:, j0:j1] for k, v in out.items()}
                analyze_device(xd, self.sr, self.nfft, self.hop, K, self.peakthresh, self._tb, frame0=frame_lo + j0,
                               nframes=j1 - j0, prev_zero=(prev_zero and j0 == 0), run_frames=run_frames, out=view,
                               refine=refine)
                ev2 = torch.cuda.Event()
                ev2.record(cur)
                _mark("analysis %d" % i, cur)
                with torch.cuda.stream(d2h):
                    d2h.wait_event(ev2)
                    for k in hb:
                        hb[k][j0:j1].copy_(out[k][0, j0:j1], non_blocking=True)
                    _mark("tables d2h %d" % i, d2h)
            if upload:
                self._xd_t = xd
                xd.record_stream(h2d)
            for t in out.values():                                # read by the copy stream: the allocator
                t.record_stream(d2h)                              # must not recycle them before it is done
            self._d2h_event = torch.cuda.Event()
            self._d2h_event.record(d2h)
        self._devout = out
        self._hostbuf = hostbuf
        self._streamed = set(hb)
        self.d2h_bytes = F * (len(snames) * K + (1 if "totalmag" in hb else 0)) * 8

    def _run_pv_chunked(self, hostbuf, budget, run_frames, refine=False):
        dev, K, hop, nfft = self._dev, self.npeaks, self.hop, self.nfft
        F = n_frames(self.nsamp, nfft, hop)
        names = ("f", "mag", "ph", "realph", "binno") + (("fine_pos", "fine_val") if refine else ())
        per_frame = hop * 4 + (len(names) * K + 1) * 8 + 4
        Fc = int(max(64, (budget // 2 - (nfft + hop) * 4) // per_frame))
        Fc = min(Fc, max(F, 1))
        cur = torch.cuda.current_stream(dev)
        h2d, d2h = _side_streams(dev)
        with torch.cuda.device(dev):
            hb = {k: _pinned(hostbuf, k, (F, K), torch.float64) for k in names}
            hb["totalmag"] = _pinned(hostbuf, "totalmag", (F,), torch.float64)
            bufs = []
            for _ in range(2 if F > Fc else 1):
                o = {k: torch.empty((1, Fc, K), dtype=torch.float64, device=dev) for k in names}
                o["npk"] = torch.empty((1, Fc), dtype=torch.int32, device=dev)
                o["totalmag"] = torch.empty((1, Fc), dtype=torch.float64, device=dev)
                bufs.append(dict(x=torch.empty((Fc * hop + nfft,), dtype=torch.float32, device=dev), out=o, free=None))
            h2d.wait_stream(cur)
            d2h.wait_stream(cur)
            last = None
            for i, j0 in enumerate(range(0, F, Fc)):
                j1 = min(F, j0 + Fc)
                b = bufs[i & 1]
                s0 = (j0 - 1) * hop if j0 > 0 else 0                     # one warm-up frame before the chunk
                s1 = (j1 - 1) * hop + nfft
                with torch.cuda.stream(h2d):
                    if b["free"] is not None:
                        h2d.wait_event(b["free"])                       # the buffer's previous tables are on the host
                    b["x"][:s1 - s0].copy_(self._xh_pinned[s0:s1], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(h2d)
                cur.wait_event(ev)
                view = {k: v[:, :j1 - j0] for k, v in b["out"].items()}
                analyze_device(b["x"][:s1 - s0], self.sr, nfft, hop, K, self.peakthresh, self._tb,
                               frame0=1 if j0 > 0 else 0, nframes=j1 - j0, prev_zero=(j0 == 0), run_frames=run_frames,
                               out=view, refine=refine)
                ev2 = torch.cuda.Event()
                ev2.record(cur)
                with torch.cuda.stream(d2h):
                    d2h.wait_event(ev2)
                    for k in names:
                        hb[k][j0:j1].copy_(b["out"][k][0, :j1 - j0], non_blocking=True)
                    hb["totalmag"][j0:j1].copy_(b["out"]["totalmag"][0, :j1 - j0], non_blocking=True)
                    b["free"] = torch.cuda.Event()
                    b["free"].record(d2h)
                    last = b["free"]
                for t in [b["x"]] + list(b["out"].values()):
                    t.record_stream(h2d), t.record_stream(d2h)
            self._d2h_event = last
        self._devout = None
        self._hostbuf = hostbuf
        self._streamed = set(hb)
        self.nframes = F
        self.chunk_frames = Fc
        self.d2h_bytes = F * (len(names) * K + 1) * 8

    def dphase2freq(self, dph, nbin):
        '''"instantaneous frequency" for the phase difference dph at bin nbin (host helper with
        the reference's arithmetic, PVAnalysis.py:133-147; the kernels do this per peak on the GPU)'''
        dphw = dph + self.wfbin[nbin] + pi2 * np.arange(-1, 2)
        freq = dphw / self.dt / pi2
        df = self.fbin[nbin] - freq
        ii = np.argmin(abs(df))
        return freq[ii], df[ii]

    def calc_fft_frame(self, pos):
        '''FFT frame at sample pos, all nfft bins, normalised by wfact (PVAnalysis.py:150-158).
        Convenience accessor (computed on the device with torch.fft in float64); run_pv does
        not use it.'''
        seg = self._xd[pos:pos + self.nfft].to(torch.float64)
        w = torch.from_numpy(np.asarray(self.win, dtype=np.float64)).to(self._dev)
        return (torch.fft.fft(seg * w) / self.wfact).cpu().numpy()

    def calc_pv_frame(self, pos):
        '''PV peaks of the frame at sample ``pos`` with the frame at ``pos - hop`` as previous
        frame (all-zero spectrum if pos < hop), like the reference when called in run order
        (PVAnalysis.py:160-211).  Returns lists f, mag, ph, realph, binno and totalmag.'''
        if pos + self.nfft > self.nsamp:
            raise ValueError("frame exceeds the signal")
        if pos >= self.hop:
            seg = self._xd[pos - self.hop:pos + self.nfft]
            o = analyze_device(seg, self.sr, self.nfft, self.hop, self.npeaks, self.peakthresh, self._tb,
                               frame0=1, nframes=1, prev_zero=False)
        else:
            seg = self._xd[pos:pos + self.nfft]
            o = analyze_device(seg, self.sr, self.nfft, self.hop, self.npeaks, self.peakthresh, self._tb,
                               frame0=0, nframes=1, prev_zero=True)
        n = int(o["npk"][0, 0].item())
        vals = [o[k][0, 0, :n].cpu().numpy().tolist() for k in ("f", "mag", "ph", "realph", "binno")]
        return vals[0], vals[1], vals[2], vals[3], [int(b) for b in vals[4]], float(o["totalmag"][0, 0].item())

    # -- tracking ----------------------------------------------------------------------
    def toSinSum(self, maxpitchjmp=0.5):
        '''
        Convert to Sine sum (PVAnalysis.py:299-322): greedy frame-to-frame partial tracking on
        the GPU.  As in the reference the argument is not forwarded: add_frame's default
        maxpitchjmp=0.5 semitones is what is applied (PVAnalysis.py:320-321,871).
        '''
        if self._devout is None and self._hostbuf is None:
            raise RuntimeError("run_pv() has not been called")
        ss = SinSum(self.sr, nfft=self.nfft, hop=self.hop, device=self._dev)
        # the reference tracks self.f / mag / ph / realph (:320): a table the caller has read (and
        # may have edited in place) or assigned is uploaded again; untouched ones stay on the device
        tabs = []
        for k in ("f", "mag", "ph", "realph"):
            if k in self._host or self._devout is None:
                a = np.asarray(self._get(k), dtype=np.float64)
                if a.ndim != 2:
                    a = a.reshape(0, self.npeaks)
                tabs.append(torch.from_numpy(np.ascontiguousarray(a)).to(self._dev))
            else:
                tabs.append(self._devout[k][0])
        ss._set_device_tables(*tabs)
        return ss

    # -- consumers (host side views over the peak tables, PVAnalysis.py:324-417) ---------
    def plot_time_freq(self, colors=True, ax=None):
        import pylab as pl
        if ax is None:
            fig, allax = pl.subplots(1)
            ax = allax
        t = np.outer(self.t, np.ones(self.npeaks))
        if colors:
            ax.scatter(t, self.f, s=6, c=20 * np.log10(self.mag), lw=0)
        else:
            ax.scatter(t, self.f, s=100 + 20 * np.log10(self.mag), lw=0)
        pl.xlabel('Time (s)')
        pl.ylabel('Frequency (Hz)')
        return ax

    def plot_time_mag(self):
        import pylab as pl
        pl.figure()
        t = np.outer(self.t, np.ones(self.npeaks))
        pl.scatter(t, 20 * np.log10(self.mag), s=10, c=self.f, lw=0, norm=pl.matplotlib.colors.LogNorm())
        pl.xlabel('Time (s)')
        pl.ylabel('Magnitude (dB)')
        cs = pl.colorbar()
        cs.set_label('Frequency (Hz)')
        return pl.gca()

    def get_time_vector(self):
        return self.t

    def get_sample_vector(self):
        return (self.t * self.sr).astype('int')

    def _on_device(self):
        """True while f / mag are the untouched device tables of the last run_pv."""
        return self._devout is not None and "f" not in self._host and "mag" not in self._host and self.nframes > 0

    def _frame_stats(self, fmin=50, fmax=10000, thr=0.1):
        key = (float(fmin), float(fmax), float(thr))
        st = getattr(self, "_stats", None)
        if st is None or st[0] != key:
            d = self._devout
            fm, idx, ps = frame_stats_device(d["f"][0], d["mag"][0], fmin, fmax, thr)
            st = (key, fm.cpu().numpy(), idx.cpu().numpy().astype('i'), ps.cpu().numpy())
            self._stats = st
        return st

    def calc_f0(self, fmin=50, fmax=10000, thr=0.1):
        """Lowest-frequency strong peak of every frame (PVAnalysis.py:371-391).  While the peak
        tables live on the device this is one pvk_frame_stats launch and a read-back of one value
        per frame (the tables are not downloaded); on host tables it is vectorised numpy."""
        if self._on_device():
            _, fm, im, _ = self._frame_stats(fmin, fmax, thr)
            self.fundamental_idx = im
            return fm.copy()
        f, mag = self.f, self.mag
        if f.ndim != 2:
            self.fundamental_idx = np.zeros(0, dtype='i')
            return np.zeros(0)
        maxmag = np.max(mag, axis=1, keepdims=True)
        ok = (f > fmin) & (f < fmax) & (mag > maxmag * thr)
        cand = np.where(ok, f, np.inf)
        im = np.argmin(cand, axis=1)
        has = ok.any(axis=1)
        im = np.where(has, im, 0).astype('i')
        fm = np.where(has, f[np.arange(f.shape[0]), im], 0.0)
        self.fundamental_idx = im
        return fm

    def calc_harmonic_power(self, f_threshold=0.01):
        """
        calculate the harmonic power of individual sine components (PVAnalysis.py:266-297):
        sets ``hpower`` and ``nharmonics`` (float64 ``[nframes, npks]``).  One pvk_harmonic_power
        launch on the device tables (host-edited ``f`` / ``mag`` are uploaded first).

        As in the reference, line :278 indexes the *rows* of ``mag`` with the peaks' column
        numbers, so ``hpower`` sums whole table rows (kept: results are identical to the
        reference's), and a peak in a column >= nframes raises IndexError.
        """
        if self._devout is None:
            raise AttributeError("f")                    # the reference fails on self.f before run_pv
        if self.nframes == 0:
            raise IndexError("tuple index out of range")     # self.f.shape[0] of an empty 1-D array (:274)
        if self._on_device():
            fd, md = self._devout["f"][0], self._devout["mag"][0]
        else:
            fd = torch.from_numpy(np.ascontiguousarray(self.f, dtype=np.float64)).to(self._dev)
            md = torch.from_numpy(np.ascontiguousarray(self.mag, dtype=np.float64)).to(self._dev)
        hp, nh, err = harmonic_power_device(fd, md, f_threshold)
        if int(err.item()):
            raise IndexError("index out of bounds for axis 0 with size %d (a peak column used as a frame index, "
                             "PVAnalysis.py:278)" % fd.shape[0])
        self.hpower = hp.cpu().numpy()
        self.nharmonics = nh.cpu().numpy()

    @property
    def fundamental_frequency(self):
        try:
            return self.f[np.arange(self.f.shape[0]), self.fundamental_idx]
        except AttributeError:
            return self.calc_f0()

    @property
    def fundamental_magnitude(self):
        try:
            return self.mag[np.arange(self.f.shape[0]), self.fundamental_idx]
        except AttributeError:
            self.calc_f0()
            return self.mag[np.arange(self.f.shape[0]), self.fundamental_idx]

    @property
    def partial_sum_magnitude(self):
        if self._on_device():
            st = getattr(self, "_stats", None)
            return (st if st is not None else self._frame_stats())[3].copy()
        return np.sqrt(np.sum(self.mag ** 2, axis=1))

    @property
    def partial_magnitude_ratio(self):
        return self.partial_sum_magnitude / self.totalmag


class PVBatch(object):
    """Clip batch (BASELINE configs[2]; SURVEY 8e): ``nclips`` independent signals of equal length
    analysed by ONE pvk_analyze_batch launch; tracking, packing and resynthesis of all clips run as
    ONE pvk_track / pvk_track_pack / pvk_resynth over the flattened peak table, in which a few
    all-zero guard rows after every clip end all partials at the clip boundary (every clip starts
    from the all-zero previous spectrum and its own partial numbering, exactly as a ``PV`` per clip:
    PVAnalysis.py:213-264, 299-322, 1053-1070 once per clip).

        pb = PVBatch(x, sr, nfft=512, hop=128, npks=20)      # x: [nclips, nsamp] numpy / torch
        pb.run_pv()
        pb.f, pb.mag, pb.ph, pb.realph, pb.binno               # float64 [nclips, nframes, npks]
        ssb = pb.toSinSum(); w = ssb.synth(sr, pb.hop)         # list of nclips float64 signals
        pb.track()["tid"]                                      # int32 CUDA [nclips, nframes, npks]
        pv3 = pb[3]                                            # a PV over clip 3 sharing the device tables

    Across GPUs a batch shards by clip with no halo and no collective
    (``dist.clip_range(nclips, rank, world)``)."""

    def __init__(self, x, sr, nfft=1024, hop=None, npks=20, pkthresh=0.005, wind=np.hanning, device=None,
                 max_edge=1.0):
        self._dev = _device(device)
        if isinstance(x, torch.Tensor):
            xd = x.detach()
        else:
            xd = torch.from_numpy(np.ascontiguousarray(np.asarray(x), dtype=np.float32))
        if xd.dim() != 2:
            raise ValueError("PVBatch expects a [nclips, nsamp] array")
        self._xd = xd.to(device=self._dev, dtype=torch.float32).contiguous()
        self.nclips, self.nsamp = (int(v) for v in self._xd.shape)
        self._kw = dict(nfft=nfft, hop=hop, npks=npks, pkthresh=pkthresh, wind=wind)
        # argument checks and host tables are PV's own
        proto = PV(self._xd[0] if self.nclips else torch.zeros(1), sr, progress=False, device=self._dev, **self._kw)
        self.sr, self.nfft, self.hop, self.npeaks, self.peakthresh = sr, proto.nfft, proto.hop, proto.npeaks, pkthresh
        self._tb = proto._tb
        # guard rows after every clip: fade-out tails (ceil(dfr*edge) blocks + 1) of one clip and the
        # fade-in heads (ceil(dfr*edge) blocks) of the next must not meet
        self.max_edge = float(max_edge)
        self.guard = 2 * int(np.ceil(self.nfft / float(self.hop) / 2. * self.max_edge)) + 3
        self._devout = None
        self._trk = None
        self._ssb = None
        self._host = {}
        self.nframes = 0

    def run_pv(self, run_frames=0):
        F = n_frames(self.nsamp, self.nfft, self.hop)
        self._devout = analyze_device(self._xd, self.sr, self.nfft, self.hop, self.npeaks, self.peakthresh, self._tb,
                                      run_frames=run_frames, nframes=F, out_rows=F + self.guard if F else 0)
        self.nframes = F
        self.rows_per_clip = F + self.guard if F else 0
        self._host = {"t": (np.arange(self.nframes) * self.hop + self.nfft / 2.0) / self.sr}
        self._trk = None
        self._ssb = None

    @property
    def device_tables(self):
        """Device tensors of the last run_pv: f mag ph realph binno float64 [nclips, nframes, npks],
        npk int32 and totalmag float64 [nclips, nframes] (views of the guard-row padded tables)."""
        if self._devout is None:
            raise RuntimeError("run_pv() has not been called")
        return {k: v[:, :self.nframes] for k, v in self._devout.items()}

    def __getattr__(self, name):
        if name in ("f", "mag", "ph", "realph", "binno", "totalmag", "t"):
            host = self.__dict__.get("_host", {})
            if name not in host:
                dev = self.__dict__.get("_devout")
                if dev is None:
                    raise AttributeError(name)
                host[name] = dev[name][:, :self.nframes].cpu().numpy()
            return host[name]
        raise AttributeError(name)

    def toSinSum(self, maxpitchjmp=0.5):
        """Tracking of every clip (PVAnalysis.py:299-322 per clip; as there, the argument is not
        forwarded) -> :class:`SinSumBatch`."""
        if self._devout is None:
            raise RuntimeError("run_pv() has not been called")
        if self._ssb is None:
            self._ssb = SinSumBatch(self)
        return self._ssb

    def track(self, maxpitchjmp=0.5):
        """Per-clip view of the batch tracking: dict(tid int32 CUDA [nclips, nframes, npks] with every
        clip's own numbering (-1 = no peak), ntracks int32 CUDA [nclips])."""
        if self._trk is None:
            ssb = self.toSinSum()
            base, _ = ssb.clip_spans()
            R, F, K = self.rows_per_clip, self.nframes, self.npeaks
            tid = ssb.ss._ensure_tracks()["tid"].view(self.nclips, R, K)[:, :F]
            b = torch.from_numpy(base[:-1].astype(np.int32)).to(self._dev).view(-1, 1, 1)
            self._trk = dict(tid=torch.where(tid >= 0, tid - b, tid),
                             ntracks=torch.from_numpy(np.diff(base).astype(np.int32)).to(self._dev))
        return self._trk

    def __len__(self):
        return self.nclips

    def __getitem__(self, i):
        """``PV`` over clip ``i``; its tables are views of the batch's device tables."""
        i = int(i)
        if i < 0:
            i += self.nclips
        if not 0 <= i < self.nclips:
            raise IndexError(i)
        pv = PV(self._xd[i], self.sr, progress=False, device=self._dev, **self._kw)
        if self._devout is not None:
            pv._devout = {k: v[i:i + 1, :self.nframes] for k, v in self._devout.items()}
            pv.nframes = self.nframes
            pv._host = {"t": self._host["t"]}
        return pv


class SinSumBatch(object):
    """Partials of every clip of a :class:`PVBatch`: ONE link / pack / resynthesis over the
    flattened, guard-row separated peak table (``ss``: the SinSum of that table; partial ids run
    clip after clip, frame indices are rows of the flattened table)."""

    def __init__(self, pb):
        self._pb = pb
        R, K = pb.rows_per_clip, pb.npeaks
        d = pb._devout
        self.ss = SinSum(pb.sr, nfft=pb.nfft, hop=pb.hop, device=pb._dev)
        self.ss._set_device_tables(*(d[k].view(pb.nclips * R, K) for k in ("f", "mag", "ph", "realph")))
        self._spans = None
        self.sr, self.nfft, self.hop = pb.sr, pb.nfft, pb.hop

    def clip_spans(self):
        """(base, last): base int64 [nclips + 1] -- clip c owns the partials base[c] .. base[c+1] of
        ``ss`` -- and last int64 [nclips] = max(SinSum.end) of clip c in its own frame numbering (-1:
        the clip has no partial).  One pvk_clip_spans launch + a read-back of 2 ints per clip."""
        if self._spans is None:
            pb = self._pb
            pk = self.ss._ensure_packed()
            nt = int(pk["tstart"].shape[0])
            cnt = torch.empty((max(pb.nclips, 1),), dtype=torch.int32, device=pb._dev)
            last = torch.empty((max(pb.nclips, 1),), dtype=torch.int32, device=pb._dev)
            with torch.cuda.device(pb._dev):
                _lib.check(_lib.lib().pvk_clip_spans(_ptr(pk["tstart"]), _ptr(pk["tlen"]), nt, max(pb.rows_per_clip, 1),
                                                     pb.nclips, _ptr(cnt), _ptr(last), _stream()), "pvk_clip_spans")
            both = torch.stack([cnt, last]).cpu().numpy().astype(np.int64)[:, :pb.nclips]
            self._spans = (np.concatenate([[0], np.cumsum(both[0])]), both[1])
        return self._spans

    @property
    def ntracks(self):
        """Number of partials of every clip (numpy int64 [nclips])."""
        return np.diff(self.clip_spans()[0])

    def __len__(self):
        return self._pb.nclips

    def synth_device(self, sr, hop, edge=1.0, minframes=3, phase_preserve=True, fscale=1.0):
        """Render all clips in one pvk_resynth: float64 CUDA tensor [nclips, rows_per_clip * hop]; row c
        holds clip c's signal from its sample 0 (then the silence of the guard rows).  ``phase_preserve``
        / ``fscale`` as in SinSum.synth (one phase scan over the flattened table, a segment per partial);
        a curve is ``[nclips, nframes]``, one ratio per clip and frame."""
        pb = self._pb
        phase_preserve, fscale = self._batch_mode(phase_preserve, fscale)
        if int(hop) != hop:
            raise TypeError("hop must be an integer number of samples")
        if edge > pb.max_edge:
            raise ValueError("edge=%r exceeds the guard rows of this batch (PVBatch(max_edge=%r))" % (edge, pb.max_edge))
        hop = int(hop)
        pk = self.ss._ensure_packed()
        tr = self.ss._trk
        nout = pb.nclips * pb.rows_per_clip * hop
        if tr["ntracks"] == 0 or nout == 0:
            return torch.zeros((pb.nclips, pb.rows_per_clip * hop), dtype=torch.float64, device=pb._dev)
        out = resynth_device(tr["tid"], pk, sr, hop, self.nfft, self.hop, edge=edge, minframes=minframes, nout=nout,
                             phase_preserve=phase_preserve, fscale=fscale)
        return out.view(pb.nclips, pb.rows_per_clip * hop)

    def _batch_mode(self, phase_preserve, fscale):
        """synth_mode() for a batch: a ``[nclips, nframes]`` curve becomes one ratio per row of the
        flattened table (the guard rows, where no partial lives, at 1) on the device."""
        pb = self._pb
        if not isinstance(fscale, (np.ndarray, torch.Tensor, list, tuple)):
            return synth_mode(phase_preserve, fscale)
        r = _curve_values(fscale)
        if r.shape != (pb.nclips, pb.nframes):
            raise ValueError("a batch fscale curve must be [nclips, nframes] = [%d, %d], not of shape %s"
                             % (pb.nclips, pb.nframes, r.shape))
        if phase_preserve:
            raise ValueError("an fscale curve needs phase_preserve=False: the analysed phases cannot be honoured "
                             "at a scaled frequency")
        rows = np.ones((pb.nclips, pb.rows_per_clip))
        rows[:, :pb.nframes] = r
        return False, _DeviceCurve(torch.from_numpy(rows.reshape(-1)).to(pb._dev))

    def clip_lengths(self, hop, edge=1.0):
        """Length of every clip's resynthesis, (max(end) + 2) * hop + edgsamp (PVAnalysis.py:1055-1059,
        1070); 0 for a clip without partials (where the reference raises ValueError)."""
        _, last = self.clip_spans()
        n = np.array([synth_geometry(int(e), int(hop), self.nfft, self.hop, edge)[0] for e in last], dtype=np.int64)
        return np.where(last >= 0, n, 0)

    def synth(self, sr, hop, edge=1.0, minframes=3, to_host=True, phase_preserve=True, fscale=1.0):
        """SinSum.synth of every clip (PVAnalysis.py:1053-1070): list of ``nclips`` float64 signals
        (numpy, or CUDA views with ``to_host=False``), each of its own length."""
        w = self.synth_device(sr, hop, edge, minframes, phase_preserve=phase_preserve, fscale=fscale)
        n = self.clip_lengths(hop, edge)
        if to_host:
            wh = w.cpu().numpy()
            return [wh[c, :n[c]] for c in range(len(n))]
        return [w[c, :n[c]] for c in range(len(n))]

    def __getitem__(self, i):
        """``SinSum`` of clip ``i`` alone (its own link / pack; for the reference's per-partial accessors)."""
        return self._pb[i].toSinSum()


class PVHarmonic(PV):
    """f0-guided phase vocoder (PVAnalysis.py:419-538): instead of picking peaks, every frame
    reads the bins at the multiples of a given fundamental.  Same constructor as PV;
    ``set_f0`` then ``run_pv`` leave ``f mag ph`` (float64 ``[nframes, npks]``), ``residuals``,
    ``t`` and ``nframes``.  One pvk_harmonic launch; no CPU fallback."""

    def __init__(self, *args, **kwargs):
        self.fmin = 30.0                                       # :421
        PV.__init__(self, *args, **kwargs)

    def set_f0(self, f0, t=None):
        '''
        Assign a f0 vector to the search (PVAnalysis.py:424-441)
        Argument:
            * f0: f0 vector over time
            * t: if present, values of time corresponding to f0
                 otherwise, the time values correspond to the hop size
        '''
        tint = np.arange(round(self.hop + self.nfft / 2), self.nsamp, self.hop) / float(self.sr)
        if t is None:
            self.f0 = f0
        else:
            self.f0 = np.interp(tint, t, f0)

    def _f0_device(self, nframes):
        f0 = self.f0
        if torch.is_tensor(f0):
            f0d = f0.detach().to(device=self._dev, dtype=torch.float64).contiguous()
        else:
            f0d = torch.from_numpy(np.ascontiguousarray(np.asarray(f0, dtype=np.float64))).to(self._dev)
        if f0d.dim() != 1 or f0d.numel() < nframes:
            # the reference fails with IndexError at f0[int(curpos/hop)] (:506)
            raise IndexError("f0 has %d values, run_pv needs one per frame (%d)" % (f0d.numel(), nframes))
        return f0d

    def run_pv(self, run_frames=0):
        if not hasattr(self, "f0"):
            raise AttributeError("PVHarmonic.run_pv: call set_f0() first")
        F = n_frames(self.nsamp, self.nfft, self.hop)
        f0d = self._f0_device(F)
        o = harmonic_device(self._xd, self.sr, self.nfft, self.hop, self.npeaks, f0d, self._tb, fmin=self.fmin,
                            nframes=F, run_frames=run_frames)
        self._hdev = o
        self._devout = None
        self._stats = None
        self.nframes = F
        self._host = {}
        empty = F == 0
        self._host["f"] = np.array([]) if empty else o["f"].cpu().numpy()
        self._host["mag"] = np.array([]) if empty else o["mag"].cpu().numpy()
        self._host["ph"] = np.array([]) if empty else o["ph"].cpu().numpy()
        self.residuals = o["residuals"].cpu().numpy()
        self.nharmonics = o["nharm"].cpu().numpy()
        self._host["t"] = (np.arange(F) * self.hop + self.nfft / 2.0) / self.sr   # :523
        if self.progress:
            self.progress.update(self.nsamp)

    @property
    def device_tables(self):
        """Device tensors of the last run_pv: f mag ph [nframes, npks], residuals, nharm."""
        if getattr(self, "_hdev", None) is None:
            raise RuntimeError("run_pv() has not been called")
        return self._hdev

    def calc_pv_frame(self, pos, f0):
        '''Harmonics of the frame at sample ``pos`` for fundamental ``f0`` with the frame at
        ``pos - hop`` as previous frame (all-zero spectrum if pos < hop), like the reference
        when called in run order (PVAnalysis.py:443-492).  Returns f, mag, ph (lists with one
        entry per harmonic, at most npks of them) and the residual.'''
        if pos + self.nfft > self.nsamp:
            raise ValueError("frame exceeds the signal")
        if pos >= self.hop:
            seg = self._xd[pos - self.hop:pos + self.nfft].contiguous()
            f0d = torch.tensor([1.0, float(f0)], dtype=torch.float64, device=self._dev)
            row = 1
        else:
            seg = self._xd[pos:pos + self.nfft].contiguous()
            f0d = torch.tensor([float(f0)], dtype=torch.float64, device=self._dev)
            row = 0
        o = harmonic_device(seg, self.sr, self.nfft, self.hop, self.npeaks, f0d, self._tb, fmin=self.fmin,
                            nframes=row + 1)
        n = min(int(o["nharm"][row].item()), self.npeaks)
        vals = [o[k][row, :n].cpu().numpy().tolist() for k in ("f", "mag", "ph")]
        return vals[0], vals[1], vals[2], float(o["residuals"][row].item())

    def toSinSum(self, maxpitchjmp=0.5):
        # the reference inherits PV.toSinSum, which needs realph (PVAnalysis.py:320) that
        # PVHarmonic.run_pv never sets (:532-538): AttributeError there, stated here
        raise AttributeError("PVHarmonic has no realph table: toSinSum is not available (as in the reference)")


# =========================================================================== partials
class RegPartial(object):
    """A quasi-sinusoidal partial with homogeneous sampling (PVAnalysis.py:585-626): view of
    one track of a SinSum.  ``f mag ph realph`` are float64 numpy arrays (the reference keeps
    python lists of the same values)."""

    def __init__(self, istart, pdict=None, overlap=0.5, fstep=None):
        self.start_idx = istart
        self.overlap = overlap
        self.fstep = fstep
        if pdict is None:
            self.f, self.mag, self.ph, self.realph = [], [], [], []
        else:
            self.f = pdict['f']
            self.mag = pdict['mag']
            self.ph = pdict['ph']
            self.realph = pdict.get('realph', pdict['ph'])

    def get_freq_at_frame(self, fr):
        relidx = fr - self.start_idx
        return self.f[relidx] if relidx >= 0 else np.nan

    def get_mag_at_frame(self, fr):
        relidx = fr - self.start_idx
        return self.mag[relidx] if relidx >= 0 else np.nan

    def synth(self, sr, hop, edge=.5, device=None):
        """Render this partial alone on the GPU (PVAnalysis.py:684-756); returns
        ``(signal, start_sample)`` like the reference: the signal starts ``edgsam`` samples
        before sample ``start_idx*hop``."""
        dev = _device(device)
        nfr = len(self.f)
        if self.fstep is None:
            raise ValueError("RegPartial.synth on the GPU needs fstep (phase correction, :715)")
        # the kernel is parameterised like SinSum (nfft, analysis hop): fstep = sr/nfft (:825),
        # overlap = hop_an/nfft (:824)
        nfft_eff = float(sr) / float(self.fstep)
        hop_an = self.overlap * nfft_eff
        if abs(nfft_eff - round(nfft_eff)) > 1e-6 or abs(hop_an - round(hop_an)) > 1e-6:
            raise ValueError("fstep / overlap must correspond to integer nfft and analysis hop")
        nfft_eff, hop_an = int(round(nfft_eff)), int(round(hop_an))
        dfr = 1. / self.overlap / 2.
        edgsam = int(dfr * hop * edge)
        dE = -(-edgsam // hop)
        rows = nfr + dE
        tid = -torch.ones((rows, 1), dtype=torch.int32, device=dev)
        tid[dE:dE + nfr, 0] = 0
        as_t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)  # noqa: E731
        pk = dict(tstart=torch.tensor([dE], dtype=torch.int32, device=dev),
                  tlen=torch.tensor([nfr], dtype=torch.int32, device=dev),
                  toff=torch.tensor([0, nfr], dtype=torch.int64, device=dev),
                  pf=as_t(self.f), pmag=as_t(self.mag), prealph=as_t(self.realph))
        out = resynth_device(tid, pk, sr, hop, nfft_eff, hop_an, edge=edge, minframes=1, max_end=dE + nfr - 1)
        s0 = dE * hop - edgsam
        sig = out[s0:s0 + hop * nfr + 2 * edgsam].cpu().numpy()
        return sig, int(self.start_idx * hop - edgsam)


class _PartialList(object):
    """Lazy ``ss.partial``: RegPartial views created from the packed track arrays on access."""

    def __init__(self, ss):
        self._ss = ss

    def __len__(self):
        return self._ss._ntracks()

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[k] for k in range(*i.indices(len(self)))]
        n = len(self)
        if i < 0:
            i += n
        if i < 0 or i >= n:
            raise IndexError(i)
        h = self._ss._host_tracks()
        a, b = int(h["toff"][i]), int(h["toff"][i + 1])
        return RegPartial(int(h["tstart"][i]),
                          dict(f=h["pf"][a:b], mag=h["pmag"][a:b], ph=h["pph"][a:b], realph=h["prealph"][a:b]),
                          overlap=self._ss.hop / float(self._ss.nfft), fstep=self._ss.sr / float(self._ss.nfft))

    def __iter__(self):
        for i in range(len(self)):
            yield self[i]


class SinSum(object):
    def __init__(self, sr, nfft=1024, hop=512, device=None):
        '''
        Sine sum object (PVAnalysis.py:797-817): a sound decomposed in a sum of quasi-sine
        waves.  Tracking (add_frame) and resynthesis (synth) run on the GPU.
            * sr   = Sampling rate
            * nfft = Number of points in FFT analysis window
            * hop  = Number of points between FFT windows
        '''
        self.nfft = nfft
        self.hop = hop
        self.sr = sr
        self._dev = _device(device)
        self._rows = {}          # host rows handed to add_frame: fr -> (f, mag, ph, realph)
        self._tables = None      # device f, mag, ph, realph [F, K]
        self._trk = None         # device tid, link, ntracks
        self._pk = None          # device packed tracks
        self._hosttrk = None
        self._maxpitchjmp = 0.5
        self._after_link = None  # hook of sharded runs: called once the link kernels are launched

    # -- construction ------------------------------------------------------------------
    def _set_device_tables(self, f, mag, ph, realph):
        self._tables = dict(f=f.contiguous(), mag=mag.contiguous(), ph=ph.contiguous(), realph=realph.contiguous())
        self._rows = None
        self._trk = self._pk = self._hosttrk = None

    def _set_device_tracks(self, tid, link, ntracks):
        """Adopt precomputed track ids (sharded runs: ids made global by the all_gather)."""
        self._trk = dict(tid=tid.contiguous(), link=link, ntracks=int(ntracks))
        self._pk = self._hosttrk = None

    def add_frame(self, fr, f, mag, ph, realph=None, maxpitchjmp=0.5):
        """Add the peaks of frame ``fr`` (PVAnalysis.py:871-957).  Rows are collected on the host;
        the greedy linking itself runs on the GPU, over all frames at once, the next time the
        partials are needed (links depend on adjacent frame pairs only)."""
        if self._rows is None:
            raise RuntimeError("this SinSum was built from device tables; add_frame is not available")
        f = np.asarray(f, dtype=np.float64)
        mag = np.asarray(mag, dtype=np.float64)
        ph = np.asarray(ph, dtype=np.float64)
        realph = ph if realph is None else np.asarray(realph, dtype=np.float64)
        self._rows[int(fr)] = (f, mag, ph, realph)
        self._maxpitchjmp = maxpitchjmp
        self._tables = self._trk = self._pk = self._hosttrk = None

    def _ensure_tables(self):
        if self._tables is None:
            if not self._rows:
                z = torch.zeros((0, 1), dtype=torch.float64, device=self._dev)
                self._tables = dict(f=z, mag=z.clone(), ph=z.clone(), realph=z.clone())
                return
            F = max(self._rows) + 1
            K = max(len(r[0]) for r in self._rows.values())
            host = np.zeros((4, F, K))
            for fr, row in self._rows.items():
                for q in range(4):
                    host[q, fr, :len(row[q])] = row[q]
            d = torch.from_numpy(host).to(self._dev)
            self._tables = dict(f=d[0], mag=d[1], ph=d[2], realph=d[3])

    def _ensure_tracks(self):
        self._ensure_tables()
        if self._trk is None:
            t = self._tables
            if t["f"].shape[0] == 0:
                # (0, npks): a rank without frames still takes part in the numbering all_gather of a
                # sharded run with 2*npks + 4 integers like everybody else (dist.StitchHandle)
                self._trk = dict(tid=torch.zeros((0, int(t["f"].shape[1])), dtype=torch.int32, device=self._dev),
                                 link=None, ntracks=0)
            else:
                tr, pk = track_pack_device(t["f"], t["mag"], t["ph"], t["realph"], self._maxpitchjmp,
                                           after_link=self._after_link)
                self._trk = tr
                if pk is not None:
                    self._pk = pk
        return self._trk

    def _ensure_packed(self):
        tr = self._ensure_tracks()
        if self._pk is None:
            t = self._tables
            if tr["ntracks"] == 0:
                e = torch.zeros((0,), dtype=torch.float64, device=self._dev)
                self._pk = dict(tstart=torch.zeros((0,), dtype=torch.int32, device=self._dev),
                                tlen=torch.zeros((0,), dtype=torch.int32, device=self._dev),
                                toff=torch.zeros((1,), dtype=torch.int64, device=self._dev),
                                pf=e, pmag=e, pph=e, prealph=e, npts=0)
            else:
                self._pk = pack_device(t["f"], t["mag"], t["ph"], t["realph"], tr["tid"], tr["link"], tr["ntracks"],
                                       npts=tr.get("npts"))
        return self._pk

    def _ntracks(self):
        return self._ensure_tracks()["ntracks"]

    def _host_tracks(self):
        if self._hosttrk is None:
            pk = self._ensure_packed()
            self._hosttrk = {k: pk[k].cpu().numpy() for k in ("tstart", "tlen", "toff", "pf", "pmag", "pph", "prealph")}
        return self._hosttrk

    # -- the reference's attributes ------------------------------------------------------
    @property
    def partial(self):
        return _PartialList(self)

    @property
    def st(self):
        return self._host_tracks()["tstart"].astype(np.int64).tolist()

    @property
    def end(self):
        h = self._host_tracks()
        return (h["tstart"].astype(np.int64) + h["tlen"] - 1).tolist()

    @property
    def track_ids(self):
        """int32 numpy [nframes, npks]: index into ``partial`` for every peak slot (-1 = none)."""
        return self._ensure_tracks()["tid"].cpu().numpy()

    @property
    def device_tracks(self):
        """Device tensors: tid, link [F, K]; tstart, tlen, toff; packed pf pmag pph prealph."""
        d = dict(self._ensure_packed())
        d.update(tid=self._trk["tid"], link=self._trk["link"])
        return d

    # -- resynthesis ---------------------------------------------------------------------
    def synth(self, sr, hop, edge=1.0, minframes=3, phase_preserve=True, to_host=True, hostbuf=None, chunks=8,
              fscale=1.0):
        """Overlap-add resynthesis of all partials with >= minframes frames
        (PVAnalysis.py:1053-1070); float64 ``[(max(end)+2)*hop + edgsamp]``.
        ``phase_preserve=False``: integrated phase instead of the analysed one -- the phase of a partial
        is the running sum of its (interpolated) frequency times ``fscale``, so ``fscale`` shifts the
        pitch and a ``hop`` other than the analysis hop stretches time (``synth(sr, round(hop_an * r),
        phase_preserve=False)``); partials with ``fscale * max(f) >= sr / 2`` are left out.
        ``fscale`` may also be a curve of one ratio per analysis frame, ``r[b]`` applying in output
        block ``b`` (glides, vibrato, intonation), e.g. ``r = ratio_of(np.arange(nframes) * hop_an /
        sr)`` with the input time of each frame row; a partial is then left out when any of its points
        has ``r[row] * f >= sr / 2`` (see synth_mode()).
        ``to_host=False`` returns the CUDA tensor instead of a numpy array.  ``hostbuf`` (a dict,
        reused across calls): render in ``chunks`` block ranges and download each finished range
        into the pinned tensor ``hostbuf['w']`` while the next one is rendered; returns a numpy view
        of it (valid until the next call with the same ``hostbuf``)."""
        nframes = None
        if isinstance(fscale, (np.ndarray, torch.Tensor, list, tuple)):
            if self._trk is None:
                self._ensure_tables()
            nframes = int((self._trk["tid"] if self._trk is not None else self._tables["f"]).shape[0])
        phase_preserve, fscale = synth_mode(phase_preserve, fscale, nframes)
        mode = dict(phase_preserve=phase_preserve, fscale=_on_device(fscale, self._dev))
        if int(hop) != hop:
            raise TypeError("hop must be an integer number of samples")
        if self._trk is None and hostbuf is not None:
            self._ensure_tables()
            if self._tables["f"].shape[0] * self._tables["f"].shape[1] > 0:
                w = self._synth_streamed_fused(sr, int(hop), edge, minframes, hostbuf, int(chunks), **mode)
                if w is not None:
                    return w
        if self._trk is None and hostbuf is None:
            # first use of the partials: link, pack and resynthesis go to the device back to back,
            # the counts are read once at the end (no host round trip between the stages)
            self._ensure_tables()
            t = self._tables
            if t["f"].shape[0] * t["f"].shape[1] > 0:
                tr, pk, out = track_pack_resynth_device(t["f"], t["mag"], t["ph"], t["realph"], sr, int(hop), self.nfft,
                                                        self.hop, edge=edge, minframes=minframes,
                                                        maxpitchjmp=self._maxpitchjmp, after_link=self._after_link,
                                                        **mode)
                self._trk = tr
                if pk is not None:
                    self._pk = pk
                if tr["ntracks"] == 0:
                    raise ValueError("max() arg is an empty sequence")     # what the reference raises (:1059)
                return out.cpu().numpy() if to_host else out
        pk = self._ensure_packed()
        tr = self._trk
        if tr["ntracks"] == 0:
            raise ValueError("max() arg is an empty sequence")     # what the reference raises (:1059)
        if hostbuf is not None:
            return self._synth_streamed(pk, tr, sr, int(hop), edge, minframes, hostbuf, int(chunks), **mode)
        out = resynth_device(tr["tid"], pk, sr, int(hop), self.nfft, self.hop, edge=edge, minframes=minframes,
                             max_end=tr.get("max_end"), **mode)
        return out.cpu().numpy() if to_host else out

    def _synth_streamed_fused(self, sr, hop, edge, minframes, hostbuf, chunks, phase_preserve=True, fscale=1.0):
        """synth(hostbuf=...) on fresh partials: link, pack, the chunked rendering and the downloads of
        the finished chunks are all queued before the host reads any count (sizes are upper bounds,
        pvk_track_pack_dev / pvk_resynth_dev); the signal is cut to its real length at the end.  Returns
        None (after setting the tracks) when the staged path has to take over: no partial at all, or
        more partials than the speculative capacity."""
        L = _lib.lib()
        dev = self._dev
        t = self._tables
        F, K = t["f"].shape
        tr = track_device(t["f"], t["mag"], self._maxpitchjmp)
        if self._after_link is not None:
            self._after_link(tr)
        raw = _pack_speculative(t["f"], t["mag"], t["ph"], t["realph"], tr)
        nt_ub, tstart, tlen, toff, packed = raw
        nout_ub, _ = synth_geometry(F - 1, hop, self.nfft, self.hop, edge)
        nblk = -(-nout_ub // hop)
        cur = torch.cuda.current_stream(dev)
        _, d2h = _side_streams(dev)
        with torch.cuda.device(dev):
            out = torch.empty((nout_ub,), dtype=torch.float64, device=dev)
            hw = _pinned(hostbuf, "w", (nout_ub,), torch.float64)
            d2h.wait_stream(cur)
            chunks = max(1, min(chunks, nblk // 64 if nblk >= 64 else 1))
            bounds = _chunk_bounds(nblk, chunks)
            ws = resynth_workspace(F, K, nt_ub, max(b - a for a, b in zip(bounds, bounds[1:])), dev, hop=hop)
            pws = _phase_ws(phase_preserve, F * K, dev)        # the phase scan runs with the first chunk
            _mark("pack queued", cur)
            for i in range(chunks):
                b0, b1 = bounds[i], bounds[i + 1]
                n0, n1 = b0 * hop, min(b1 * hop, nout_ub)
                _resynth_ex(L, tr["tid"], F, K, nt_ub, tr["ntracks"], tstart, tlen, toff, packed[0], packed[1], packed[3],
                            sr, hop, self.nfft, self.hop, edge, minframes, out[n0:n1], nout_ub, b0, b1 - b0, ws, i > 0,
                            phase_preserve, fscale, pws)
                ev = torch.cuda.Event()
                ev.record(cur)
                _mark("resynth %d" % i, cur)
                with torch.cuda.stream(d2h):
                    d2h.wait_event(ev)
                    hw[n0:n1].copy_(out[n0:n1], non_blocking=True)
                    _mark("w d2h %d" % i, d2h)
            out.record_stream(d2h)
            nt, npts, last = track_counts(tr)                    # the one read-back; the downloads keep running
            tr["ntracks_dev"] = tr["ntracks"]
            tr["ntracks"], tr["npts"], tr["max_end"] = nt, npts, last
            self._trk = tr
            if nt == 0 or nt > nt_ub:
                d2h.synchronize()
                return None
            self._pk = _pack_sliced(raw, nt, npts)
            d2h.synchronize()
        nout, _ = synth_geometry(last, hop, self.nfft, self.hop, edge)
        self.d2h_bytes = nout_ub * 8
        self._last_out = out
        return hw[:nout].numpy()

    def _synth_streamed(self, pk, tr, sr, hop, edge, minframes, hostbuf, chunks, phase_preserve=True, fscale=1.0):
        dev = self._dev
        F, K = tr["tid"].shape
        max_end = tr.get("max_end")
        if max_end is None:
            max_end = int((pk["tstart"] + pk["tlen"] - 1).max().item())
        nout, _ = synth_geometry(max_end, hop, self.nfft, self.hop, edge)
        nblk = -(-nout // hop)
        cur = torch.cuda.current_stream(dev)
        _, d2h = _side_streams(dev)
        with torch.cuda.device(dev):
            out = torch.empty((nout,), dtype=torch.float64, device=dev)
            hw = _pinned(hostbuf, "w", (nout,), torch.float64)
            d2h.wait_stream(cur)
            chunks = max(1, min(chunks, nblk // 64 if nblk >= 64 else 1))
            bounds = _chunk_bounds(nblk, chunks)
            ws = resynth_workspace(F, K, int(pk["tstart"].shape[0]), max(b - a for a, b in zip(bounds, bounds[1:])), dev,
                                   hop=hop)
            pws = _phase_ws(phase_preserve, pk["pf"].numel(), dev)  # the phase scan runs with the first chunk
            _mark("pack done", cur)
            for i in range(chunks):
                b0, b1 = bounds[i], bounds[i + 1]
                n0, n1 = b0 * hop, min(b1 * hop, nout)
                resynth_device(tr["tid"], pk, sr, hop, self.nfft, self.hop, edge=edge, minframes=minframes,
                               max_end=max_end, block0=b0, nblocks=b1 - b0, out=out[n0:n1], ws=ws, reuse_tracks=i > 0,
                               phase_preserve=phase_preserve, fscale=fscale, phase_ws=pws)
                ev = torch.cuda.Event()
                ev.record(cur)
                _mark("resynth %d" % i, cur)
                with torch.cuda.stream(d2h):
                    d2h.wait_event(ev)
                    hw[n0:n1].copy_(out[n0:n1], non_blocking=True)
                    _mark("w d2h %d" % i, d2h)
            d2h.synchronize()
        self.d2h_bytes = nout * 8
        self._last_out = out
        return hw[:nout].numpy()

    def partial_samples(self, hop, edge=1.0, minframes=3):
        """Work units of synth(): sum over rendered partials of hop*nfr + 2*edgsam."""
        h = self._host_tracks()
        dfr = self.nfft / self.hop / 2.
        e = int(dfr * hop * edge)
        tl = h["tlen"][h["tlen"] >= minframes].astype(np.int64)
        return int((tl * hop + 2 * e).sum())

    # -- summaries (PVAnalysis.py:960-994,1072-1111) ---------------------------------------
    def get_partials_idx_at_frame(self, fr):
        h = self._host_tracks()
        s = h["tstart"].astype(np.int64)
        return np.flatnonzero((fr >= s) & (fr <= s + h["tlen"] - 1))

    def get_partials_at_frame(self, fr):
        return [self.partial[int(i)] for i in self.get_partials_idx_at_frame(fr)]

    def get_partials_idx_ending_at_frame(self, fr):
        h = self._host_tracks()
        s = h["tstart"].astype(np.int64)
        return np.flatnonzero((fr >= s) & (fr == s + h["tlen"] - 1))

    def _track_means(self, key):
        h = self._host_tracks()
        if len(h["tlen"]) == 0:
            return np.zeros(0)
        return np.add.reduceat(h[key], h["toff"][:-1]) / h["tlen"]

    def get_avfreq(self):
        return self._track_means("pf")

    def get_avmag(self):
        return self._track_means("pmag")

    def get_summary(self, minlen=10):
        h = self._host_tracks()
        sel = np.flatnonzero(h["tlen"] > minlen)
        psum = np.zeros(len(sel), dtype=[('idx', 'i4'), ('n', 'i4'), ('f', 'f4'), ('mag', 'f4')])
        psum['idx'] = sel
        psum['n'] = h["tlen"][sel]
        psum['f'] = self.get_avfreq()[sel]
        psum['mag'] = self.get_avmag()[sel]
        psum.sort(order='mag')
        return psum

    def get_nframes(self):
        return max(self.end)
