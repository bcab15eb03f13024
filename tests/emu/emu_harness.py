"""TEST INFRASTRUCTURE ONLY -- drive tests/emu/libpvk_emu.so (the kernels compiled for the
CPU SIMT emulator) through the same C ABI, with numpy arrays standing in for device memory.
Used to debug kernel logic on the GPU-less build container; the real parity tests are the
``-m gpu`` ones that go through pypevoc_b200 -> libpvk.so on the B200."""
import ctypes as C
import os
import subprocess

import numpy as np

from pypevoc_b200 import _lib as binding

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "libpvk_emu.so")


def build(force=False):
    srcs = [os.path.join(HERE, f) for f in ("cuda_emu.h", "cuda_emu.cc")]
    csrc = os.path.join(os.path.dirname(os.path.dirname(HERE)), "pypevoc_b200", "csrc")
    srcs += [os.path.join(csrc, f) for f in os.listdir(csrc)]
    srcs.append(os.path.join(os.path.dirname(os.path.dirname(HERE)), "include", "pvk.h"))
    if force or not os.path.isfile(SO) or any(os.path.getmtime(s) > os.path.getmtime(SO) for s in srcs):
        subprocess.check_call([os.path.join(HERE, "build_emu.sh")], stdout=subprocess.DEVNULL)
    return SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = binding.declare(C.CDLL(build()), strict=False)
    return _lib


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def check(st):
    if st != 0:
        raise RuntimeError("emu libpvk: %s" % lib().pvk_last_error().decode())


def host_tables(sr, nfft, hop, wind=np.hanning):
    """Same expressions as PV.__init__ (PVAnalysis.py:97-118)."""
    win = wind(nfft)
    wfact = np.sqrt(sum(win ** 2) * nfft) / 2.0
    fstep = float(sr) / float(nfft)
    dt = float(hop) / float(sr)
    fbin = np.arange(float(nfft)) * fstep
    pi2 = 2.0 * np.pi
    wfbin = np.round(pi2 * fbin * dt / pi2) * pi2
    return dict(win_scaled=np.ascontiguousarray((win / wfact).astype(np.float32)), fbin=fbin,
                wfbin=wfbin, dt=dt, fstep=fstep, wfact=wfact)


def analyze(x, sr, nfft, hop, npks, pkthresh=0.005, nclips=1, frame0=0, nframes=None,
            prev_zero=1, run_frames=0, spectra=False, wind=np.hanning, refine=False, out_rows=None):
    """``out_rows`` (>= nframes): pvk_analyze_batch -- tables [nclips, out_rows, npks] (fine_pos /
    fine_val with ``refine``) whose rows beyond nframes are zero guard rows."""
    L = lib()
    x = np.ascontiguousarray(x, dtype=np.float32)
    if x.ndim == 1:
        x = x[None, :]
    nclips, nsamp = x.shape
    tb = host_tables(sr, nfft, hop, wind)
    if nframes is None:
        span = nsamp - nfft
        nframes = 0 if span <= 0 else -(-span // hop)
        nframes -= frame0
    tbytes = L.pvk_analyze_tables_bytes(nfft)
    assert tbytes > 0
    tables = np.zeros(tbytes, dtype=np.uint8)
    check(L.pvk_analyze_init(nfft, ptr(tables), None))
    shp = (nclips, nframes, npks)
    out = {k: np.full(shp, np.nan) for k in ("f", "mag", "ph", "realph", "binno")}
    npk = np.full((nclips, nframes), -7, dtype=np.int32)
    totalmag = np.full((nclips, nframes), np.nan)
    spec = np.zeros((nclips, nframes, nfft // 2, 2), dtype=np.float32) if spectra else None
    if out_rows is not None:
        assert not spectra and out_rows >= nframes
        shp = (nclips, out_rows, npks)
        names = ("f", "mag", "ph", "realph", "binno") + (("fine_pos", "fine_val") if refine else ())
        out = {k: np.full(shp, np.nan) for k in names}
        for v in out.values():
            v[:, nframes:] = 0.0
        npk = np.zeros((nclips, out_rows), dtype=np.int32)
        totalmag = np.zeros((nclips, out_rows))
        check(L.pvk_analyze_batch(ptr(x), nclips, x.strides[0] // 4, nsamp, ptr(tb["win_scaled"]), ptr(tb["fbin"]),
                                  ptr(tb["wfbin"]), ptr(tables), nfft, hop, npks, pkthresh, tb["dt"], tb["fstep"],
                                  frame0, nframes, prev_zero, run_frames, ptr(out["f"]), ptr(out["mag"]),
                                  ptr(out["ph"]), ptr(out["realph"]), ptr(out["binno"]), ptr(npk), ptr(totalmag),
                                  None, ptr(out.get("fine_pos")), ptr(out.get("fine_val")), out_rows, None))
    elif refine:
        out["fine_pos"], out["fine_val"] = np.full(shp, np.nan), np.full(shp, np.nan)
        check(L.pvk_analyze_ex(ptr(x), nclips, x.strides[0] // 4, nsamp, ptr(tb["win_scaled"]), ptr(tb["fbin"]),
                               ptr(tb["wfbin"]), ptr(tables), nfft, hop, npks, pkthresh, tb["dt"], tb["fstep"],
                               frame0, nframes, prev_zero, run_frames, ptr(out["f"]), ptr(out["mag"]),
                               ptr(out["ph"]), ptr(out["realph"]), ptr(out["binno"]), ptr(npk), ptr(totalmag),
                               ptr(spec), ptr(out["fine_pos"]), ptr(out["fine_val"]), None))
    else:
        check(L.pvk_analyze(ptr(x), nclips, x.strides[0] // 4, nsamp, ptr(tb["win_scaled"]), ptr(tb["fbin"]),
                            ptr(tb["wfbin"]), ptr(tables), nfft, hop, npks, pkthresh, tb["dt"], tb["fstep"],
                            frame0, nframes, prev_zero, run_frames, ptr(out["f"]), ptr(out["mag"]),
                            ptr(out["ph"]), ptr(out["realph"]), ptr(out["binno"]), ptr(npk), ptr(totalmag),
                            ptr(spec), None))
    out.update(npk=npk, totalmag=totalmag, nframes=nframes)
    if spectra:
        out["fx"] = spec[..., 0] + 1j * spec[..., 1]
    return out


def harmonic(x, sr, f0, nfft, hop, npks, fmin=30.0, run_frames=0, wind=np.hanning):
    """pvk_harmonic on host arrays (PVHarmonic.run_pv)."""
    L = lib()
    x = np.ascontiguousarray(x, dtype=np.float32)
    nsamp = len(x)
    tb = host_tables(sr, nfft, hop, wind)
    span = nsamp - nfft
    nframes = 0 if span <= 0 else -(-span // hop)
    f0 = np.ascontiguousarray(f0, dtype=np.float64)
    assert len(f0) >= nframes
    tables = np.zeros(L.pvk_analyze_tables_bytes(nfft), dtype=np.uint8)
    check(L.pvk_analyze_init(nfft, ptr(tables), None))
    out = {k: np.full((nframes, npks), np.nan) for k in ("f", "mag", "ph")}
    res = np.full(nframes, -5.0)
    nharm = np.full(nframes, -7, dtype=np.int32)
    check(L.pvk_harmonic(ptr(x), nsamp, ptr(tb["win_scaled"]), ptr(tb["fbin"]), ptr(tb["wfbin"]), ptr(tables),
                         nfft, hop, npks, tb["dt"], float(sr), float(fmin), ptr(f0), nframes, run_frames,
                         ptr(out["f"]), ptr(out["mag"]), ptr(out["ph"]), ptr(res), ptr(nharm), None))
    out.update(residuals=res, nharm=nharm, nframes=nframes)
    return out


def frame_stats(f, mag, fmin=50, fmax=10000, thr=0.1):
    """pvk_frame_stats on host arrays [F, K]."""
    L = lib()
    f = np.ascontiguousarray(f, dtype=np.float64)
    mag = np.ascontiguousarray(mag, dtype=np.float64)
    F, K = f.shape
    fm = np.full(F, np.nan)
    idx = np.full(F, -9, dtype=np.int32)
    ps = np.full(F, np.nan)
    check(L.pvk_frame_stats(ptr(f), ptr(mag), F, K, float(fmin), float(fmax), float(thr), ptr(fm), ptr(idx), ptr(ps), None))
    return fm, idx, ps


def harmonic_power(f, mag, f_threshold=0.01):
    """pvk_harmonic_power on host arrays [F, K] -> (hpower, nharmonics, err)."""
    L = lib()
    f = np.ascontiguousarray(f, dtype=np.float64)
    mag = np.ascontiguousarray(mag, dtype=np.float64)
    F, K = f.shape
    hp, nh = np.full((F, K), np.nan), np.full((F, K), np.nan)
    rowpow = np.full(max(min(F, K), 1), np.nan)
    err = np.zeros(1, dtype=np.int32)
    check(L.pvk_harmonic_power(ptr(f), ptr(mag), F, K, float(f_threshold), ptr(rowpow), ptr(hp), ptr(nh), ptr(err), None))
    return hp, nh, int(err[0])


def track(f, mag, maxpitchjmp=0.5):
    """pvk_track on host arrays; f, mag [F, K] or [nclips, F, K]."""
    L = lib()
    f = np.ascontiguousarray(f, dtype=np.float64)
    mag = np.ascontiguousarray(mag, dtype=np.float64)
    if f.ndim == 2:
        f, mag = f[None], mag[None]
    nclips, F, K = f.shape
    tid = np.full((nclips, F, K), -99, dtype=np.int32)
    link = np.full((nclips, F, K), -99, dtype=np.int32)
    ntracks = np.full(nclips, -1, dtype=np.int32)
    wsb = L.pvk_track_workspace_bytes(nclips, F, K)
    ws = np.zeros(max(wsb, 8), dtype=np.uint8)
    check(L.pvk_track(ptr(f), ptr(mag), nclips, F, K, maxpitchjmp, ptr(tid), ptr(link), ptr(ntracks),
                      ptr(ws), wsb, None))
    stats = np.full((3, nclips), -77, dtype=np.int64)
    check(L.pvk_track_stats(ptr(tid), ptr(ntracks), nclips, F, K, ptr(stats), None))
    return dict(tid=tid, link=link, ntracks=ntracks, stats=stats)


def track_pack(f, mag, ph, realph, tid, link, ntracks):   # link unused (kept for call sites)
    """pvk_track_pack for one clip ([F, K] arrays)."""
    L = lib()
    F, K = f.shape
    arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in (f, mag, ph, realph)]
    tid = np.ascontiguousarray(tid, dtype=np.int32)
    npts = int((tid >= 0).sum())
    tstart = np.full(max(ntracks, 1), -1, dtype=np.int32)
    tlen = np.full(max(ntracks, 1), -1, dtype=np.int32)
    toff = np.full(ntracks + 1, -1, dtype=np.int64)
    packed = [np.full(max(npts, 1), np.nan) for _ in range(4)]
    wsb = L.pvk_track_pack_workspace_bytes(ntracks)
    ws = np.zeros(max(wsb, 8), dtype=np.uint8)
    check(L.pvk_track_pack(ptr(arrs[0]), ptr(arrs[1]), ptr(arrs[2]), ptr(arrs[3]), ptr(tid), F, K,
                           ntracks, ptr(tstart), ptr(tlen), ptr(toff), ptr(packed[0]), ptr(packed[1]),
                           ptr(packed[2]), ptr(packed[3]), ptr(ws), int(wsb), None))
    return dict(tstart=tstart[:ntracks], tlen=tlen[:ntracks], toff=toff, pf=packed[0][:npts],
                pmag=packed[1][:npts], pph=packed[2][:npts], prealph=packed[3][:npts])


def resynth(tid, pk, sr, hop, nfft, hop_an, edge=1.0, minframes=3, block0=0, nblocks=-1, nout=None,
            ws_blocks=None):
    """pvk_resynth for one clip: tid [F, K], pk = dict from track_pack; ``ws_blocks``: see
    resynth_emu.workspace."""
    import resynth_emu              # tests/resynth_emu.py imports this module
    L = lib()
    tid = np.ascontiguousarray(tid, dtype=np.int32)
    F, K = tid.shape
    nt = len(pk["tstart"])
    max_end = int((pk["tstart"] + pk["tlen"] - 1).max()) if nt else -1
    dfr = 1.0 / (hop_an / float(nfft)) / 2.0
    E = int(dfr * hop * edge)
    if nout is None:
        nout = (max_end + 2) * hop + E
    nblk = -(-nout // hop)
    nb = nblk - block0 if nblocks < 0 else nblocks
    out = np.full(min(nb * hop, nout - block0 * hop), np.nan)
    ts = np.ascontiguousarray(pk["tstart"], dtype=np.int32)
    tl = np.ascontiguousarray(pk["tlen"], dtype=np.int32)
    ws = resynth_emu.workspace(F, K, nt, nb, ws_blocks)
    check(L.pvk_resynth(ptr(tid), F, K, nt, ptr(ts), ptr(tl), ptr(pk["toff"]), ptr(pk["pf"]), ptr(pk["pmag"]),
                        ptr(pk["prealph"]), float(sr), int(hop), int(nfft), int(hop_an), float(edge),
                        int(minframes), ptr(out), nout, block0, nblocks, ptr(ws), ws.size, 0, None))
    return out


def segment_stitch(tids, plans, store="rename"):
    """pvk_segment_summary -> (concatenate = all_gather) -> pvk_segment_resolve -> the renaming store of
    every segment; tids[r]: local ids int32 [rows, K] of segment r.  ``store``: "rename"
    (pvk_segment_rename) writes each segment's renamed own rows to an array of their own; "push"
    (pvk_segment_rename_push) stores them into the tables of ALL ranks (here: `world` numpy arrays
    standing in for local + peer memory); "mcast" (pvk_segment_rename_mcast) stores them once, to one
    table standing in for the multicast address of all ranks' tables.  Returns (the arrays written: the
    own rows of every segment, or the tables, each of which must be the complete global table; total
    partials; last frame with a point)."""
    L = lib()
    world = len(plans)
    K = tids[0].shape[1]
    F = sum(p["nown"] for p in plans)
    summ = np.zeros((world, 2 * K + 4), dtype=np.int32)
    tids = [np.ascontiguousarray(t, dtype=np.int32) for t in tids]
    for r, p in enumerate(plans):
        check(L.pvk_segment_summary(ptr(tids[r]), K, p["own0"], p["nown"], p["j0"], ptr(summ[r]), None))
    out = [np.full((F, K), -7, dtype=np.int32) for _ in range({"rename": 0, "push": world, "mcast": 1}[store])]
    dst = np.array([t.ctypes.data for t in out], dtype=np.uint64)
    cap = max(max(q["own0"] for q in plans) * K, 1)          # scratch holds any segment's back-halo ids
    for r, p in enumerate(plans):
        scratch = np.zeros(cap, dtype=np.int32)
        gidlow = np.zeros(cap, dtype=np.int32)
        params = np.zeros(8, dtype=np.int32)
        check(L.pvk_segment_resolve(ptr(summ), world, K, r, ptr(scratch), cap, ptr(gidlow), ptr(params), None))
        own = np.ascontiguousarray(tids[r][p["own0"]:p["own0"] + p["nown"]])
        if store == "rename":
            out.append(np.empty_like(own))
            check(L.pvk_segment_rename(ptr(own), own.size, ptr(gidlow), ptr(params), ptr(out[-1]), None))
        elif store == "push":
            check(L.pvk_segment_rename_push(ptr(own), own.size, ptr(gidlow), ptr(params), ptr(dst), world,
                                            p["j0"] * K, None))
        else:
            check(L.pvk_segment_rename_mcast(ptr(own), own.size, ptr(gidlow), ptr(params), ptr(out[0]), p["j0"] * K,
                                             None))
    return out, int(params[3]), int(params[4])


def stft_bank(x, win, nfft, hop, nframes, fb_folded=None, fb_lo=None, fb_hi=None, flux_bins=None, inv_wsum2=None,
              run_frames=0):
    """pvk_stft_bank through the emulator; returns dict(bank, flux, rms) of the requested outputs."""
    L = lib()
    x = np.ascontiguousarray(x, dtype=np.float32)
    win = np.ascontiguousarray(win, dtype=np.float32)
    tables = np.zeros(L.pvk_analyze_tables_bytes(nfft), dtype=np.uint8)
    check(L.pvk_analyze_init(nfft, ptr(tables), None))
    out = {}
    nfilt = 0
    if fb_folded is not None:
        fb_folded = np.ascontiguousarray(fb_folded, dtype=np.float64)
        fb_lo = np.ascontiguousarray(fb_lo, dtype=np.int32)
        fb_hi = np.ascontiguousarray(fb_hi, dtype=np.int32)
        nfilt = fb_folded.shape[0]
        out["bank"] = np.full((nframes, nfilt), np.nan)
    if flux_bins is not None:
        out["flux"] = np.full((max(nframes - 1, 0),), np.nan)
    if inv_wsum2 is not None:
        out["rms"] = np.full((nframes,), np.nan)
    lo, hi = flux_bins if flux_bins is not None else (0, 0)
    check(L.pvk_stft_bank(ptr(x), x.size, ptr(win), ptr(tables), nfft, hop, nframes, run_frames, ptr(fb_folded),
                          ptr(fb_lo), ptr(fb_hi), nfilt, ptr(out.get("bank")), int(lo), int(hi), ptr(out.get("flux")),
                          float(inv_wsum2 or 0.0), ptr(out.get("rms")), None))
    return out
