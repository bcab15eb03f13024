"""CPU: the CUDA sources compiled for the SIMT emulator (tests/emu) reproduce the reference.

This runs the *same kernel code* as the GPU (tests/emu/cuda_emu.h turns threads into fibers)
through the same C ABI, so kernel logic regressions are caught on the GPU-less build
container.  It is test infrastructure: the product never loads the emulator library, and
the parity tests proper are the ``-m gpu`` ones."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

from oracle import pv_oracle as orc
from golden_util import CASES, case_golden, case_signal, pv_kwargs
import parity_util as pu

eh = pytest.importorskip("emu_harness")

FAST = ["two_sines", "readme_vibrato", "noisy_odd_hop", "cfg3_clip", "cfg5_like"]


@pytest.fixture(scope="module", autouse=True)
def _build():
    eh.build()


@pytest.mark.parametrize("name", FAST)
def test_emu_analysis_vs_reference_golden(name):
    x, sr = case_signal(name)
    kw = pv_kwargs(name)
    hop = kw["hop"] or kw["nfft"] // 2
    g = case_golden(name)
    o = eh.analyze(x, sr, kw["nfft"], hop, kw["npks"], spectra=True)
    got = {k: o[k][0] for k in ("f", "mag", "ph", "realph", "binno", "totalmag", "npk")}
    ref = {k: g[k] for k in ("f", "mag", "ph", "realph", "binno", "totalmag")}
    pu.compare_analysis(got, ref, sr, kw["nfft"])
    oo = orc.analyze(np.zeros(1), sr, nfft=kw["nfft"], hop=hop, npks=kw["npks"], fx_given=o["fx"][0].astype(np.complex64))
    pu.compare_exact_on_spectrum(got, oo)


@pytest.mark.parametrize("name", FAST)
def test_emu_tracking_and_resynthesis_vs_reference_golden(name):
    g = case_golden(name)
    _, sr = case_signal(name)
    kw = pv_kwargs(name)
    tr = eh.track(g["f"], g["mag"])
    assert np.array_equal(tr["tid"][0], g["tid"])
    nt = int(tr["ntracks"][0])
    pk = eh.track_pack(g["f"], g["mag"], g["ph"], g["realph"], tr["tid"][0], tr["link"][0], nt)
    assert np.array_equal(pk["tstart"], g["st"])
    assert np.array_equal(pk["tstart"] + pk["tlen"] - 1, g["end"])
    for h in CASES[name]["synth_hops"]:
        w = eh.resynth(tr["tid"][0], pk, sr, h, kw["nfft"], int(g["hop"]))
        ref = g["synth_%d" % h]
        assert w.shape == ref.shape
        assert pu.snr_db(w, ref) > 110.0
        # a small workspace renders the same signal chunk by chunk; a block sub-range matches too
        w2 = eh.resynth(tr["tid"][0], pk, sr, h, kw["nfft"], int(g["hop"]), ws_blocks=5)
        assert np.array_equal(w, w2)
        w3 = eh.resynth(tr["tid"][0], pk, sr, h, kw["nfft"], int(g["hop"]), block0=3, nblocks=4)
        assert np.array_equal(w[3 * h:7 * h], w3)


def test_emu_degenerate_and_select_paths():
    rng = np.random.RandomState(3)
    sr = 44100
    cases = []
    cases.append((rng.randn(2048 * 4).astype(np.float32), 2048, 1024, 50, 0.005))    # C > K: radix select
    cases.append((rng.randn(1024 * 4).astype(np.float32), 1024, 512, 3, 0.0))
    z = np.zeros(1024 * 4, dtype=np.float32); cases.append((z, 1024, 256, 20, 0.005))
    imp = np.zeros(1024 * 4, dtype=np.float32); imp[1500] = 1.0; cases.append((imp, 1024, 256, 20, 0.005))
    flat = np.zeros(256 * 4, dtype=np.float32); flat[300] = 1.0; flat[301] = 1e-4; cases.append((flat, 256, 64, 5, 0.5))
    tr_ = np.zeros(512 * 6, dtype=np.float32); tr_[::32] = 1.0; cases.append((tr_, 512, 128, 30, 0.005))
    cases.append((rng.randn(256 * 5).astype(np.float32), 256, 64, 200, -0.1))         # th < 0: every bin a candidate
    cases.append((rng.randn(256 * 5).astype(np.float32), 256, 64, 40, -0.1))          # ... with C > K
    for x, nfft, hop, npks, th in cases:
        o = eh.analyze(x, sr, nfft, hop, npks, pkthresh=th, spectra=True)
        got = {k: o[k][0] for k in ("f", "mag", "ph", "realph", "binno", "totalmag", "npk")}
        oo = orc.analyze(np.zeros(1), sr, nfft=nfft, hop=hop, npks=npks, pkthresh=th,
                         fx_given=o["fx"][0].astype(np.complex64))
        pu.compare_exact_on_spectrum(got, oo)


def test_emu_segment_warmup_and_batch():
    from pypevoc_b200 import signals
    x = signals.harm(44100, 0.4, 220, 90, 0.5, 0.01, 1)
    full = eh.analyze(x, 44100, 2048, 256, 60)
    seg = eh.analyze(x[6 * 256:], 44100, 2048, 256, 60, frame0=1, prev_zero=0)
    for k in ("f", "mag", "ph", "realph", "binno", "npk", "totalmag"):
        assert np.array_equal(full[k][0][7:], seg[k][0]), k
    clips = np.stack([x[:12000], x[3000:15000], np.zeros(12000, dtype=np.float32)])
    b = eh.analyze(clips, 44100, 1024, 256, 20, run_frames=5)
    for i in range(3):
        one = eh.analyze(clips[i], 44100, 1024, 256, 20)
        for k in ("f", "binno", "npk"):
            assert np.array_equal(one[k][0], b[k][i])


def test_emu_track_stitch_across_tiles():
    """Long partials crossing many 128-frame chunks and more than one shared-memory tile of the
    stitch pass (npks = 1024 -> 23 chunks per tile), peaks in random slots."""
    rng = np.random.RandomState(11)
    F, K = 128 * 30 + 17, 1024
    f = np.zeros((F, K)); mag = np.zeros((F, K))
    base = np.array([440.0, 1000.0, 3000.0])
    for j in range(F):
        cols = np.sort(rng.choice(K, 3, replace=False))
        alive = [True, (j // 500) % 2 == 0, j % 97 != 0]       # partial 1 dies / is reborn, 2 has gaps
        for q in range(3):
            if alive[q]:
                f[j, cols[q]] = base[q] * (1 + 0.001 * np.sin(j / 50.0 + q))
                mag[j, cols[q]] = 0.5 / (q + 1) + 0.01 * rng.rand()
    o = orc.track(f, mag)
    tr = eh.track(f, mag)
    assert np.array_equal(tr["tid"][0], o["tid"])
    assert int(tr["ntracks"][0]) == len(o["st"])


def test_emu_track_long_table_scans_stitch_rounds_and_stats():
    """38 400 frames x 8 slots: ten scan tiles, 300 chunk boundary rows = two pointer-jumping tiles of
    256 rows with 9 rounds; partials of every length (short ones die inside a chunk, one lives for
    the whole table, one is reborn every 1000 frames); pvk_track_stats against the oracle."""
    rng = np.random.RandomState(5)
    F, K = 128 * 300, 8
    f = np.zeros((F, K)); mag = np.zeros((F, K))
    for j in range(F):
        cols = rng.permutation(K)
        f[j, cols[0]] = 440.0 * (1 + 0.002 * np.sin(j / 40.0)); mag[j, cols[0]] = 0.5
        if j % 1000 != 999:
            f[j, cols[1]] = 1500.0 + 0.01 * (j % 1000); mag[j, cols[1]] = 0.3
        if rng.rand() < 0.3:
            f[j, cols[2]] = 3000.0 + 900.0 * rng.rand(); mag[j, cols[2]] = 0.1 * rng.rand() + 0.01
    f[-3:] = 0.0; mag[-3:] = 0.0                              # the table ends with empty frames
    o = orc.track(f, mag)
    tr = eh.track(f, mag)
    assert np.array_equal(tr["tid"][0], o["tid"])
    assert int(tr["ntracks"][0]) == len(o["st"])
    assert tr["stats"][:, 0].tolist() == [int((o["tid"] >= 0).sum()), int(np.max(o["end"])), len(o["st"])]
    pk = eh.track_pack(f, mag, f, f, tr["tid"][0], None, len(o["st"]))
    assert np.array_equal(pk["tstart"], o["st"]) and np.array_equal(pk["tstart"] + pk["tlen"] - 1, o["end"])
    assert pk["toff"][-1] == tr["stats"][0, 0] and np.array_equal(np.diff(pk["toff"]), pk["tlen"])


@pytest.mark.parametrize("world", [2, 5])
def test_emu_segment_numbering_kernels(world):
    """pvk_segment_summary / _resolve / _rename (global numbering of per-segment linked partials)
    against the reference's numbering of the unsharded table."""
    from pypevoc_b200 import dist as D
    g = case_golden("cfg3_clip")
    F, K = g["f"].shape
    plans = D.plan_segments((F - 1) * 128 + 512 + 1, 512, 128, world)
    tids = [orc.track(g["f"][p["w0"]:p["w1"]], g["mag"][p["w0"]:p["w1"]])["tid"] for p in plans]
    rows, ntot, max_end = eh.segment_stitch(tids, plans)
    assert np.array_equal(np.concatenate(rows), g["tid"])
    assert ntot == len(g["st"]) and max_end == int(np.max(g["end"]))
    # the fused variant: every segment stores its renamed rows into the tables of all ranks
    for table in eh.segment_stitch(tids, plans, store="push")[0]:
        assert np.array_equal(table, g["tid"])


@pytest.mark.parametrize("K,mode", [(150, "asc"), (300, "asc_dense"), (200, "gaps"), (160, "shuffled"), (130, "ties"),
                                    (400, "ties"), (600, "asc_dense"), (520, "gaps")])
def test_emu_large_row_link_kernel(K, mode):
    """Rows wider than 128 peaks: the propose/commit kernel with window re-scans (K <= 512) and the
    sequential sorted-rank / windowed kernel above that -- ascending gap-free rows
    (binary-searched window), rows with holes or out of order (full scan fallback), magnitude
    ties, all against the oracle's sequential greedy loop, bit for bit."""
    f, mag = pu.wide_rows(K, mode)
    tr = eh.track(f, mag)
    ref = orc.track(f, mag)
    assert np.array_equal(tr["tid"][0], ref["tid"])
    assert int(tr["ntracks"][0]) == int(ref["tid"].max()) + 1


def test_emu_pack_respects_capacity():
    """A pack sized for fewer partials than the table holds (the speculative pack of
    pv.track_pack_device above its cap) writes nothing out of bounds and packs the partials below
    the capacity exactly as a full pack does (ADVICE r1: ids were not bound-checked)."""
    import ctypes as C
    rng = np.random.RandomState(5)
    F, K = 70, 12
    f = np.zeros((F, K)); mag = np.zeros((F, K))
    for j in range(F):                                        # many short partials: births in most frames
        n = rng.randint(3, K + 1)
        cols = np.sort(rng.choice(K, n, replace=False))
        f[j, cols] = np.sort(rng.uniform(100, 8000, n)); mag[j, cols] = rng.uniform(0.1, 1.0, n)
    ph = rng.uniform(-3, 3, (F, K)); rph = rng.uniform(-3, 3, (F, K))
    tr = eh.track(f, mag)
    tid = np.ascontiguousarray(tr["tid"][0])
    nt = int(tr["ntracks"][0])
    full = eh.track_pack(f, mag, ph, rph, tid, None, nt)
    cap = nt // 3
    assert cap >= 4
    L = eh.lib()
    G = 64                                                    # canary elements either side
    tstart = np.full(cap + 2 * G, -77, dtype=np.int32); tlen = np.full(cap + 2 * G, -77, dtype=np.int32)
    toff = np.full(cap + 1 + 2 * G, -77, dtype=np.int64)
    packed = [np.full(F * K + 2 * G, -77.0) for _ in range(4)]
    wsb = L.pvk_track_pack_workspace_bytes(cap)
    ws = np.zeros(max(wsb, 8), dtype=np.uint8)
    at = lambda a: C.c_void_p(a.ctypes.data + G * a.itemsize)  # noqa: E731
    arrs = [np.ascontiguousarray(a) for a in (f, mag, ph, rph)]
    eh.check(L.pvk_track_pack(eh.ptr(arrs[0]), eh.ptr(arrs[1]), eh.ptr(arrs[2]), eh.ptr(arrs[3]), eh.ptr(tid), F, K, cap,
                              at(tstart), at(tlen), at(toff), at(packed[0]), at(packed[1]), at(packed[2]), at(packed[3]),
                              eh.ptr(ws), int(wsb), None))
    for a in (tstart, tlen, toff) + tuple(packed):
        assert np.all(a[:G] == -77) and np.all(a[-G:] == -77)
    assert np.array_equal(tstart[G:G + cap], full["tstart"][:cap]) and np.array_equal(tlen[G:G + cap], full["tlen"][:cap])
    assert np.array_equal(toff[G:G + cap + 1], full["toff"][:cap + 1])
    n = int(full["toff"][cap])
    for q, k in enumerate(("pf", "pmag", "pph", "prealph")):
        assert np.array_equal(packed[q][G:G + n], full[k][:n])
        assert np.all(packed[q][G + n:] == -77)


def test_emu_clip_batch_flattened_with_guard_rows():
    """Clip batches (BASELINE configs[2]): pvk_analyze_batch writes every clip's rows into one table
    with zero guard rows between the clips; ONE pvk_track / pvk_track_pack / pvk_resynth over the
    flattened table equals the per-clip runs -- ids up to the clip's base, signals bit for bit."""
    from pypevoc_b200 import signals
    sr, nfft, hop, npks = 16000, 512, 128, 20
    clips = np.stack([signals.speech_like_clip(s, sr=sr, dur=0.5) for s in (3, 4, 5)])
    F = -(-(clips.shape[1] - nfft) // hop)
    dfr = nfft / hop / 2.0
    E = int(dfr * hop)
    G = 2 * (-(-E // hop)) + 3
    b = eh.analyze(clips, sr, nfft, hop, npks, out_rows=F + G)
    flat = {k: b[k].reshape(-1, npks) for k in ("f", "mag", "ph", "realph")}
    trb = eh.track(flat["f"], flat["mag"])
    ntb = int(trb["ntracks"][0])
    pkb = eh.track_pack(flat["f"], flat["mag"], flat["ph"], flat["realph"], trb["tid"][0], None, ntb)
    wb = eh.resynth(trb["tid"][0], pkb, sr, hop, nfft, hop, nout=clips.shape[0] * (F + G) * hop)
    base = 0
    for c in range(clips.shape[0]):
        a = eh.analyze(clips[c], sr, nfft, hop, npks)
        for k in ("f", "mag", "ph", "realph", "binno"):
            assert np.array_equal(a[k][0], b[k][c, :F]), k
            assert not b[k][c, F:].any()
        tr = eh.track(a["f"][0], a["mag"][0])
        nt = int(tr["ntracks"][0])
        tb = trb["tid"][0][c * (F + G):c * (F + G) + F]
        assert np.array_equal(np.where(tb >= 0, tb - base, -1), tr["tid"][0])
        assert (trb["tid"][0][c * (F + G) + F:(c + 1) * (F + G)] == -1).all()
        pk = eh.track_pack(a["f"][0], a["mag"][0], a["ph"][0], a["realph"][0], tr["tid"][0], None, nt)
        assert np.array_equal(pkb["tstart"][base:base + nt] - c * (F + G), pk["tstart"])
        assert np.array_equal(pkb["tlen"][base:base + nt], pk["tlen"])
        w = eh.resynth(tr["tid"][0], pk, sr, hop, nfft, hop)
        s0 = c * (F + G) * hop
        assert np.array_equal(wb[s0:s0 + len(w)], w)
        assert not wb[s0 + len(w):(c + 1) * (F + G) * hop - E].any()     # (the next clip's fade-in heads come after)
        base += nt
    assert base == ntb


def _many_births_table(seed=5, F=70, K=12):
    rng = np.random.RandomState(seed)
    f = np.zeros((F, K)); mag = np.zeros((F, K))
    for j in range(F):                                        # many short partials: births in most frames
        n = rng.randint(3, K + 1)
        cols = np.sort(rng.choice(K, n, replace=False))
        f[j, cols] = np.sort(rng.uniform(100, 8000, n)); mag[j, cols] = rng.uniform(0.1, 1.0, n)
    return f, mag, rng.uniform(-3, 3, (F, K)), rng.uniform(-3, 3, (F, K))


def test_emu_pack_and_resynth_with_device_side_counts():
    """pvk_track_pack_dev / pvk_resynth_dev (index arrays sized by an upper bound, the real number of
    partials read on the device): same packed tracks and the same signal as the exact-size calls; with
    a capacity BELOW the real count nothing is read or written out of bounds (ids beyond the capacity
    are ignored by every kernel that indexes with them)."""
    import ctypes as C
    f, mag, ph, rph = _many_births_table()
    F, K = f.shape
    tr = eh.track(f, mag)
    tid = np.ascontiguousarray(tr["tid"][0])
    nt = int(tr["ntracks"][0])
    full = eh.track_pack(f, mag, ph, rph, tid, None, nt)
    sr, nfft, hop = 16000, 512, 128
    wfull = eh.resynth(tid, full, sr, hop, nfft, hop)
    L = eh.lib()
    ntd = np.array([nt], dtype=np.int32)
    arrs = [np.ascontiguousarray(a) for a in (f, mag, ph, rph)]
    G = 64
    at = lambda a: C.c_void_p(a.ctypes.data + G * a.itemsize)  # noqa: E731
    for cap in (F * K, nt, nt // 3):
        tstart = np.full(cap + 2 * G, -77, dtype=np.int32); tlen = np.full(cap + 2 * G, -77, dtype=np.int32)
        toff = np.full(cap + 1 + 2 * G, -77, dtype=np.int64)
        packed = [np.full(F * K + 2 * G, -77.0) for _ in range(4)]
        wsb = L.pvk_track_pack_workspace_bytes(cap)
        ws = np.zeros(max(wsb, 8), dtype=np.uint8)
        eh.check(L.pvk_track_pack_dev(eh.ptr(arrs[0]), eh.ptr(arrs[1]), eh.ptr(arrs[2]), eh.ptr(arrs[3]), eh.ptr(tid), F, K,
                                      cap, eh.ptr(ntd), at(tstart), at(tlen), at(toff), at(packed[0]), at(packed[1]),
                                      at(packed[2]), at(packed[3]), eh.ptr(ws), int(wsb), None))
        for a in (tstart, tlen, toff) + tuple(packed):
            assert np.all(a[:G] == -77) and np.all(a[-G:] == -77)
        m = min(cap, nt)
        assert np.array_equal(tstart[G:G + m], full["tstart"][:m]) and np.array_equal(tlen[G:G + m], full["tlen"][:m])
        assert np.array_equal(toff[G:G + m + 1], full["toff"][:m + 1])
        n = int(full["toff"][m])
        for q, k in enumerate(("pf", "pmag", "pph", "prealph")):
            assert np.array_equal(packed[q][G:G + n], full[k][:n])
        # rendering with the upper-bound sizes: (F + 1) * hop + E samples, cut afterwards
        E = int(nfft / hop / 2.0 * hop)
        nout_ub = (F + 1) * hop + E
        out = np.full(nout_ub + 2 * G, -77.0)
        rwsb = int(L.pvk_resynth_workspace_bytes(F, K, cap, -(-nout_ub // hop)))
        rws = np.zeros(max(rwsb, 8), dtype=np.uint8)
        eh.check(L.pvk_resynth_dev(eh.ptr(tid), F, K, cap, eh.ptr(ntd), at(tstart), at(tlen), at(toff), at(packed[0]),
                                   at(packed[1]), at(packed[3]), float(sr), hop, nfft, hop, 1.0, 3, at(out), nout_ub, 0, -1,
                                   eh.ptr(rws), rwsb, 0, None))
        assert np.all(out[:G] == -77) and np.all(out[-G:] == -77)
        if cap >= nt:
            assert np.array_equal(out[G:G + len(wfull)], wfull)
            assert not out[G + len(wfull):G + nout_ub].any()       # beyond the real length: silence


def test_emu_segment_rename_mcast_equals_push():
    """pvk_segment_rename_mcast (one store per id to the multicast address of all ranks' tables; in
    the emulator a plain table) writes what pvk_segment_rename_push writes into every table."""
    from pypevoc_b200 import dist as D
    f, mag, _, _ = _many_births_table(seed=9, F=90, K=10)
    F, K = f.shape
    world = 3
    plans = D.plan_segments(512 + (F - 1) * 128 + 1, 512, 128, world)
    assert plans[-1]["frames_total"] == F
    tids = [np.ascontiguousarray(eh.track(f[p["w0"]:p["w1"]], mag[p["w0"]:p["w1"]])["tid"][0]) for p in plans]
    tables = eh.segment_stitch(tids, plans, store="push")[0]
    (mc,), _, _ = eh.segment_stitch(tids, plans, store="mcast")
    full = eh.track(f, mag)["tid"][0]
    assert np.array_equal(mc, full)
    for t in tables:
        assert np.array_equal(t, mc)
