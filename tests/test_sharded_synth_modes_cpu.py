"""CPU: integrated-phase resynthesis of a segment-sharded signal (``ShardedSinSum.synth_local(
phase_preserve=False, fscale=...)``), with the kernels run in the SIMT emulator (tests/emu).  Ranks
are simulated one after another (tests/sharded_emu_util.py) and the concatenated own signals must
equal the unsharded ``pvk_resynth_ex(phase_preserve=0)`` render bit for bit: on goldens, on synthetic
tables that put partial starts and ends at every row around a boundary, and on degenerate plans."""
import ctypes as C

import numpy as np
import pytest

import sharded_emu_util as su
from golden_util import case_golden, case_signal, pv_kwargs
from pypevoc_b200 import dist as D

eh = su.eh

SEMITONES7 = 2 ** (7 / 12.)


@pytest.fixture(scope="module", autouse=True)
def _build():
    eh.build()


def golden(name):
    g = case_golden(name)
    _, sr = case_signal(name)
    kw = pv_kwargs(name)
    tr = eh.track(g["f"], g["mag"])
    tid, pk = su.pack(np.ascontiguousarray(tr["tid"][0]), g["f"], g["mag"], g["realph"])
    return g, sr, kw["nfft"], int(g["hop"]), tid, pk


def max_end(tid):
    return int(np.nonzero((tid >= 0).any(axis=1))[0].max())


def check_equal(tid, pk, f, mag, realph, sr, hop, nfft, hop_an, fscale, world, edge=1.0, minframes=3):
    ref = su.unsharded(tid, pk, sr, hop, nfft, hop_an, edge, minframes, fscale, max_end(tid))
    sig, ranks = su.sharded(tid, f, mag, realph, sr, hop, nfft, hop_an, edge, minframes, fscale, world)
    assert sig.shape == ref.shape
    assert np.array_equal(sig, ref), np.max(np.abs(sig - ref))
    return ref, ranks


CASES = [(name, world, hop_mult, fscale) for name in ("cfg3_clip", "metric_1s") for world in (2, 3, 5)
         for hop_mult, fscale in ((1, 1.0), (2, SEMITONES7), (None, 0.5))]


@pytest.mark.parametrize("name,world,hop_mult,fscale", CASES)
def test_golden_sharded_equals_unsharded(name, world, hop_mult, fscale):
    """hop = the analysis hop, twice it (time stretch) and 200 (the general resynth_kernel path)."""
    g, sr, nfft, hop_an, tid, pk = golden(name)
    hop = 200 if hop_mult is None else hop_mult * hop_an
    check_equal(tid, pk, g["f"], g["mag"], g["realph"], sr, hop, nfft, hop_an, fscale, world)


def test_golden_cases_need_the_handover():
    g, sr, nfft, hop_an, tid, pk = golden("cfg3_clip")
    ref = su.unsharded(tid, pk, sr, 256, nfft, hop_an, 1.0, 3, SEMITONES7, max_end(tid))
    sig, _ = su.sharded(tid, g["f"], g["mag"], g["realph"], sr, 256, nfft, hop_an, 1.0, 3, SEMITONES7, 3,
                        handover=False)
    assert not np.array_equal(sig, ref)


# ------------------------------------------------------------------ synthetic tables
NFFT, HOP_AN, SR = 1024, 256, 16000.0          # dfr 2: Af 2, dE 2; minframes 3: Lb 6, Lf 7


def synthetic(F=60, world=3, seed=0):
    """Partial starts and ends at every row from j0 - Lb to j0 + Lf of every boundary, plus:
    column 0 spans every rank; column 1 exceeds the Nyquist limit at 2^(7/12) only in the last rank's
    own rows; column 2 is born in [j1, j1 + dE] of rank 0 (whose own blocks hold its fade-in head) and
    exceeds the limit only in rank 1's own rows."""
    rng = np.random.default_rng(seed)
    plans = su.plans_for(F, NFFT, HOP_AN, world, 1.0, 3)
    Lb, Lf = D.halos(NFFT, HOP_AN, 1.0, 3)
    j1 = plans[0]["j1"]
    spans = [(0, F - 1, None), (min(5, F - 1), max(F - 3, min(5, F - 1)), None),
             (min(j1 + 1, F - 1), min(j1 + 15, F - 1), None)]
    hi = {1: [max(F - 6, spans[1][0])], 2: [min(j1 + 10, F - 1)]}
    for p in plans[1:]:
        if p["nown"] == 0:
            continue
        for r in range(max(p["j0"] - Lb, 0), min(p["j0"] + Lf + 1, F)):
            spans.append((r, min(r + r % 5, F - 1), None))                     # starts at r
            spans.append((max(r - 1 - r % 4, 0), r, None))                     # ends at r
    K = len(spans)
    tid = np.full((F, K), -1, dtype=np.int32)
    f = np.zeros((F, K))
    mag = np.zeros((F, K))
    realph = np.zeros((F, K))
    for c, (s, e, _) in enumerate(spans):
        n = e - s + 1
        tid[s:e + 1, c] = c
        f[s:e + 1, c] = (300.0 + 170.0 * c % 2900.0) + 15.0 * np.sin(np.arange(n) / 3.0) + rng.standard_normal(n)
        mag[s:e + 1, c] = 0.05 + 0.02 * rng.random(n)
        realph[s:e + 1, c] = rng.uniform(-np.pi, np.pi, n)
    f[:, 1] = np.where(tid[:, 1] >= 0, 3000.0, 0.0)
    for c, rows in hi.items():
        f[rows, c] = 5600.0                                       # 5600 * 2^(7/12) >= 8000 > 5600
    tid, pk = su.pack(tid, f, mag, realph)
    return tid, pk, f, mag, realph, plans


@pytest.mark.parametrize("world", [2, 3, 5])
@pytest.mark.parametrize("hop,fscale", [(256, 1.0), (512, SEMITONES7), (200, 0.5), (200, SEMITONES7)])
def test_synthetic_boundaries(world, hop, fscale):
    tid, pk, f, mag, realph, _ = synthetic(F=60, world=world, seed=world)
    check_equal(tid, pk, f, mag, realph, SR, hop, NFFT, HOP_AN, fscale, world)


def test_synthetic_nyquist_flags_cross_ranks():
    tid, pk, f, mag, realph, plans = synthetic(F=60, world=3)
    ref, ranks = check_equal(tid, pk, f, mag, realph, SR, 256, NFFT, HOP_AN, SEMITONES7, 3)
    g1, g2 = tid[5, 1], tid[plans[0]["j1"] + 1, 2]
    assert [int(r["flags"][g1]) for r in ranks] == [0, 0, 1]        # the last rank alone sees it
    assert [int(r["flags"][g2]) for r in ranks] == [0, 1, 0]        # rank 1 sees it, rank 0 renders its head
    sig, _ = su.sharded(tid, f, mag, realph, SR, 256, NFFT, HOP_AN, 1.0, 3, SEMITONES7, 3, global_flags=False)
    assert not np.array_equal(sig, ref)


@pytest.mark.parametrize("F,world", [(11, 3), (7, 4), (20, 5), (13, 3), (24, 2)])
def test_degenerate_plans(F, world):
    """Too short to shard (rank 0 owns everything, the others nothing), own ranges shorter than the
    halos (a window spans several neighbours, windows starting at frame 0 on ranks > 0), uneven shares."""
    tid, pk, f, mag, realph, plans = synthetic(F=F, world=world, seed=F)
    if F < 4 * world:
        assert all(p["nown"] == 0 for p in plans[1:])
    check_equal(tid, pk, f, mag, realph, SR, 200, NFFT, HOP_AN, SEMITONES7, world)
    check_equal(tid, pk, f, mag, realph, SR, 256, NFFT, HOP_AN, 1.0, world)


def test_handover_rows_follow_the_halos():
    Lb, Lf = D.halos(2048, 512, 1.0, 3)
    plans = D.plan_segments(44100 * 60, 2048, 512, 4)
    dE = 2
    Af = 2
    for p in plans:
        lo, hi = D.handover_rows(p, plans, 2048, 512, 1.0)
        if p["w0"] > 0:
            assert lo == max(Af + 2, 3) == Lb - dE and p["w0"] + lo == p["j0"] - dE
        else:
            assert lo == -1
        if p["rank"] + 1 < len(plans):
            assert p["w0"] + hi == plans[p["rank"] + 1]["j0"] - dE and hi < p["nframes"]


# ------------------------------------------------------------------ argument checks
def _args(**kw):
    F, K, nt = 10, 4, 3
    a = dict(tid=np.zeros((F, K), dtype=np.int32), F=F, K=K, nt=nt, ts=np.zeros(nt, dtype=np.int32),
             tl=np.ones(nt, dtype=np.int32), toff=np.arange(nt + 1, dtype=np.int64), pf=np.full(nt, 100.0),
             ws=np.zeros(1 << 16, dtype=np.uint8), pws=np.zeros(16), rec=np.zeros(2 * K, dtype=np.int64),
             lo=2, hi=5, world=2, rank=1, flags=np.zeros(8, dtype=np.uint8), table=np.zeros((F, K), dtype=np.int32))
    a.update(kw)
    return a


def _scan(a):
    L = eh.lib()
    return L.pvk_resynth_scan(eh.ptr(a["tid"]), a["F"], a["K"], a["nt"], eh.ptr(a["ts"]), eh.ptr(a["tl"]),
                              eh.ptr(a["toff"]), eh.ptr(a["pf"]), eh.ptr(a["pf"]), 16000.0, 16, 64, 16, 1.0,
                              eh.ptr(a["ws"]), a["ws"].size if a["ws"] is not None else 0, eh.ptr(a["pws"]),
                              a["pws"].size if a["pws"] is not None else 0, a["lo"], a["hi"], eh.ptr(a["rec"]),
                              a.get("rec_len", 2 * a["K"]), None)


def _handover(a):
    L = eh.lib()
    recs = a["rec"]
    return L.pvk_resynth_handover(eh.ptr(a["tid"]), a["F"], a["K"], a["nt"], eh.ptr(a["ts"]), eh.ptr(a["tl"]),
                                  eh.ptr(a["toff"]), eh.ptr(a["pws"]), a["pws"].size, eh.ptr(recs),
                                  a.get("recs_len", a["world"] * 2 * a["K"]), a["world"], a["rank"], a["lo"],
                                  eh.ptr(a["ws"]), a["ws"].size, None)


def _flags(a):
    L = eh.lib()
    return L.pvk_nyquist_flags(eh.ptr(a["pf"]), eh.ptr(a["ts"]), a.get("n", a["nt"]), 16000.0, a.get("fscale", 1.0),
                               eh.ptr(a["flags"]), a.get("nflags", 8), None)


def _import(a):
    L = eh.lib()
    return L.pvk_resynth_import_flags(eh.ptr(a["tid"]), a["F"], a["K"], a["nt"], eh.ptr(a["ts"]), eh.ptr(a["table"]),
                                      a.get("table_rows", a["F"]), a.get("row0", 0), eh.ptr(a["flags"]), 8,
                                      eh.ptr(a["ws"]), a["ws"].size, None)


@pytest.mark.parametrize("fn,kw,needle", [
    (_scan, dict(hi=10), "outside"), (_scan, dict(lo=6, hi=5), "after"), (_scan, dict(rec_len=7), "rec_len"),
    (_scan, dict(pws=None), "phase_ws"), (_scan, dict(ws=np.zeros(64, dtype=np.uint8)), "workspace"),
    (_scan, dict(tid=None), "NULL"), (_scan, dict(K=0), "npks"),
    (_handover, dict(rank=2), "rank"), (_handover, dict(lo=10), "outside"), (_handover, dict(recs_len=15), "recs_len"),
    (_handover, dict(rec=None), "recs_len"), (_handover, dict(ws=np.zeros(64, dtype=np.uint8)), "workspace"),
    (_flags, dict(fscale=0.0), "fscale"), (_flags, dict(flags=None), "flags"), (_flags, dict(n=-1), "negative"),
    (_import, dict(row0=1), "outside"), (_import, dict(table_rows=5), "outside"), (_import, dict(table=None), "NULL"),
    (_import, dict(flags=None), "flags"),
])
def test_new_exports_reject_arguments(fn, kw, needle):
    a = _args(**kw)
    before = {k: v.copy() for k, v in a.items() if isinstance(v, np.ndarray)}
    n0 = eh.lib().pvk_launch_count()
    assert fn(a) != 0
    assert needle in eh.lib().pvk_last_error().decode()
    assert eh.lib().pvk_launch_count() == n0                       # refused before anything was launched
    for k, v in before.items():
        assert np.array_equal(a[k], v, equal_nan=True), k


def test_render_refuses_phase_preserve():
    L = eh.lib()
    a = _args()
    out = np.zeros(64)
    st = L.pvk_resynth_render(eh.ptr(a["tid"]), 10, 4, 3, None, eh.ptr(a["ts"]), eh.ptr(a["tl"]), eh.ptr(a["toff"]),
                              eh.ptr(a["pf"]), eh.ptr(a["pf"]), eh.ptr(a["pf"]), 16000.0, 16, 64, 16, 1.0, 1, eh.ptr(out),
                              64, 0, -1, eh.ptr(a["ws"]), a["ws"].size, 0, 1, 1.0, eh.ptr(a["pws"]), 16, None)
    assert st != 0 and "phase_preserve" in L.pvk_last_error().decode()


def test_new_exports_declared():
    from pypevoc_b200 import _lib
    for name in ("pvk_resynth_scan", "pvk_resynth_handover", "pvk_nyquist_flags", "pvk_resynth_import_flags",
                 "pvk_resynth_render"):
        assert _lib.SIGNATURES[name][0] is C.c_int
    assert _lib.SIGNATURES["pvk_resynth_render"][1] == _lib.SIGNATURES["pvk_resynth_ex"][1]
