"""CPU: the time map of the resynthesis (``synth(time_map=...)``, ``pvk_time_map``) with the kernels run in
the SIMT emulator (tests/emu): the kernel against the float64 model of tests/time_map_oracle.py bit for bit
(synthetic tables of 1 to 1024 peaks per row, goldens, every kind of map), the identity map through pack
and render against the render without a map, mapped renders against the float64 reference of the render
contract (tests/render_contract.py), and the argument checks of the host and of the export."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

import render_contract as rc
import resynth_emu as rem
import time_map_emu as tme
import time_map_oracle as tmo
from golden_util import case_golden, case_signal, pv_kwargs
from pypevoc_b200 import pv as P

eh = rem.eh

TAU_EMU = 2e-6          # the render contract's bound for the emulated kernels (test_render_contract_cpu)
FLOOR = 1e-9


@pytest.fixture(scope="module", autouse=True)
def _build():
    eh.build()


def run_table(F, K, seed, minframes=3):
    """A ``make_table`` peak table (F >= 8) whose partials are the runs of its columns (the table is
    written so that the tracker finds exactly these), packed by the emulated pvk_track_pack: (tid, pk, table)."""
    t = rc.make_table(F, K, rc.SR, seed=seed, minframes=minframes, stationary=K > 64)
    t["mag"][[5, 7], 0] = 0.0                                       # column 0: a partial of one row at row 6
    on = t["mag"] > 0
    starts = on & ~np.vstack([np.zeros((1, K), dtype=bool), on[:-1]])
    run = np.cumsum(starts.T.reshape(-1)).reshape(K, F).T - 1     # run number, column after column
    tid, _ = rem.pack(np.where(on, run, -1).astype(np.int32), t["f"], t["mag"], t["realph"])
    nt = int(tid.max()) + 1
    pk = eh.track_pack(t["f"], t["mag"], t["ph"], t["realph"], tid, None, nt)
    return tid, pk, t


def golden(name):
    """A golden case tracked and packed by the emulated kernels: (sr, nfft, hop_an, tid, pk)."""
    g = case_golden(name)
    sr = float(g["sr"]) if "sr" in g.files else case_signal(name)[1]
    nfft = int(g["nfft"]) if "nfft" in g.files else pv_kwargs(name)["nfft"]
    tr = eh.track(g["f"], g["mag"])
    tid = np.ascontiguousarray(tr["tid"][0])
    pk = eh.track_pack(g["f"], g["mag"], g["ph"], g["realph"], tid, None, int(tr["ntracks"][0]))
    return sr, nfft, int(g["hop"]), tid, pk


@pytest.mark.parametrize("K", [1, 3, 50, 400, 1024])
def test_kernel_matches_oracle_synthetic(K):
    F = 10 if K >= 400 else 30
    tid, pk, _ = run_table(F, K, seed=K)
    assert (pk["tlen"] == 1).any()                                  # partials of length 1
    for name, tau in tmo.example_maps(F).items():
        tmo.check_bits(tme.time_map(tid, pk, tau), tmo.time_map(tid, pk, tau))


@pytest.mark.parametrize("name", ["metric_1s", "real_speech", "cfg5_like"])
def test_kernel_matches_oracle_goldens(name):
    sr, nfft, hop_an, tid, pk = golden(name)
    F = tid.shape[0]
    speed = 0.8 + 0.45 * (0.5 + 0.5 * np.sin(np.arange(2 * F) * 0.05))
    for tau in list(tmo.example_maps(F).values()) + [tmo.speed_map(speed, F)]:
        tmo.check_bits(tme.time_map(tid, pk, tau), tmo.time_map(tid, pk, tau))


def test_ids_beyond_ntracks_are_no_points():
    tid, pk, _ = run_table(20, 6, seed=3)
    tau = np.arange(0.0, 19.0, 0.6)
    nt = len(pk["tstart"])
    got = tme.time_map(tid, pk, tau, ntracks=nt - 3)
    ref = list(tmo.time_map(tid, pk, tau))
    cut = ref[0] >= nt - 3
    ref[0] = np.where(cut, -1, ref[0]).astype(np.int32)
    for j in (1, 2, 3):
        ref[j] = np.where(cut, 0.0, ref[j])
    tmo.check_bits(got, ref)


def test_jumps_leave_partials_without_points():
    """A map that jumps over rows keeps the ids of the partials it skips, packed with tlen 0."""
    tid, pk, _ = run_table(30, 12, seed=9)
    tm, pkm, last = tme.time_map_pack(tid, pk, tmo.example_maps(30)["jump35"])
    assert len(pkm["tstart"]) == len(pk["tstart"])
    assert (pkm["tlen"] == 0).any() and (pkm["tlen"] > 0).any()
    assert last == rem.max_end(tm)
    assert np.array_equal(np.diff(pkm["toff"]), pkm["tlen"])


# ------------------------------------------------------------------ render
def gains(tid, pk, q):
    """pvk_formant_gains through the emulator: the magnitudes a formant-shifting render takes."""
    L = eh.lib()
    F, K = tid.shape
    out = np.full(max(len(pk["pmag"]), 1), np.nan)
    if np.ndim(q) == 0:
        qa = (float(q), None, 0)
    else:
        qc = np.ascontiguousarray(q, dtype=np.float64)
        qa = (1.0, eh.ptr(qc), qc.size)
    eh.check(L.pvk_formant_gains(eh.ptr(np.ascontiguousarray(tid, dtype=np.int32)), F, K, len(pk["tstart"]), None,
                                 eh.ptr(pk["tstart"]), eh.ptr(pk["toff"]), eh.ptr(pk["pf"]), eh.ptr(pk["pmag"]), *qa,
                                 eh.ptr(out), out.size, None))
    return out


@pytest.mark.parametrize("hop", [256, 512, 200])
def test_identity_map_renders_bit_for_bit(hop):
    F, K, nfft, hop_an = 36, 10, 1024, 256
    tid, pk, _ = run_table(F, K, seed=hop)
    tm, pkm, last = tme.time_map_pack(tid, pk, np.arange(F, dtype=np.float64))
    assert np.array_equal(tm, tid) and last == rem.max_end(tid)
    for n in ("tstart", "tlen", "toff", "pf", "pmag", "prealph"):
        assert np.array_equal(pkm[n], pk[n]), n
    nout = P.synth_geometry(last, hop, nfft, hop_an)[0]
    vib = rc.vibrato(F, hop_an, rc.SR, semis=2.0)
    for r, phi in ((1.0, None), (2 ** (7 / 12.), None), (vib, None), (1.5, 1.0), (vib, vib[::-1])):
        pm, pmm = None, None
        if phi is not None:
            q = P.formant_ratio(False, r, phi)
            pm, pmm = gains(tid, pk, q), gains(tm, pkm, q)
            assert np.array_equal(pm, pmm)
        a = rem.render(tid, pk, rc.SR, hop, nfft, hop_an, fscale=r, pmag=pm, nout=nout)
        b = rem.render(tm, pkm, rc.SR, hop, nfft, hop_an, fscale=r, pmag=pmm, nout=nout)
        assert np.all(np.isfinite(a)) and np.array_equal(a, b)


def mapped_reference_check(tid, pk, tau, sr, hop, nfft, hop_an, r, minframes=3, edge=1.0, label=""):
    tm, pkm, last = tme.time_map_pack(tid, pk, tau)
    nout = P.synth_geometry(last, hop, nfft, hop_an, edge)[0]
    w = rem.render(tm, pkm, sr, hop, nfft, hop_an, edge, minframes, fscale=r, nout=nout)
    parts = [p for p in rem.parts(pkm) if len(p["f"]) > 0]
    ref = rc.reference(parts, sr, hop, nfft, hop_an, edge, minframes, "free", r)
    scale = rc.amp_scale(parts, sr, hop, nfft, hop_an, edge, minframes, r)
    rc.check_render(w, ref, scale, TAU_EMU, FLOOR, label, hop)
    return pkm


@pytest.mark.parametrize("hop", [256, 512, 200])
def test_mapped_render_matches_reference(hop):
    """Stretch curves, a freeze and jumps that leave partials without points, rendered from the mapped
    pack and checked sample by sample against the float64 integrated-phase reference of its partials."""
    F, K, nfft, hop_an = 40, 10, 1024, 256
    tid, pk, _ = run_table(F, K, seed=100 + hop)
    speed = 0.8 + 0.45 * (np.arange(60) % 20) / 19.0                # 1.25x .. 0.8x stretch
    cases = dict(stretch2=np.arange(0.0, F - 1, 0.5), curve=tmo.speed_map(speed, F), freeze=tmo.example_maps(F)["freeze"],
                 jump35=tmo.example_maps(F)["jump35"], late_early=tmo.example_maps(F)["late_early"])
    skipped = False
    for name, tau in cases.items():
        B = len(tau)
        for r in (1.0, rc.vibrato(B, hop_an, rc.SR, semis=2.0)):
            pkm = mapped_reference_check(tid, pk, tau, rc.SR, hop, nfft, hop_an, r,
                                         label="%s %s" % (name, "curve" if np.ndim(r) else "scalar"))
            skipped |= bool((pkm["tlen"] == 0).any())
    assert skipped                                                  # the cases hold partials with tlen' = 0


def test_mapped_golden_render_matches_reference():
    sr, nfft, hop_an, tid, pk = golden("real_speech")
    F = tid.shape[0]
    tau = tmo.speed_map(np.where(np.arange(3 * F) < F // 2, 0.5, 1.5), F)
    mapped_reference_check(tid, pk, tau, sr, hop_an, nfft, hop_an, 1.0, label="real_speech 0.5x then 1.5x")


# ------------------------------------------------------------------ argument checks
def test_host_checks():
    F = 12
    for bad in ([0.0, 2.0, 1.0],                          # decreasing
                [0.0, np.nan], [0.0, np.inf],
                [-0.5, 1.0], [0.0, F - 1 + 1e-9],          # out of range
                np.zeros((2, 3)), [],                      # 2-D, empty
                np.zeros(0)):
        with pytest.raises(ValueError):
            P.time_map_values(bad, F)
    for bad in ("0 1 2", 3.0, None, np.array(["a"]), np.array([True, False]), np.array([1 + 1j])):
        with pytest.raises(TypeError):
            P.time_map_values(bad, F)
    assert np.array_equal(P.time_map_values(np.arange(F), F), np.arange(F, dtype=np.float64))
    assert P.time_map_values([3, 3, 3], F).dtype == np.float64     # a freeze


def fake_sinsum(F, K):
    """A SinSum with host rows only (no device is touched before the checks that fail)."""
    ss = P.SinSum.__new__(P.SinSum)
    ss.nfft, ss.hop, ss.sr, ss._dev = 1024, 256, rc.SR, "cpu"
    ss._rows, ss._pk, ss._hosttrk, ss._maxpitchjmp, ss._after_link = None, None, None, 0.5, None
    ss._trk = None
    z = np.zeros((F, K))
    import torch
    ss._tables = dict(f=torch.from_numpy(z), mag=torch.from_numpy(z), ph=torch.from_numpy(z),
                      realph=torch.from_numpy(z))
    return ss


def test_synth_checks_before_any_launch():
    ss = fake_sinsum(12, 4)
    tau = np.arange(0.0, 11.0, 0.5)                                 # B = 22
    with pytest.raises(ValueError, match="phase_preserve"):
        ss.synth(rc.SR, 256, time_map=tau)
    with pytest.raises(ValueError, match="phase_preserve"):
        ss.synth(rc.SR, 256, phase_preserve=True, time_map=tau)
    with pytest.raises(ValueError):
        ss.synth(rc.SR, 256, phase_preserve=False, time_map=tau[::-1])
    with pytest.raises(ValueError):
        ss.synth(rc.SR, 256, phase_preserve=False, time_map=np.array([0.0, 11.5]))
    with pytest.raises(ValueError, match="22 frames"):
        ss.synth(rc.SR, 256, phase_preserve=False, time_map=tau, fscale=np.ones(12))      # one per table row
    with pytest.raises(ValueError, match="22 frames"):
        ss.synth(rc.SR, 256, phase_preserve=False, time_map=tau, fscale=1.2, formant_shift=np.ones(21))
    with pytest.raises(TypeError):
        ss.synth(rc.SR, 256, phase_preserve=False, time_map="fast")


def test_export_argument_errors():
    """pvk_time_map checks sizes, npks and pointers before any CUDA call."""
    L = eh.lib()
    tid, pk, _ = run_table(8, 4, seed=2)
    tau = np.array([0.0, 1.5, 3.0])
    to = np.zeros((3, 4), dtype=np.int32)
    fo, mo, ro = (np.zeros((3, 4)) for _ in range(3))
    nt = len(pk["tstart"])

    def call(nframes=8, npks=4, ntracks=nt, B=3, tid_p=eh.ptr(tid), tmap=eh.ptr(tau), f_out=eh.ptr(fo),
             pf=eh.ptr(pk["pf"])):
        return L.pvk_time_map(tid_p, nframes, npks, ntracks, eh.ptr(pk["tstart"]), eh.ptr(pk["tlen"]), eh.ptr(pk["toff"]),
                              pf, eh.ptr(pk["pmag"]), eh.ptr(pk["prealph"]), tmap, B, eh.ptr(to), f_out, eh.ptr(mo),
                              eh.ptr(ro), None)
    assert call() == 0
    assert call(B=0, tid_p=None, tmap=None) == 0                    # nothing to map: no pointer is read
    for kw in (dict(npks=0), dict(npks=1025), dict(nframes=-1), dict(ntracks=-1), dict(B=-1), dict(nframes=0),
               dict(tid_p=None), dict(tmap=None), dict(f_out=None), dict(pf=None)):
        assert call(**kw) != 0, kw
        assert b"pvk_time_map" in L.pvk_last_error()
