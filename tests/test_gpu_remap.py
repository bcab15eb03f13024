"""GPU: the remap of the partials (``SinSum.remap(tau)``, ``pvk_track_relink``) on the B200: the relink, the stats
and the pack against the float64 model of tests/remap_oracle.py bit for bit (synthetic tables, goldens, the
60 s benchmark prefix under a ping-pong map), a non-decreasing remap against ``synth(time_map=...)`` bit for
bit on every ``SinSum.synth`` path, remapped renders against the float64 render reference (per sample, within
the bound of tests/test_gpu_render_contract.py), the state of a remapped SinSum, and two behavioural checks by
re-analysis: a rising glide played backwards falls, and a looped sustained tone keeps one partial and its
level across the loop point."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import remap_oracle as rmo
import render_contract as rc
import time_map_oracle as tmo
from golden_util import case_golden
from test_gpu_render_contract import FLOOR, GPU_CASES, TAU_GPU
from test_gpu_time_map import host_pk, rc_parts, tracked

pytestmark = pytest.mark.gpu

SR = rc.SR


@pytest.fixture(scope="module")
def P():
    from pypevoc_b200 import _lib, pv
    _lib.lib()
    return pv


def check_device(P, tid, pk, tau):
    """pv.remap_device against the model, bit for bit: ids, links, counts and every packed array."""
    tables, tr, pkr = P.remap_device(tid, pk, torch.from_numpy(np.ascontiguousarray(tau, dtype=np.float64)).cuda())
    ref_tid, ref_link, ref_pk, _ = rmo.remap(tid.cpu().numpy(), host_pk(pk), tau)
    assert np.array_equal(tr["link"].cpu().numpy(), ref_link)
    assert np.array_equal(tr["tid"].cpu().numpy(), ref_tid)
    assert tr["ntracks"] == len(ref_pk["tstart"]) and tr["npts"] == len(ref_pk["pf"])
    assert int(tr["ntracks_dev"][0].item()) == tr["ntracks"]
    assert tr["max_end"] == (int(np.nonzero((ref_tid >= 0).any(axis=1))[0].max()) if tr["ntracks"] else -1)
    rmo.check_pack(host_pk(pkr), ref_pk)
    return tr


@pytest.mark.parametrize("K", [1, 32, 33, 100, 513, 1024])
def test_gpu_relink_matches_model_synthetic(P, K):
    F = 40
    t = rc.make_table(F, K, SR, seed=K, stationary=K > 64)
    tid, pk = tracked(P, t)
    for tau in rmo.all_maps(F).values():
        check_device(P, tid, pk, tau)


@pytest.mark.parametrize("name", ["metric_1s", "real_speech", "real_guitar"])
def test_gpu_relink_matches_model_goldens(P, name):
    g = case_golden(name)
    tid, pk = tracked(P, dict(f=g["f"], mag=g["mag"], ph=g["ph"], realph=g["realph"]))
    for tau in rmo.all_maps(tid.shape[0]).values():
        check_device(P, tid, pk, tau)


@pytest.fixture(scope="module")
def metric_ss(P):
    """The partials of the 60 s prefix of the benchmark signal, nfft 2048 / hop 512 / npks 50."""
    from pypevoc_b200 import signals
    sr = 44100
    x = signals.harm_torch(sr, 60 * sr, 220.0, 90, 0.5, 0.01, 1, torch.device("cuda"), scale=0.25)
    x = (x * float(np.float32(0.9 / float(x.abs().max())))).cpu().numpy()
    pv = P.PV(x, sr, nfft=2048, hop=512, npks=50, progress=False)
    pv.run_pv()
    ss = pv.toSinSum()
    ss.device_tracks
    return ss


def pingpong(F):
    """A ping-pong over the whole table at 1x: forwards from row 0 to row F - 1, then backwards to row 0."""
    return np.concatenate([np.arange(0.0, F), np.arange(F - 2.0, -1.0, -1.0)])


def test_gpu_relink_matches_model_metric_prefix(P, metric_ss):
    d = metric_ss.device_tracks
    tr = check_device(P, d["tid"], d, pingpong(d["tid"].shape[0]))
    assert tr["ntracks"] > len(metric_ss.st)                        # partials come apart at the turns


def test_gpu_metric_prefix_remapped_per_sample(P, metric_ss):
    sr, nfft, hop_an, hop = 44100, 2048, 512, 512
    rs = metric_ss.remap(pingpong(metric_ss.track_ids.shape[0]))
    w = rs.synth(sr, hop, phase_preserve=False, fscale=1.25)
    parts = rc_parts(rs._host_tracks())
    ref = rc.reference(parts, sr, hop, nfft, hop_an, 1.0, 3, "free", 1.25)
    scale = rc.amp_scale(parts, sr, hop, nfft, hop_an, 1.0, 3, 1.25)
    worst = rc.check_render(np.asarray(w), ref, scale, TAU_GPU, FLOOR, "metric 60 s ping-pong", hop,
                            rc.render_branch(hop, 50, nfft, hop_an, 1.0))
    print("metric 60 s ping-pong worst %.2e" % worst)


@pytest.mark.parametrize("name", ["tile16_taylor_dE2", "tile8", "g8_G2"])
def test_gpu_remapped_render_per_sample(P, name):
    hop, nfft, hop_an, edge, K, F, minframes, ws_blocks = GPU_CASES[name]
    t = rc.make_table(F, K, SR, seed=sum(map(ord, name)), minframes=minframes, stationary=K > 64)
    tid, pk = tracked(P, t)
    br = rc.case_branch(GPU_CASES[name])
    for label, tau in rmo.remap_maps(F).items():
        _, tr, pkr = P.remap_device(tid, pk, torch.from_numpy(tau).cuda())
        parts = rc_parts(host_pk(pkr))
        for r in (1.0, rc.vibrato(len(tau), hop_an, SR, semis=2.0)):
            w = P.resynth_device(tr["tid"], pkr, SR, hop, nfft, hop_an, edge, minframes, max_end=tr["max_end"],
                                 phase_preserve=False, fscale=r).cpu().numpy()
            ref = rc.reference(parts, SR, hop, nfft, hop_an, edge, minframes, "free", r)
            scale = rc.amp_scale(parts, SR, hop, nfft, hop_an, edge, minframes, r)
            lab = "%s %s %s" % (name, label, "curve" if np.ndim(r) else "scalar")
            worst = rc.check_render(w, ref, scale, TAU_GPU, FLOOR, lab, hop, br)
            print("%-40s worst %.2e" % (lab, worst))


def _fresh(P, x, sr):
    pv = P.PV(x, sr, nfft=2048, hop=512, npks=50, progress=False)
    pv.run_pv()
    return pv.toSinSum()


@pytest.mark.parametrize("mode", ["scalar", "curve", "formant", "formant curve"])
def test_gpu_monotone_remap_is_the_time_map(P, mode):
    """For non-decreasing maps, ss.remap(tau).synth(...) renders the bits of ss.synth(..., time_map=tau) on the
    staged and the hostbuf paths and with to_host=False; the source SinSum does not change."""
    from pypevoc_b200 import signals
    sr = 44100
    x = signals.harm(sr, 3.0, 220, 30, 0.5, 0.02, 9)
    ss = _fresh(P, x, sr)
    F = ss.track_ids.shape[0]
    st0, end0, f0, ids0 = list(ss.st), list(ss.end), np.array(ss.partial[3].f, copy=True), ss.track_ids.copy()
    maps = dict(identity=np.arange(F, dtype=np.float64), slow=tmo.speed_map(np.full(2 * F, 0.6), F),
                curve=tmo.speed_map(np.linspace(0.8, 1.25, 2 * F), F), jump35=tmo.example_maps(F)["jump35"])
    for label, tau in maps.items():
        B = len(tau)
        vib = rc.vibrato(B, 512, sr, semis=2.0)
        kw = dict(scalar=dict(fscale=1.5), curve=dict(fscale=vib), formant=dict(fscale=1.5, formant_shift=1.0),
                  **{"formant curve": dict(fscale=vib, formant_shift=vib[::-1])})[mode]
        kw["phase_preserve"] = False
        ref = np.array(ss.synth(sr, 512, time_map=tau, **kw))
        rs = ss.remap(tau)
        assert np.array_equal(np.array(rs.synth(sr, 512, **kw)), ref), label
        assert np.array_equal(np.array(rs.synth(sr, 512, hostbuf={}, chunks=4, **kw)), ref), label
        w = rs.synth(sr, 512, to_host=False, **kw)
        assert torch.is_tensor(w) and w.is_cuda and np.array_equal(w.cpu().numpy(), ref), label
        assert np.array_equal(np.array(_fresh(P, x, sr).remap(tau).synth(sr, 512, **kw)), ref), label
    assert ss.st == st0 and ss.end == end0 and np.array_equal(ss.partial[3].f, f0)
    assert np.array_equal(ss.track_ids, ids0)


def test_gpu_remapped_sinsum_state(P):
    """A remapped SinSum answers partial / st / end / track_ids / device_tracks from its runs, renders with
    time_map, remaps again, and refuses phase_preserve=True; a reversal of a reversal gives back the partials."""
    from pypevoc_b200 import signals
    sr = 44100
    ss = _fresh(P, signals.harm(sr, 2.0, 220, 20, 0.5, 0.02, 5), sr)
    F = ss.track_ids.shape[0]
    rev = np.arange(F - 1, -1, -1.0)
    rs = ss.remap(rev)
    d = rs.device_tracks
    ids = rs.track_ids
    assert ids.shape == (F, ss.track_ids.shape[1]) and np.array_equal(ids, d["tid"].cpu().numpy())
    assert len(rs.partial) == len(ss.partial) == len(rs.st) == len(rs.end)
    ends = np.asarray(ss.end)
    assert sorted(rs.st) == sorted((F - 1 - ends).tolist())
    p = rs.partial[0]
    n = rs.end[0] - rs.st[0] + 1
    assert len(p.f) == n and np.array_equal(np.asarray(p.ph), np.asarray(p.realph))
    with pytest.raises(ValueError, match="phase_preserve"):
        rs.synth(sr, 512)
    back = rs.remap(torch.from_numpy(rev))
    key = lambda s: sorted((s.st[i], tuple(s.partial[i].f), tuple(s.partial[i].mag)) for i in range(len(s.partial)))
    assert key(back) == key(ss)
    a = np.array(rs.synth(sr, 512, phase_preserve=False, time_map=np.arange(0.0, F - 1, 0.5)))
    assert np.array_equal(a, np.array(rs.remap(np.arange(0.0, F - 1, 0.5)).synth(sr, 512, phase_preserve=False)))


# ------------------------------------------------------------------ behaviour, by re-analysis
SR_B, NFFT_B, HOP_B = 16000.0, 1024, 256


def _analyse(P, x, npks=8):
    pv = P.PV(np.asarray(x, dtype=np.float64), SR_B, nfft=NFFT_B, hop=HOP_B, npks=npks, progress=False)
    pv.run_pv()
    return pv


def _dominant(pv):
    f, m = np.asarray(pv.f), np.asarray(pv.mag)
    j = np.argmax(m, axis=1)
    return f[np.arange(len(j)), j]


def test_gpu_reversed_glide_falls(P):
    """A glide 300 -> 600 Hz over 2 s, played backwards, re-analyses as a glide 600 -> 300 Hz: the dominant
    frequency of output frame b is the analysed one of input frame F - 1 - b."""
    t = np.arange(int(2 * SR_B)) / SR_B
    x = 0.5 * np.sin(2 * np.pi * np.cumsum(300.0 * 2 ** (t / 2.0)) / SR_B)
    pv = _analyse(P, x)
    F = pv.f.shape[0]
    fin = _dominant(pv)
    w = pv.toSinSum().remap(np.arange(F - 1, -1, -1.0)).synth(SR_B, HOP_B, phase_preserve=False)
    fd = _dominant(_analyse(P, w))
    core = np.arange(8, F - 8)
    assert np.all(np.diff(fd[core]) < 0.0)
    assert np.max(np.abs(fd[core] / fin[F - 1 - core] - 1.0)) < 1e-2          # two frames of the glide
    assert fd[8] > 560.0 and fd[F - 9] < 320.0


def test_gpu_loop_keeps_one_partial_and_its_level(P):
    """A sustained 500 Hz tone looped from frame 60 back to frame 30 three times: its partial is one partial
    across every loop point (the same id on both sides of each jump), and its RMS in 10 ms windows around
    the jumps stays within 0.5 dB of the steady state."""
    n = int(2 * SR_B)
    x = 0.5 * np.sin(2 * np.pi * 500.0 * np.arange(n) / SR_B)              # 10 ms = 5 periods
    pv = _analyse(P, x, npks=3)
    F = pv.f.shape[0]
    j0, j1 = 30, 60
    tau = np.concatenate([np.arange(0.0, j1 + 1.0)] + [np.arange(j0, j1 + 1.0)] * 3 + [np.arange(j1 + 1.0, F)])
    rs = pv.toSinSum().remap(tau)
    ids = rs.track_ids
    jumps = [j1 + 1 + k * (j1 - j0 + 1) for k in range(3)]
    for b in jumps:
        pa = ids[b - 1][np.argmax(np.where(ids[b - 1] >= 0, rs._tables["mag"][b - 1].cpu().numpy(), -1))]
        pb = ids[b][np.argmax(np.where(ids[b] >= 0, rs._tables["mag"][b].cpu().numpy(), -1))]
        assert pa == pb >= 0, b
    w = np.asarray(rs.synth(SR_B, HOP_B, phase_preserve=False))
    win = int(0.01 * SR_B)
    dfr = NFFT_B / HOP_B / 2.0

    def rms(c):
        return np.sqrt(np.mean(w[c - win // 2:c + win // 2] ** 2))
    steady = np.median([rms(int((b + dfr) * HOP_B)) for b in range(20, len(tau) - 20, 3)])
    for b in jumps:
        centre = int((b + dfr) * HOP_B)                             # output time of the first block after the jump
        for c in range(centre - 2 * HOP_B, centre + 2 * HOP_B + 1, win // 2):
            assert abs(20 * np.log10(rms(c) / steady)) < 0.5, (b, c, rms(c), steady)
