"""GPU: the time map of the resynthesis (``synth(time_map=...)``, ``pvk_time_map``) on the B200: the kernel
against the float64 model of tests/time_map_oracle.py bit for bit (synthetic tables, goldens, the 60 s
benchmark prefix under a stretch curve), the identity map against no map through every ``SinSum.synth``
path bit for bit, mapped renders against the float64 render reference (per sample, within the bound of
tests/test_gpu_render_contract.py), and two behavioural checks by re-analysis: a freeze holds the
frequency of its input frame, and a two-tone sequence under a 0.5x-then-2x map switches where the map
says."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import render_contract as rc
import time_map_oracle as tmo
from golden_util import case_golden
from test_gpu_render_contract import FLOOR, GPU_CASES, TAU_GPU

pytestmark = pytest.mark.gpu

SR = rc.SR


@pytest.fixture(scope="module")
def P():
    from pypevoc_b200 import _lib, pv
    _lib.lib()
    return pv


def tracked(P, t):
    dev = torch.device("cuda")
    fd, magd, phd, realphd = (torch.from_numpy(np.ascontiguousarray(t[k])).to(dev) for k in ("f", "mag", "ph", "realph"))
    tr = P.track_device(fd, magd)
    nt = int(tr["ntracks"][0].item())
    pk = P.pack_device(fd, magd, phd, realphd, tr["tid"], tr["link"], nt)
    return tr["tid"], pk


def host_pk(pk):
    return {k: (v.cpu().numpy() if torch.is_tensor(v) else v) for k, v in pk.items()}


def device_map(P, tid, pk, tau):
    """pvk_time_map on the device: the mapped tables (tid', f', mag', realph') as numpy arrays."""
    from pypevoc_b200 import _lib
    L = _lib.lib()
    dev = tid.device
    F, K = tid.shape
    td = torch.from_numpy(np.ascontiguousarray(tau, dtype=np.float64)).to(dev)
    B = td.numel()
    to = torch.full((B, K), -99, dtype=torch.int32, device=dev)
    outs = [torch.full((B, K), float("nan"), dtype=torch.float64, device=dev) for _ in range(3)]
    p = P._ptr
    _lib.check(L.pvk_time_map(p(tid), F, K, int(pk["tstart"].shape[0]), p(pk["tstart"]), p(pk["tlen"]), p(pk["toff"]),
                              p(pk["pf"]), p(pk["pmag"]), p(pk["prealph"]), p(td), B, p(to), *(p(o) for o in outs),
                              P._stream()), "pvk_time_map")
    return [to.cpu().numpy()] + [o.cpu().numpy() for o in outs]


def check_kernel(P, tid, pk, tau):
    tmo.check_bits(device_map(P, tid, pk, tau), tmo.time_map(tid.cpu().numpy(), host_pk(pk), tau))


@pytest.mark.parametrize("K", [1, 3, 50, 400, 1024])
def test_gpu_kernel_matches_oracle_synthetic(P, K):
    F = 40
    t = rc.make_table(F, K, SR, seed=K, stationary=K > 64)
    tid, pk = tracked(P, t)
    for tau in tmo.example_maps(F).values():
        check_kernel(P, tid, pk, tau)


@pytest.mark.parametrize("name", ["metric_1s", "real_speech", "cfg5_like"])
def test_gpu_kernel_matches_oracle_goldens(P, name):
    g = case_golden(name)
    tid, pk = tracked(P, dict(f=g["f"], mag=g["mag"], ph=g["ph"], realph=g["realph"]))
    F = tid.shape[0]
    for tau in list(tmo.example_maps(F).values()) + [tmo.speed_map(np.linspace(0.8, 1.25, 2 * F), F)]:
        check_kernel(P, tid, pk, tau)


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


def stretch_curve(F):
    """A map of the whole table whose stretch moves between 0.8x and 1.25x (speed 1.25 .. 0.8)."""
    b = np.arange(2 * F)
    return tmo.speed_map(1.025 + 0.225 * np.sin(2 * np.pi * b / 700.0), F)


def test_gpu_kernel_matches_oracle_metric_prefix(P, metric_ss):
    d = metric_ss.device_tracks
    tau = stretch_curve(d["tid"].shape[0])
    check_kernel(P, d["tid"], d, tau)


def test_gpu_metric_prefix_mapped_per_sample(P, metric_ss):
    sr, nfft, hop_an, hop = 44100, 2048, 512, 512
    d = metric_ss.device_tracks
    tau = stretch_curve(d["tid"].shape[0])
    w = metric_ss.synth(sr, hop, phase_preserve=False, fscale=1.25, time_map=tau)
    tm, pkm, last = P.time_map_device(d["tid"], d, torch.from_numpy(tau).cuda())
    parts = [p for p in rc_parts(host_pk(pkm)) if len(p["f"]) > 0]
    ref = rc.reference(parts, sr, hop, nfft, hop_an, 1.0, 3, "free", 1.25)
    scale = rc.amp_scale(parts, sr, hop, nfft, hop_an, 1.0, 3, 1.25)
    worst = rc.check_render(np.asarray(w), ref, scale, TAU_GPU, FLOOR, "metric 60 s mapped", hop,
                            rc.render_branch(hop, 50, nfft, hop_an, 1.0))
    print("metric 60 s mapped worst %.2e" % worst)


def rc_parts(pk):
    o = pk["toff"]
    return [dict(start_idx=int(pk["tstart"][v]), f=pk["pf"][o[v]:o[v + 1]], mag=pk["pmag"][o[v]:o[v + 1]],
                 realph=pk["prealph"][o[v]:o[v + 1]]) for v in range(len(pk["tstart"]))]


@pytest.mark.parametrize("name", ["tile16_taylor_dE2", "tile8", "g8_G2"])
def test_gpu_mapped_render_per_sample(P, name):
    hop, nfft, hop_an, edge, K, F, minframes, ws_blocks = GPU_CASES[name]
    t = rc.make_table(F, K, SR, seed=sum(map(ord, name)), minframes=minframes, stationary=K > 64)
    tid, pk = tracked(P, t)
    br = rc.case_branch(GPU_CASES[name])
    maps = dict(stretch2=np.arange(0.0, F - 1, 0.5), freeze=tmo.example_maps(F)["freeze"],
                jump35=tmo.example_maps(F)["jump35"], curve=tmo.speed_map(np.linspace(0.8, 1.25, 3 * F), F))
    for label, tau in maps.items():
        tm, pkm, last = P.time_map_device(tid, pk, torch.from_numpy(tau).cuda())
        parts = [p for p in rc_parts(host_pk(pkm)) if len(p["f"]) > 0]
        for r in (1.0, rc.vibrato(len(tau), hop_an, SR, semis=2.0)):
            w = P.resynth_device(tm, pkm, SR, hop, nfft, hop_an, edge, minframes, max_end=last, phase_preserve=False,
                                 fscale=r).cpu().numpy()
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
def test_gpu_identity_map_is_no_map(P, mode):
    """time_map=np.arange(F) renders the same bits as no map on the staged and the hostbuf paths, on
    first use and after; the partials of the SinSum stay as they were."""
    from pypevoc_b200 import signals
    sr = 44100
    x = signals.harm(sr, 3.0, 220, 30, 0.5, 0.02, 9)
    ss = _fresh(P, x, sr)
    F = ss.track_ids.shape[0]
    st0, end0, f0 = list(ss.st), list(ss.end), np.array(ss.partial[3].f, copy=True)
    vib = rc.vibrato(F, 512, sr, semis=2.0)
    kw = dict(scalar=dict(fscale=1.5), curve=dict(fscale=vib), formant=dict(fscale=1.5, formant_shift=1.0),
              **{"formant curve": dict(fscale=vib, formant_shift=vib[::-1])})[mode]
    kw["phase_preserve"] = False
    ident = np.arange(F, dtype=np.float64)
    plain = np.array(ss.synth(sr, 512, **kw))
    assert np.array_equal(np.array(ss.synth(sr, 512, time_map=ident, **kw)), plain)
    assert np.array_equal(np.array(ss.synth(sr, 512, hostbuf={}, chunks=4, time_map=ident, **kw)), plain)
    assert np.array_equal(np.array(_fresh(P, x, sr).synth(sr, 512, time_map=ident, **kw)), plain)
    assert np.array_equal(np.array(_fresh(P, x, sr).synth(sr, 512, hostbuf={}, chunks=4, time_map=ident, **kw)), plain)
    w = ss.synth(sr, 512, time_map=torch.from_numpy(ident), to_host=False, **kw)
    assert torch.is_tensor(w) and w.is_cuda and np.array_equal(w.cpu().numpy(), plain)
    tau = tmo.speed_map(np.full(2 * F, 0.6), F)                     # a real stretch: staged == streamed
    kw2 = dict(kw)
    for k in ("fscale", "formant_shift"):
        if np.ndim(kw2.get(k)) > 0:
            kw2[k] = rc.vibrato(len(tau), 512, sr, semis=2.0)
    a = np.array(ss.synth(sr, 512, time_map=tau, **kw2))
    assert np.array_equal(np.array(ss.synth(sr, 512, hostbuf={}, chunks=4, time_map=tau, **kw2)), a)
    assert len(a) > 1.5 * len(plain)
    assert ss.st == st0 and ss.end == end0 and np.array_equal(ss.partial[3].f, f0)


# ------------------------------------------------------------------ behaviour, by re-analysis
SR_B, NFFT_B, HOP_B = 16000.0, 1024, 256


def _analyse(P, x):
    pv = P.PV(np.asarray(x, dtype=np.float64), SR_B, nfft=NFFT_B, hop=HOP_B, npks=8, progress=False)
    pv.run_pv()
    return pv


def _dominant(pv):
    f, m = np.asarray(pv.f), np.asarray(pv.mag)
    j = np.argmax(m, axis=1)
    return f[np.arange(len(j)), j]


def test_gpu_freeze_holds_the_frozen_frame(P):
    """A glide 300 -> 600 Hz frozen at its middle frame for 120 output blocks: the re-analysed frequency
    of the frozen stretch is the analysed frequency of that frame."""
    t = np.arange(int(2 * SR_B)) / SR_B
    x = 0.5 * np.sin(2 * np.pi * np.cumsum(300.0 * 2 ** (t / 2.0)) / SR_B)
    pv = _analyse(P, x)
    F = pv.f.shape[0]
    j0 = F // 2
    fz = pv.f[j0, np.argmax(pv.mag[j0])]
    tau = np.concatenate([np.arange(0.0, j0), np.full(120, float(j0)), np.arange(j0, F, 1.0)])
    w = pv.toSinSum().synth(SR_B, HOP_B, phase_preserve=False, time_map=tau)
    fd = _dominant(_analyse(P, w))
    held = fd[j0 + 20:j0 + 100]                                     # frames well inside the freeze
    assert np.max(np.abs(held / fz - 1.0)) < 1e-4, (fz, held.min(), held.max())
    assert abs(fd[j0 + 140] / fz - 1.0) > 0.01                     # and the glide goes on after it


def test_gpu_two_tones_switch_where_the_map_says(P):
    """440 Hz for 1 s then 660 Hz for 1 s, played at half speed up to 1.5 s of input and at double speed
    after: the tone switches at 2x its input time (one hop either way) and the output has the length of
    the map."""
    n = int(SR_B)
    x = np.concatenate([0.5 * np.sin(2 * np.pi * 440.0 * np.arange(n) / SR_B),
                        0.5 * np.sin(2 * np.pi * 660.0 * np.arange(n, 2 * n) / SR_B)])
    pv = _analyse(P, x)
    F = pv.f.shape[0]
    jcut = 1.5 * SR_B / HOP_B
    b = np.arange(4 * F)
    tau = np.where(b <= 2 * jcut, 0.5 * b, jcut + 2.0 * (b - 2 * jcut))
    tau = tau[tau <= F - 1]
    w = pv.toSinSum().synth(SR_B, HOP_B, phase_preserve=False, time_map=tau)
    assert len(w) == P.synth_geometry(len(tau) - 1, HOP_B, NFFT_B, HOP_B)[0]
    assert abs(len(w) / SR_B - 3.25) < 0.1                          # 1.5 s at half speed + 0.5 s at double
    dfr = NFFT_B / HOP_B / 2.0
    j_sw = (n - NFFT_B / 2.0) / HOP_B                               # input frame centred on the switch
    pred = 2.0 * j_sw * HOP_B + dfr * HOP_B                         # output block 2 j_sw, centred like it
    fd = _dominant(_analyse(P, w))
    late = np.nonzero(np.abs(fd - 660.0) < np.abs(fd - 440.0))[0]
    late = late[late > 10]
    det = late[0] * HOP_B + NFFT_B / 2.0
    assert abs(det - pred) <= HOP_B, (det, pred)
    assert np.all(np.abs(fd[late[0]:len(fd) - 8] - 660.0) < 5.0)


def test_gpu_map_over_rows_without_points_is_silence(P):
    """A map that reads only rows without any point renders the silence of an empty table, (-1 + 2) * hop + E
    samples, on the staged and the hostbuf paths."""
    ss = P.SinSum(SR_B, nfft=NFFT_B, hop=HOP_B)
    for fr in range(20):
        on = fr < 10
        ss.add_frame(fr, [440.0, 880.0] if on else [0.0, 0.0], [0.5, 0.25] if on else [0.0, 0.0], [0.1, 0.2])
    n = P.synth_geometry(-1, HOP_B, NFFT_B, HOP_B)[0]
    for kw in (dict(), dict(hostbuf={})):
        w = np.asarray(ss.synth(SR_B, HOP_B, phase_preserve=False, time_map=[12.0, 13.5, 19.0], **kw))
        assert w.shape == (n,) and not w.any()
    assert len(ss.synth(SR_B, HOP_B, phase_preserve=False, time_map=[0.0, 4.5, 9.0])) == (2 + 2) * HOP_B + 2 * HOP_B
