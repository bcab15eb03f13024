"""GPU: time-varying pitch shift, ``SinSum.synth(phase_preserve=False, fscale=curve)``: the numpy model
(tests/synth_curve_oracle.py) on the 60 s metric prefix, glides and vibrato checked by re-analysis,
fused / staged / streamed / clip-batch paths bit for bit, a constant curve against the scalar ratio,
``ShardedSinSum.synth_local`` with a curve, and the launch count."""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import parity_util as pu
import synth_curve_oracle as sco
from pypevoc_b200 import signals

pytestmark = pytest.mark.gpu

SR, NFFT, HOP = 44100, 2048, 512


@pytest.fixture(scope="module")
def P():
    from pypevoc_b200 import _lib, pv
    _lib.lib()
    return pv


def host_parts(ss):
    h = ss._host_tracks()
    o = h["toff"]
    return [dict(start_idx=int(h["tstart"][v]), f=h["pf"][o[v]:o[v + 1]], mag=h["pmag"][o[v]:o[v + 1]],
                 realph=h["prealph"][o[v]:o[v + 1]]) for v in range(len(h["tstart"]))]


def vibrato(F, rate=5.0, semis=1.0, hop_an=HOP, sr=SR):
    t = np.arange(F) * hop_an / sr                            # input time of each frame row
    return 2.0 ** (semis * np.sin(2 * np.pi * rate * t) / 12.0)


def glide(F, octaves=1.0):
    return 2.0 ** (octaves * (np.arange(F) / max(F - 1, 1) - 0.5))


@pytest.fixture(scope="module")
def metric_pv(P):
    """60 s prefix of the benchmark signal, nfft 2048 / hop 512 / npks 50."""
    x = signals.harm_torch(SR, 60 * SR, 220.0, 90, 0.5, 0.01, 1, torch.device("cuda"), scale=0.25)
    x = (x * float(np.float32(0.9 / float(x.abs().max())))).cpu().numpy()
    pv = P.PV(x, SR, nfft=NFFT, hop=HOP, npks=50, progress=False)
    pv.run_pv()
    return pv


def test_metric_prefix_vs_oracle(P, metric_pv):
    ss = metric_pv.toSinSum()
    F = metric_pv.nframes
    for hop, r in ((512, vibrato(F)), (200, glide(F, 0.5)), (1024, vibrato(F, 3.0, 2.0))):
        w = ss.synth(SR, hop, phase_preserve=False, fscale=r)
        ref = sco.synth(host_parts(ss), SR, hop, NFFT, HOP, r)
        assert w.shape == ref.shape
        snr = pu.snr_db(w, ref)
        print("metric prefix hop %d: SNR %.1f dB" % (hop, snr))
        assert snr > 90.0


def tone(dur=6.0, f0=220.0, nharm=5):
    t = np.arange(int(SR * dur)) / SR
    return sum(np.sin(2 * np.pi * f0 * h * t + 0.3 * h) / h for h in range(1, nharm + 1)).astype(np.float32) * 0.3


@pytest.mark.parametrize("kind,hop", [("glide", 512), ("vibrato", 512), ("glide", 1024), ("vibrato", 1024)])
def test_curve_by_reanalysis(P, kind, hop):
    """The strongest partial of each frame of the re-analysed output sits at f0 times the ratio the
    output carries between that frame's and the previous frame's window centres (the analysis measures
    the phase advance between them), within 1e-3, away from the ends.  The ratio steps once per
    synthesis block, and the 2048-sample analysis window straddles those steps, which biases its
    estimate by a fraction of a step: the vibrato (0.5 Hz, +-1 semitone) keeps the steps under 0.25 %
    also when a block is 1024 samples long."""
    f0 = 220.0
    pv = P.PV(tone(f0=f0), SR, nfft=NFFT, hop=HOP, npks=20, progress=False)
    pv.run_pv()
    F = pv.nframes
    r = glide(F) if kind == "glide" else vibrato(F, rate=0.5)
    y = pv.toSinSum().synth(SR, hop, phase_preserve=False, fscale=r)
    pa = P.PV(np.asarray(y, dtype=np.float32), SR, nfft=NFFT, hop=HOP, npks=20, progress=False)
    pa.run_pv()
    f, mag = np.asarray(pa.f), np.asarray(pa.mag)
    got = f[np.arange(len(f)), np.argmax(mag, axis=1)]
    rs = np.repeat(r, hop)                                    # ratio of every output sample
    c = np.arange(len(f)) * HOP + NFFT // 2                   # window centres
    margin = 12 * max(1, hop // HOP)
    bad, worst = [], 0.0
    for j in range(margin, len(f) - margin):
        if c[j] >= len(rs):
            break
        want = f0 * rs[c[j - 1]:c[j]].mean()
        worst = max(worst, abs(got[j] / want - 1))
        if abs(got[j] / want - 1) >= 1e-3:
            bad.append((j, got[j], want))
    print("re-analysis %s hop %d: worst relative error %.2e" % (kind, hop, worst))
    assert (len(f) - 2 * margin) > 100 and not bad, bad[:5]


@pytest.mark.parametrize("hop", [512, 200])
def test_paths_bit_identical(P, metric_pv, hop):
    F = metric_pv.nframes
    r = vibrato(F)
    kw = dict(phase_preserve=False, fscale=r)
    ss = metric_pv.toSinSum()
    fused = ss.synth(SR, hop, **kw)
    staged = ss.synth(SR, hop, **kw)
    assert np.array_equal(fused, staged)
    assert np.array_equal(ss.synth(SR, hop, hostbuf={}, chunks=8, **kw), fused)
    ss2 = metric_pv.toSinSum()
    assert np.array_equal(ss2.synth(SR, hop, hostbuf={}, chunks=8, **kw), fused)
    assert np.array_equal(ss.synth(SR, hop, phase_preserve=False, fscale=torch.from_numpy(r).cuda()), fused)
    assert not np.array_equal(ss.synth(SR, hop, phase_preserve=False, fscale=1.0), fused)


@pytest.mark.parametrize("hop", [512, 200])
def test_constant_curve_is_the_scalar(P, metric_pv, hop):
    F = metric_pv.nframes
    for c in (1.0, 1.12):
        a = metric_pv.toSinSum().synth(SR, hop, phase_preserve=False, fscale=np.full(F, c))      # fused
        ss = metric_pv.toSinSum()
        b = ss.synth(SR, hop, phase_preserve=False, fscale=c)
        assert np.array_equal(a, b), (hop, c)
        assert np.array_equal(ss.synth(SR, hop, phase_preserve=False, fscale=[c] * F), b)       # staged
        assert np.array_equal(ss.synth(SR, hop, hostbuf={}, phase_preserve=False, fscale=np.full(F, c)), b)


def test_launch_count_of_scalar_and_curve(P, metric_pv):
    from pypevoc_b200 import _lib
    L = _lib.lib()
    ss = metric_pv.toSinSum()
    ss.synth(SR, 512)
    counts = []
    for kw in (dict(), dict(phase_preserve=False, fscale=1.1), dict(phase_preserve=False, fscale=vibrato(metric_pv.nframes))):
        torch.cuda.synchronize()
        n0 = int(L.pvk_launch_count())
        ss.synth(SR, 512, **kw)
        torch.cuda.synchronize()
        counts.append(int(L.pvk_launch_count()) - n0)
    assert counts[1] == counts[2] and counts[0] < counts[1], counts


def test_clip_batch_equals_single_clips(P):
    import pypevoc_b200 as pb200
    clips = np.stack([signals.speech_like_clip(seed=1000 + i, sr=16000, dur=0.8) for i in range(5)]).astype(np.float32)
    pb = pb200.PVBatch(clips, 16000, nfft=512, hop=128, npks=20)
    pb.run_pv()
    ssb = pb.toSinSum()
    F = pb.nframes
    curves = np.stack([vibrato(F, 4.0 + i, 1.0 + 0.5 * i, 128, 16000) for i in range(5)])
    for hop in (128, 200):
        wb = ssb.synth(16000, hop, phase_preserve=False, fscale=curves)
        for i in range(5):
            pv = pb200.PV(clips[i], 16000, nfft=512, hop=128, npks=20, progress=False)
            pv.run_pv()
            w = pv.toSinSum().synth(16000, hop, phase_preserve=False, fscale=curves[i])
            assert wb[i].shape == w.shape and np.array_equal(wb[i], w), (hop, i)
    with pytest.raises(ValueError):
        ssb.synth(16000, 128, phase_preserve=False, fscale=curves[:, :-1])


def test_errors_before_launching(P, metric_pv):
    from pypevoc_b200 import _lib
    ss = metric_pv.toSinSum()
    F = metric_pv.nframes
    n0 = int(_lib.lib().pvk_launch_count())
    for bad in (np.ones(F - 1), np.ones((F, 1)), np.r_[np.ones(F - 1), np.nan], np.r_[np.ones(F - 1), 0.0]):
        with pytest.raises(ValueError):
            ss.synth(SR, 512, phase_preserve=False, fscale=bad)
    with pytest.raises(ValueError):
        ss.synth(SR, 512, phase_preserve=True, fscale=np.ones(F))
    with pytest.raises(TypeError):
        ss.synth(SR, 512, phase_preserve=False, fscale=np.ones(F, dtype=bool))
    assert int(_lib.lib().pvk_launch_count()) == n0


# ------------------------------------------------------------------ sharded
GAP_NPKS = 30


def _sharded_world1(x):
    from pypevoc_b200 import dist as D
    p = D.plan_segments(len(x), NFFT, HOP, 1)[0]
    xl = np.ascontiguousarray(x[p["sample0"]:p["sample0"] + p["nsamp"]])
    spv = D.ShardedPV(torch.from_numpy(xl).cuda(), SR, len(x), nfft=NFFT, hop=HOP, npks=GAP_NPKS, rank=0, world=1,
                      device=torch.device("cuda"))
    spv.run_pv()
    return spv.toSinSum()


@pytest.mark.parametrize("path", ["first_use", "staged", "streamed"])
def test_synth_local_world1(P, path):
    x = tone(4.0)
    pv0 = P.PV(x, SR, nfft=NFFT, hop=HOP, npks=GAP_NPKS, progress=False)
    pv0.run_pv()
    ss0 = pv0.toSinSum()
    r = vibrato(pv0.nframes)
    for hop in (HOP, 2 * HOP):
        ref = ss0.synth(SR, hop, phase_preserve=False, fscale=r)
        ss = _sharded_world1(x)
        if path == "staged":
            assert ss.ntracks == len(ss0.st)
        if path == "streamed":
            w, s0 = ss.synth_local(hop=hop, hostbuf={}, chunks=4, phase_preserve=False, fscale=r)
        else:
            w, s0 = ss.synth_local(hop=hop, to_host=True, phase_preserve=False, fscale=r)
        assert s0 == 0 and np.array_equal(np.asarray(w), ref), (path, hop)
    with pytest.raises(ValueError):
        _sharded_world1(x).synth_local(phase_preserve=False, fscale=r[:-1])


def _worker(rank, world, port, result_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    from pypevoc_b200 import dist as D
    x = tone(4.0)
    plans = D.plan_segments(len(x), NFFT, HOP, world)
    p = plans[rank]
    r = vibrato(plans[0]["frames_total"])
    xl = torch.from_numpy(np.ascontiguousarray(x[p["sample0"]:p["sample0"] + p["nsamp"]])).cuda()
    spv = D.ShardedPV(xl, SR, len(x), nfft=NFFT, hop=HOP, npks=GAP_NPKS, rank=rank, world=world,
                      device=torch.device("cuda", rank))
    spv.run_pv()
    w, s0 = spv.toSinSum().synth_local(hop=HOP, to_host=True, phase_preserve=False, fscale=r)
    np.savez(os.path.join(result_dir, "r%d.npz" % rank), w=np.asarray(w), s0=s0)
    dist.barrier()
    dist.destroy_process_group()


def test_real_ranks_over_nccl(P, tmp_path):
    import torch.multiprocessing as mp
    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs at least 2 GPUs")
    x = tone(4.0)
    pv0 = P.PV(x, SR, nfft=NFFT, hop=HOP, npks=GAP_NPKS, progress=False)
    pv0.run_pv()
    ref = pv0.toSinSum().synth(SR, HOP, phase_preserve=False, fscale=vibrato(pv0.nframes))
    mp.spawn(_worker, args=(world, 29600 + (os.getpid() % 200), str(tmp_path)), nprocs=world, join=True)
    sig = np.zeros_like(ref)
    covered = 0
    for k in range(world):
        z = np.load(os.path.join(str(tmp_path), "r%d.npz" % k))
        w, s0 = z["w"], int(z["s0"])
        sig[s0:s0 + len(w)] = w
        covered += len(w)
    assert covered == len(ref) and np.array_equal(sig, ref)
