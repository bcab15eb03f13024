"""GPU: formant gains of the resynthesis (``synth(formant_shift=...)``, ``pvk_formant_gains``) on the
B200: the kernel against the float64 model of tests/formant_oracle.py, the render against the float64
render reference fed with the model's gained magnitudes (per sample, within the bound of
tests/test_gpu_render_contract.py), every render path against the staged call bit for bit, and real
ranks (>= 2 GPUs) against the unsharded render bit for bit."""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import formant_oracle as fo
import render_contract as rc
from golden_util import case_golden
from test_gpu_render_contract import FLOOR, GPU_CASES, TAU_GPU

pytestmark = pytest.mark.gpu

SR = rc.SR
SEMITONES7 = 2 ** (7 / 12.)


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
    return tr, pk


def device_gains(P, tr, pk, q):
    qd = P._on_device(q if np.ndim(q) == 0 else np.ascontiguousarray(q, dtype=np.float64), torch.device("cuda"))
    g = P._formant_gains(qd, tr["tid"], int(pk["tstart"].shape[0]), None, pk["tstart"], pk["toff"], pk["pf"], pk["pmag"],
                         pk["pf"].numel())
    return g[:pk["pf"].numel()].cpu().numpy()


def host_pk(pk):
    return {k: (v.cpu().numpy() if torch.is_tensor(v) else v) for k, v in pk.items()}


@pytest.mark.parametrize("K", [1, 3, 50, 400, 1024])
def test_gpu_kernel_matches_oracle_synthetic(P, K):
    F = 40
    t = rc.make_table(F, K, SR, seed=K, stationary=K > 64)
    rng = np.random.default_rng(K)
    perm = rng.permutation(K)
    for k in ("f", "mag", "ph", "realph"):
        t[k][F // 2] = t[k][F // 2, perm]                          # a row out of frequency order
    tr, pk = tracked(P, t)
    tid = tr["tid"].cpu().numpy()
    for q in (1.5, 1 / 1.3, 0.6 + 0.9 * rng.random(F)):
        got = device_gains(P, tr, pk, q)
        ref = fo.gained_packed(tid, host_pk(pk), q)
        assert np.max(np.abs(got - ref) / np.abs(ref)) <= 1e-12


@pytest.mark.parametrize("name", ["metric_1s", "real_speech", "cfg5_like"])
def test_gpu_kernel_matches_oracle_goldens(P, name):
    g = case_golden(name)
    t = dict(f=g["f"], mag=g["mag"], ph=g["ph"], realph=g["realph"])
    tr, pk = tracked(P, t)
    tid = tr["tid"].cpu().numpy()
    F = tid.shape[0]
    for q in (1.5, 1.0 / SEMITONES7, rc.vibrato(F, int(g["hop"]), 44100.0) / 1.2):
        got = device_gains(P, tr, pk, q)
        ref = fo.gained_packed(tid, host_pk(pk), q)
        assert np.max(np.abs(got - ref) / np.abs(ref)) <= 1e-12


def _modes(F, hop_an):
    vib = rc.vibrato(F, hop_an, SR)
    # (label, mode, fscale, formant_shift)
    return [("preserve formant 1.3", "preserve", 1.0, 1.3),
            ("free 1.5 formant 1", "free", 1.5, 1.0),
            ("vibrato formant curve", "free", vib, 1.0 / vib ** 0.5)]


@pytest.mark.parametrize("name", ["tile16_taylor_dE2", "tile8", "tile4_taylor", "g8_G2", "g16_700", "g8_chunked",
                                  "g8_K1024", "g16_K1024", "tile16_edge0p3"])
def test_gpu_render_with_gains_per_sample(P, name):
    case = GPU_CASES[name]
    hop, nfft, hop_an, edge, K, F, minframes, ws_blocks = case
    t = rc.make_table(F, K, SR, seed=sum(map(ord, name)), minframes=minframes, stationary=K > 64)
    tr, pk = tracked(P, t)
    tid = tr["tid"].cpu().numpy()
    br = rc.case_branch(case)
    for label, mode, r, phi in _modes(F, hop_an):
        q = P.formant_ratio(mode == "preserve", r, phi, F)
        w = P.resynth_device(tr["tid"], pk, SR, hop, nfft, hop_an, edge, minframes, phase_preserve=mode == "preserve",
                             fscale=r, formant=P._on_device(q, torch.device("cuda"))).cpu().numpy()
        gm = fo.gained_table(tid, t["f"], t["mag"], q)
        parts = rc.parts_from_tid(tid, t["f"], gm, t["ph"], t["realph"])
        ref = rc.reference(parts, SR, hop, nfft, hop_an, edge, minframes, mode, r)
        scale = rc.amp_scale(parts, SR, hop, nfft, hop_an, edge, minframes, None if mode == "preserve" else r)
        worst = rc.check_render(w, ref, scale, TAU_GPU, FLOOR, "%s %s" % (name, label), hop, br)
        print("%-44s worst %.2e  %s" % ("%s %s" % (name, label), worst, rc.branch_label(br)))


@pytest.fixture(scope="module")
def metric_pv(P):
    """60 s prefix of the benchmark signal, nfft 2048 / hop 512 / npks 50."""
    from pypevoc_b200 import signals
    sr = 44100
    x = signals.harm_torch(sr, 60 * sr, 220.0, 90, 0.5, 0.01, 1, torch.device("cuda"), scale=0.25)
    x = (x * float(np.float32(0.9 / float(x.abs().max())))).cpu().numpy()
    pv = P.PV(x, sr, nfft=2048, hop=512, npks=50, progress=False)
    pv.run_pv()
    return pv


def test_gpu_metric_prefix_with_gains_per_sample(P, metric_pv):
    sr, nfft, hop_an, hop = 44100, 2048, 512, 512
    ss = metric_pv.toSinSum()
    h = ss._host_tracks()
    tid = ss.track_ids
    q = P.formant_ratio(False, 1.25, 1.0)
    gmag = fo.gained_packed(tid, h, q)
    o = h["toff"]
    parts = [dict(start_idx=int(h["tstart"][v]), f=h["pf"][o[v]:o[v + 1]], mag=gmag[o[v]:o[v + 1]],
                  realph=h["prealph"][o[v]:o[v + 1]]) for v in range(len(h["tstart"]))]
    w = ss.synth(sr, hop, phase_preserve=False, fscale=1.25, formant_shift=1.0)
    br = rc.render_branch(hop, 50, nfft, hop_an, 1.0)
    ref = rc.reference(parts, sr, hop, nfft, hop_an, 1.0, 3, "free", 1.25)
    scale = rc.amp_scale(parts, sr, hop, nfft, hop_an, 1.0, 3, 1.25)
    worst = rc.check_render(np.asarray(w), ref, scale, TAU_GPU, FLOOR, "metric 60 s formant", hop, br)
    print("metric 60 s formant worst %.2e" % worst)
    assert np.array_equal(ss.partial[3].mag, h["pmag"][o[3]:o[4]])          # the analysed values stay


def _fresh(P, x, sr):
    pv = P.PV(x, sr, nfft=2048, hop=512, npks=50, progress=False)
    pv.run_pv()
    return pv.toSinSum()


@pytest.mark.parametrize("mode", ["preserve formant 1.3", "free 1.5 formant 1", "vibrato formant curve"])
def test_gpu_render_paths_agree_bit_for_bit(P, mode):
    """Fused first use, staged, hostbuf streamed fused and hostbuf streamed give the same bits; the
    analysed magnitudes stay as they were; formant_shift = fscale (and 1 at phase_preserve) is None."""
    from pypevoc_b200 import signals
    sr = 44100
    x = signals.harm(sr, 3.0, 220, 30, 0.5, 0.02, 9)
    ss = _fresh(P, x, sr)
    F = ss.track_ids.shape[0]
    pmag0 = ss.device_tracks["pmag"].clone()                      # the analysed values, before any formant render
    mag0 = np.array(ss.partial[3].mag, copy=True)
    label, m, r, phi = [c for c in _modes(F, 512) if c[0] == mode][0]
    kw = dict(phase_preserve=m == "preserve", fscale=r, formant_shift=phi)
    fused = np.array(_fresh(P, x, sr).synth(sr, 512, **kw))
    streamed_fused = np.array(_fresh(P, x, sr).synth(sr, 512, hostbuf={}, chunks=4, **kw))
    staged = np.array(ss.synth(sr, 512, **kw))
    streamed = np.array(ss.synth(sr, 512, hostbuf={}, chunks=4, **kw))
    assert np.array_equal(fused, staged) and np.array_equal(streamed_fused, staged)
    assert np.array_equal(streamed, staged)
    plain = dict(kw, formant_shift=None)
    assert not np.array_equal(staged, np.array(ss.synth(sr, 512, **plain)))
    same = dict(kw, formant_shift=r)
    assert np.array_equal(np.array(ss.synth(sr, 512, **same)), np.array(ss.synth(sr, 512, **plain)))
    assert torch.equal(ss.device_tracks["pmag"], pmag0)
    assert np.array_equal(ss.partial[3].mag, mag0)


def test_gpu_batch_equals_clips(P):
    from pypevoc_b200 import PVBatch, signals
    sr = 16000
    xs = np.stack([signals.harm(sr, 1.0, 150 + 40 * c, 12, 0.5, 0.02, 9) for c in range(3)]).astype(np.float32)
    pb = PVBatch(xs, sr, nfft=1024, hop=256, npks=20)
    pb.run_pv()
    sb = pb.toSinSum()
    F = pb.nframes
    r = np.stack([rc.vibrato(F, 256, sr, rate=3.0 + c) for c in range(3)])
    phi = np.stack([np.linspace(0.8, 1.3, F) for _ in range(3)])
    ws = sb.synth(sr, 256, phase_preserve=False, fscale=r, formant_shift=phi)
    for c in range(3):
        one = pb[c].toSinSum().synth(sr, 256, phase_preserve=False, fscale=r[c], formant_shift=phi[c])
        assert np.array_equal(ws[c], one), c
    w1 = sb.synth(sr, 256, formant_shift=1.2)
    for c in range(3):
        assert np.array_equal(w1[c], pb[c].toSinSum().synth(sr, 256, formant_shift=1.2)), c
    with pytest.raises(ValueError):
        sb.synth(sr, 256, formant_shift=np.ones(F))


def _worker(rank, world, port, result_dir):
    import torch.distributed as dist
    from pypevoc_b200 import dist as D, signals
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    sr, nfft, hop, npks = 44100, 2048, 512, 50
    x = signals.harm(sr, 6.0, 220, 90, 0.5, 0.02, 9)
    plans = D.plan_segments(len(x), nfft, hop, world)
    p = plans[rank]
    F = plans[0]["frames_total"]
    xl = torch.from_numpy(np.ascontiguousarray(x[p["sample0"]:p["sample0"] + p["nsamp"]]))
    out = {}
    for i, (m, r, phi) in enumerate(_multi_modes(F)):
        kw = dict(to_host=True, phase_preserve=m == "preserve", fscale=r, formant_shift=phi)
        for hb in (None, {}):
            spv = D.ShardedPV(xl.cuda(), sr, len(x), nfft=nfft, hop=hop, npks=npks, rank=rank, world=world,
                              device=torch.device("cuda", rank))
            spv.run_pv()
            ss = spv.toSinSum()
            # first call on fresh partials (fused first use with phase_preserve and no hostbuf), then a second
            # call on the same ShardedSinSum (the staged path)
            for name in ("first", "again"):
                w, s0 = ss.synth_local(hostbuf=hb, **kw)
                key = "%d_%s_%s" % (i, "host" if hb is None else "hostbuf", name)
                out["w" + key] = np.array(w)
                out["s" + key] = s0
    np.savez(os.path.join(result_dir, "r%d.npz" % rank), **out)
    dist.barrier()
    dist.destroy_process_group()


def _multi_modes(F):
    vib = rc.vibrato(F, 512, 44100)
    return [("preserve", 1.0, 1.3), ("free", SEMITONES7, 1.0), ("free", vib, 1.0 / vib)]


def test_gpu_sharded_ranks_equal_unsharded(P, tmp_path):
    import torch.multiprocessing as mp
    from pypevoc_b200 import signals
    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs at least 2 GPUs")
    sr = 44100
    x = signals.harm(sr, 6.0, 220, 90, 0.5, 0.02, 9)
    ss = _fresh(P, x, sr)
    F = ss.track_ids.shape[0]
    port = 29600 + (os.getpid() % 200)
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    zs = [np.load(os.path.join(str(tmp_path), "r%d.npz" % r)) for r in range(world)]
    for i, (m, r, phi) in enumerate(_multi_modes(F)):
        ref = np.array(ss.synth(sr, 512, phase_preserve=m == "preserve", fscale=r, formant_shift=phi))
        for path in ("host_first", "host_again", "hostbuf_first", "hostbuf_again"):
            key = "%d_%s" % (i, path)
            sig = np.zeros_like(ref)
            for z in zs:
                w, s0 = z["w" + key], int(z["s" + key])
                sig[s0:s0 + len(w)] = w
            assert np.array_equal(sig, ref), key
