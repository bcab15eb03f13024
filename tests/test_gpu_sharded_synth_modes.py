"""GPU: integrated-phase resynthesis of a segment-sharded signal, ``ShardedSinSum.synth_local(
phase_preserve=False, fscale=...)``.  Simulated ranks run one after another on one B200 with the
collectives replaced by their definition (the record all_gather by a concatenation, the flag
all_reduce by a maximum); ``synth_local`` itself at world 1 on every path; real NCCL ranks when the
machine has two GPUs or more.  Every result must equal the unsharded ``SinSum.synth(
phase_preserve=False, fscale=...)`` bit for bit."""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

SR, NFFT, HOP, NPKS = 44100, 2048, 512, 50
MODES = [(512, 1.0), (512, 2 ** (7 / 12.)), (1024, 1.0), (200, 0.5)]


def gap_signal():
    from pypevoc_b200 import signals
    x = signals.harm(SR, 4.0, 220, 90, 0.5, 0.02, 9)
    x[int(2.2 * SR):int(2.6 * SR)] = 0.0                      # a silent gap: partials end and restart
    return x


def metric_prefix():
    from pypevoc_b200 import signals
    x = signals.harm_torch(SR, 60 * SR, 220.0, 90, 0.5, 0.01, 1, torch.device("cuda"), scale=0.25)
    return (x * float(np.float32(0.9 / float(x.abs().max())))).cpu().numpy()


@pytest.fixture(scope="module")
def signals_():
    return {"gap": gap_signal(), "metric60": metric_prefix()}


def simulated(x, world, hop, fscale, table, ntracks, max_end):
    """Every rank's stages through the dist.py *_device helpers; returns the assembled signal."""
    from pypevoc_b200 import dist as D
    from pypevoc_b200 import pv as P
    plans = D.plan_segments(len(x), NFFT, HOP, world)
    tb = P.host_tables(SR, NFFT, HOP)
    ranks = []
    for p in plans:
        xs = torch.from_numpy(np.ascontiguousarray(x[p["sample0"]:p["sample0"] + p["nsamp"]])).cuda()
        a = P.analyze_device(xs, SR, NFFT, HOP, NPKS, 0.005, tb, frame0=p["frame0"], nframes=p["nframes"],
                             prev_zero=p["prev_zero"])
        tab = {k: a[k][0] for k in ("f", "mag", "ph", "realph")}
        tr, pk = P.track_pack_device(tab["f"], tab["mag"], tab["ph"], tab["realph"])
        F = tab["f"].shape[0]
        if pk is None:
            e = torch.zeros((0,), dtype=torch.float64, device="cuda")
            pk = dict(tstart=torch.zeros((0,), dtype=torch.int32, device="cuda"), tlen=torch.zeros((0,), dtype=torch.int32,
                      device="cuda"), toff=torch.zeros((1,), dtype=torch.int64, device="cuda"), pf=e, pmag=e, prealph=e)
        b0, b1, nout = D.render_range(p, plans, max_end, hop, NFFT, HOP)
        ws = P.resynth_workspace(F, NPKS, int(pk["tstart"].shape[0]), max(b1 - b0, 1), torch.device("cuda"))
        pws = P._phase_ws(False, pk["pf"].numel(), torch.device("cuda"))
        rec = D.handover_scan_device(tr["tid"], pk, p, plans, SR, hop, NFFT, HOP, fscale, ws, pws)
        ranks.append(dict(p=p, tab=tab, tid=tr["tid"], pk=pk, ws=ws, pws=pws, rec=rec, b=(b0, b1)))
    recs = torch.cat([r["rec"] for r in ranks])
    flags = None
    for r in ranks:
        p = r["p"]
        D.handover_apply_device(r["tid"], r["pk"], p, plans, recs, NFFT, HOP, r["ws"], r["pws"])
        o0, n = p["own0"], p["nown"]
        fl = D.nyquist_flags_device(r["tab"]["f"][o0:o0 + n], table[p["j0"]:p["j1"]], ntracks, SR, fscale)
        flags = fl if flags is None else torch.maximum(flags, fl)
    out = np.zeros(P.synth_geometry(max_end, hop, NFFT, HOP)[0])
    for r in ranks:
        p = r["p"]
        D.nyquist_import_device(r["tid"], r["pk"], p, table, flags, ntracks, r["ws"])
        w = D.resynth_local(r["tid"], r["pk"], p, plans, max_end, SR, hop, NFFT, HOP, ws=r["ws"], phase_preserve=False,
                            fscale=fscale, phase_ws=r["pws"], scanned=True).cpu().numpy()
        b0 = r["b"][0]
        out[b0 * hop:b0 * hop + len(w)] = w
    return out


@pytest.mark.parametrize("sig", ["gap", "metric60"])
@pytest.mark.parametrize("world", [2, 3, 5])
def test_simulated_ranks_equal_unsharded(signals_, sig, world):
    from pypevoc_b200 import PV
    x = signals_[sig]
    pv0 = PV(x, SR, nfft=NFFT, hop=HOP, npks=NPKS, progress=False)
    pv0.run_pv()
    ss0 = pv0.toSinSum()
    table = torch.from_numpy(np.ascontiguousarray(ss0.track_ids, dtype=np.int32)).cuda()
    ntracks, max_end = len(ss0.st), max(ss0.end)
    for hop, fscale in (MODES if sig == "gap" or world == 3 else MODES[1:2]):
        ref = ss0.synth(SR, hop, phase_preserve=False, fscale=fscale)
        w = simulated(x, world, hop, fscale, table, ntracks, max_end)
        assert w.shape == ref.shape
        assert np.array_equal(w, ref), (sig, world, hop, fscale, float(np.max(np.abs(w - ref))))


def _sharded_world1(x, **kw):
    from pypevoc_b200 import dist as D
    p = D.plan_segments(len(x), NFFT, HOP, 1)[0]
    xl = np.ascontiguousarray(x[p["sample0"]:p["sample0"] + p["nsamp"]])
    spv = D.ShardedPV(torch.from_numpy(xl).cuda(), SR, len(x), nfft=NFFT, hop=HOP, npks=NPKS, rank=0, world=1,
                      device=torch.device("cuda"))
    spv.run_pv()
    return spv.toSinSum()


@pytest.mark.parametrize("path", ["first_use", "staged", "streamed"])
def test_synth_local_world1_paths(signals_, path):
    from pypevoc_b200 import PV
    x = signals_["gap"]
    pv0 = PV(x, SR, nfft=NFFT, hop=HOP, npks=NPKS, progress=False)
    pv0.run_pv()
    ss0 = pv0.toSinSum()
    for hop, fscale in MODES:
        ref = ss0.synth(SR, hop, phase_preserve=False, fscale=fscale)
        ss = _sharded_world1(x)
        if path == "staged":
            assert ss.ntracks == len(ss0.st)                      # an accessor first
        if path == "streamed":
            w, s0 = ss.synth_local(hop=hop, hostbuf={}, chunks=4, phase_preserve=False, fscale=fscale)
        else:
            w, s0 = ss.synth_local(hop=hop, to_host=True, phase_preserve=False, fscale=fscale)
        assert s0 == 0 and np.array_equal(np.asarray(w), ref), (path, hop, fscale)


def test_phase_preserve_keyword_is_the_old_path(signals_):
    from pypevoc_b200 import _lib
    x = signals_["gap"]
    L = _lib.lib()
    res = []
    for kw in ({}, dict(phase_preserve=True), dict(phase_preserve=True, fscale=1.0)):
        ss = _sharded_world1(x)
        n0 = int(L.pvk_launch_count())
        w, _ = ss.synth_local(to_host=True, **kw)
        torch.cuda.synchronize()
        res.append((int(L.pvk_launch_count()) - n0, np.asarray(w)))
    assert res[0][0] == res[1][0] == res[2][0]
    assert np.array_equal(res[0][1], res[1][1]) and np.array_equal(res[0][1], res[2][1])


def test_synth_local_rejects_before_launching(signals_):
    from pypevoc_b200 import _lib
    ss = _sharded_world1(signals_["gap"])
    n0 = int(_lib.lib().pvk_launch_count())
    with pytest.raises(ValueError):
        ss.synth_local(phase_preserve=True, fscale=1.5)
    with pytest.raises(ValueError):
        ss.synth_local(phase_preserve=False, fscale=0.0)
    with pytest.raises(TypeError):
        ss.synth_local(phase_preserve=False, fscale="2")
    assert int(_lib.lib().pvk_launch_count()) == n0


def _worker(rank, world, port, result_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    from pypevoc_b200 import dist as D
    x = gap_signal()
    plans = D.plan_segments(len(x), NFFT, HOP, world)
    p = plans[rank]
    out = {}
    for i, (hop, fscale) in enumerate(((HOP, 2 ** (7 / 12.)), (2 * HOP, 1.0))):
        xl = torch.from_numpy(np.ascontiguousarray(x[p["sample0"]:p["sample0"] + p["nsamp"]])).cuda()
        spv = D.ShardedPV(xl, SR, len(x), nfft=NFFT, hop=HOP, npks=NPKS, rank=rank, world=world,
                          device=torch.device("cuda", rank))
        spv.run_pv()
        w, s0 = spv.toSinSum().synth_local(hop=hop, to_host=True, phase_preserve=False, fscale=fscale)
        out["w%d" % i], out["s%d" % i] = np.asarray(w), s0
    np.savez(os.path.join(result_dir, "r%d.npz" % rank), **out)
    dist.barrier()
    dist.destroy_process_group()


def test_real_ranks_over_nccl(tmp_path):
    import torch.multiprocessing as mp
    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs at least 2 GPUs")
    from pypevoc_b200 import PV
    x = gap_signal()
    pv0 = PV(x, SR, nfft=NFFT, hop=HOP, npks=NPKS, progress=False)
    pv0.run_pv()
    ss0 = pv0.toSinSum()
    port = 29400 + (os.getpid() % 200)
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    for i, (hop, fscale) in enumerate(((HOP, 2 ** (7 / 12.)), (2 * HOP, 1.0))):
        ref = ss0.synth(SR, hop, phase_preserve=False, fscale=fscale)
        sig = np.zeros_like(ref)
        covered = 0
        for r in range(world):
            z = np.load(os.path.join(str(tmp_path), "r%d.npz" % r))
            w, s0 = z["w%d" % i], int(z["s%d" % i])
            sig[s0:s0 + len(w)] = w
            covered += len(w)
        assert covered == len(ref) and np.array_equal(sig, ref), (hop, fscale)
