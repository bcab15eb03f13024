#!/usr/bin/env python
"""bench.py -- phase-vocoder hot path on B200: STFT frames/s + resynthesis partial-samples/s.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR     (+ the last timed step's outputs)

Workload (BASELINE.json): the 10-minute mono 44.1 kHz synthetic harmonic tone + noise of
configs[1], analysed with the parameters the metric is quoted on (nfft=2048, hop=512,
npks=50), followed by tracking and full resynthesis.  One "step" = one pass of the whole hot
path (PV.run_pv -> toSinSum -> SinSum.synth) over that signal.

  value      frames / step time with the signal already resident in HBM (kernel path)
  e2e        same metric through the public API with HOST buffers: pinned host signal -> H2D
             -> PV.run_pv -> toSinSum -> synth -> D2H of the peak tables and the signal
  roofline   the step's dominant kernel against the measured HBM copy peak
  cpu_baseline  the unmodified reference (baseline/_ref; the numpy oracle port where it is absent) on
             one host core, on a bounded prefix of the same samples
N > 1 is weak scaling: every rank owns its own hop-aligned 10-minute segment of an N x 10
minute signal (plus a few halo frames either side), analyses, links and resynthesises it from
local data with one 24-byte read-back at the end of the step; a 2K+4-integer all_gather makes the
partial numbering global and ONE gather collects the int32 track table on a high-priority side
stream (NVSwitch multicast stores of the rename kernel up to 4 ranks, NCCL beyond -- dist.py).
Before any N > 1 measurement a short sharded run is compared bit for bit with the unsharded one
(exit status 3 on a mismatch).  `--workload cfg4 / cfg3`: the 8-hour signal (strong scaling) and the
4096-clip batch of BASELINE.json as auxiliary lines.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# signal: SURVEY 8d "metric" recipe (f0 = 220 Hz so that harmonics are > 5 bins apart at
# nfft 2048 and survive the salience filter: ~40 peaks per frame), 10 minutes long
CFG = dict(sr=44100, seconds=600, nfft=2048, hop=512, npks=50, pkthresh=0.005,
           f0=220.0, nharm=90, p=0.5, sigma=0.01, seed=1)
# other BASELINE.json configs (`--workload`; auxiliary lines for profiles/, the driver runs the default):
#   cfg4  configs[3]: ONE 8-hour signal, nfft 2048 / hop 256 / npks 100, segment-sharded: STRONG scaling
#   cfg3  configs[2]: 4096 speech-like 3 s clips @ 16 kHz, nfft 512 / hop 128 / npks 20, split by clip: STRONG scaling
CFG4 = dict(sr=44100, seconds=8 * 3600, nfft=2048, hop=256, npks=100, pkthresh=0.005,
            f0=200.0, nharm=100, p=0.4, sigma=0.01, seed=4000)
CFG3 = dict(sr=16000, seconds=3, nclips=4096, nfft=512, hop=128, npks=20, pkthresh=0.005)
E2E_TABLES = ("f", "mag", "ph", "totalmag")      # what the end-to-end step downloads (the arrays north_star names)
DUMP_BYTES = 60 << 20                            # --dump-outputs: data bytes of all files, under 64 MB with headers
METRIC = "STFT frames/sec (nfft=2048,hop=512,npks=50) + resynth partial-samples/sec"
WORKLOAD = ("10 min mono 44.1 kHz synthetic harmonic tone+noise (configs[1] length; 220 Hz, 90 harmonics, "
            "sigma 0.01), metric parameters nfft=2048 hop=512 npks=50, analysis + tracking + full resynthesis")


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return json.load(fh), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------- clocks
class ClockSampler(object):
    """SM clock and throttle reasons sampled DURING the timed region: an NVML polling thread
    (2 ms period -- the timed region lasts tens of milliseconds, too short for `nvidia-smi -lms`),
    with `nvidia-smi` as the fallback when NVML is not importable."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.thread = None
        self.samples = []
        self.period = float(os.environ.get("PVK_CLOCK_PERIOD_MS", "2")) * 1e-3
        self.path = "/tmp/pvk_clocks_%d_%d.csv" % (os.getpid(), index)
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll(self):
        n = self.nvml
        bits = (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40),
                ("sw_power_cap", 0x4))
        while not self._stop:
            try:
                clk = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                try:
                    r = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                except Exception:
                    r = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.samples.append((clk, tuple(name for name, b in bits if r & b)))
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self.nvml is not None:
            import threading
            self._stop = False
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=self.fh, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.thread is not None:
            self._stop = True
            self.thread.join(timeout=1.0)
            if self.samples:
                sm = [c for c, _ in self.samples]
                hi = [v for v in sm if v >= 0.5 * max(sm)]
                reasons = sorted({r for _, rs in self.samples for r in rs})
                out = {"sm_mhz": float(np.median(hi)), "sm_max_mhz": self.smax, "reasons": reasons,
                       "samples": len(sm), "source": "nvml, 2 ms polling during the timed steps"}
            return out
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
            self.fh.close()
            sm, smax, reasons = [], [], set()
            for line in open(self.path):
                p = [s.strip() for s in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1])); smax.append(float(p[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            if sm:
                hi = [v for v in sm if v >= 0.5 * max(sm)]
                out = {"sm_mhz": float(np.median(hi)), "sm_max_mhz": float(max(smax)),
                       "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 20"}
            os.unlink(self.path)
        except Exception:
            pass
        return out


# --------------------------------------------------------------------------- sharded parity self-check
def sharded_selfcheck(rank, world, dev):
    """N > 1 only, before the warm-up: a 6 s signal with a silent gap and a silent tail goes through
    the sharded path (ShardedPV over NCCL / peer memory, exactly the calls the timed step makes) and
    through the unsharded single-GPU path; every rank compares its own analysis rows, the gathered
    track table, the spans and its rendered block range BIT FOR BIT.  Any mismatch on any rank makes
    every rank exit with status 3, so a green N-GPU bench line carries multi-GPU parity."""
    import torch
    import torch.distributed as dist
    from pypevoc_b200 import PV, signals
    from pypevoc_b200 import dist as D
    sr, nfft, hop, npks = 44100, 2048, 512, 50
    x = signals.harm(sr, 6.0, 220, 90, 0.5, 0.02, 9)
    x[int(2.2 * sr):int(2.6 * sr)] = 0.0
    x[int(5.3 * sr):] = 0.0
    pv0 = PV(x, sr, nfft=nfft, hop=hop, npks=npks, progress=False, device=dev)
    pv0.run_pv()
    ss0 = pv0.toSinSum()
    w0 = ss0.synth(sr, hop)
    tid0 = ss0.track_ids
    plans = D.plan_segments(len(x), nfft, hop, world)
    p = plans[rank]
    xl = torch.from_numpy(np.ascontiguousarray(x[p["sample0"]:p["sample0"] + p["nsamp"]]))
    bad = []
    peer = mcast = None
    for rep in range(3):                               # both alternating peer tables + one reuse
        spv = D.ShardedPV(xl.to(dev), sr, len(x), nfft=nfft, hop=hop, npks=npks, rank=rank, world=world, device=dev)
        spv.run_pv()
        ss = spv.toSinSum()
        w, s0 = ss.synth_local(to_host=True)
        peer = bool(ss._h.peer_used)
        mcast = bool(getattr(ss._h, "multicast_used", False))
        for k in ("f", "mag", "ph", "realph", "binno"):
            if not np.array_equal(np.asarray(getattr(spv.pv, k))[spv.own_rows], getattr(pv0, k)[p["j0"]:p["j1"]]):
                bad.append("rep %d: own rows of %s" % (rep, k))
        if not np.array_equal(ss.track_ids, tid0):
            bad.append("rep %d: gathered track table" % rep)
        if ss.st != ss0.st or ss.end != ss0.end or ss.ntracks != len(ss0.st) or ss.max_end != max(ss0.end):
            bad.append("rep %d: spans / counts" % rep)
        if not np.array_equal(np.asarray(w), w0[s0:s0 + len(w)]):
            bad.append("rep %d: rendered block range [%d, %d)" % (rep, s0, s0 + len(w)))
    cover = torch.tensor([len(w), len(bad)], dtype=torch.int64, device=dev)
    dist.all_reduce(cover)
    if int(cover[0].item()) != len(w0):
        bad.append("block ranges cover %d of %d samples" % (int(cover[0].item()), len(w0)))
    if bad or int(cover[1].item()):
        sys.stderr.write("rank %d: SHARDED PARITY FAILED: %s\n" % (rank, "; ".join(bad) or "(another rank)"))
        sys.stderr.flush()
        dist.barrier()
        os._exit(3)
    return {"sharded_vs_unsharded": "bit-exact (own rows f/mag/ph/realph/binno, gathered track table, st/end, "
                                    "rendered block ranges; 3 passes)", "frames": int(pv0.nframes),
            "partials": len(ss0.st), "ranks": world, "peer_memory_gather": peer, "nvswitch_multicast": mcast}


# --------------------------------------------------------------------------- clip batch (configs[2])
def clips_main(args, world, rank, dev, real_stdout):
    """--workload cfg3: 4096 speech-like clips split by clip over the ranks (dist.clip_range; no halo,
    no collective): PVBatch.run_pv -> toSinSum (ONE link + pack over the flattened table) ->
    synth_device (ONE resynthesis launch), device resident.  Strong scaling."""
    import torch
    import torch.distributed as dist
    from pypevoc_b200 import PVBatch, signals
    from pypevoc_b200 import pv as P
    from pypevoc_b200 import dist as D
    from pypevoc_b200 import _lib
    c = dict(CFG3, nclips=args.cfg3_clips)
    sr, nfft, hop, npks = c["sr"], c["nfft"], c["hop"], c["npks"]
    c0, c1 = D.clip_range(c["nclips"], rank, world)
    # 64 distinct clips tiled to the batch size (numpy generation of 4096 distinct clips takes minutes;
    # throughput does not depend on it); clip i of the batch = base[i % 64]
    base = np.stack([signals.speech_like_clip(1000 + i, sr=sr, dur=float(c["seconds"])) for i in range(64)])
    xd = torch.from_numpy(base).to(dev)[torch.arange(c0, c1, device=dev) % 64].contiguous()
    pb = PVBatch(xd, sr, nfft=nfft, hop=hop, npks=npks, pkthresh=c["pkthresh"], device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    state = {}

    def step(timed):
        e = [ev() for _ in range(4)]
        state.clear()
        e[0].record()
        pb.run_pv()
        e[1].record()
        ssb = pb.toSinSum()
        ssb.ss._ensure_packed()                          # link + pack of all clips; one 24-byte read-back
        e[2].record()
        w = ssb.synth_device(sr, hop)
        e[3].record()
        state.update(ssb=ssb, w=w)
        timed.append(e)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
    import gc
    count = _lib.lib().pvk_launch_count
    sampler = ClockSampler(dev.index)
    sampler.start()
    t_wait = time.perf_counter()
    while sampler.thread is not None and len(sampler.samples) < 5 and time.perf_counter() - t_wait < 2.0:
        time.sleep(0.005)
    gc.collect()
    gc.disable()
    settle = max(0, 5 - args.warmup)
    nwarm = settle + args.warmup
    timed, warm, launches0 = [], [], 0
    for i in range(nwarm + args.steps):
        if i == nwarm:
            barrier()
            del sampler.samples[:]
            launches0 = int(count())
        torch.cuda.synchronize()
        flush.fill_(1)
        step(timed if i >= nwarm else warm)
    barrier()
    launches = int(count()) - launches0
    clocks = sampler.stop()
    gc.enable()
    st = np.array([[e[i].elapsed_time(e[i + 1]) for i in range(3)] for e in timed])
    sys.stderr.write("rank %d per-step stage ms [analysis, tracking+pack, resynth]:\n%s\n" % (rank, np.round(st, 3)))
    ssb = state["ssb"]
    tl = ssb.ss._ensure_packed()["tlen"].cpu().numpy().astype(np.int64)
    _, E = P.synth_geometry(0, hop, nfft, hop)
    F = pb.nframes
    t = torch.tensor([float(st.sum(axis=1).mean())] + st.mean(axis=0).tolist() +
                     [float((c1 - c0) * F), float((tl[tl >= 3] * hop + 2 * E).sum()), float(len(tl))],
                     device=dev, dtype=torch.float64)
    if world > 1:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        t[:4] = tmax[:4]
    ms_step, ms_an, ms_trk, ms_syn, frames_total, psamp_total, tracks_total = [float(v) for v in t.tolist()]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk_, how = peaks()
    hbm = float(pk_["hbm_gbs"])
    alg_an = (4 * hop + 20 * npks + 8) * (c1 - c0) * F
    line = {
        "metric": "STFT frames/sec (nfft=512,hop=128,npks=20, clip batch) + resynth partial-samples/sec",
        "value": frames_total / (ms_step * 1e-3), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32 FFT, f64 per-peak/phase", "data": "synthetic",
        "config": {"workload": "%d synthetic speech-like %d s clips @ %d Hz (configs[2]; 64 distinct clips tiled), nfft=%d "
                               "hop=%d npks=%d, clip-batched analysis + tracking + full resynthesis"
                               % (c["nclips"], c["seconds"], sr, nfft, hop, npks),
                   "sr": sr, "nclips": c["nclips"], "clips_per_gpu": c1 - c0, "frames_per_clip": F, "nfft": nfft, "hop": hop,
                   "npks": npks, "frames_total": frames_total, "partial_samples_total": psamp_total,
                   "tracks_total": tracks_total, "guard_rows_per_clip": pb.guard,
                   "l2": "256 MiB buffer written between timed steps; per-step CUDA events on the launch stream",
                   "settle_passes_before_warmup": settle,
                   "parallelism": "clips split x%d (dist.clip_range; independent units, no halo, no collective)" % world},
        "stages": {"analysis_ms": ms_an, "tracking_pack_ms": ms_trk, "resynth_ms": ms_syn,
                   "analysis_frames_per_s": frames_total / (ms_an * 1e-3),
                   "resynth_partial_samples_per_s": psamp_total / (ms_syn * 1e-3)},
        "roofline": {"kernel": "analyze_kernel<8>", "bound": "hbm", "achieved": alg_an / (ms_an * 1e-3) / 1e9, "peak": hbm,
                     "unit": "GB/s", "frac": alg_an / (ms_an * 1e-3) / 1e9 / hbm, "traffic": None, "ms": ms_an,
                     "alg_bytes_per_launch": alg_an, "peak_source": how},
        "clocks": clocks, "gpu_launches": launches, "e2e": None,
    }
    sys.stdout.flush()
    os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------- GPU arm
def gpu_main(args):
    # everything else that writes to fd 1 (NCCL's version banner, library chatter) goes to stderr:
    # the contract is ONE JSON line on stdout
    real_stdout = os.dup(1)
    sys.stdout.flush()
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    from pypevoc_b200 import PV, signals
    from pypevoc_b200 import pv as P
    from pypevoc_b200 import dist as D

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if args.workload == "cfg3":
        return clips_main(args, world, rank, dev, real_stdout)
    strong = args.workload == "cfg4"
    c = dict(CFG4, seconds=int(round(args.cfg4_hours * 3600))) if strong else CFG
    sr, nfft, hop, npks = c["sr"], c["nfft"], c["hop"], c["npks"]
    nsamp_seg = sr * c["seconds"]
    nsamp_total = nsamp_seg if strong else world * nsamp_seg

    # ---- synthetic signal: rank r owns frames [r*Fseg, (r+1)*Fseg) of an N*10-minute signal and
    #      analyses a window with a few halo rows either side (pypevoc_b200/dist.py)
    plans = D.plan_segments(nsamp_total, nfft, hop, world)
    plan = plans[rank]
    xd = signals.harm_torch(sr, plan["nsamp"], c["f0"], c["nharm"], c["p"], c["sigma"], c["seed"], dev,
                            t0_samples=plan["sample0"], scale=0.25)
    # SURVEY 8d: peak 0.9 (the max over the whole N x 10-minute signal; one fp32 factor on every rank, so
    # the overlapping windows of neighbouring ranks stay bit-identical)
    peak = xd.abs().max().to(torch.float64)
    if world > 1:
        dist.all_reduce(peak, op=dist.ReduceOp.MAX)
    xd.mul_(float(np.float32(0.9 / float(peak.item()))))
    tb = P.host_tables(sr, nfft, hop)
    selfcheck = sharded_selfcheck(rank, world, dev) if world > 1 else None
    F = plan["nown"]                                 # own frames (halo rows are not counted)
    frames_total = plan["frames_total"]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    trace = bool(os.environ.get("PVK_BENCH_TRACE"))
    state = {}

    def step(timed=None):
        """One pass of the hot path over this rank's segment (device resident)."""
        e = [ev() for _ in range(5)] if timed is not None else None
        state.clear()                                     # (the previous step's tensors go back to the allocator)
        ht = [time.perf_counter()] if trace else None     # PVK_BENCH_TRACE=1: host-side launch timeline
        if e: e[0].record()
        a = P.analyze_device(xd, sr, nfft, hop, npks, c["pkthresh"], tb, frame0=plan["frame0"],
                             nframes=plan["nframes"], prev_zero=plan["prev_zero"])
        if e: e[1].record()
        if ht: ht.append(time.perf_counter())
        tab = {k: a[k][0] for k in ("f", "mag", "ph", "realph")}
        box = []

        def after_link(tr):
            # global numbering (2K+4-int all_gather) and THE all_gather of the track table go to a
            # side stream, queued behind the link kernels while those still run (their host-side
            # launch cost hides behind analysis + linking); packing and resynthesis below use LOCAL
            # ids and overlap them
            if ht: ht.append(time.perf_counter())
            if world > 1:
                box.append(D.StitchHandle(tr["tid"], plan, plans))
            if ht: ht.append(time.perf_counter())
            if e: e[2].record()
        if world == 1:
            # link, id resolution, pack and resynthesis are queued back to back (pack and resynthesis sized
            # by upper bounds, the real counts are read on the device); the step's one host read-back
            # (24 bytes: partials, points, last frame) comes at the very end
            tr, pk, w = P.track_pack_resynth_device(tab["f"], tab["mag"], tab["ph"], tab["realph"], sr, hop, nfft, hop,
                                                    after_link=after_link,
                                                    after_pack=(lambda tr_: e[3].record()) if e else None)
            if e: e[4].record()
            state.update(a=a, tr=tr, pk=pk, w=w, st=dict(ntracks=tr["ntracks"], max_end=tr["max_end"]), table=tr["tid"],
                         spans=(pk["tstart"], pk["tlen"]), peer=None)
            if timed is not None:
                timed.append(e)
            return
        # N > 1: the same back half on this rank's window (dist.track_pack_resynth_local): link -> [numbering +
        # gather of the track table on a side stream] -> pack -> rendering of the rank's own block range, all
        # queued back to back; one 24-byte read-back at the end, then the 8 integers of the numbering pass
        def after_pack(tr_):
            if e: e[3].record()
            box[0].join_before_render()                  # (only with PVK_GATHER_JOIN=pack; default: joined at the end)
        glob = {}

        def before_sync(tr_):
            # queued behind the rendering, before the host waits for anything on the main stream: the 8
            # integers of the numbering pass (the side stream finished long ago), the join of the gathered
            # table and the spans pass over it
            glob["ntg"], glob["max_end"] = box[0].counts()
            with torch.cuda.stream(box[0].side):         # the spans pass over the N x longer table runs beside the
                glob["spans"] = P.spans_device(box[0].table_on_side(), glob["ntg"])   # rendering, not after it
            glob["table"] = box[0].table()               # (joins the side stream into the main one)
        tr, pk, w, b0 = D.track_pack_resynth_local(tab, plan, plans, sr, hop, nfft, hop, after_link=after_link,
                                                   after_pack=after_pack, before_sync=before_sync)
        sh = box[0]
        ntg, max_end, table, spans = glob["ntg"], glob["max_end"], glob["table"], glob["spans"]
        st = dict(ntracks=ntg, max_end=max_end)
        w = w[:D.trim_local(w.numel(), b0, plan, plans, max_end, hop, nfft, hop)[0]]
        if e: e[4].record()
        if ht:
            ht.append(time.perf_counter())
            torch.cuda.synchronize()
            ht.append(time.perf_counter())
            sys.stderr.write("trace rank %d: host ms since step start [analysis launched, track launched, stitch "
                             "launched, counts read, pack launched, resynth launched, global counts read, all "
                             "launched, gpu idle] = %s\n" % (rank, ["%.3f" % (1e3 * (v - ht[0])) for v in ht[1:]]))
        state.update(a=a, tr=tr, pk=pk, w=w, st=st, table=table, spans=spans, peer=bool(sh.peer_used) if sh else None)
        if timed is not None:
            timed.append(e)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    import gc
    from pypevoc_b200 import _lib
    count = _lib.lib().pvk_launch_count
    sampler = ClockSampler(local)
    sampler.start()                                      # NVML's first queries are slow: wait them out here
    t_wait = time.perf_counter()
    while sampler.thread is not None and len(sampler.samples) < 5 and time.perf_counter() - t_wait < 2.0:
        time.sleep(0.005)
    gc.collect()
    gc.disable()                                         # no collector pauses inside the timed steps
    # --warmup W is honoured exactly: W warm-up steps directly before the K timed ones.  The caching
    # allocator / driver / NCCL channels settle within ~5 passes, so `settle` extra untimed passes
    # (reported in config) run BEFORE the counted warm-up when W is small.
    settle = max(0, 8 - args.warmup)
    nwarm = settle + args.warmup
    timed, warm, launches0 = [], [], 0                   # (warm-up events stay alive until the end)
    # one loop, one step form: settle + warm-up steps are passes of exactly the timed code (events, L2
    # flush, idle device at the start), so nothing but the barrier separates them from the K timed steps
    for i in range(nwarm + args.steps):
        if i == nwarm:
            barrier()
            del sampler.samples[:]                       # clocks are sampled DURING the timed steps only
            launches0 = int(count())
        torch.cuda.synchronize()                         # every step starts from an idle device
        flush.fill_(1)                                   # L2 flush between timed iterations
        step(timed if i >= nwarm else warm)
    barrier()
    launches = int(_lib.lib().pvk_launch_count()) - launches0     # libpvk kernels launched by the timed steps
    clocks = sampler.stop()
    gc.enable()
    if args.dump_outputs:
        own = slice(plan["own0"], plan["own0"] + plan["nown"]) if world > 1 else slice(None)
        outs = {k: state["a"][k][0][own] for k in ("f", "mag", "ph", "realph", "binno", "totalmag")}
        outs["track_ids"] = state["table"][plan["j0"]:plan["j1"]] if world > 1 else state["table"]
        outs["partial_start"], outs["partial_length"] = state["spans"]
        outs["synth"] = state["w"]
        dump_outputs(args.dump_outputs, outs, DUMP_BYTES // world, "_rank%d" % rank if world > 1 else "")
    st = np.array([[e[i].elapsed_time(e[i + 1]) for i in range(4)] for e in timed])   # ms per stage
    ms_step_local = float(st.sum(axis=1).mean())
    sys.stderr.write("rank %d per-step stage ms [analysis, tracking, pack, resynth]:\n%s\n" % (rank, np.round(st, 3)))
    t = torch.tensor([ms_step_local] + st.mean(axis=0).tolist(), device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step, ms_an, ms_trk, ms_pack, ms_syn = [float(v) for v in t.tolist()]

    tl = state["spans"][1].cpu().numpy().astype(np.int64)         # global table (every rank has it)
    _, E = P.synth_geometry(state["st"]["max_end"], hop, nfft, hop)
    psamp_total = float((tl[tl >= 3] * hop + 2 * E).sum())
    psamp_local = psamp_total / world

    # ---- end to end through the public API with host buffers (pinned), per rank
    e2e = None
    if not args.no_e2e and not strong:
        xh = torch.empty(plan["nsamp"], dtype=torch.float32).pin_memory()
        xh.copy_(xd)
        hostbuf = {}
        times = []

        def e2e_step():
            t0 = time.perf_counter()
            if world == 1:
                pv = PV(xh, sr, nfft=nfft, hop=hop, npks=npks, pkthresh=c["pkthresh"], progress=False, device=dev)
                pv.run_pv(hostbuf=hostbuf, stream_tables=E2E_TABLES)   # upload, analysis and table download overlap
                ss = pv.toSinSum()
                w = ss.synth(sr, hop, hostbuf=hostbuf)     # rendering and signal download overlap
                assert pv.f.shape == (pv.nframes, npks) and w.dtype == np.float64   # host views (synchronises)
                nb = pv.d2h_bytes + ss.d2h_bytes
            else:
                spv = D.ShardedPV(xh, sr, nsamp_total, nfft=nfft, hop=hop, npks=npks, pkthresh=c["pkthresh"],
                                  rank=rank, world=world, device=dev)
                spv.run_pv(hostbuf=hostbuf, stream_tables=E2E_TABLES)
                ss = spv.toSinSum()
                w, _ = ss.synth_local(hostbuf=hostbuf)
                tids = ss.device_track_table                 # the gathered track table (stays on the device)
                assert spv.pv.f.shape[1] == npks and w.dtype == np.float64 and tids.shape[0] == frames_total
                nb = spv.pv.d2h_bytes + ss.d2h_bytes
            torch.cuda.synchronize()
            return time.perf_counter() - t0, nb
        for _ in range(4):
            e2e_step()
        for _ in range(args.steps):
            flush.fill_(1)
            barrier()
            dt, nb = e2e_step()
            times.append(dt)
        tt = torch.tensor([float(np.mean(times)), float(nb), float(xh.numel() * 4)], device=dev, dtype=torch.float64)
        if world > 1:
            tmax = tt.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(tt, op=dist.ReduceOp.SUM)
            tt[0] = tmax[0]
        e2e = {"value": frames_total / float(tt[0].item()), "unit": "frames/s",
               "h2d_bytes_per_step": int(tt[2].item()), "d2h_bytes_per_step": int(tt[1].item()),
               "ms_per_step": 1e3 * float(tt[0].item()),
               "note": "PV(pinned host signal).run_pv(hostbuf, stream_tables=f/mag/ph/totalmag) -> toSinSum -> "
                       "synth(hostbuf): the float64 f / mag / ph tables, totalmag and the float64 resynthesis land in "
                       "pinned host memory (copies overlap the kernels on side streams); realph / binno stay on the "
                       "device and are downloaded on first access of the attribute; host wall clock, max over ranks"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk_, how = peaks()
    hbm = float(pk_["hbm_gbs"])
    alg_an = (4 * hop + 20 * npks + 8) * F                       # bytes per launch (SURVEY 8d)
    pbar = psamp_local / max(1.0, float(state["w"].numel()))
    alg_syn = (16.0 / hop + 4.0 / max(pbar, 1e-9)) * psamp_local
    roof_an = {"kernel": "analyze_kernel<10>", "bound": "hbm", "achieved": alg_an / (ms_an * 1e-3) / 1e9, "peak": hbm,
               "unit": "GB/s", "frac": alg_an / (ms_an * 1e-3) / 1e9 / hbm, "traffic": _traffic("analyze"),
               "ms": ms_an, "alg_bytes_per_launch": alg_an, "peak_source": how,
               "note": "fused framing+FFT+peak-pick+IF: issue / latency bound at 16 resident warps per SM (ncu r2x: issue "
                       "slots 57 % busy, DRAM 5 %), see DESIGN.md 4.1"}
    roof_syn = {"kernel": "resynth stage (resynth_tracks_kernel + resynth_tile_kernel, partial bodies built in-kernel)", "bound": "hbm", "achieved": alg_syn / (ms_syn * 1e-3) / 1e9, "peak": hbm,
                "unit": "GB/s", "frac": alg_syn / (ms_syn * 1e-3) / 1e9 / hbm, "traffic": _traffic("resynth"),
                "ms": ms_syn, "alg_bytes_per_launch": alg_syn, "peak_source": how,
                "partial_samples_per_s": psamp_local / (ms_syn * 1e-3),
                "note": "compute bound by construction (one MUFU cosine per partial-sample; ncu r2x: XU pipe 76 % busy, issue "
                        "slots 76 %), see DESIGN.md 4.3"}
    # `roofline` is reported on the same kernel at every N: analyze_kernel, the one launch of the analysis stage
    # (the metric's frames/s; ncu launch list r2x: 439 us).  The other long kernel, resynth_tile_kernel (472 us
    # of the resynthesis stage, which also holds resynth_tracks_kernel and the step's read-back), is reported
    # beside it as `roofline_resynth`.
    dominant = roof_an
    line = {
        "metric": METRIC, "value": frames_total / (ms_step * 1e-3), "unit": "frames/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "f32 FFT, f64 per-peak/phase", "data": "synthetic",
        "config": {"workload": WORKLOAD if not strong else (
                       "%g h mono 44.1 kHz synthetic harmonic tone+noise (configs[3]; 200 Hz, 100 harmonics, sigma 0.01), "
                       "nfft=2048 hop=256 npks=100, ONE signal segment-sharded over the GPUs, analysis + tracking + "
                       "full resynthesis" % args.cfg4_hours),
                   "sr": sr, "seconds_per_gpu": c["seconds"] if not strong else c["seconds"] / float(world),
                   "nfft": nfft, "hop": hop,
                   "npks": npks, "frames_per_gpu": F, "frames_total": frames_total,
                   "partial_samples_total": psamp_total, "tracks_total": int(state["st"]["ntracks"]),
                   "l2": "256 MiB buffer written between timed steps; per-step CUDA events on the launch stream",
                   "settle_passes_before_warmup": settle, "signal_peak": 0.9,
                   "parallelism": "segment-sharded x%d (hop-aligned frame ranges + %d/%d halo rows; local "
                                  "resynthesis; track table gathered by %s)" % ((world,) + D.halos(nfft, hop) + (
                                      "P2P stores of the rename kernel into symmetric-memory tables over NVLink"
                                      if state.get("peer") else "one NCCL all_gather",))},
        "stages": {"analysis_ms": ms_an, "tracking_ms": ms_trk, "pack_ms": ms_pack, "resynth_ms": ms_syn,
                   "analysis_frames_per_s": frames_total / (ms_an * 1e-3),
                   "resynth_partial_samples_per_s": psamp_total / (ms_syn * 1e-3)},
        "roofline": dominant, "roofline_analysis": roof_an, "roofline_resynth": roof_syn,
        "clocks": clocks, "gpu_launches": launches,
    }
    if e2e is not None:
        line["e2e"] = e2e
    if selfcheck is not None:
        line["selfcheck"] = selfcheck
    if strong:
        line["metric"] = "STFT frames/sec (nfft=2048,hop=256,npks=100) + resynth partial-samples/sec"
        line["e2e"] = None
    if world == 1 and not args.no_cpu and not strong:
        line["cpu_baseline"] = cpu_baseline(xd[:sr * args.cpu_seconds + nfft].cpu().numpy(), 1)
    sys.stdout.flush()
    os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(outdir, arrays, budget, suffix=""):
    """Write device arrays as float64 `outdir/<name><suffix>.npy`.  An array larger than its equal share
    of `budget` bytes keeps a fixed, seeded sample of its rows (sorted; the same rows for arrays of the
    same length), so two builds run with the same arguments can be compared output for output."""
    import torch
    os.makedirs(outdir, exist_ok=True)
    cap = budget // len(arrays)
    for name, t in arrays.items():
        t = t.to(torch.float64)
        n = t.shape[0]
        rows = max(1, cap // max(1, t[:1].numel() * 8))
        if n > rows:
            idx = np.sort(np.random.default_rng(0).choice(n, rows, replace=False))
            t = t.index_select(0, torch.from_numpy(idx).to(t.device))
        np.save(os.path.join(outdir, name + suffix + ".npy"), t.cpu().numpy())


def _traffic(which):
    """DRAM bytes per launch from the committed ncu capture (profiles/traffic.json), else null."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            return json.load(fh).get(which)
    except Exception:
        return None


# --------------------------------------------------------------------------- CPU arms
def _oracle_pipeline(x):
    """analysis -> tracking -> resynthesis with the numpy oracle; returns (frames, partial-samples, stage times)."""
    from oracle import pv_oracle as orc
    c = CFG
    t0 = time.perf_counter()
    o = orc.analyze(x, c["sr"], nfft=c["nfft"], hop=c["hop"], npks=c["npks"], pkthresh=c["pkthresh"])
    t1 = time.perf_counter()
    tr = orc.track(o["f"], o["mag"])
    parts = orc.partials_from_tracks(tr, o["f"], o["mag"], o["ph"], o["realph"])
    t2 = time.perf_counter()
    orc.synth(parts, c["sr"], c["hop"], c["nfft"], c["hop"])
    t3 = time.perf_counter()
    ps = orc.partial_samples(parts, c["hop"], c["nfft"], c["hop"])
    return o["nframes"], ps, (t1 - t0, t2 - t1, t3 - t2)


def _reference_pipeline(x):
    """analysis -> tracking -> resynthesis with the UNMODIFIED reference (pypevoc.PV.run_pv,
    PV.toSinSum, RegPartial.synth through the documented Python-3 overlap-add shim of
    oracle/ref_loader.py); same return values as _oracle_pipeline."""
    from oracle import ref_loader as rl
    c = CFG
    t0 = time.perf_counter()
    pv = rl.ref_run_pv(np.asarray(x, dtype=np.float64), c["sr"], c["nfft"], c["hop"], c["npks"], c["pkthresh"])
    t1 = time.perf_counter()
    ss = pv.toSinSum()
    t2 = time.perf_counter()
    rl.ref_sinsum_synth(ss, c["sr"], c["hop"])
    t3 = time.perf_counter()
    E = int(c["hop"] * c["nfft"] / c["hop"] / 2.)
    ps = sum(len(p.f) * c["hop"] + 2 * E for p in ss.partial if len(p.f) >= 3)
    return pv.nframes, ps, (t1 - t0, t2 - t1, t3 - t2)


def _reference_kind():
    try:
        from oracle import ref_loader as rl
        if rl.available():
            rl.load()
            return "reference"
    except Exception as e:
        sys.stderr.write("bench: the reference under baseline/_ref could not be imported (%r); timing the port\n" % (e,))
    return "port"


def _worker(args):
    seed_off, nsamp, kind = args
    from pypevoc_b200 import signals
    c = CFG
    x = signals.harm(c["sr"], nsamp / float(c["sr"]), c["f0"], c["nharm"], c["p"], c["sigma"], c["seed"] + seed_off)
    import warnings
    warnings.simplefilter("ignore")
    t0 = time.perf_counter()
    fr, ps, st = (_reference_pipeline if kind == "reference" else _oracle_pipeline)(x)
    return fr, ps, st, time.perf_counter() - t0


def cpu_baseline(x, cores):
    import warnings
    warnings.simplefilter("ignore")
    kind = _reference_kind()
    t0 = time.perf_counter()
    fr, ps, st = (_reference_pipeline if kind == "reference" else _oracle_pipeline)(x)
    dt = time.perf_counter() - t0
    what = ("unmodified reference PV.run_pv + toSinSum + synth (baseline/_ref)" if kind == "reference"
            else "numpy oracle analyze+track+synth")
    return {"value": fr / dt, "unit": "frames/s", "cores": cores, "kind": kind,
            "sample": "first %.0f s of the same samples (%d frames): %s" % (len(x) / CFG["sr"], fr, what),
            "analysis_frames_per_s": fr / st[0], "tracking_s": st[1],
            "resynth_partial_samples_per_s": ps / st[2]}


def reference_main(args):
    """--impl reference: the reference's own CPU implementation of the path on all host cores, one
    disjoint segment of the workload signal per process: the UNMODIFIED reference from baseline/_ref
    (offline pip install done by __graft_entry__.build(); kind "reference") when it is there, else
    the numpy oracle port (kind "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    kind = _reference_kind()
    cores = os.cpu_count() or 1
    c = CFG
    seg = c["sr"] * args.ref_seconds + c["nfft"]
    ctx = mp.get_context("fork")
    times, frames = [], 0
    with ctx.Pool(cores) as pool:
        for it in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            res = pool.map(_worker, [(100 * it + i, seg, kind) for i in range(cores)])
            dt = time.perf_counter() - t0
            if it >= args.warmup:
                times.append(max(r[3] for r in res))
                frames = sum(r[0] for r in res)
    ms = 1e3 * float(np.mean(times))
    val = frames / (ms * 1e-3)
    what = ("unmodified reference (baseline/_ref): PV.run_pv + toSinSum + RegPartial.synth" if kind == "reference"
            else "numpy oracle analyze+track+synth")
    sample = "%d disjoint %d s segments of the workload signal per step, one process per core, %s" % (
        cores, args.ref_seconds, what)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sr": c["sr"], "seconds_per_gpu": c["seconds"], "nfft": c["nfft"],
                       "hop": c["hop"], "npks": c["npks"], "sample": sample},
            "cpu_baseline": {"value": val, "unit": "frames/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-seconds", type=int, default=15)
    ap.add_argument("--ref-seconds", type=int, default=8)
    ap.add_argument("--workload", default="metric", choices=["metric", "cfg3", "cfg4"])
    ap.add_argument("--cfg4-hours", type=float, default=8.0)
    ap.add_argument("--cfg3-clips", type=int, default=4096)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's outputs (analysis tables, track ids, partial "
                         "spans, resynthesis) as float64 DIR/<name>.npy, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload == "cfg3"):
        ap.error("--dump-outputs covers the GPU path of the metric and cfg4 workloads")
    if args.impl == "reference":
        reference_main(args)
    else:
        gpu_main(args)


if __name__ == "__main__":
    main()
