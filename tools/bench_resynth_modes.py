"""Time the resynthesis stage (tracks + phase scan + render) in its two phase models on one GPU.

Workload: the benchmark's metric signal (10 minutes, SURVEY 8d recipe, 44.1 kHz), analysed with
nfft 2048 / hop 512 / npks 50 and tracked once; then, alternating in every round, with an L2 flush
(256 MB written) before each timed pass:

  preserve      phase_preserve=True (what bench.py times)
  free          phase_preserve=False, fscale 1
  free_shift    phase_preserve=False, fscale 2^(7/12)      (partials scaled to >= sr/2 are left out)
  free_stretch  phase_preserve=False, synthesis hop 1024   (2x time stretch)
  free_curve    phase_preserve=False, a per-frame fscale curve: +-1 semitone vibrato at 5 Hz
                (uploaded once before the timed passes; the upload is not part of the stage)

The phase scan alone (its three kernels) is timed from a torch.profiler capture of its own.  A
second leg does the same at the cfg4 length (one 8-hour signal, nfft 2048 / hop 256 / npks 100),
where single partials span hundreds of thousands of frames.

    python tools/bench_resynth_modes.py [--out profiles/x.json] [--rounds 10] [--cfg4-hours 8 | 0]

Prints one JSON document (card name and power limit included)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from pypevoc_b200 import pv as P, signals  # noqa: E402

METRIC = dict(sr=44100, seconds=600, nfft=2048, hop=512, npks=50, pkthresh=0.005, f0=220.0, nharm=90, p=0.5,
              sigma=0.01, seed=1)
CFG4 = dict(sr=44100, seconds=8 * 3600, nfft=2048, hop=256, npks=100, pkthresh=0.005, f0=200.0, nharm=100, p=0.4,
            sigma=0.01, seed=4000)
SCAN_KERNELS = ("phase_scan_groups_kernel", "phase_scan_carry_kernel", "phase_scan_fixup_kernel")


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
    except Exception as e:                                   # the reading is reported, not required
        q = "unavailable (%r)" % (e,)
    return dict(name=name, power_limit_and_max_sm_clock=q)


def tracked(c, dev):
    """Signal -> analysis -> tracks + packed partials (device), as bench.py builds them."""
    sr = c["sr"]
    x = signals.harm_torch(sr, sr * c["seconds"], c["f0"], c["nharm"], c["p"], c["sigma"], c["seed"], dev, scale=0.25)
    x.mul_(float(np.float32(0.9 / float(x.abs().max()))))
    tb = P.host_tables(sr, c["nfft"], c["hop"])
    a = P.analyze_device(x, sr, c["nfft"], c["hop"], c["npks"], c["pkthresh"], tb)
    del x
    tab = {k: a[k][0] for k in ("f", "mag", "ph", "realph")}
    tr, pk = P.track_pack_device(tab["f"], tab["mag"], tab["ph"], tab["realph"])
    del a, tab
    torch.cuda.synchronize()
    return tr, pk


def vibrato_curve(F, hop_an, sr, rate=5.0, semitones=1.0):
    """One ratio per frame row from its input time row * hop_an / sr."""
    t = np.arange(F) * hop_an / float(sr)
    return 2.0 ** (semitones * np.sin(2 * np.pi * rate * t) / 12.0)


def partial_samples(pk, hop, nfft, hop_an, sr, fscale=None, edge=1.0, minframes=3):
    """Work units: sum over rendered partials of hop * nfr + 2 * edge samples (fscale: Nyquist rule;
    a numpy curve: each point at the ratio of its row)."""
    tl = pk["tlen"].to(torch.int64)
    keep = tl >= minframes
    if fscale is not None:
        ids = torch.repeat_interleave(torch.arange(tl.numel(), device=tl.device), tl)
        f = pk["pf"]
        if isinstance(fscale, np.ndarray):
            rows = pk["tstart"].to(torch.int64)[ids] + torch.arange(ids.numel(), device=tl.device) - pk["toff"][ids]
            f, fscale = f * torch.from_numpy(fscale).to(tl.device)[rows], 1.0
        fmax = torch.full((tl.numel(),), -1.0, dtype=torch.float64, device=tl.device)
        fmax.scatter_reduce_(0, ids, f, reduce="amax")
        keep &= fscale * fmax < 0.5 * sr
    E = int(nfft / hop_an / 2. * hop * edge)
    return int((tl[keep] * hop + 2 * E).sum().item())


def run_leg(c, dev, rounds, label):
    sr, nfft, hop_an = c["sr"], c["nfft"], c["hop"]
    t0 = time.time()
    tr, pk = tracked(c, dev)
    prep_s = time.time() - t0
    tid, max_end = tr["tid"], tr["max_end"]
    F, K = tid.shape
    modes = [("preserve", hop_an, True, 1.0), ("free", hop_an, False, 1.0),
             ("free_shift", hop_an, False, 2 ** (7 / 12.)), ("free_stretch", 2 * hop_an, False, 1.0),
             ("free_curve", hop_an, False, vibrato_curve(F, hop_an, sr))]
    dcurve = P._on_device(modes[-1][3], dev)
    bufs = {}
    for name, hop, pp, fs in modes:
        nout, _ = P.synth_geometry(max_end, hop, nfft, hop_an)
        nb = -(-nout // hop)
        bufs[name] = dict(out=torch.empty(nout, dtype=torch.float64, device=dev),
                          ws=P.resynth_workspace(F, K, len(pk["tstart"]), nb, dev, hop=hop),
                          pws=None if pp else torch.empty(max(pk["pf"].numel(), 1), dtype=torch.float64, device=dev))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def render(name, hop, pp, fs):
        b = bufs[name]
        P.resynth_device(tid, pk, sr, hop, nfft, hop_an, max_end=max_end, out=b["out"], ws=b["ws"],
                         phase_preserve=pp, fscale=dcurve if name == "free_curve" else fs, phase_ws=b["pws"])

    for m in modes:                                          # warm-up: module load, every shape once
        render(*m)
    torch.cuda.synchronize()
    times = {m[0]: [] for m in modes}
    for _ in range(rounds):
        for m in modes:
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            render(*m)
            e1.record()
            e1.synchronize()
            times[m[0]].append(e0.elapsed_time(e1))
    # the scan alone: kernel times of a separate profiled run of the free mode
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(rounds):
            flush.fill_(1)
            render(*modes[1])
        torch.cuda.synchronize()
    scan_us, kern = 0.0, {}
    for evt in prof.key_averages():
        if any(k in evt.key for k in SCAN_KERNELS) or "resynth" in evt.key:
            t = getattr(evt, "device_time_total", None)
            if t is None:
                t = evt.cuda_time_total
            kern[evt.key] = round(t / rounds, 2)
            if any(k in evt.key for k in SCAN_KERNELS):
                scan_us += t / rounds
    res = dict(leg=label, workload=dict((k, c[k]) for k in ("sr", "seconds", "nfft", "hop", "npks")),
               frames=int(F), partials=int(tr["ntracks"]), points=int(pk["pf"].numel()),
               longest_partial_frames=int(pk["tlen"].max().item()), setup_s=round(prep_s, 1), rounds=rounds,
               l2_flush="256 MB written before every timed pass", modes={})
    for name, hop, pp, fs in modes:
        t = np.array(times[name])
        ps = partial_samples(pk, hop, nfft, hop_an, sr, None if pp else fs)
        fs_doc = "vibrato +-1 semitone, 5 Hz, per frame" if isinstance(fs, np.ndarray) else fs
        res["modes"][name] = dict(hop=hop, phase_preserve=pp, fscale=fs_doc, median_ms=round(float(np.median(t)), 4),
                                  min_ms=round(float(t.min()), 4), max_ms=round(float(t.max()), 4),
                                  partial_samples=ps, partial_samples_per_s=float("%.4g" % (ps / (np.median(t) * 1e-3))))
    base = res["modes"]["preserve"]["median_ms"]
    for name in res["modes"]:
        res["modes"][name]["vs_preserve"] = round(res["modes"][name]["median_ms"] / base, 3)
    res["scan_only_ms"] = round(scan_us / 1e3, 4)
    res["scan_share_of_free"] = round(scan_us / 1e3 / res["modes"]["free"]["median_ms"], 3)
    res["free_curve_vs_free"] = round(res["modes"]["free_curve"]["median_ms"] / res["modes"]["free"]["median_ms"], 3)
    res["profiled_kernels_us_per_pass"] = kern
    del bufs, flush, tr, pk, dcurve
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--cfg4-hours", type=float, default=8.0, help="length of the long-partial leg (0: skip it)")
    ap.add_argument("--out", default=None, help="also write the JSON document here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_resynth_modes.py needs a GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    doc = dict(card=card(), legs=[])

    def emit():                                              # after every leg: a failing long leg keeps the first
        s = json.dumps(doc, indent=1)
        print(s, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as fh:
                fh.write(s + "\n")
    doc["legs"].append(run_leg(METRIC, dev, args.rounds, "metric"))
    emit()
    if args.cfg4_hours > 0:
        c = dict(CFG4, seconds=int(round(args.cfg4_hours * 3600)))
        doc["legs"].append(run_leg(c, dev, max(3, args.rounds // 3), "cfg4"))
        emit()


if __name__ == "__main__":
    main()
