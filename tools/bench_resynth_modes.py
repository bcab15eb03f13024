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
  formant       free_shift with formant_shift=1.0: the formant gain kernel runs inside the timed stage
  formant_curve free_curve with formant_shift=1.0 (a per-row ratio curve for the gain kernel)
  time_map      phase_preserve=False, time_map: a stretch curve between 0.8x and 1.25x over the whole
                signal.  Timed twice: the map stage alone (pvk_time_map, pvk_track_stats and its 24-byte
                read-back, pvk_track_pack of the mapped tables) and the whole stage (map stage + render
                of the mapped partials, allocations included, as SinSum.synth(time_map=...) runs it)
  remap         SinSum.remap(tau) of a ping-pong loop at 1x over the first half of the signal (forwards,
                then backwards: as many output blocks as the time_map row),
                rendered with phase_preserve=False.  Timed twice, alternating with the time_map passes: the
                remap stage alone (pvk_time_map, pvk_track_relink, pvk_track_stats and its 24-byte
                read-back, pvk_track_pack) and the whole stage (remap stage + render of the runs)

The phase scan alone (its three kernels) is timed from a torch.profiler capture of the free mode, the
formant gain kernel from one capture per formant mode.  A
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


def stretch_map(F, period=700.0):
    """A time map over the whole table whose local stretch moves between 0.8x and 1.25x (speed 1.25 ..
    0.8 analysis frames per output block, a sine of ``period`` output blocks)."""
    b = np.arange(2 * F)
    tau = np.concatenate([[0.0], np.cumsum(1.025 + 0.225 * np.sin(2 * np.pi * b / period))])
    return tau[tau <= F - 1]


def pingpong_map(F):
    """A ping-pong loop at 1x over the first half of the table: forwards from row 0 to row F // 2, then
    backwards to row 0 (about F output blocks, as many as stretch_map)."""
    h = F // 2
    return np.concatenate([np.arange(0.0, h + 1.0), np.arange(h - 1.0, -1.0, -1.0)])


def time_leg_map(tid, pk, sr, nfft, hop_an, dev, rounds, flush):
    """Median / min / max ms of the map stage and of the whole stage of the time map (stretch_map) and of
    the remap (pingpong_map), the four timed passes alternating in every round."""
    F = tid.shape[0]
    tau = stretch_map(F)
    td = torch.from_numpy(tau).to(dev)
    pp = pingpong_map(F)
    ppd = torch.from_numpy(pp).to(dev)

    def whole():
        tm, pkm, last = P.time_map_device(tid, pk, td)
        P.resynth_device(tm, pkm, sr, hop_an, nfft, hop_an, max_end=last, phase_preserve=False)
        return pkm

    def remap_whole():
        _, tr, pkr = P.remap_device(tid, pk, ppd)
        P.resynth_device(tr["tid"], pkr, sr, hop_an, nfft, hop_an, max_end=tr["max_end"], phase_preserve=False)
        return tr, pkr

    pkm = whole()                                            # warm-up
    trr, pkr = remap_whole()
    torch.cuda.synchronize()
    ps = partial_samples(pkm, hop_an, nfft, hop_an, sr, 1.0)
    ps_r = partial_samples(pkr, hop_an, nfft, hop_an, sr, 1.0)
    runs = dict(partials=int(trr["ntracks"]), points=int(trr["npts"]))
    del pkm, trr, pkr
    times = dict(map=[], whole=[], remap=[], remap_whole=[])
    for _ in range(rounds):
        for name, fn in (("map", lambda: P.time_map_device(tid, pk, td)), ("whole", whole),
                         ("remap", lambda: P.remap_device(tid, pk, ppd)), ("remap_whole", remap_whole)):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1))
    t = {k: np.array(v) for k, v in times.items()}
    tm = dict(output_blocks=int(len(tau)), stretch="0.8x .. 1.25x (speed sine, 700-block period)",
              temp_table_bytes=int(len(tau) * tid.shape[1] * 28),
              median_ms=round(float(np.median(t["whole"])), 4), min_ms=round(float(t["whole"].min()), 4),
              max_ms=round(float(t["whole"].max()), 4), map_stage_median_ms=round(float(np.median(t["map"])), 4),
              map_stage_min_ms=round(float(t["map"].min()), 4), partial_samples=ps,
              partial_samples_per_s=float("%.4g" % (ps / (np.median(t["whole"]) * 1e-3))))
    rm = dict(output_blocks=int(len(pp)), map="ping-pong loop at 1x over the first half of the table (forwards, then backwards)",
              temp_table_bytes=int(len(pp) * tid.shape[1] * 36), runs=runs,
              median_ms=round(float(np.median(t["remap_whole"])), 4), min_ms=round(float(t["remap_whole"].min()), 4),
              max_ms=round(float(t["remap_whole"].max()), 4),
              remap_stage_median_ms=round(float(np.median(t["remap"])), 4),
              remap_stage_min_ms=round(float(t["remap"].min()), 4), partial_samples=ps_r,
              partial_samples_per_s=float("%.4g" % (ps_r / (np.median(t["remap_whole"]) * 1e-3))))
    return tm, rm


def run_leg(c, dev, rounds, label):
    sr, nfft, hop_an = c["sr"], c["nfft"], c["hop"]
    t0 = time.time()
    tr, pk = tracked(c, dev)
    prep_s = time.time() - t0
    tid, max_end = tr["tid"], tr["max_end"]
    F, K = tid.shape
    modes = [("preserve", hop_an, True, 1.0), ("free", hop_an, False, 1.0),
             ("free_shift", hop_an, False, 2 ** (7 / 12.)), ("free_stretch", 2 * hop_an, False, 1.0),
             ("free_curve", hop_an, False, vibrato_curve(F, hop_an, sr)),
             ("formant", hop_an, False, 2 ** (7 / 12.)), ("formant_curve", hop_an, False, vibrato_curve(F, hop_an, sr))]
    dcurve = P._on_device(modes[4][3], dev)
    # formant_shift=1.0 (formant preservation) at the shift / vibrato: the gain kernel runs inside the timed render
    formant = {"formant": P.formant_ratio(False, modes[5][3], 1.0), "formant_curve": dcurve}
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
                         phase_preserve=pp, fscale=dcurve if name in ("free_curve", "formant_curve") else fs,
                         phase_ws=b["pws"], formant=formant.get(name))

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
    # the formant gain kernel alone: a capture of its own per formant mode (the scan of the free capture
    # above stays the only one counted in scan_only_ms)
    gain_us = {}
    for m in (modes[5], modes[6]):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(rounds):
                flush.fill_(1)
                render(*m)
            torch.cuda.synchronize()
        gain_us[m[0]] = 0.0
        for evt in prof.key_averages():
            if "formant_gain_kernel" in evt.key:
                t = getattr(evt, "device_time_total", None)
                if t is None:
                    t = evt.cuda_time_total
                gain_us[m[0]] += t / rounds
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
    res["formant_vs_free_shift"] = round(res["modes"]["formant"]["median_ms"] / res["modes"]["free_shift"]["median_ms"], 3)
    res["formant_curve_vs_free_curve"] = round(res["modes"]["formant_curve"]["median_ms"] /
                                               res["modes"]["free_curve"]["median_ms"], 3)
    res["formant_gain_kernel_us"] = {k: round(v, 2) for k, v in gain_us.items()}
    res["formant_gain_share"] = {k: round(v / 1e3 / res["modes"][k]["median_ms"], 4) for k, v in gain_us.items()}
    res["profiled_kernels_us_per_pass"] = kern
    del bufs                                                 # room for the mapped tables (13.6 GB at cfg4)
    torch.cuda.empty_cache()
    tmr, rmr = time_leg_map(tid, pk, sr, nfft, hop_an, dev, rounds, flush)
    res["modes"]["time_map"] = dict(hop=hop_an, phase_preserve=False, fscale=1.0, **tmr)
    res["time_map_vs_free"] = round(tmr["median_ms"] / res["modes"]["free"]["median_ms"], 3)
    res["time_map_stage_share"] = round(tmr["map_stage_median_ms"] / tmr["median_ms"], 3)
    res["modes"]["remap"] = dict(hop=hop_an, phase_preserve=False, fscale=1.0, **rmr)
    res["remap_stage_vs_time_map_stage_per_block"] = round(
        (rmr["remap_stage_median_ms"] / rmr["output_blocks"]) / (tmr["map_stage_median_ms"] / tmr["output_blocks"]), 3)
    res["remap_stage_share"] = round(rmr["remap_stage_median_ms"] / rmr["median_ms"], 3)
    del flush, tr, pk, dcurve, formant
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
