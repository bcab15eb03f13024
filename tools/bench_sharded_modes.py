"""Time the sharded resynthesis stage of ``ShardedSinSum.synth_local`` in its phase models.

Runs under torchrun (one process per GPU, NCCL) or as a plain process (world 1).  Workloads:

  metric  the benchmark's metric signal, 10 minutes PER RANK (weak scaling), nfft 2048 / hop 512 / npks 50
  cfg4    one signal of --cfg4-hours hours split over the ranks (strong scaling), nfft 2048 / hop 256 /
          npks 100 (0 = skip)

Every rank analyses and links its window once; then, alternating in every round, with an L2 flush
(256 MB written) before each timed pass, the stage synth_local runs (tracks + scan + hand-over +
collectives + render, output left on the device) is timed with a host clock around work that ends in
a device synchronise, max over the ranks:

  preserve      phase_preserve=True
  free          phase_preserve=False, fscale 1
  free_shift    phase_preserve=False, fscale 2^(7/12)
  free_stretch  phase_preserve=False, synthesis hop 2x the analysis hop
  free_curve    phase_preserve=False, a per-frame fscale curve over the global frames: +-1 semitone
                vibrato at 5 Hz (checked and uploaded inside the timed call, as a user's call does)

``handover`` times dist.integrated_phase_local alone (scan + records + all_gather + seed / fix-up +
flags + all_reduce + import) at fscale 2^(7/12).

    [torchrun --nproc_per_node N] python tools/bench_sharded_modes.py [--out F.json] [--rounds 5]

Rank 0 prints one JSON document (card name and power limit included)."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from pypevoc_b200 import dist as D, pv as P, signals  # noqa: E402
from bench_resynth_modes import card, vibrato_curve  # noqa: E402

METRIC = dict(sr=44100, seconds=600, nfft=2048, hop=512, npks=50, f0=220.0, nharm=90, p=0.5, sigma=0.01, seed=1)
CFG4 = dict(sr=44100, seconds=3600, nfft=2048, hop=256, npks=100, f0=200.0, nharm=100, p=0.4, sigma=0.01, seed=4000)
MODES = [("preserve", 1, dict()), ("free", 1, dict(phase_preserve=False)),
         ("free_shift", 1, dict(phase_preserve=False, fscale=2 ** (7 / 12.))),
         ("free_stretch", 2, dict(phase_preserve=False))]


def sharded_sinsum(c, rank, world, dev, group):
    sr, nfft, hop = c["sr"], c["nfft"], c["hop"]
    x = signals.harm_torch(sr, sr * c["seconds"], c["f0"], c["nharm"], c["p"], c["sigma"], c["seed"], dev, scale=0.25)
    x.mul_(float(np.float32(0.9 / float(x.abs().max()))))
    plans = D.plan_segments(x.numel(), nfft, hop, world)
    p = plans[rank]
    xl = x[p["sample0"]:p["sample0"] + p["nsamp"]].contiguous()
    spv = D.ShardedPV(xl, sr, x.numel(), nfft=nfft, hop=hop, npks=c["npks"], rank=rank, world=world, device=dev,
                      group=group)
    spv.run_pv()
    ss = spv.toSinSum()
    _ = ss.ntracks, ss.device_track_table, ss.local._ensure_packed()     # link + numbering + gather + pack
    torch.cuda.synchronize()
    return ss


def timed(fn, world, flush):
    flush.zero_()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=flush.device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()) * 1e3


def run(c, rank, world, dev, group, rounds, flush):
    ss = sharded_sinsum(c, rank, world, dev, group)
    hop = c["hop"]
    curve = vibrato_curve(ss._spv.plans[0]["frames_total"], hop, c["sr"])
    modes = MODES + [("free_curve", 1, dict(phase_preserve=False, fscale=curve))]
    res = {m: [] for m, _, _ in modes}
    res["handover"] = []

    def handover():
        tidl, pk = ss.local._trk["tid"], ss.local._pk
        F, K = tidl.shape
        ws = P.resynth_workspace(F, K, int(pk["tstart"].shape[0]), 1, dev, hop=hop)
        pws = P._phase_ws(False, pk["pf"].numel(), dev)
        spv = ss._spv
        D.integrated_phase_local(tidl, pk, ss.local._tables["f"], spv.plan, spv.plans, ss.tid_own,
                                 ss.device_track_table, ss.ntracks, c["sr"], hop, c["nfft"], hop, 2 ** (7 / 12.), ws, pws,
                                 group=group)
    for r in range(rounds + 1):                                    # round 0: warm-up
        for name, hm, kw in modes:
            ms = timed(lambda: ss.synth_local(hop=hm * hop, **kw), world, flush)
            if r:
                res[name].append(ms)
        ms = timed(handover, world, flush)
        if r:
            res["handover"].append(ms)
    return {k: dict(median_ms=float(np.median(v)), min_ms=float(np.min(v)), max_ms=float(np.max(v))) for k, v in res.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--cfg4-hours", type=float, default=1.0)
    a = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if world > 1:
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
        dist.init_process_group("nccl")
    dev = torch.device("cuda", torch.cuda.current_device())
    flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)            # 256 MB > 126 MB of L2
    out = dict(card=card(), world=world, rounds=a.rounds, timing="host clock around a device synchronise, max over ranks")
    m = dict(METRIC, seconds=METRIC["seconds"] * world)
    out["metric_10min_per_rank"] = run(m, rank, world, dev, None, a.rounds, flush)
    if a.cfg4_hours > 0:
        out["cfg4_%gh" % a.cfg4_hours] = run(dict(CFG4, seconds=int(3600 * a.cfg4_hours)), rank, world, dev, None,
                                             a.rounds, flush)
    if rank == 0:
        doc = json.dumps(out, indent=1)
        print(doc)
        if a.out:
            with open(a.out, "w") as fh:
                fh.write(doc + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
