"""GPU: the per-sample accuracy contract of the resynthesis render (tests/render_contract.py) on the
device, where the cosines are the hardware's ``__cosf``.  The emulator's case table
(tests/test_render_contract_cpu.py) plus the shapes the emulator cannot afford: K 600 and 1024 at
non-tile hops (shared-memory opt-in), more than 32768 blocks (several prepare + render chunks),
windowed hops 2100 and 4100, the tile shapes of hops 2048 / 768 / 384 / 640, fade lengths from 0 to
2.5 hops, knots inside chunks, and the 60 s metric prefix.  Each render is checked sample by sample
against the float64 reference in the three modes; every case prints its worst ratio and branch."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import parity_util as pu
import render_contract as rc
from pypevoc_b200 import signals

pytestmark = pytest.mark.gpu

# Worst per-sample ratio |w - ref| / scale measured on a B200 (1000 W power limit), per branch, over the
# three modes of every case (the MUFU cosine sees larger arguments at larger RS, see render_bodies):
#   tile<16>: 4.0e-6 (E 102, MUFU + partial fades), 3.2e-6 (E 0), 2.4e-6 (2048/384 knots, dE 7),
#             1.8e-6 (hop 2048, tpb 4), 1.1e-6 (knot inside a chunk), 3.5e-7 (60 s metric prefix)
#   tile<8>: 1.4e-6 (hop 768, E 30)          tile<4>: 1.1e-6 (hop 640, E 0)
#   resynth<16> windowed: 2.8e-6 (hop 2100, 1024/300), 1.0e-6 (hop 4100)
#   resynth<16>: 8.8e-7 (hop 700); with the shared-memory opt-in (K 600 / 1024): 4.9e-7
#   resynth<8>: 2.2e-6 (hop 300, E 5), 1.3e-6 (33000 blocks, 2 chunks), 1.1e-6 (G 2, just under the
#               Nyquist rule); with the shared-memory opt-in: 2.1e-7
# The overall worst is 4.0e-6; the bound is 2.5 times that (4 times would be looser than 1e-5).
TAU_GPU = 1e-5
FLOOR = 1e-9

# name: (hop, nfft, hop_an, edge, K, F, minframes, ws_blocks), as rc.CASES
GPU_CASES = dict(rc.CASES)
GPU_CASES.update({
    "g8_K600": (300, 1024, 256, 1.0, 600, 8, 1, None),
    "g8_K1024": (300, 1024, 256, 0.3, 1024, 8, 1, None),
    "g16_K600": (700, 1024, 256, 0.1, 600, 8, 1, None),
    "g16_K1024": (700, 1024, 256, 1.0, 1024, 8, 1, None),
    "g8_33000_blocks": (300, 1024, 256, 1.0, 4, 33000, 3, None),        # 2 chunks of 32768 blocks
    "g16_windowed_4100": (4100, 1024, 256, 1.0, 8, 8, 3, None),
    "g16_windowed_2100_knots": (2100, 1024, 300, 0.3, 8, 8, 3, None),
    "tile16_2048_edge1": (2048, 1024, 256, 1.0, 12, 10, 3, None),
    "tile8_768_edge0p02": (768, 1024, 256, 0.02, 12, 12, 3, None),      # E 30: MUFU + partial
    "tile4_384_knots": (384, 2048, 384, 1.0, 12, 12, 3, None),
    "tile4_640_edge0p1": (640, 1024, 256, 0.1, 12, 12, 3, None),
    "tile16_edge0p1": (512, 1024, 256, 0.1, 16, 24, 3, None),           # E 102
    "tile16_edge0p3": (512, 1024, 256, 0.3, 16, 24, 3, None),           # E 307
    "tile16_edge0": (512, 1024, 256, 0.0, 16, 24, 3, None),
    "tile16_edge2p5_knots": (512, 2048, 384, 2.5, 16, 24, 3, None),
    "g8_300_knots_edge0p02": (300, 1024, 300, 0.02, 16, 24, 3, None),
    "g8_300_knots_edge2p5": (300, 1024, 300, 2.5, 16, 24, 3, None),
})
NAMES = sorted(GPU_CASES)
SR = rc.SR
WORST = {}                                                   # label -> (worst ratio, branch label)


@pytest.fixture(scope="module")
def P():
    from pypevoc_b200 import _lib, pv
    _lib.lib()
    return pv


def gpu_render(P, t, case, mode, r):
    """track_device -> pack_device -> resynth_device of a synthetic table; returns (w, partials)."""
    hop, nfft, hop_an, edge, K, F, minframes, ws_blocks = case
    dev = torch.device("cuda")
    fd, magd, phd, realphd = (torch.from_numpy(np.ascontiguousarray(t[k])).to(dev) for k in ("f", "mag", "ph", "realph"))
    tr = P.track_device(fd, magd)
    nt = int(tr["ntracks"][0].item())
    pk = P.pack_device(fd, magd, phd, realphd, tr["tid"], tr["link"], nt)
    ws = None
    if ws_blocks is not None:
        from pypevoc_b200 import _lib
        wsb = int(_lib.lib().pvk_resynth_workspace_bytes(F, K, nt, 0)) + (ws_blocks - 1) * rc.row_ws_bytes(K)
        ws = torch.zeros(wsb, dtype=torch.uint8, device=dev)
    w = P.resynth_device(tr["tid"], pk, SR, hop, nfft, hop_an, edge, minframes, ws=ws,
                         phase_preserve=mode == "preserve", fscale=r).cpu().numpy()
    parts = rc.parts_from_tid(tr["tid"].cpu().numpy(), t["f"], t["mag"], t["ph"], t["realph"])
    return w, parts


def check(w, parts, sr, hop, nfft, hop_an, edge, minframes, mode, r, label, br):
    ref = rc.reference(parts, sr, hop, nfft, hop_an, edge, minframes, mode, r)
    scale = rc.amp_scale(parts, sr, hop, nfft, hop_an, edge, minframes, None if mode == "preserve" else r)
    worst = rc.check_render(w, ref, scale, TAU_GPU, FLOOR, label, hop, br)
    WORST[label] = (worst, rc.branch_label(br))
    print("%-44s worst %.2e  %s" % (label, worst, rc.branch_label(br)))
    return ref


@pytest.mark.parametrize("name", NAMES)
def test_gpu_render_per_sample(P, name):
    case = GPU_CASES[name]
    hop, nfft, hop_an, edge, K, F, minframes, ws_blocks = case
    t = rc.make_table(F, K, SR, seed=sum(map(ord, name)), minframes=minframes, stationary=K > 64)
    br = rc.case_branch(case)
    for label, mode, r in rc.modes(case, NAMES.index(name)):
        w, parts = gpu_render(P, t, case, mode, r)
        check(w, parts, SR, hop, nfft, hop_an, edge, minframes, mode, r, "%s %s" % (name, label), br)


def test_gpu_just_under_nyquist(P):
    """The highest partial at fscale * max(f) just under sr / 2 is rendered and within the bound."""
    name = "g8_G2"
    case = GPU_CASES[name]
    hop, nfft, hop_an, edge, K, F, minframes, ws_blocks = case
    t = rc.make_table(F, K, SR, seed=sum(map(ord, name)), minframes=minframes)
    fmax = float(t["f"].max())
    fs = np.nextafter(0.5 * SR / fmax, 0.0)
    while fs * fmax >= 0.5 * SR:
        fs = np.nextafter(fs, 0.0)
    w, parts = gpu_render(P, t, case, "free", fs)
    check(w, parts, SR, hop, nfft, hop_an, edge, minframes, "free", fs, "%s fscale %.17g" % (name, fs),
          rc.case_branch(case))


def test_gpu_cases_cover_every_branch():
    seen = set()
    for name in NAMES:
        seen |= rc.branch_features(rc.case_branch(GPU_CASES[name]))
    assert rc.BRANCHES <= seen, sorted(rc.BRANCHES - seen)


@pytest.fixture(scope="module")
def metric_pv(P):
    """60 s prefix of the benchmark signal, nfft 2048 / hop 512 / npks 50."""
    sr = 44100
    x = signals.harm_torch(sr, 60 * sr, 220.0, 90, 0.5, 0.01, 1, torch.device("cuda"), scale=0.25)
    x = (x * float(np.float32(0.9 / float(x.abs().max())))).cpu().numpy()
    pv = P.PV(x, sr, nfft=2048, hop=512, npks=50, progress=False)
    pv.run_pv()
    return pv


@pytest.mark.parametrize("mode", ["preserve", "fscale 1.25", "vibrato"])
def test_gpu_metric_prefix_per_sample(P, metric_pv, mode):
    sr, nfft, hop_an, hop = 44100, 2048, 512, 512
    ss = metric_pv.toSinSum()
    h = ss._host_tracks()
    o = h["toff"]
    parts = [dict(start_idx=int(h["tstart"][v]), f=h["pf"][o[v]:o[v + 1]], mag=h["pmag"][o[v]:o[v + 1]],
                  realph=h["prealph"][o[v]:o[v + 1]]) for v in range(len(h["tstart"]))]
    F = metric_pv.nframes
    r = {"preserve": 1.0, "fscale 1.25": 1.25, "vibrato": rc.vibrato(F, hop_an, sr)}[mode]
    m = "preserve" if mode == "preserve" else "free"
    w = ss.synth(sr, hop, phase_preserve=m == "preserve", fscale=r)
    br = rc.render_branch(hop, 50, nfft, hop_an, 1.0)
    ref = check(np.asarray(w), parts, sr, hop, nfft, hop_an, 1.0, 3, m, r, "metric 60 s %s" % mode, br)
    assert pu.snr_db(w, ref) > 90.0


def test_gpu_worst_ratios_summary():
    """Runs last (file order): the worst ratio of every render above, by branch."""
    byb = {}
    for label, (worst, b) in WORST.items():
        if worst > byb.get(b, (0.0, ""))[0]:
            byb[b] = (worst, label)
    for b, (worst, label) in sorted(byb.items(), key=lambda kv: -kv[1][0]):
        print("worst %.2e  %-44s %s" % (worst, label, b))
    if WORST:
        print("overall worst %.2e (TAU_GPU %.1e)" % (max(v[0] for v in WORST.values()), TAU_GPU))
