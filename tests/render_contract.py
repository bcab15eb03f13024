"""Per-sample accuracy contract of the resynthesis render (pypevoc_b200/csrc/pvk_resynth.cu).

An aggregate SNR over a whole signal cannot see an error confined to a few samples: a wrong fade, a
wrong knot segment or a wrong last block.  The tests built on this module compare every output
sample with a float64 reference, relative to the local amplitude scale at that sample:

    |w[n] - ref[n]| <= tau * scale[n] + floor

``scale[n]`` (:func:`amp_scale`) is the sum over the rendered partials of ``|msig|`` at ``n``, with each
fade held at the amplitude of its un-faded end (near the silent end of a fade the faded envelope goes
to zero, but the fp32 phase error of the sample does not).

Helpers (no tests here):

- :func:`render_branch` restates the dispatch of ``resynth_run`` / ``render_fades`` / ``render_bodies``
  and names the branch a case renders through; :func:`branch_features` turns it into the set of
  branches a coverage test checks.
- :func:`make_table` writes a synthetic peak table with controlled columns (partial lengths, positions,
  frequencies, glides, amplitudes).
- :func:`reference` is the float64 reference of each mode.  With integrated phase it is
  :func:`free_synth`, whose block start phases are an exact sum of the per-block advances, so it stays
  accurate on partials of any length (the sample-by-sample ``cumsum`` of the numpy models accumulates
  rounding error along the partial).
"""
import math

import numpy as np

from oracle import pv_oracle as orc
import synth_curve_oracle as sco
import synth_modes_oracle as smo

pi2 = 2.0 * np.pi
CHUNK_BLOCKS = 32768          # blocks per prepare + render chunk of the staged kernels (full workspace)
BODY_ITEM_BYTES = 80          # sizeof(BodyItem) in pvk_resynth.cu: one staged partial body


def row_ws_bytes(K):
    """Workspace bytes of one staged block of a table K peaks wide: K BodyItems and a 4-byte count
    (``resynth_row_ws`` in pvk_resynth.cu)."""
    return K * BODY_ITEM_BYTES + 4


# ------------------------------------------------------------------ dispatch
def geometry(hop, nfft, hop_an, edge):
    """(E, dE, qk, qkm) as ``resynth_run`` / ``synth_params`` compute them."""
    dfr = 1.0 / (hop_an / float(nfft)) / 2.0
    E = int(dfr * hop * edge)
    af, am = dfr + 0.5, dfr
    qk = int(math.ceil((af - math.floor(af)) * hop))
    qkm = int(math.ceil((am - math.floor(am)) * hop))
    return E, -(-E // hop), qk, qkm


def render_branch(hop, npks, nfft, hop_an, edge, nblocks=None, chunk_blocks=CHUNK_BLOCKS):
    """The render branch of one launch: kernel, RS samples per thread, nchp chunk threads per item
    group, G item groups, tiles per block (tile kernels), windowed (hop > bd * RS), shared-memory
    opt-in (> 48 KB), number of prepare + render chunks (``nblocks`` blocks, ``chunk_blocks`` per chunk),
    the fade regimes, and whether a knot falls inside a chunk (the per-sample body path)."""
    E, dE, qk, qkm = geometry(hop, nfft, hop_an, edge)
    tile = hop % 128 == 0
    if tile:
        RS = 16 if hop % 512 == 0 else 8 if hop % 256 == 0 else 4
        br = dict(kernel="tile<%d>" % RS, RS=RS, nchp=32, G=1, tpb=hop // (32 * RS), windowed=False,
                  smem=False, chunks=1)
    else:
        RS = 16 if hop >= 512 else 8
        nch = -(-hop // RS)
        bd = 128 if nch >= 32 else 64
        nchp = min(nch, bd)
        smem = npks * BODY_ITEM_BYTES + RS * (bd + 32 // RS) * 4 > 48 * 1024
        chunks = 1 if nblocks is None else -(-nblocks // chunk_blocks)
        br = dict(kernel="resynth<%d>" % RS, RS=RS, nchp=nchp, G=min(bd // nchp, npks), tpb=None,
                  windowed=nch > bd, smem=smem, chunks=chunks)
    fades = set()
    if E > 0:
        if E >= RS:
            # whole-chunk fades: cubic Taylor envelope when the envelope angle moves <= 0.05 rad per
            # half chunk, else one MUFU cosine per sample (the fp32 test of render_fades)
            e1 = np.float32(3.14159265358979) * np.float32(1.0 / E)
            fades.add("taylor" if e1 * np.float32(RS // 2) <= np.float32(0.05) else "mufu")
        if E % RS or hop % RS:
            fades.add("partial")              # a fade edge (or a block end) inside a chunk
    inside = lambda k: 0 < k < hop and k % RS != 0                       # noqa: E731
    br.update(E=E, dE=dE, qk=qk, qkm=qkm, fades=fades,
              body_slow=inside(qk) or inside(qkm) or (not tile and hop % RS != 0))
    return br


def branch_features(br):
    """The branches one launch renders through, as strings (the rows of the dispatch table)."""
    s = {br["kernel"]}
    if br["kernel"].startswith("tile") and br["tpb"] > 2:
        s.add("tile tpb>2")
    if br["kernel"] == "resynth<8>" and br["G"] > 1:
        s.add("resynth<8> G>1")
    if br["windowed"]:
        s.add("%s windowed" % br["kernel"])
    if br["smem"]:
        s.add("smem opt-in")
    if br["chunks"] > 1:
        s.add("chunks>1")
    s.update("fade " + f for f in br["fades"])
    if br["body_slow"]:
        s.add("body slow")
    if br["E"] == 0:
        s.add("E=0")
    elif br["E"] < br["RS"]:
        s.add("E<RS")
    if br["dE"] > 1:
        s.add("dE>1")
    return s


# every branch of resynth_run / render_fades / render_bodies; the case tables must reach each one
BRANCHES = {"tile<16>", "tile<8>", "tile<4>", "tile tpb>2", "resynth<8>", "resynth<8> G>1", "resynth<16>",
            "resynth<16> windowed", "smem opt-in", "chunks>1", "fade taylor", "fade mufu", "fade partial",
            "body slow", "E=0", "E<RS", "dE>1"}


def branch_label(br):
    parts = [br["kernel"], "RS%d" % br["RS"], "nchp%d" % br["nchp"], "G%d" % br["G"]]
    if br["tpb"] is not None:
        parts.append("tpb%d" % br["tpb"])
    for k in ("windowed", "smem", "body_slow"):
        if br[k]:
            parts.append(k)
    if br["chunks"] > 1:
        parts.append("chunks%d" % br["chunks"])
    parts.append("E%d dE%d fades=%s" % (br["E"], br["dE"], "+".join(sorted(br["fades"])) or "none"))
    return " ".join(parts)


# ------------------------------------------------------------------ the case table
# name: (hop, nfft, hop_an, edge, K, F, minframes, ws_blocks)
#   ws_blocks: render the staged kernels in chunks of that many blocks (None: one chunk)
CASES = {
    "tile16_taylor_dE2": (512, 1024, 256, 1.0, 12, 14, 3, None),       # E 1024: Taylor fades, dE 2
    "tile16_tpb4": (2048, 1024, 256, 0.3, 6, 6, 3, None),              # 4 tiles per block, E 1228 partial
    "tile16_knot_in_chunk": (512, 2048, 384, 0.2, 8, 10, 3, None),     # qk 86: knot inside a chunk
    "tile16_mufu_fade": (512, 1024, 256, 0.1, 8, 10, 2, None),         # E 102: MUFU envelope, partial
    "tile16_edge_2p5": (512, 1024, 256, 2.5, 6, 8, 1, None),           # E 2560 > hop: dE 5
    "tile8": (256, 1024, 256, 0.3, 12, 14, 3, None),                   # E 153: MUFU + partial-chunk fades
    "tile8_tpb3": (768, 1024, 256, 0.5, 8, 8, 3, None),
    "tile4_taylor": (128, 512, 128, 0.5, 12, 16, 3, None),             # E 128, RS 4: Taylor
    "tile4_tpb3": (384, 1024, 256, 1.0, 8, 10, 3, None),
    "tile4_tpb5_E0": (640, 1024, 256, 0.0, 8, 8, 3, None),             # no fades
    "g8_G2": (200, 1024, 256, 0.1, 12, 14, 3, None),                   # 2 item groups, knot inside
    "g8_odd_small_edge": (300, 1024, 300, 0.01, 10, 12, 2, None),      # E 5 < RS; knots inside
    "g8_G3_edge0": (136, 1024, 256, 0.0, 8, 14, 3, None),              # 3 item groups, E 0
    "g8_chunked": (300, 1024, 256, 1.0, 8, 16, 3, 3),                  # prepare + render in 6 chunks
    "g16_700": (700, 1024, 256, 0.3, 8, 8, 3, None),
    "g16_windowed": (2100, 1024, 256, 0.5, 6, 5, 3, None),             # hop > 128 * 16: windows
    "g16_smem_optin": (700, 1024, 256, 1.0, 616, 4, 1, None),          # K 616: > 48 KB shared memory
}
FSCALES = (0.5, 1.0, 1.5)
SR = 16000.0


def case_branch(case):
    """render_branch of a case tuple (its block count is the output length of a table of F rows)."""
    hop, nfft, hop_an, edge, K, F, minframes, ws_blocks = case
    E = geometry(hop, nfft, hop_an, edge)[0]
    nblocks = -(-((F + 1) * hop + E) // hop)
    return render_branch(hop, K, nfft, hop_an, edge, nblocks=nblocks, chunk_blocks=ws_blocks or CHUNK_BLOCKS)


def modes(case, i):
    """(label, mode, r) of the renders of the ``i``-th case: phase-preserving, integrated phase at
    FSCALES[i % 3] and a fast +-2 semitone vibrato curve."""
    hop, nfft, hop_an, edge, K, F = case[:6]
    fs = FSCALES[i % len(FSCALES)]
    return [("preserve", "preserve", 1.0), ("fscale %g" % fs, "free", fs),
            ("vibrato", "free", vibrato(F, hop_an, SR, rate=40.0, semis=2.0))]


# ------------------------------------------------------------------ synthetic peak tables
def make_table(F, K, sr, seed=0, fmin=1.0, fmax_frac=0.49, glide=0.025, minframes=3, stationary=False):
    """A peak table ``[F, K]`` (f, mag, ph, realph) written row by row.  Column ``c`` holds partials near
    its own base frequency, spaced geometrically from ``fmin`` to ``fmax_frac * sr``, one after the other
    with one empty row between them, so the tracker finds exactly these partials when the columns are
    more than half a semitone apart:

    - column 0 holds one partial from row 0 to the last row, the top column ends at the last row;
    - the other columns cycle through lengths 1 .. minframes + 1 and longer ones, from staggered starts;
    - every other column glides (frequency times ``1 +- glide`` per frame, under the tracker's half
      semitone), the others wobble by 0.1 %; a glide never leaves its column's band;
    - partial amplitudes are log-uniform over 1e-4 .. 1e2 and change by up to 2x from frame to frame;
    - realph and ph are uniform phases.

    ``stationary``: no glides and no wobble (many columns, closer than the tracker's limit)."""
    rng = np.random.default_rng(seed)
    f = np.zeros((F, K))
    mag = np.zeros((F, K))
    ph = np.zeros((F, K))
    realph = np.zeros((F, K))
    fb = fmin * (fmax_frac * sr / fmin) ** (np.arange(K) / max(K - 1, 1))
    lens = list(range(1, minframes + 2)) + [F, 7, 2 * minframes + 3, F // 2]
    for c in range(K):
        row = 0 if c in (0, K - 1) else int(rng.integers(0, 4))
        j = c
        while row < F:
            n = F if c == 0 else lens[j % len(lens)]
            j += 1
            n = min(n, F - row)
            if c == K - 1:
                n = F - row                              # the top column ends at the last row
            k = np.arange(n)
            if stationary:
                fr = np.full(n, fb[c])
            elif c % 2 == 1 and 0 < c < K - 1:
                g = glide if (c // 2) % 2 == 0 else -glide
                span = min(n, 16)                        # glide up (down) then back, inside the band
                tri = np.minimum(k % (2 * span), 2 * span - k % (2 * span))
                fr = fb[c] * (1.0 + g) ** tri
            else:
                fr = fb[c] * (1.0 + 1e-3 * np.sin(1.3 * k + c))
            if c == K - 1:
                fr = np.minimum(fr, fmax_frac * sr)
            m0 = 10.0 ** rng.uniform(-4.0, 2.0)
            f[row:row + n, c] = fr
            mag[row:row + n, c] = m0 * 2.0 ** rng.uniform(-1.0, 1.0, n)
            ph[row:row + n, c] = rng.uniform(-np.pi, np.pi, n)
            realph[row:row + n, c] = rng.uniform(-np.pi, np.pi, n)
            row += n + 1
    return dict(f=f, mag=mag, ph=ph, realph=realph, sr=float(sr))


def parts_from_tid(tid, f, mag, ph, realph):
    """The partials of a track-id table (from the tracking kernel), as :func:`oracle.pv_oracle.partials_from_tracks`
    gives them to the numpy models."""
    tid = np.asarray(tid)
    nt = int(tid.max()) + 1 if tid.size and tid.max() >= 0 else 0
    rows, cols = np.nonzero(tid >= 0)
    st = np.full(nt, np.iinfo(np.int64).max, dtype=np.int64)
    np.minimum.at(st, tid[rows, cols], rows)
    return orc.partials_from_tracks(dict(tid=tid, st=st), f, mag, ph, realph)


def vibrato(F, hop_an, sr, rate=5.0, semis=1.0):
    """A +-``semis`` semitone vibrato at ``rate`` Hz: one ratio per frame row."""
    t = np.arange(F) * hop_an / float(sr)
    return 2.0 ** (semis * np.sin(2 * np.pi * rate * t) / 12.0)


# ------------------------------------------------------------------ references
def _rendered(parts, sr, minframes, mode, r):
    if mode == "preserve":
        return [p for p in parts if len(p["f"]) >= minframes]
    if np.ndim(r) == 0:
        return [p for p in parts if smo.renders(p, sr, minframes, False, float(r))]
    return [p for p in parts if sco.renders(p, sr, minframes, r)]


def _overlap_add(parts, hop, nfft, hop_an, edge, render_one, max_end=None):
    """SinSum.synth's output length and placement (PVAnalysis.py:1055-1070)."""
    dfr = nfft / hop_an / 2.
    edgsamp = int(edge * hop * dfr)
    if max_end is None:
        max_end = max(p["start_idx"] + len(p["f"]) - 1 for p in parts)
    w = np.zeros((max_end + 2) * hop + 2 * edgsamp)
    for p in parts:
        wi, e = render_one(p)
        s = int(p["start_idx"] * hop - e) + edgsamp
        if s >= 0:
            w[s:s + len(wi)] += wi
    return w[edgsamp:]


def block_start_phases(p0, adv):
    """Start phase (cycles in [0, 1)) of every block: ``p0`` plus the exact sum of the advances of the
    blocks before it, mod 1.  Each advance is reduced mod 1 (exact) and truncated to 2^-64 cycles, and
    the sums are taken in 64-bit integers, which wrap exactly mod 1 cycle: the error is below 2^-64
    cycles per block, whatever the partial's length (a float64 running sum would lose ~1e-16 of its
    growing magnitude at every step)."""
    a = np.floor(np.mod(adv, 1.0) * 2.0 ** 64).astype(np.uint64)
    s = np.zeros(len(adv), dtype=np.uint64)
    if len(adv) > 1:
        s[1:] = np.cumsum(a[:-1], dtype=np.uint64)
    return np.mod(p0 + s.astype(np.float64) * 2.0 ** -64, 1.0)


def free_partial(pf, pmag, prealph, sr, hop, overlap, rp, edge=1.0):
    """One partial in integrated-phase mode with the ratios ``rp`` of its own rows: the model of
    :mod:`synth_curve_oracle` (a constant ``rp`` is :mod:`synth_modes_oracle`'s ``fscale``), with the
    phase kept in cycles as (block start phase from :func:`block_start_phases`) + (in-block sum of the
    scaled frequency).  Returns ``(signal, start_sample)``."""
    pf = np.asarray(pf, dtype=np.float64)
    pmag = np.asarray(pmag, dtype=np.float64)
    rp = np.asarray(rp, dtype=np.float64)
    nfr = len(pf)
    hop = int(hop)
    dfr = 1. / overlap / 2.
    newt = np.arange(hop * (nfr + dfr))
    fsig = np.interp(newt, hop * (dfr + .5 + np.arange(nfr)), pf)
    msig = np.interp(newt, hop * (dfr + np.arange(nfr)), pmag)
    n = hop * nfr
    fc = fsig[:n].reshape(nfr, hop) * (rp / float(sr))[:, None]           # cycles per sample
    inb = np.zeros((nfr, hop))
    inb[:, 1:] = np.cumsum(fc[:, :-1], axis=1)
    p0 = float(np.mod(prealph[0] / pi2, 1.0))
    th = block_start_phases(p0, inb[:, -1] + fc[:, -1])[:, None] + inb   # cycles
    body = msig[:n] * np.cos(pi2 * np.mod(th.ravel(), 1.0))
    E = int(dfr * hop * edge)
    q = np.arange(E)
    hmag = msig[0] * (1 - np.cos(np.pi * q / float(E))) / 2.
    hth = p0 - rp[0] * pf[0] * (E - q) / float(sr)
    tmag = msig[n] * (1 + np.cos(np.pi * q / float(E))) / 2.
    tth = np.mod(th[-1, -1], 1.0) + rp[-1] * pf[-1] * (q + 1) / float(sr)
    return np.concatenate((hmag * np.cos(pi2 * np.mod(hth, 1.0)), body, tmag * np.cos(pi2 * np.mod(tth, 1.0)))), E


def free_synth(parts, sr, hop, nfft, hop_an, r, edge=1.0, minframes=3, max_end=None):
    """Integrated-phase overlap-add with :func:`free_partial`; ``r``: a scalar ratio or one per frame row."""
    overlap = hop_an / float(nfft)
    if max_end is None:
        max_end = max(p["start_idx"] + len(p["f"]) - 1 for p in parts)

    def one(p):
        rp = np.full(len(p["f"]), float(r)) if np.ndim(r) == 0 else sco.part_ratios(p, r)
        return free_partial(p["f"], p["mag"], p["realph"], sr, hop, overlap, rp, edge)
    return _overlap_add(_rendered(parts, sr, minframes, "free", r), hop, nfft, hop_an, edge, one, max_end)


def reference(parts, sr, hop, nfft, hop_an, edge, minframes, mode, r=1.0):
    """The float64 reference of a render: ``mode`` "preserve" (:func:`oracle.pv_oracle.synth`) or "free"
    (``r`` a scalar fscale or a per-row curve, :func:`free_synth`)."""
    if mode == "preserve":
        return orc.synth(parts, sr, hop, nfft, hop_an, edge, minframes)
    return free_synth(parts, sr, hop, nfft, hop_an, r, edge, minframes)


def model(parts, sr, hop, nfft, hop_an, edge, minframes, mode, r=1.0):
    """The numpy models of the tests (sample-by-sample cumsum of the integrated phase)."""
    if mode == "preserve":
        return orc.synth(parts, sr, hop, nfft, hop_an, edge, minframes)
    if np.ndim(r) == 0:
        return smo.synth(parts, sr, hop, nfft, hop_an, edge, minframes, phase_preserve=False, fscale=float(r))
    return sco.synth(parts, sr, hop, nfft, hop_an, r, edge, minframes)


def amp_scale(parts, sr, hop, nfft, hop_an, edge, minframes, r=None):
    """Local amplitude scale of every output sample: the sum over the rendered partials of ``|msig|``
    (the ``msig`` lines of :func:`oracle.pv_oracle.synth_partial`) without the raised cosine of the
    fades, i.e. a head holds ``|msig[0]|`` and a tail ``|msig[hop * nfr]|``.  ``r`` (a scalar ratio or a
    per-row curve): integrated phase, where the partials the Nyquist rule skips are left out."""
    hop = int(hop)
    overlap = hop_an / float(nfft)
    dfr = 1. / overlap / 2.

    def one(p):
        pmag = np.asarray(p["mag"], dtype=np.float64)
        nfr = len(pmag)
        newt = np.arange(hop * (nfr + dfr))
        msig = np.abs(np.interp(newt, hop * (dfr + np.arange(nfr)), pmag))
        E = int(dfr * hop * edge)
        n = hop * nfr
        return np.concatenate((np.full(E, msig[0]), msig[:n], np.full(E, msig[n]))), E
    max_end = max(p["start_idx"] + len(p["f"]) - 1 for p in parts)
    rendered = _rendered(parts, sr, minframes, "preserve" if r is None else "free", r)
    return _overlap_add(rendered, hop, nfft, hop_an, edge, one, max_end)


# ------------------------------------------------------------------ the check
def worst_ratio(w, ref, scale, floor, tau=1.0):
    """(worst ratio, its sample): the smallest tau with ``|w - ref| <= tau * scale + floor`` everywhere
    (inf where the scale is 0 and the error exceeds the floor, or where w is not finite)."""
    err = np.abs(np.asarray(w, dtype=np.float64) - ref)
    ex = np.maximum(err - floor, 0.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(ex > 0, ex / scale, 0.0)
    ratio[~np.isfinite(err)] = np.inf
    if ratio.size == 0:
        return 0.0, -1
    i = int(np.argmax(ratio))
    return float(ratio[i]), i


def check_render(w, ref, scale, tau, floor, label, hop=None, branch=None):
    """Assert ``|w - ref| <= tau * scale + floor`` at every sample and ``w.shape == ref.shape``; returns
    the worst ratio (see :func:`worst_ratio`).  On failure the message names the worst sample, its block
    and offset in the block (``hop``) and the branch that rendered it (``branch``, from render_branch)."""
    w = np.asarray(w)
    assert w.shape == ref.shape, "%s: shape %s != reference %s" % (label, w.shape, ref.shape)
    worst, i = worst_ratio(w, ref, scale, floor)
    if not worst <= tau:
        where = "sample %d" % i
        if hop:
            where += " (block %d, offset %d of %d)" % (i // hop, i % hop, hop)
        msg = "%s: |w - ref| = %.3e at %s, scale %.3e: ratio %.3e > tau %.1e" % (
            label, abs(float(w[i]) - float(ref[i])), where, scale[i], worst, tau)
        if branch is not None:
            msg += "; branch: " + branch_label(branch)
        nbad = int(np.sum(~(np.abs(w - ref) <= tau * scale + floor)))
        raise AssertionError(msg + "; %d samples out of bound" % nbad)
    return worst
