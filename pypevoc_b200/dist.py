"""Segment sharding of one long signal over the GPUs of a box (SURVEY section 8e).

One process per GPU (torchrun).  Rank g *owns* the contiguous, hop-aligned frame range
[j0, j1) and analyses a slightly larger *window* of frames [w0, w1) = [j0 - Lb, j1 + Lf):

  * analysis needs the previous frame's spectrum: one extra warm-up frame before w0
    (recomputed, not emitted), i.e. the rank reads samples [(w0-1)*hop, (w1-1)*hop + nfft);
  * the link of frame j to frame j-1 depends on those two peak rows only (SURVEY A5), so local
    tracking over the window rows reproduces the global links of every own row;
  * one block of resynthesised samples depends on a few neighbouring frames of each partial that
    sounds in it: Af + 1 frames back and one frame ahead for the body (PVAnalysis.py:701-736),
    ceil(dfr*edge) further frames for fade-in heads / fade-out tails of partials that start
    after / end before the block (:740-751), and `minframes` frames to know that a partial is
    rendered at all (:1061).  With Lb = dE + max(Af + 2, minframes) and Lf = dE + minframes + 2
    halo rows the partials cut by the window edges cannot influence an own block, so every rank
    renders its own block range [j0, j1) from LOCAL tables, bit-identical to the unsharded run.

Hence no collective runs on the hot path.  What has to be global is the numbering of the
partials (the reference numbers them in order of creation, PVAnalysis.py:819-830): every rank
contributes 2*K + 4 integers (the local ids in the row before its first own row and in its
last own row, and how many partials were born before / inside its own rows), one tiny
all_gather distributes them and each rank renames its own rows.  ONE all_gather over NVLink
then collects the track table (global ids of every frame, int32 [F, K]); first frame and length
of every partial follow from it (pvk_track_spans).  The peak tables stay sharded;
`ShardedSinSum.gather_tables()` collects them on request (second, optional collective).
"""
import os

import numpy as np
import torch

from . import pv as P


def halos(nfft, hop, edge=1.0, minframes=3):
    """(Lb, Lf): frame rows a rank needs before / after its own range to render its own blocks."""
    dfr = nfft / float(hop) / 2.
    Af = int(np.floor(dfr + 0.5))
    dE = int(np.ceil(dfr * edge))
    return dE + max(Af + 2, int(minframes)), dE + int(minframes) + 2


def plan_segments(nsamp_total, nfft, hop, world, edge=1.0, minframes=3):
    """Frame ranges and sample windows of every rank.  Keys: j0, j1 (own global frames), w0, w1
    (window = emitted rows), own0 (local row of j0), nown, sample0 / nsamp (window of the global
    signal the rank reads), frame0 (local index of the first emitted row), nframes (emitted
    rows), prev_zero, frames_total."""
    F = P.n_frames(nsamp_total, nfft, hop)
    Lb, Lf = halos(nfft, hop, edge, minframes)
    plans = []
    shard = F >= 4 * world          # too short to shard: rank 0 takes everything
    # equal shares of ceil(F / world) rows with a short LAST rank: the all_gather of the track table
    # then lands in frame order without a copy.  If that would leave a rank empty (F barely above
    # 4 * world) the rows are spread evenly instead (gather_track_table concatenates in that case).
    per = -(-F // world)
    equal = per * (world - 1) < F
    for g in range(world):
        if not shard:
            j0, j1 = (0, F) if g == 0 else (F, F)
        elif equal:
            j0, j1 = g * per, min((g + 1) * per, F)
        else:
            j0, j1 = (F * g) // world, (F * (g + 1)) // world
        if j1 <= j0:
            plans.append(dict(rank=g, j0=j0, j1=j1, w0=j0, w1=j0, own0=0, nown=0, sample0=0, nsamp=0, frame0=0,
                              nframes=0, prev_zero=True, frames_total=F))
            continue
        w0, w1 = max(0, j0 - Lb), min(F, j1 + Lf)
        if w0 == 0:
            s0, frame0, prev_zero = 0, 0, True
        else:
            s0, frame0, prev_zero = (w0 - 1) * hop, 1, False
        plans.append(dict(rank=g, j0=j0, j1=j1, w0=w0, w1=w1, own0=j0 - w0, nown=j1 - j0, sample0=s0,
                          nsamp=(w1 - 1) * hop + nfft - s0, frame0=frame0, nframes=w1 - w0, prev_zero=prev_zero,
                          frames_total=F))
    return plans


def clip_range(nclips, rank, world):
    """Clips [c0, c1) of a batch that rank ``rank`` analyses (SURVEY 8e, clip batches): independent
    units split evenly, no halo, no collective -- every rank runs a ``PVBatch`` on its slice."""
    return (nclips * rank) // world, (nclips * (rank + 1)) // world


# --------------------------------------------------------------------------- global numbering
def local_summary(tid_local, plan):
    """int32 [2K + 4]: local ids of the row before the first own row (-1 = none), local ids of the
    last own row, nb = partials born before the own rows, n_own = partials born in the own rows,
    global index of the last own row that holds a point (-1 = none), number of own rows.
    Local ids count partials in order of creation, so ids born in rows < r are exactly the ids
    below 1 + max(tid[:r])."""
    K = tid_local.shape[1]
    dev = tid_local.device
    own0, nown = plan["own0"], plan["nown"]
    out = torch.full((2 * K + 4,), -1, dtype=torch.int32, device=dev)
    if nown == 0 or tid_local.shape[0] == 0:
        out[2 * K:] = torch.tensor([0, 0, -1, 0], dtype=torch.int32, device=dev)
        return out
    if own0 > 0:
        out[:K] = tid_local[own0 - 1]
        nb = tid_local[:own0].max().clamp(min=-1) + 1
    else:
        nb = torch.zeros((), dtype=torch.int32, device=dev)
    own = tid_local[own0:own0 + nown]
    out[K:2 * K] = own[-1]
    nbo = torch.maximum(own.max().clamp(min=-1) + 1, nb)
    rows = torch.nonzero((own >= 0).any(dim=1)).flatten()
    last = (rows[-1] + plan["j0"]) if rows.numel() else torch.full((), -1, device=dev)
    out[2 * K] = nb
    out[2 * K + 1] = nbo - nb
    out[2 * K + 2] = last
    out[2 * K + 3] = nown
    return out


def resolve_ids(summ_all, K):
    """Sequential pass over the ranks' summaries (numpy int [world, 2K+4], host): returns
    (base[g], Gprev[g]) -- global id of the first partial born in rank g's own rows and global
    ids of the row before its first own row -- plus the total number of partials and the global
    index of the last frame that holds a point."""
    world = summ_all.shape[0]
    base, G = 0, np.full(K, -1, dtype=np.int64)
    bases, gprevs, max_end = [], [], -1
    for g in range(world):
        prev_tid, last_tid = summ_all[g, :K], summ_all[g, K:2 * K]
        nb, n_own, last_row, nown = (int(v) for v in summ_all[g, 2 * K:2 * K + 4])
        bases.append(base)
        gprevs.append(G.copy())
        if nown == 0:
            continue
        # global ids of this rank's last own row: born in the own rows -> base + rank of birth,
        # born before them -> the id the partial carries in the row before the first own row
        Gl = np.full(K, -1, dtype=np.int64)
        cols = np.flatnonzero(last_tid >= 0)
        if len(cols):
            L = last_tid[cols].astype(np.int64)
            newborn = L >= nb
            Gl[cols[newborn]] = base + (L[newborn] - nb)
            old = cols[~newborn]
            if len(old):
                inv = np.full(max(nb, 1), -1, dtype=np.int64)      # local id -> column in the previous row
                pc = np.flatnonzero(prev_tid >= 0)
                inv[prev_tid[pc]] = pc
                Gl[old] = G[inv[last_tid[old]]]
        G = Gl
        base += n_own
        max_end = max(max_end, last_row)
    return bases, gprevs, base, max_end


def global_ids(tid_local, plan, base, gprev, nb, n_own):
    """Global ids of the own rows (int32 [nown, K]) from the local ids of the window."""
    dev = tid_local.device
    own0, nown = plan["own0"], plan["nown"]
    own = tid_local[own0:own0 + nown].long()
    if nown == 0:
        return own.to(torch.int32)
    nt = max(int(nb + n_own), 1)
    gid = torch.full((nt,), -1, dtype=torch.int64, device=dev)
    if n_own > 0:
        gid[nb:nb + n_own] = base + torch.arange(n_own, device=dev)
    if own0 > 0 and nb > 0:
        prev = tid_local[own0 - 1].long()
        cols = torch.nonzero(prev >= 0).flatten()
        gid[prev[cols]] = torch.as_tensor(np.asarray(gprev), dtype=torch.int64, device=dev)[cols]
    return torch.where(own >= 0, gid[own.clamp(min=0, max=nt - 1)], torch.full_like(own, -1)).to(torch.int32)


def segment_summary_device(tid_local, plan):
    """pvk_segment_summary of this rank's window (CUDA int32 [2K + 4]); slot 2K+1 holds nb + n_own."""
    import ctypes as C
    from . import _lib
    L = _lib.lib()
    K = tid_local.shape[1]
    dev = tid_local.device
    with torch.cuda.device(dev):
        mine = torch.empty((2 * K + 4,), dtype=torch.int32, device=dev)
        _lib.check(L.pvk_segment_summary(C.c_void_p(tid_local.data_ptr()), K, plan["own0"], plan["nown"], plan["j0"],
                                         C.c_void_p(mine.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)),
                   "pvk_segment_summary")
    return mine


def segment_rename_device(tid_local, plan, world, allv, max_own0=None, sync=True):
    """pvk_segment_resolve + pvk_segment_rename: global ids of the own rows from the gathered
    summaries ``allv`` (CUDA int32 [world * (2K + 4)]).  One host read-back (8 ints) at the end;
    ``sync=False`` leaves it to the caller (``params`` int32 [8] on the device: slot 3 = total
    number of partials, slot 4 = global index of the last frame holding a point)."""
    import ctypes as C
    from . import _lib
    L = _lib.lib()
    K = tid_local.shape[1]
    dev = tid_local.device
    own0, nown, g = plan["own0"], plan["nown"], plan["rank"]
    ptr = lambda t: C.c_void_p(t.data_ptr())                                   # noqa: E731
    with torch.cuda.device(dev):
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        # the pass walks every segment: scratch must hold the back-halo ids of the largest one
        cap = max((own0 if max_own0 is None else max_own0) * K, 1)
        scratch = torch.empty((2, cap), dtype=torch.int32, device=dev)
        params = torch.zeros((8,), dtype=torch.int32, device=dev)
        _lib.check(L.pvk_segment_resolve(ptr(allv), world, K, g, ptr(scratch[0]), cap, ptr(scratch[1]), ptr(params),
                                         stream), "pvk_segment_resolve")
        own = tid_local[own0:own0 + nown]
        tid_own = torch.empty_like(own)
        _lib.check(L.pvk_segment_rename(ptr(own), own.numel(), ptr(scratch[1]), ptr(params), ptr(tid_own), stream),
                   "pvk_segment_rename")
        if not sync:
            return dict(tid_own=tid_own, params=params)
        ph = params.cpu().numpy()
    return dict(tid_own=tid_own, ntracks=int(ph[3]), max_end=int(ph[4]))


def segment_rename_push_device(tid_local, plan, world, allv, tables, max_own0=None):
    """pvk_segment_resolve + pvk_segment_rename_push: the renamed own rows are stored straight into
    every table of ``tables`` (int32 CUDA tensors [frames_total, K]: the local one and, in a
    multi-GPU run, the peers' tables mapped over NVLink) at this segment's row offset -- the gather
    of the track table as P2P stores of the kernel that computes the ids, no collective call.
    The caller owns the cross-rank barriers around it.  Returns ``params`` (device int32 [8], as
    segment_rename_device(sync=False))."""
    import ctypes as C
    from . import _lib
    L = _lib.lib()
    K = tid_local.shape[1]
    dev = tid_local.device
    own0, nown, g = plan["own0"], plan["nown"], plan["rank"]
    ptr = lambda t: C.c_void_p(t.data_ptr())                                   # noqa: E731
    with torch.cuda.device(dev):
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        cap = max((own0 if max_own0 is None else max_own0) * K, 1)
        scratch = torch.empty((2, cap), dtype=torch.int32, device=dev)
        params = torch.zeros((8,), dtype=torch.int32, device=dev)
        _lib.check(L.pvk_segment_resolve(ptr(allv), world, K, g, ptr(scratch[0]), cap, ptr(scratch[1]), ptr(params),
                                         stream), "pvk_segment_resolve")
        own = tid_local[own0:own0 + nown].contiguous()
        dst = torch.tensor([int(t.data_ptr()) for t in tables], dtype=torch.int64, device=dev)
        _lib.check(L.pvk_segment_rename_push(ptr(own), own.numel(), ptr(scratch[1]), ptr(params), ptr(dst), len(tables),
                                             plan["j0"] * K, stream), "pvk_segment_rename_push")
        # keep the operands alive until the stream has consumed them
        params._pvk_keep = (own, dst, scratch)
    return params


def _stitch_device(tid_local, plan, plans, group):
    """stitch() for CUDA tables: summary / resolve / rename run as three small libpvk kernels."""
    import torch.distributed as dist
    world = len(plans)
    tid_local = tid_local.contiguous()
    mine = segment_summary_device(tid_local, plan)
    if world > 1:
        allv = torch.empty((world * mine.numel(),), dtype=torch.int32, device=mine.device)
        dist.all_gather_into_tensor(allv, mine, group=group)
    else:
        allv = mine
    return segment_rename_device(tid_local, plan, world, allv, max(p["own0"] for p in plans))


def stitch(tid_local, plan, plans, group=None):
    """Global numbering of this rank's own rows: one tiny all_gather (2K + 4 ints per rank) and a
    sequential pass over the ranks.  Returns dict(tid_own int32 [nown, K] global ids, ntracks
    (total), max_end (global index of the last frame with a point)).  CUDA tables take the libpvk
    kernels; CPU tensors (gloo tests) the equivalent torch / numpy statement below."""
    if tid_local.is_cuda:
        return _stitch_device(tid_local, plan, plans, group)
    import torch.distributed as dist
    world = len(plans)
    K = tid_local.shape[1]
    mine = local_summary(tid_local, plan)
    if world > 1:
        flat = torch.empty((world * mine.numel(),), dtype=torch.int32, device=mine.device)
        dist.all_gather_into_tensor(flat, mine, group=group)
        allv = flat.view(world, mine.numel())
    else:
        allv = mine.unsqueeze(0)
    summ = allv.cpu().numpy()
    bases, gprevs, ntot, max_end = resolve_ids(summ, K)
    g = plan["rank"]
    tid_own = global_ids(tid_local, plan, bases[g], gprevs[g], int(summ[g, 2 * K]), int(summ[g, 2 * K + 1]))
    return dict(tid_own=tid_own, ntracks=ntot, max_end=max_end)


_STITCH_STREAMS = {}
_PEER_TABLES = {}            # (device, world, rows, K) -> symmetric-memory track tables (PVK_PEER_GATHER=1)


def _peer_gather_wanted(world):
    """PVK_PEER_GATHER=1 / 0 forces the fused rename + peer-store gather / the NCCL all_gather.  Unset:
    chosen by measurement (profiles/r2u_*, r2w_*: B200 x 2 / x 8, NVSwitch): equal within noise on 2 GPUs
    (1.375 vs 1.393 ms per step), NCCL -- which uses the switch's multicast itself -- 4 % ahead on 8
    (1.441 vs 1.499 ms), so the peer-store kernel is the default up to 4 ranks and NCCL beyond."""
    v = os.environ.get("PVK_PEER_GATHER")
    if v is not None:
        return v != "0"
    return world <= 4


def _stitch_stream(dev):
    """The side stream the numbering + gather run on (one per device; not the copy streams of
    pv._side_streams: the collectives must not queue behind table downloads)."""
    key = (dev.type, dev.index)
    if key not in _STITCH_STREAMS:
        # high priority: its kernels are tiny (summary, resolve, rename + stores, barriers, the collective's
        # copy CTAs) and must not queue behind the thousands of CTAs of the rendering kernel they overlap
        _STITCH_STREAMS[key] = torch.cuda.Stream(device=dev, priority=-1)
    return _STITCH_STREAMS[key]


class StitchHandle(object):
    """Global numbering and THE all_gather of the track table, launched on a side stream so that
    neither the collectives nor their host-side launch cost sit on the hot path: packing and
    resynthesis of the rank's own blocks use LOCAL ids and run meanwhile on the main stream.
    ``counts()`` is the one host read-back (8 ints); ``table()`` joins the streams."""

    def __init__(self, tid_local, plan, plans, group=None):
        import torch.distributed as dist
        self.plans, self.plan = plans, plan
        world = len(plans)
        dev = tid_local.device
        self.dev = dev
        cur = torch.cuda.current_stream(dev)
        self.side = _stitch_stream(dev)
        self.side.wait_stream(cur)
        tid_local = tid_local.contiguous()
        tid_local.record_stream(self.side)
        self._counts = None
        self._joined = False
        with torch.cuda.stream(self.side):
            mine = segment_summary_device(tid_local, plan)
            if world > 1:
                allv = torch.empty((world * mine.numel(),), dtype=torch.int32, device=dev)
                dist.all_gather_into_tensor(allv, mine, group=group)
            else:
                allv = mine
            self.peer_used = False
            self.multicast_used = False
            if world > 1 and _peer_gather_wanted(world) and self._peer_gather(tid_local, allv, group):
                return
            r = segment_rename_device(tid_local, plan, world, allv, max(p["own0"] for p in plans), sync=False)
            self._tid_own, self._params = r["tid_own"], r["params"]
            _, finish = gather_track_table(self._tid_own, plans, group, async_op=False)
            self._table = finish()                        # queued behind the gather on the side stream

    def _peer_gather(self, tid_local, allv, group):
        """(Default up to 4 ranks, see _peer_gather_wanted.)  Rename fused with the gather --
        pvk_segment_rename_push stores the renamed rows straight into the track tables of all ranks,
        which are symmetric-memory buffers mapped over NVLink; two signal-pad barriers replace the
        NCCL all_gather (verified bit for bit against the unsharded run on 2 GPUs, profiles/r2a_*).  Two buffers alternate, so a returned table stays valid until the second
        next call.  Returns False (and the NCCL path runs) if symmetric memory cannot be set up or the
        plan is not the equal-share one."""
        import sys
        import torch.distributed as dist
        plans, plan = self.plans, self.plan
        world = len(plans)
        K = tid_local.shape[1]
        rows_max = max(p["nown"] for p in plans)
        F = sum(p["nown"] for p in plans)
        if any(p["nown"] and p["j0"] != p["rank"] * rows_max for p in plans):
            return False
        try:
            key = (self.dev.index, world, rows_max, K)
            ent = _PEER_TABLES.get(key)
            if ent is None:
                import torch.distributed._symmetric_memory as sm
                grp = group if group is not None else dist.group.WORLD
                bufs = [sm.empty(world * rows_max * K, dtype=torch.int32, device=self.dev) for _ in range(2)]
                ent = dict(bufs=bufs, hdls=[sm.rendezvous(b, grp) for b in bufs], turn=0)
                _PEER_TABLES[key] = ent
            i = ent["turn"]
            ent["turn"] = 1 - i
            buf, hdl = ent["bufs"][i], ent["hdls"][i]
            hdl.barrier()                                 # every rank is done with this buffer's previous content
            import ctypes as C
            from . import _lib
            L = _lib.lib()
            own0, nown, g = plan["own0"], plan["nown"], plan["rank"]
            cap = max(max(p["own0"] for p in plans) * K, 1)
            scratch = torch.empty((2, cap), dtype=torch.int32, device=self.dev)
            params = torch.zeros((8,), dtype=torch.int32, device=self.dev)
            ptr = lambda t: C.c_void_p(t.data_ptr())                           # noqa: E731
            stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            _lib.check(L.pvk_segment_resolve(ptr(allv), world, K, g, ptr(scratch[0]), cap, ptr(scratch[1]), ptr(params),
                                             stream), "pvk_segment_resolve")
            own = tid_local[own0:own0 + nown].contiguous()
            mc = 0
            if os.environ.get("PVK_PEER_MULTICAST", "1") != "0":
                try:
                    mc = int(hdl.multicast_ptr or 0)                # 0: no multicast object behind this buffer
                except Exception:
                    mc = 0
            if mc:
                # ONE store per 16 bytes, replicated into every rank's table by the NVSwitch
                _lib.check(L.pvk_segment_rename_mcast(ptr(own), own.numel(), ptr(scratch[1]), ptr(params),
                                                      C.c_void_p(mc), plan["j0"] * K, stream), "pvk_segment_rename_mcast")
            else:
                _lib.check(L.pvk_segment_rename_push(ptr(own), own.numel(), ptr(scratch[1]), ptr(params),
                                                     C.c_void_p(int(hdl.buffer_ptrs_dev)), world, plan["j0"] * K, stream),
                           "pvk_segment_rename_push")
            self.multicast_used = bool(mc)
            hdl.barrier()                                 # all ranks' stores have landed
            table = buf.view(world * rows_max, K)[:F]
            self._keep = (own, scratch)
            self._params = params
            self._table = table
            self._tid_own = table[plan["j0"]:plan["j0"] + nown]
            self.peer_used = True
            return True
        except Exception as e:                            # no symmetric memory here: the NCCL path runs
            if not _PEER_TABLES.get("warned"):
                _PEER_TABLES["warned"] = True
                sys.stderr.write("pypevoc_b200: the peer-memory gather is unavailable (%r); "
                                 "using the NCCL all_gather\n" % (e,))
            return False

    def join_before_render(self):
        """PVK_GATHER_JOIN=pack: make the current stream wait for the numbering + gather before the
        rendering kernels are queued on it.  Default ("end"): the gather runs beside the rendering on the
        high-priority stitch stream and is joined when the table is needed -- measured on 8 GPUs
        (profiles/r2w_*): 1.44 - 1.50 ms per step against 1.58 with the early join."""
        if os.environ.get("PVK_GATHER_JOIN", "end") != "end":
            torch.cuda.current_stream(self.dev).wait_stream(self.side)

    def counts(self):
        """(total number of partials, global index of the last frame holding a point)."""
        if self._counts is None:
            with torch.cuda.stream(self.side):
                ph = self._params.cpu().numpy()          # synchronises the side stream only
            self._counts = (int(ph[3]), int(ph[4]))
        return self._counts

    def _join(self):
        cur = torch.cuda.current_stream(self.dev)
        cur.wait_stream(self.side)
        return cur

    @property
    def tid_own(self):
        cur = self._join()
        if not self.peer_used:                            # (symmetric-memory buffers are not the caching allocator's)
            self._tid_own.record_stream(cur)
        return self._tid_own

    def table_on_side(self):
        """The gathered table for work queued on the stitch stream itself (``with
        torch.cuda.stream(handle.side)``): no join, the consumer runs beside the main stream's kernels."""
        return self._table

    def table(self):
        """int32 [F, K] global ids of every frame (the main stream waits for the gather)."""
        if not self._joined:
            cur = self._join()
            if not self.peer_used:
                self._table.record_stream(cur)
            self._joined = True
        return self._table


def render_range_local(plan, plans, local_last, hop, nfft, hop_an, edge=1.0):
    """render_range() without knowing the GLOBAL last frame: ``local_last`` is the global index of
    the last frame holding a point inside this rank's window (-1 = none).  The rank owning the
    last frames sees the signal's last point in its window whenever its range is not empty (the
    back halo is longer than the fade-out), so its range equals render_range(); every other rank
    renders its whole own range [j0, j1) -- samples at or beyond the true output length are
    simply dropped afterwards (trim_local), rendering them is harmless.  Returns (b0, b1, bound)
    with ``bound`` = the sample count stores are clipped at."""
    if plan["nown"] == 0:
        return 0, 0, 0
    last = max(p["rank"] for p in plans if p["nown"] > 0)
    if plan["rank"] != last:
        return plan["j0"], plan["j1"], plan["j1"] * hop
    if local_last < 0:
        return 0, 0, 0
    nout, _ = P.synth_geometry(local_last, hop, nfft, hop_an, edge)
    nblk = -(-nout // hop)
    return min(plan["j0"], nblk), nblk, nout


def trim_local(n_rendered, b0, plan, plans, max_end, hop, nfft, hop_an, edge=1.0):
    """Samples of a render_range_local() rendering that belong to the output signal, once the
    global ``max_end`` is known: (count, first global sample) exactly as render_range() has them."""
    g0, g1, nout = render_range(plan, plans, max_end, hop, nfft, hop_an, edge)
    n = max(min(g1 * hop, nout) - g0 * hop, 0)
    if n == 0:
        return 0, g0 * hop
    assert g0 == b0 and n <= n_rendered, (g0, b0, n, n_rendered)
    return n, g0 * hop


def gather_track_table(tid_own, plans, group=None, async_op=False):
    """THE all_gather of the track table: global ids of every frame, int32 [F, K], on every rank.
    Returns (work handle or None, finish()) -- finish() waits and returns the table."""
    import torch.distributed as dist
    world = len(plans)
    K = tid_own.shape[1]
    rows_max = max(p["nown"] for p in plans)
    if world == 1:
        return None, (lambda: tid_own)
    if tid_own.shape[0] == rows_max and tid_own.is_contiguous():
        mine = tid_own
    else:
        mine = torch.full((rows_max, K), -1, dtype=torch.int32, device=tid_own.device)
        mine[:tid_own.shape[0]] = tid_own
    flat1 = torch.empty((world * rows_max * K,), dtype=torch.int32, device=tid_own.device)
    work = dist.all_gather_into_tensor(flat1, mine.view(-1), group=group, async_op=async_op)
    flat = flat1.view(world, rows_max, K)
    F = sum(p["nown"] for p in plans)
    # plan_segments gives every rank but the last non-empty one rows_max rows: the gathered buffer
    # is then the table itself (plus padding at the end)
    in_order = all(p["nown"] == rows_max or all(q["nown"] == 0 for q in plans[i + 1:]) for i, p in enumerate(plans))

    def finish():
        if work is not None:
            work.wait()
        if in_order:
            return flat1.view(world * rows_max, K)[:F]
        return torch.cat([flat[g, :plans[g]["nown"]] for g in range(world)]).contiguous()
    return work, finish


def gather_rows(t_own, plans, group=None):
    """all_gather of one sharded per-frame table (own rows of every rank, any dtype) -> [F, ...]."""
    import torch.distributed as dist
    world = len(plans)
    if world == 1:
        return t_own
    rows_max = max(p["nown"] for p in plans)
    mine = torch.zeros((rows_max,) + tuple(t_own.shape[1:]), dtype=t_own.dtype, device=t_own.device)
    mine[:t_own.shape[0]] = t_own
    flat1 = torch.empty((world * mine.numel(),), dtype=t_own.dtype, device=t_own.device)
    dist.all_gather_into_tensor(flat1, mine.contiguous().view(-1), group=group)
    flat = flat1.view((world,) + tuple(mine.shape))
    return torch.cat([flat[g, :plans[g]["nown"]] for g in range(world)]).contiguous()


def render_range(plan, plans, max_end, hop, nfft, hop_an, edge=1.0):
    """Blocks this rank renders, in global and local (window row) coordinates, and the length of
    the whole signal: own blocks [j0, j1), clipped to the signal; the rank owning the last frames
    also renders the blocks after them.  Returns (b0, b1, nout_total)."""
    nout, _ = P.synth_geometry(max_end, hop, nfft, hop_an, edge)
    if max_end < 0:
        return 0, 0, 0
    nblk = -(-nout // hop)
    last = max(p["rank"] for p in plans if p["nown"] > 0)
    b0 = min(plan["j0"], nblk)
    b1 = nblk if plan["rank"] == last else min(plan["j1"], nblk)
    if plan["nown"] == 0:
        b0 = b1 = 0
    return b0, b1, nout


def resynth_local(tid_local, pk_local, plan, plans, max_end, sr, hop, nfft, hop_an, edge=1.0, minframes=3,
                  out=None, ws=None, block_range=None, reuse_tracks=False, local_last=None, **mode):
    """Render this rank's block range (or the sub-range ``block_range`` of it, global block
    indices) from its LOCAL tables: float64 device tensor holding global samples
    [b0*hop, min(b1*hop, nout)).  ``local_last`` (instead of the global ``max_end``): the range
    of render_range_local(), to be cut with trim_local() once ``max_end`` is known.  ``mode``:
    phase_preserve / fscale / phase_ws / scanned of resynth_device (integrated phase: after
    integrated_phase_local)."""
    if local_last is not None:
        b0, b1, nout = render_range_local(plan, plans, local_last, hop, nfft, hop_an, edge)
    else:
        b0, b1, nout = render_range(plan, plans, max_end, hop, nfft, hop_an, edge)
    if block_range is not None:
        b0, b1 = block_range
    if b1 <= b0:
        return torch.zeros((0,), dtype=torch.float64, device=tid_local.device)
    w0 = plan["w0"]
    nout_local = nout - w0 * hop                       # same signal, local sample origin w0*hop
    return P.resynth_device(tid_local, pk_local, sr, hop, nfft, hop_an, edge=edge, minframes=minframes,
                            block0=b0 - w0, nblocks=b1 - b0, nout=nout_local, out=out, ws=ws,
                            reuse_tracks=reuse_tracks, **mode)


def track_pack_resynth_local(tab, plan, plans, sr, hop, nfft, hop_an, edge=1.0, minframes=3, maxpitchjmp=0.5,
                             after_link=None, after_pack=None, before_sync=None, formant=None):
    """Back half of the path for one rank's window, queued without a host round trip
    (pv.track_pack_resynth_device): link, pack and the rendering of the rank's block range.  No count
    is needed to know the range: every rank but the one owning the last frames renders its own blocks
    [j0, j1); the last one renders up to the bound its window allows (its last window row as "last
    frame") -- cut with trim_local() once the global last frame is known.  ``tab``: device tables f mag
    ph realph [window rows, K].  ``formant``: the formant ratio q of the window rows (pv.formant_ratio(),
    float or pv._DeviceCurve).  Returns (tr, pk, w, b0): w holds global samples [b0*hop, ...)."""
    w1 = plan["w1"]
    b0, b1, bound = render_range_local(plan, plans, (w1 - 1) if plan["nown"] > 0 else -1, hop, nfft, hop_an, edge)
    w0 = plan["w0"]
    rng = (b0 - w0, max(b1 - b0, 0), max(bound - w0 * hop, 0))
    tr, pk, w = P.track_pack_resynth_device(tab["f"], tab["mag"], tab["ph"], tab["realph"], sr, hop, nfft, hop_an, edge=edge,
                                            minframes=minframes, maxpitchjmp=maxpitchjmp, after_link=after_link,
                                            after_pack=after_pack, block_range=rng, before_sync=before_sync,
                                            formant=formant)
    if w is None:
        w = torch.zeros((0,), dtype=torch.float64, device=tab["f"].device)
    return tr, pk, w, b0


# --------------------------------------------------------------------------- integrated phase
def handover_rows(plan, plans, nfft, hop, edge=1.0):
    """(h_lo, h_hi): local rows of this rank's hand-over row h(g) = j0 - dE and of the next rank's,
    h(g+1) (-1: none).  h(g) = w0 + max(Af + 2, minframes) is where the local advances stop reading
    frames clamped at the cut w0 (the first Af + 1 advances of a cut partial do), and no P an own block
    reads lies before it: bodies start at j0, tails read the last row of partials ending at or after
    j0 - dE.  A window starting at frame 0 cuts nothing: h_lo = -1, the local scan is exact."""
    if plan["nframes"] == 0:
        return -1, -1
    dE = int(np.ceil(nfft / float(hop) / 2. * edge))
    w0, g = plan["w0"], plan["rank"]
    lo = plan["j0"] - dE - w0 if w0 > 0 else -1
    nxt = plans[g + 1] if g + 1 < len(plans) else None
    hi = nxt["j0"] - dE - w0 if nxt is not None and nxt["nframes"] > 0 and nxt["w0"] > 0 else -1
    return lo, hi


def _pk_args(pk):
    return pk["tstart"], pk["tlen"], pk["toff"], int(pk["tstart"].shape[0])


def handover_scan_device(tid_local, pk, plan, plans, sr, hop, nfft, hop_an, fscale, ws, phase_ws, edge=1.0):
    """pvk_resynth_scan of this rank's window partials (block start phases into ``phase_ws``, local
    Nyquist flags into ``ws``) + its hand-over record, CUDA int64 [2K] -- gathered over the ranks by
    the caller (all_gather, world x 2K).  ``fscale``: a float, or a pv._DeviceCurve of the window rows
    (pvk_resynth_scan_curve)."""
    import ctypes as C
    from . import _lib
    L = _lib.lib()
    F, K = tid_local.shape
    tstart, tlen, toff, nt = _pk_args(pk)
    lo, hi = handover_rows(plan, plans, nfft, hop_an, edge)
    dev = tid_local.device
    with torch.cuda.device(dev):
        rec = torch.empty((2 * K,), dtype=torch.int64, device=dev)
        if isinstance(fscale, P._DeviceCurve):
            fn, ratio = L.pvk_resynth_scan_curve, (1.0, P._ptr(fscale.t), int(fscale.t.numel()))
        else:
            fn, ratio = L.pvk_resynth_scan, (float(fscale),)
        _lib.check(fn(P._ptr(tid_local), F, K, nt, P._ptr(tstart), P._ptr(tlen), P._ptr(toff), P._ptr(pk["pf"]),
                      P._ptr(pk["prealph"]), float(sr), int(hop), int(nfft), int(hop_an), *ratio, P._ptr(ws),
                      int(ws.numel()), P._ptr(phase_ws), int(phase_ws.numel()), lo, hi, P._ptr(rec), rec.numel(),
                      P._stream()), "pvk_resynth_scan")
    return rec


def handover_apply_device(tid_local, pk, plan, plans, recs, nfft, hop_an, ws, phase_ws, edge=1.0):
    """pvk_resynth_handover: the true block start phases of the partials alive at this rank's hand-over
    row, from the records of all ranks ``recs`` (CUDA int64 [world * 2K])."""
    from . import _lib
    L = _lib.lib()
    F, K = tid_local.shape
    tstart, tlen, toff, nt = _pk_args(pk)
    lo, _ = handover_rows(plan, plans, nfft, hop_an, edge)
    with torch.cuda.device(tid_local.device):
        _lib.check(L.pvk_resynth_handover(P._ptr(tid_local), F, K, nt, P._ptr(tstart), P._ptr(tlen), P._ptr(toff),
                                          P._ptr(phase_ws), int(phase_ws.numel()), P._ptr(recs), recs.numel(),
                                          len(plans), plan["rank"], lo, P._ptr(ws), int(ws.numel()), P._stream()),
                   "pvk_resynth_handover")


def nyquist_flags_device(f_own, tid_own, ntracks, sr, fscale):
    """uint8 CUDA [ntracks]: 1 for the global partials with a point of this rank's own rows at
    fscale * f >= sr / 2.  The own rows partition the frames, so the element-wise max over the ranks
    (all_reduce MAX, by the caller) is the unsharded Nyquist rule.  ``fscale``: a float, or a
    pv._DeviceCurve of the own rows (each point tested at its row's ratio)."""
    from . import _lib
    L = _lib.lib()
    dev = tid_own.device
    flags = torch.zeros((max(int(ntracks), 1),), dtype=torch.uint8, device=dev)
    f_own = f_own.contiguous()
    tid_own = tid_own.contiguous()
    with torch.cuda.device(dev):
        if isinstance(fscale, P._DeviceCurve):
            _lib.check(L.pvk_nyquist_flags_curve(P._ptr(f_own), P._ptr(tid_own), tid_own.numel(), float(sr), 1.0,
                                                 P._ptr(fscale.t), int(fscale.t.numel()), int(tid_own.shape[1]),
                                                 P._ptr(flags), int(ntracks), P._stream()), "pvk_nyquist_flags_curve")
        else:
            _lib.check(L.pvk_nyquist_flags(P._ptr(f_own), P._ptr(tid_own), tid_own.numel(), float(sr), float(fscale),
                                           P._ptr(flags), int(ntracks), P._stream()), "pvk_nyquist_flags")
    return flags


def nyquist_import_device(tid_local, pk, plan, table, flags, ntracks, ws):
    """pvk_resynth_import_flags: the global flags of this rank's window partials into ``ws`` (where the
    render reads them), through the global track table ``table`` (CUDA int32 [F, K])."""
    from . import _lib
    L = _lib.lib()
    F, K = tid_local.shape
    tstart, _, _, nt = _pk_args(pk)
    with torch.cuda.device(tid_local.device):
        _lib.check(L.pvk_resynth_import_flags(P._ptr(tid_local), F, K, nt, P._ptr(tstart), P._ptr(table),
                                              int(table.shape[0]), plan["w0"], P._ptr(flags), int(ntracks), P._ptr(ws),
                                              int(ws.numel()), P._stream()), "pvk_resynth_import_flags")


def integrated_phase_local(tid_local, pk, f_local, plan, plans, tid_own, table, ntracks, sr, hop, nfft, hop_an, fscale,
                           ws, phase_ws, edge=1.0, group=None):
    """Scan, hand-over and Nyquist flags of one rank (phase_preserve=False): afterwards ``ws`` and
    ``phase_ws`` hold what the unsharded scan would give for every partial point an own block reads, and
    resynth_device(..., scanned=True) renders the own blocks.  COLLECTIVE: one all_gather of world x 2K
    int64 records and one all_reduce(MAX) of ntracks bytes.  ``fscale``: a float, or a pv._DeviceCurve
    of the window rows [w0, w1) (the flags take its own-row part)."""
    import torch.distributed as dist
    world = len(plans)
    rec = handover_scan_device(tid_local, pk, plan, plans, sr, hop, nfft, hop_an, fscale, ws, phase_ws, edge)
    if world > 1:
        recs = torch.empty((world * rec.numel(),), dtype=torch.int64, device=rec.device)
        dist.all_gather_into_tensor(recs, rec, group=group)
    else:
        recs = rec
    handover_apply_device(tid_local, pk, plan, plans, recs, nfft, hop_an, ws, phase_ws, edge)
    o0, n = plan["own0"], plan["nown"]
    own = P._DeviceCurve(fscale.t[o0:o0 + n]) if isinstance(fscale, P._DeviceCurve) else fscale
    flags = nyquist_flags_device(f_local[o0:o0 + n], tid_own, ntracks, sr, own)
    if world > 1:
        dist.all_reduce(flags, op=dist.ReduceOp.MAX, group=group)
    nyquist_import_device(tid_local, pk, plan, table, flags, ntracks, ws)


# --------------------------------------------------------------------------- host API
class ShardedSinSum(object):
    """Result of ShardedPV.toSinSum(): the global track table on every rank + this rank's local
    partials (window rows, local ids) for resynthesis."""

    def __init__(self, spv, local_ss, handle=None):
        self._spv = spv
        self.local = local_ss
        self._handle = handle                # StitchHandle: numbering + gather in flight on a side stream
        self._spans = None
        self._first = None                   # (w, b0) rendered together with the first link / pack
        self.sr, self.nfft, self.hop = spv.sr, spv.nfft, spv.hop

    def _hook(self, tr):
        self._handle = StitchHandle(tr["tid"], self._spv.plan, self._spv.plans, self._spv.group)

    @property
    def _h(self):
        """The stitch handle; created right behind the link kernels the first time the partials are
        needed (by synth_local together with pack + rendering, or by any accessor)."""
        if self._handle is None:
            ss = self.local
            ss._after_link = self._hook
            try:
                tr = ss._ensure_tracks()                             # link -> [numbering + gather] -> pack -> counts
            finally:
                ss._after_link = None
            if self._handle is None:                                 # (no frames on this rank: nothing was launched)
                self._handle = StitchHandle(tr["tid"], self._spv.plan, self._spv.plans, self._spv.group)
        return self._handle

    @property
    def ntracks(self):
        """Total number of partials of the whole signal (host read-back of the numbering pass)."""
        return self._h.counts()[0]

    @property
    def max_end(self):
        """Global index of the last frame holding a point."""
        return self._h.counts()[1]

    @property
    def tid_own(self):
        """int32 CUDA tensor [nown, K]: global ids of this rank's own rows."""
        return self._h.tid_own

    @property
    def device_track_table(self):
        """int32 CUDA tensor [F, K]: global partial id of every peak slot of every frame."""
        return self._h.table()

    @property
    def track_ids(self):
        return self.device_track_table.cpu().numpy()

    def device_spans(self):
        """(tstart, tlen) int32 CUDA tensors [ntracks]: first frame and length of every partial."""
        if self._spans is None:
            self._spans = P.spans_device(self.device_track_table, self.ntracks)
        return self._spans

    @property
    def st(self):
        return self.device_spans()[0].cpu().numpy().astype(np.int64).tolist()

    @property
    def end(self):
        s, n = self.device_spans()
        return (s.cpu().numpy().astype(np.int64) + n.cpu().numpy() - 1).tolist()

    def gather_tables(self, group=None):
        """Second, optional collective: collect the sharded peak tables and return an ordinary
        SinSum (identical on every rank) with the global numbering, e.g. to read ``partial[i]``."""
        spv = self._spv
        d = spv.pv.device_tables
        o0, n = spv.plan["own0"], spv.plan["nown"]
        glob = {k: gather_rows(d[k][o0:o0 + n], spv.plans, group) for k in ("f", "mag", "ph", "realph")}
        ss = P.SinSum(self.sr, nfft=self.nfft, hop=self.hop, device=spv.pv._dev)
        ss._set_device_tables(glob["f"], glob["mag"], glob["ph"], glob["realph"])
        ss._set_device_tracks(self.device_track_table, None, self.ntracks)
        return ss

    def synth_local(self, sr=None, hop=None, edge=1.0, minframes=3, hostbuf=None, chunks=8, to_host=False,
                    phase_preserve=True, fscale=1.0, formant_shift=None):
        """Render this rank's own block range of the resynthesised signal (the last rank also renders
        the tail): global samples [b0*hop, ...).  Returns (signal, first global sample).  ``hostbuf``:
        render in ``chunks`` ranges and download each into pinned ``hostbuf['w']`` meanwhile.
        ``phase_preserve`` / ``fscale`` as in SinSum.synth: with ``phase_preserve=False`` the ranks hand
        the integrated phases of the partials crossing their boundaries on to each other and agree on the
        Nyquist rule (integrated_phase_local: one all_gather of world x 2K int64 and one all_reduce of
        ntracks bytes), so the concatenated own signals equal the unsharded render bit for bit.
        COLLECTIVE in that mode: every rank makes the same call.  ``fscale`` may be a curve over the
        GLOBAL frames, ``[frames_total]`` (see pv.synth_mode()); each rank uses its window's rows.  It is
        checked on every rank before anything is launched.  ``formant_shift`` as in SinSum.synth (a curve over
        the global frames, too): a row's formant gains depend on that row's points only, all of which are
        in the window, so this needs no collective of its own."""
        spv = self._spv
        nf = spv.plans[0]["frames_total"]
        phase_preserve, fscale = P.synth_mode(phase_preserve, fscale, nframes=nf)
        formant = P.formant_ratio(phase_preserve, fscale, formant_shift, nframes=nf)
        win = slice(spv.plan["w0"], spv.plan["w1"])
        if isinstance(fscale, np.ndarray):
            fscale = P._on_device(np.ascontiguousarray(fscale[win]), spv.pv._dev)
        if isinstance(formant, np.ndarray):
            formant = P._on_device(np.ascontiguousarray(formant[win]), spv.pv._dev)
        sr = spv.sr if sr is None else sr
        hop = spv.hop if hop is None else int(hop)
        if (edge, minframes) != (spv.edge, spv.minframes):
            raise ValueError("the segment halos were planned for edge=%r, minframes=%r" % (spv.edge, spv.minframes))
        if (phase_preserve and self._handle is None and hostbuf is None and self.local._trk is None
                and spv.plan["nframes"] > 0):
            # first use: link, numbering + gather (side stream), pack and rendering are queued back to back;
            # the counts are read once at the end
            t = self.local._tables
            tr, pk, w, b0 = track_pack_resynth_local(t, spv.plan, spv.plans, sr, hop, self.nfft, self.hop, edge, minframes,
                                                     maxpitchjmp=self.local._maxpitchjmp, after_link=self._hook,
                                                     after_pack=lambda tr_: self._handle.join_before_render(),
                                                     formant=formant)
            self.local._trk = tr
            if pk is not None:
                self.local._pk = pk
            n, s0 = trim_local(w.numel(), b0, spv.plan, spv.plans, self.max_end, hop, self.nfft, self.hop, edge)
            w = w[:n]
            return (w.cpu().numpy() if to_host else w), s0
        self._h                                                      # (numbering + gather go out before the pack)
        pk = self.local._ensure_packed()
        tidl = self.local._trk["tid"]
        # block range from LOCAL knowledge (the numbering / gather may still be in flight); the
        # few samples beyond the true output length are cut below, once max_end is known
        ll = self.local._trk.get("max_end", -1)
        ll = ll + spv.plan["w0"] if ll is not None and ll >= 0 else -1
        args = (spv.plan, spv.plans)
        b0, b1, bound = render_range_local(spv.plan, spv.plans, ll, hop, self.nfft, self.hop, edge)
        n_local = max(min(b1 * hop, bound) - b0 * hop, 0)
        dev = tidl.device
        nblk = b1 - b0
        chunks = max(1, min(chunks, nblk // 64 if nblk >= 64 else 1)) if hostbuf is not None else 1
        F, K = tidl.shape
        ws, mode = None, {}
        if not phase_preserve:
            # scan -> hand-over -> flags -> render: the hand-over needs the gathered track table and the
            # global partial count, so the integrated-phase render starts behind them
            ws = P.resynth_workspace(F, K, int(pk["tstart"].shape[0]), max(-(-nblk // chunks), 1), dev, hop=hop)
            pws = P._phase_ws(False, pk["pf"].numel(), dev)
            integrated_phase_local(tidl, pk, self.local._tables["f"], spv.plan, spv.plans, self.tid_own,
                                   self.device_track_table, self.ntracks, sr, hop, self.nfft, self.hop, fscale, ws, pws,
                                   edge, spv.group)
            mode = dict(phase_preserve=False, fscale=fscale, phase_ws=pws, scanned=True)
        if formant is not None:
            mode["pmag"] = P._formant_gains(formant, tidl, int(pk["tstart"].shape[0]), None, pk["tstart"], pk["toff"],
                                            pk["pf"], pk["pmag"], pk["pf"].numel())
        if hostbuf is None:
            w = resynth_local(tidl, pk, *args, None, sr, hop, self.nfft, self.hop, edge, minframes, ws=ws,
                              local_last=ll, **mode)
            n, s0 = trim_local(w.numel(), b0, *args, self.max_end, hop, self.nfft, self.hop, edge)
            w = w[:n]
            return (w.cpu().numpy() if to_host else w), s0
        cur = torch.cuda.current_stream(dev)
        _, d2h = P._side_streams(dev)
        with torch.cuda.device(dev):
            out = torch.empty((n_local,), dtype=torch.float64, device=dev)
            hw = P._pinned(hostbuf, "w", (n_local,), torch.float64)
            d2h.wait_stream(cur)
            if ws is None and nblk:
                ws = P.resynth_workspace(F, K, int(pk["tstart"].shape[0]), -(-nblk // chunks), dev)
            for i in range(chunks if nblk else 0):
                c0, c1 = b0 + (nblk * i) // chunks, b0 + (nblk * (i + 1)) // chunks
                n0, n1 = (c0 - b0) * hop, min((c1 - b0) * hop, n_local)
                resynth_local(tidl, pk, *args, None, sr, hop, self.nfft, self.hop, edge, minframes, out=out[n0:n1],
                              ws=ws, block_range=(c0, c1), reuse_tracks=i > 0, local_last=ll, **mode)
                ev = torch.cuda.Event()
                ev.record(cur)
                with torch.cuda.stream(d2h):
                    d2h.wait_event(ev)
                    hw[n0:n1].copy_(out[n0:n1], non_blocking=True)
            d2h.synchronize()
        n, s0 = trim_local(n_local, b0, *args, self.max_end, hop, self.nfft, self.hop, edge)
        self.d2h_bytes = n_local * 8
        self._last_out = out
        return hw[:n].numpy(), s0


class ShardedPV(object):
    """PV over one long signal sharded across the ranks of a torch.distributed job.

    Every rank constructs it with ITS window of the signal (``plan['sample0']`` ..
    ``+plan['nsamp']``; see :func:`plan_segments`), host or device.  ``run_pv`` analyses the
    rank's window rows, ``toSinSum`` links them locally, makes the numbering global and gathers
    the track table (the one all_gather), ``ShardedSinSum.synth_local`` renders the rank's own
    block range of the output signal from local data.
    """

    def __init__(self, x_local, sr, nsamp_total, nfft=1024, hop=None, npks=20, pkthresh=0.005, wind=np.hanning,
                 rank=None, world=None, device=None, edge=1.0, minframes=3, group=None):
        import torch.distributed as dist
        self.rank = dist.get_rank() if rank is None else rank
        self.world = dist.get_world_size() if world is None else world
        hop = int(nfft / 2) if hop is None else int(hop)
        self.edge, self.minframes, self.group = edge, minframes, group
        self.plans = plan_segments(nsamp_total, nfft, hop, self.world, edge, minframes)
        self.plan = self.plans[self.rank]
        self.pv = P.PV(x_local, sr, nfft=nfft, hop=hop, npks=npks, pkthresh=pkthresh, wind=wind, progress=False,
                       device=device)
        if self.pv.nsamp != self.plan["nsamp"]:
            raise ValueError("rank %d expects %d samples starting at global sample %d, got %d" % (
                self.rank, self.plan["nsamp"], self.plan["sample0"], self.pv.nsamp))
        self.sr, self.nfft, self.hop = sr, nfft, hop

    def run_pv(self, hostbuf=None, chunks=8, stream_tables=None):
        """Analyse this rank's window rows [w0, w1) (own rows: ``own_rows``).  ``hostbuf``: stream the
        tables (``stream_tables``: which of them) into pinned host memory as in PV.run_pv."""
        p, pv = self.plan, self.pv
        pv._hostbuf = None
        pv._d2h_event = None
        if hostbuf is not None and p["nframes"] > 0:
            pv._run_pv_streamed(hostbuf, int(chunks), 0, frame_lo=p["frame0"], nframes=p["nframes"],
                                prev_zero=p["prev_zero"], stream_tables=stream_tables)
        else:
            pv._devout = P.analyze_device(pv._xd, pv.sr, pv.nfft, pv.hop, pv.npeaks, pv.peakthresh, pv._tb,
                                          frame0=p["frame0"], nframes=p["nframes"], prev_zero=p["prev_zero"])
        pv.nframes = p["nframes"]
        pv._host = {}
        pv._host["t"] = ((np.arange(pv.nframes) + p["w0"]) * pv.hop + pv.nfft / 2.0) / pv.sr

    @property
    def own_rows(self):
        """slice of the window rows (pv.f etc.) this rank owns."""
        return slice(self.plan["own0"], self.plan["own0"] + self.plan["nown"])

    def toSinSum(self, async_gather=True):
        """Local linking + global numbering + the gather of the track table.  Nothing is launched
        here: the work is queued the first time the result is used -- by ``synth_local`` in one go with
        packing and rendering (one host read-back at the end), or by any accessor.  COLLECTIVE: every
        rank must make the same first use (the numbering all_gather and the table gather need all ranks)."""
        d = self.pv.device_tables
        ss = P.SinSum(self.sr, nfft=self.nfft, hop=self.hop, device=self.pv._dev)
        ss._set_device_tables(d["f"], d["mag"], d["ph"], d["realph"])
        return ShardedSinSum(self, ss)
