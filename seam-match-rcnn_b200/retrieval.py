"""Retrieval front-ends over the engine: single-GPU search, the gallery-sharded multi-GPU
search (one process per GPU; the exchange is done by the kernels themselves over NVLink peer
memory, an NCCL all-gather path is kept for stacks without symmetric memory), and the
evaluation-script outputs (rank of the true shop item, top-k hit counts).

The reference scores one query at a time on the CPU (evaluate_movingfashion.py:157-277,
evaluate_multiDF2.py:209-230); here all queries go through one fused pass.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist

from .engine import PreparedGallery, SeamEngine

K_THRESHOLDS = (1, 5, 10, 20)       # evaluate_movingfashion.py:15


# ----------------------------------------------------------------------------------------
# partitioning (pure host logic, exercised on CPU with gloo in tests/)
# ----------------------------------------------------------------------------------------
def shard_bounds(n: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous balanced split of n rows over `world` ranks: [lo, hi) of `rank`."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError("bad world/rank")
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def all_gather_rows(x: torch.Tensor, group=None) -> torch.Tensor:
    """All-gather tensors that differ in their first dimension (padded to the maximum)."""
    world = dist.get_world_size(group)
    n = torch.tensor([x.shape[0]], device=x.device, dtype=torch.int64)
    ns = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(ns, n, group=group)
    sizes = [int(v) for v in ns]
    m = max(sizes)
    pad = x
    if x.shape[0] < m:
        pad = torch.cat([x, x.new_zeros((m - x.shape[0],) + tuple(x.shape[1:]))], 0)
    outs = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(outs, pad.contiguous(), group=group)
    return torch.cat([o[:s] for o, s in zip(outs, sizes)], 0)


# ----------------------------------------------------------------------------------------
# host placement
# ----------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(device) -> Optional[int]:
    """Pin this process to the CPUs of the NUMA node the GPU hangs off (Linux sysfs), so that the pinned host
    buffers it allocates afterwards are first-touched on that node: on a two-socket 8-GPU box a rank whose buffers
    live on the other socket moves its tracks over the inter-socket link and gets a fraction of its PCIe bandwidth.
    Returns the node, or None when it cannot be determined (nothing is changed then).  Call it before allocating
    pinned memory; one process per GPU."""
    import os
    try:
        dev = torch.device(device)
        idx = dev.index if dev.index is not None else torch.cuda.current_device()
        bus = torch.cuda.get_device_properties(idx).pci_bus_id if hasattr(torch.cuda.get_device_properties(idx), "pci_bus_id") else None
        if bus is None:
            import pynvml
            pynvml.nvmlInit()
            bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(idx)).busId
            bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:                      # NVML prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return node
    except Exception:                                        # noqa: BLE001 -- placement is an optimisation, never an error
        return None


# ----------------------------------------------------------------------------------------
# single GPU
# ----------------------------------------------------------------------------------------
def search(engine: SeamEngine, seq: torch.Tensor, mask: Optional[torch.Tensor], gallery, k: int = 20):
    """aggregation -> scorer -> top-k for all tracks.  Returns (scores, margins, idx int32)."""
    if not isinstance(gallery, PreparedGallery):
        gallery = engine.prepare_gallery(gallery)
    return engine.search(seq, mask, gallery, k)[1:]


# ----------------------------------------------------------------------------------------
# from HOST memory (the reference's eval keeps every feature in host memory between the detector
# and the scorer, evaluate_movingfashion.py:45-92, and moves one product's frames to the device per
# query, :253-262)
# ----------------------------------------------------------------------------------------
class HostTrackStream:
    """Streams a host ``x3_1_seq (1+Tmax, Q, 256)`` / ``x3_1_mask (Q, 1+Tmax)`` pair to the device in
    ``nchunk`` slices of tracks on a private copy stream and aggregates each slice as soon as it has
    landed, so that the PCIe transfer of slice i+1 overlaps the kernels of slice i.  Only the frame rows
    1..Tmax cross the bus: row 0 is the layout's dummy (models/match_head.py:101-111) and is never read.
    Pinned host tensors make the copies asynchronous; pageable ones work but serialise."""

    def __init__(self, engine: SeamEngine, nchunk: int = 4):
        self.engine = engine
        self.nchunk = int(nchunk)
        self.copy_stream = torch.cuda.Stream(device=engine.device)

    def h2d_bytes(self, seq_h: torch.Tensor, mask_h: Optional[torch.Tensor]) -> int:
        n = (seq_h.shape[0] - 1) * seq_h.shape[1] * seq_h.shape[2] * seq_h.element_size()
        return n + (mask_h.numel() * mask_h.element_size() if mask_h is not None else 0)

    def uploads(self, seq_h: torch.Tensor, mask_h: Optional[torch.Tensor]):
        """Yields (lo, hi, tracks (1+Tmax, hi-lo, 256), mask or None) per slice, in order, usable on the current
        stream: all copies are enqueued on the copy stream first, the current stream waits for each slice's event."""
        eng, dev = self.engine, self.engine.device
        Q = seq_h.shape[1]
        main = torch.cuda.current_stream(dev)
        self.copy_stream.wait_stream(main)
        staged = []
        with torch.cuda.stream(self.copy_stream):
            for c in range(self.nchunk):
                lo, hi = shard_bounds(Q, self.nchunk, c)
                if hi == lo:
                    continue
                s_d = eng.upload_tracks(seq_h, lo, hi)               # one pitched copy of rows 1..Tmax
                m_d = mask_h[lo:hi].to(dev, non_blocking=True) if mask_h is not None else None
                ev = torch.cuda.Event()
                ev.record(self.copy_stream)
                staged.append((lo, hi, s_d, m_d, ev))
        for lo, hi, s_d, m_d, ev in staged:
            main.wait_event(ev)
            s_d.record_stream(main)
            if m_d is not None:
                m_d.record_stream(main)
            yield lo, hi, s_d, m_d

    def chunks(self, seq_h: torch.Tensor, mask_h: Optional[torch.Tensor]):
        """Yields (lo, hi, descriptors (hi-lo,256) on the device) per slice, in order, on the current stream."""
        for lo, hi, s_d, m_d in self.uploads(seq_h, mask_h):
            yield lo, hi, self.engine.aggregate(s_d, m_d)


def search_host(engine: SeamEngine, seq_h: torch.Tensor, mask_h: Optional[torch.Tensor], gallery_h: torch.Tensor,
                k: int = 20, out: Optional[Sequence[torch.Tensor]] = None, stream: Optional[HostTrackStream] = None,
                index_offset: int = 0):
    """Host tensors in, host tensors out: gallery upload + preparation, chunked track upload overlapped
    with aggregation and scoring, results copied back per chunk into ``out`` (three (Q,k) host tensors:
    scores fp32, margins fp32, idx int32; allocated pinned when not given).  Returns ``out``; the caller
    synchronises the current stream before reading it."""
    dev = engine.device
    stream = stream or HostTrackStream(engine)
    Q = seq_h.shape[1]
    if out is None:
        out = [torch.empty((Q, k), dtype=dt).pin_memory() for dt in (torch.float32, torch.float32, torch.int32)]
    main = torch.cuda.current_stream(dev)
    stream.copy_stream.wait_stream(main)
    with torch.cuda.stream(stream.copy_stream):
        g_d = gallery_h.to(dev, non_blocking=True)
        ev_g = torch.cuda.Event()
        ev_g.record(stream.copy_stream)
    main.wait_event(ev_g)
    g_d.record_stream(main)
    gallery = engine.prepare_gallery(g_d, index_offset=index_offset)
    for lo, hi, q_c in stream.chunks(seq_h, mask_h):
        res = engine.score_topk(q_c, gallery, k)
        for dst, src in zip(out, res):
            dst[lo:hi].copy_(src, non_blocking=True)
    return out


# ----------------------------------------------------------------------------------------
# gallery-sharded multi-GPU search
# ----------------------------------------------------------------------------------------
class ShardedRetriever:
    """Each rank holds a contiguous slice of the gallery (prepared once) and scores every
    query against it; queries are aggregated in slices and all-gathered; the per-rank
    (Q,k) candidate lists are all-gathered and merged.  `ops` is the compute provider -- a
    SeamEngine in production; tests inject a CPU stand-in to exercise the collective logic
    with gloo.
    """

    def __init__(self, ops, gallery_shard: torch.Tensor, shard_offset: int, group=None, world: Optional[int] = None,
                 rank: Optional[int] = None):
        self.ops = ops
        self.group = group
        self.world = world if world is not None else (dist.get_world_size(group) if dist.is_initialized() else 1)
        self.rank = rank if rank is not None else (dist.get_rank(group) if dist.is_initialized() else 0)
        self.gallery = (gallery_shard if isinstance(gallery_shard, PreparedGallery)
                        else ops.prepare_gallery(gallery_shard, index_offset=shard_offset))
        self.shard_offset = shard_offset
        self.shard_rows = gallery_shard.G if isinstance(gallery_shard, PreparedGallery) else gallery_shard.shape[0]
        self._gallery_rows: Optional[int] = None     # rows of the whole gallery, found on first use

    @classmethod
    def from_full_gallery(cls, ops, gallery: torch.Tensor, group=None):
        world = dist.get_world_size(group) if dist.is_initialized() else 1
        rank = dist.get_rank(group) if dist.is_initialized() else 0
        lo, hi = shard_bounds(gallery.shape[0], world, rank)
        return cls(ops, gallery[lo:hi], lo, group)

    def aggregate(self, seq: torch.Tensor, mask: Optional[torch.Tensor]) -> torch.Tensor:
        """Every rank aggregates Q/N tracks; the (Q/N,256) results are all-gathered."""
        Q = seq.shape[1]
        if self.world == 1:
            return self.ops.aggregate(seq, mask)
        lo, hi = shard_bounds(Q, self.world, self.rank)
        part = self.ops.aggregate(seq[:, lo:hi], None if mask is None else mask[lo:hi])
        return all_gather_rows(part, self.group)

    def search_descriptors(self, q: torch.Tensor, k: int):
        sc, mg, ix = self.ops.score_topk(q, self.gallery, k)
        if self.world == 1:
            return sc, mg, ix
        packs = []
        for t in (sc, mg, ix):
            outs = [torch.empty_like(t) for _ in range(self.world)]
            dist.all_gather(outs, t.contiguous(), group=self.group)
            packs.append(torch.stack(outs, 0))
        return self.ops.merge_topk(packs[0], packs[1], packs[2])

    def search(self, seq: torch.Tensor, mask: Optional[torch.Tensor], k: int = 20):
        return self.search_descriptors(self.aggregate(seq, mask), k)

    def gallery_rows(self, device) -> int:
        """Rows of the whole gallery (the end of the last shard): one MAX all-reduce on first use."""
        if self._gallery_rows is None:
            end = self.shard_offset + self.shard_rows
            if self.world > 1:
                t = torch.tensor([end], dtype=torch.int64, device=device)
                dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
                end = int(t)
            self._gallery_rows = end
        return self._gallery_rows

    def rank_of_target(self, q: torch.Tensor, target: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """Rank (0 = best) of the global gallery row ``target[i]`` for every query over the whole sharded gallery,
        and its margin: ``(rank int32 (Q,), margin fp32 (Q,))``, the same integers and bits as ``rank_of_target`` on
        the unsharded gallery (evaluate_movingfashion.py:268-269).  The shard holding the target computes its margin
        (``-inf`` on the others), a MAX all-reduce hands it to every shard, each counts the rows ranking before it
        (ties by global row) and a SUM all-reduce adds the counts.  ``q`` holds every query on every rank."""
        dev = self.gallery.g.device if isinstance(self.gallery, PreparedGallery) else q.device
        G = self.gallery_rows(dev)
        if q.shape[0] and (int(target.min()) < 0 or int(target.max()) >= G):
            raise ValueError(f"target index out of range [0, {G})")
        if self.world == 1:
            return self.ops.rank_of_target(q, self.gallery, target)
        Q = q.shape[0]
        if self.shard_rows == 0:          # nothing to compute here; the library takes no empty shard
            margin = torch.full((Q,), -float("inf"), dtype=torch.float32, device=dev)
        else:
            margin = self.ops.target_margin(q, self.gallery, target)
        dist.all_reduce(margin, op=dist.ReduceOp.MAX, group=self.group)
        if self.shard_rows == 0:
            rank = torch.zeros((Q,), dtype=torch.int32, device=dev)
        else:
            rank = self.ops.rank_count(q, self.gallery, target, margin)
        dist.all_reduce(rank, op=dist.ReduceOp.SUM, group=self.group)
        return rank, margin

    def evaluate_aggregated(self, seq, mask, target: torch.Tensor,
                            k_thresholds: Sequence[int] = K_THRESHOLDS) -> "RetrievalReport":
        """``evaluate_aggregated`` over the sharded gallery: the same ``RetrievalReport`` as the single-GPU function
        on the whole gallery, from the sharded aggregation, search and rank.  ``seq`` / ``mask`` hold all tracks."""
        q = self.aggregate(seq, mask)
        kmax = min(max(k_thresholds), 32)
        sc, _, ix = self.search_descriptors(q, kmax)
        ranks, _ = self.rank_of_target(q, target)
        return _report(ranks, k_thresholds, sc, ix)

    def search_peer(self, seq: torch.Tensor, mask: Optional[torch.Tensor], peer: "PeerExchange", lens=None):
        """Same result as ``search`` with the exchange done by the kernels themselves (``PeerExchange``): three
        library calls, no collective, no copy, no barrier -- capturable into one CUDA graph.  ``seq`` / ``mask`` hold
        ALL Q tracks (each rank aggregates the slice it owns); returns the complete ``(Q,k)`` result on every rank
        (views of the exchange's final buffers) or, for a non-replicating exchange, the owner's rows."""
        lo, hi = peer.q_lo[self.rank], peer.q_lo[self.rank + 1]
        self.ops.sharded_aggregate(peer, seq[:, lo:hi], None if mask is None else mask[lo:hi],
                                   None if lens is None else lens[lo:hi])
        self.ops.sharded_score_topk(peer, self.gallery)
        return self.ops.sharded_merge(peer)


# ----------------------------------------------------------------------------------------
# the exchange steps done by the kernels over NVLink peer memory (csrc/exchange.cuh)
# ----------------------------------------------------------------------------------------
def exchange_layout(Q: int, k: int, world: int):
    """Pure host logic of the sharded search: who owns which queries and how big the exchange buffers are.
    Rank r owns queries ``[q_lo[r], q_lo[r+1])`` (contiguous, balanced): it aggregates their tracks and merges their
    per-shard lists.  Returns a dict of ``q_lo`` (world+1 ints), ``own_max`` and the per-rank buffer shapes."""
    if world < 1 or world > 8:
        raise ValueError("the sharded search supports 1..8 ranks (one NVSwitch box)")
    bounds = [shard_bounds(Q, world, r) for r in range(world)]
    q_lo = [b[0] for b in bounds] + [Q]
    own_max = max(max(hi - lo for lo, hi in bounds), 1)
    return {"q_lo": q_lo, "own_max": own_max,
            "q_all": (2, max(Q, 1), 256), "lists": (2, world, own_max, k), "final": (max(Q, 1), k), "flags": (3 * 8,)}


class PeerExchange:
    """Buffers + descriptor (``struct seam_exchange``) of the gallery-sharded search.

    The two things that cross GPUs per step -- every rank's aggregated descriptors (everybody needs all Q) and the
    per-shard top-k lists (they meet at the rank that owns the query) -- plus the merged rows when every rank wants
    the complete result are STORED BY THE PRODUCING KERNELS straight into the consumers' memory: the buffers are
    symmetric memory (``torch.distributed._symmetric_memory``: every peer's buffer is mapped into this process),
    the stores travel over NVLink / NVSwitch, and flag words written after the last store (release) and polled by
    the consuming kernel before its first load (acquire) order them.  Descriptor and list buffers are
    double-buffered by the parity of a device-side step counter, so there is no barrier anywhere in a step and the
    whole step replays as ONE CUDA graph without a host-side argument changing.

    ``world == 1`` (or ``local_peers``) uses plain device tensors -- the same kernels and protocol on one GPU."""

    def __init__(self, engine: SeamEngine, Q: int, k: int, group=None, replicate: bool = True, local_peers=None):
        from ._lib import SeamExchange
        self.engine = engine
        dev = engine.device
        self.Q, self.k, self.replicate = int(Q), int(k), bool(replicate)
        if local_peers is not None:                        # several "ranks" inside one process (protocol tests)
            self.world, self.rank = local_peers["world"], local_peers["rank"]
        elif group is None and not dist.is_initialized():
            self.world, self.rank = 1, 0
        else:
            self.group = group if group is not None else dist.group.WORLD
            self.world, self.rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        lay = exchange_layout(self.Q, self.k, self.world)
        self.q_lo, self.own_max = lay["q_lo"], lay["own_max"]
        names = ["q_all", "list_margin", "list_idx", "flags"] + (["final_score", "final_margin", "final_idx"] if replicate else [])
        shapes = {"q_all": lay["q_all"], "list_margin": lay["lists"], "list_idx": lay["lists"], "flags": lay["flags"],
                  "final_score": lay["final"], "final_margin": lay["final"], "final_idx": lay["final"]}
        dtypes = {"q_all": torch.float32, "list_margin": torch.float32, "list_idx": torch.int32, "flags": torch.int32,
                  "final_score": torch.float32, "final_margin": torch.float32, "final_idx": torch.int32}
        self._bufs, self._peers = {}, {}
        if local_peers is not None:
            shared = local_peers["shared"]                 # {rank: {name: tensor}} filled by every local rank
            mine = {n: torch.zeros(shapes[n], dtype=dtypes[n], device=dev) for n in names}
            shared[self.rank] = mine
            self._bufs = mine
            self._shared = shared
        elif self.world == 1:
            self._bufs = {n: torch.zeros(shapes[n], dtype=dtypes[n], device=dev) for n in names}
            self._peers = {n: [self._bufs[n]] for n in names}
        else:
            import torch.distributed._symmetric_memory as symm
            for n in names:
                t = symm.empty(shapes[n], dtype=dtypes[n], device=dev)
                t.zero_()
                h = symm.rendezvous(t, self.group)
                self._bufs[n] = t
                self._handle = h
                self._peers[n] = [t if r == self.rank else h.get_buffer(r, shapes[n], dtypes[n]) for r in range(self.world)]
                # multicast pays when a row has several destinations (N = 8: step -4 %); with one peer it only adds the
                # copy the switch reflects back (measured slower at N = 2)
                self._mc = getattr(self, "_mc", {})
                self._mc[n] = self._multicast_address(h, t) if self.world > 2 else 0
            torch.cuda.synchronize(dev)
            dist.barrier(self.group)                       # nobody signals into flags a peer has not zeroed yet
        self._step = torch.ones(1, dtype=torch.int32, device=dev)
        self._done = torch.zeros(4, dtype=torch.int32, device=dev)
        self.struct = SeamExchange()
        if local_peers is None:
            self._fill_struct()

    def _fill_struct(self):
        """(Re)build the C descriptor from the peer tensors (local-peer mode: once every rank has allocated)."""
        if hasattr(self, "_shared"):
            names = list(self._bufs)
            self._peers = {n: [self._shared[r][n] for r in range(self.world)] for n in names}
        x = self.struct
        x.world, x.rank, x.Q, x.k, x.own_max = self.world, self.rank, self.Q, self.k, self.own_max
        for i, v in enumerate(self.q_lo):
            x.q_lo[i] = v
        for n, tensors in self._peers.items():
            arr = getattr(x, n)
            for r, t in enumerate(tensors):
                arr[r] = t.data_ptr()
        x.step = self._step.data_ptr()
        x.done = self._done.data_ptr()
        mc = getattr(self, "_mc", {})
        x.q_all_mc = mc.get("q_all", 0) or None
        fin = [mc.get(n, 0) for n in ("final_score", "final_margin", "final_idx")]
        x.final_score_mc, x.final_margin_mc, x.final_idx_mc = fin if all(fin) else (None, None, None)

    @staticmethod
    def _multicast_address(handle, t: torch.Tensor) -> int:
        """Address of ``t`` in the NVSwitch multicast mapping of its symmetric allocation (0: none -- no NVLS on this
        box, or switched off with SEAM_NO_MULTICAST=1).  A store to it lands in every rank's copy of the tensor."""
        import os
        if os.environ.get("SEAM_NO_MULTICAST", "0") == "1":
            return 0
        try:
            base = int(handle.multicast_ptr)
            local = int(handle.buffer_ptrs[handle.rank])
        except Exception:                                    # noqa: BLE001 -- an optimisation, never an error
            return 0
        off = t.data_ptr() - local
        if base == 0 or off < 0 or off + t.numel() * t.element_size() > int(handle.buffer_size):
            return 0
        return base + off

    def device_barrier(self) -> None:
        """Enqueue a cross-rank barrier KERNEL on the current stream (symmetric-memory signal pads): every rank's
        stream passes it at the same moment.  Not part of the search (the kernels order themselves by flag words);
        measurements use it so that a step timed on the device does not include the host's launch skew between ranks."""
        h = getattr(self, "_handle", None)
        if h is not None:
            h.barrier(channel=0)

    @property
    def multicast(self) -> bool:
        """Whether the descriptors travel by NVSwitch multicast (one store per row instead of world - 1)."""
        return bool(getattr(self, "_mc", {}).get("q_all", 0))

    @property
    def final(self):
        """(scores, margins, idx): this rank's copy of the complete (Q,k) result of the last finished step."""
        return self._bufs["final_score"], self._bufs["final_margin"], self._bufs["final_idx"]

    def descriptors(self) -> torch.Tensor:
        """Both parity halves of this rank's (Q,256) descriptor buffer (diagnostics / tests)."""
        return self._bufs["q_all"]

    @property
    def steps_done(self) -> int:
        return int(self._step.item()) - 1


# ----------------------------------------------------------------------------------------
# evaluation-script outputs
# ----------------------------------------------------------------------------------------
@dataclass
class RetrievalReport:
    """What evaluate_movingfashion.py:268-277, 360-367 derives from the aggregated-descriptor
    ranking: per-query rank of the true shop item and the top-k accuracies."""
    ranks: torch.Tensor                 # (Q,) int32, 0 = best
    hits: List[int]                     # k_accs_aggr_desc
    accuracies: List[float]             # hits / Q
    topk_scores: torch.Tensor
    topk_idx: torch.Tensor


def evaluate_aggregated(engine: SeamEngine, seq, mask, gallery: torch.Tensor, target: torch.Tensor,
                        k_thresholds: Sequence[int] = K_THRESHOLDS) -> RetrievalReport:
    """The "AGGR DESC" block of the eval loop for all products at once.

    Per product the reference aggregates the track (evaluate_movingfashion.py:253-262), scores
    it against every shop descriptor (:263-267), argsorts (:268), reads the rank of the true
    shop item (:269) and counts hits for k in k_thresholds (:270-277).
    """
    q = engine.aggregate(seq, mask)
    gal = engine.prepare_gallery(gallery)
    kmax = min(max(k_thresholds), 32)
    sc, mg, ix = engine.score_topk(q, gal, kmax)
    ranks, _ = engine.rank_of_target(q, gal, target)
    return _report(ranks, k_thresholds, sc, ix)


def _report(ranks: torch.Tensor, k_thresholds: Sequence[int], sc: torch.Tensor, ix: torch.Tensor) -> RetrievalReport:
    r = ranks.cpu()
    hits = [int((r < k).sum()) for k in k_thresholds]
    n = max(1, ranks.shape[0])
    return RetrievalReport(ranks=ranks, hits=hits, accuracies=[h / n for h in hits], topk_scores=sc, topk_idx=ix)


@dataclass
class ProductReport:
    """The four accuracy rows the eval script writes to its CSV (evaluate_movingfashion.py:435-443, in per
    cent) and its return values (:340, :351, :356), plus the per-frame rank statistics (:425-429)."""
    perf: torch.Tensor                  # (4, len(k_thresholds)) float32, per cent: per frame / best frame of the
                                        # product / average descriptor / aggregated descriptor
    ret: Tuple[float, float, float]     # (ret1, ret2, ret3) = top-1 of rows 0, 2, 3 as fractions
    frame_ranks: torch.Tensor           # (N,) int32
    product_ranks: torch.Tensor         # (3, P) int32: best frame, average descriptor, aggregated descriptor
    rank_median: float
    rank_q1: float
    rank_q3: float


def evaluate_products(engine: SeamEngine, frame_desc: torch.Tensor, frame_product: torch.Tensor,
                      shop_desc: torch.Tensor, target: torch.Tensor, frame_last: Tuple[torch.Tensor, torch.Tensor],
                      seq: torch.Tensor, mask: Optional[torch.Tensor], shop_aggr: torch.Tensor,
                      aggr_last: Tuple[torch.Tensor, torch.Tensor],
                      k_thresholds: Sequence[int] = K_THRESHOLDS) -> ProductReport:
    """The per-product loop of the eval script (evaluate_movingfashion.py:157-330) for all products at once,
    for the variants that rank with a single descriptor per query:

    row 0  every tracked frame box on its own: ``compute_ranking`` (:95-100) with ``match_predictor.last``
           (``frame_last`` = the ``w, b`` the detector emits, models/video_matchrcnn.py:297-314), hits :223-232;
    row 1  the product's best frame ("Product Max", :233-241): minimum of its frames' ranks;
    row 2  the average of the product's frame descriptors (:279-292), same scorer;
    row 3  the aggregated descriptor (:252-277) with ``temporal_aggregator.last`` (``aggr_last``).

    ``frame_desc (N,256)`` are the match features of the tracked boxes, ``frame_product (N,)`` the product
    (0..P-1) each belongs to, ``shop_desc (G,256)`` / ``shop_aggr (G,256)`` the shop boxes' match features
    and aggregator descriptors, ``target (P,)`` each product's shop row; ``seq`` / ``mask`` the aggregator
    input of the P tracks.  Ranks come from ``seam_rank_of_target_prepared`` (tensor-core count + fp32 verdicts near the target), i.e.
    the position the reference reads out of its full argsort, without sorting.  The reference runs rows 0-2 in
    numpy fp16 (:82-100); these are the fp32 values of the same formulas (SURVEY.md section 0, fact 5).
    The average / maximum *distance* fusions (:294-316) reduce a (frames x gallery) score matrix per product
    and are not covered here."""
    dev = engine.device
    frame_desc = frame_desc.to(dev, torch.float32)
    fp = frame_product.to(dev, torch.int64)
    target = target.to(dev, torch.int64)
    P = int(target.shape[0])
    ks = list(k_thresholds)

    big = torch.iinfo(torch.int32).max
    with engine.scorer(*frame_last):                     # the caller's scorer is put back on exit
        shop = engine.prepare_gallery(shop_desc)         # operands depend on the scorer just loaded
        fr, _ = engine.rank_of_target(frame_desc, shop, target[fp])
        best = torch.full((P,), big, dtype=torch.int32, device=dev).scatter_reduce(0, fp, fr, "amin")
        cnt = torch.zeros((P,), dtype=torch.float32, device=dev).index_add_(0, fp, torch.ones_like(fr, dtype=torch.float32))
        avg = torch.zeros((P, frame_desc.shape[1]), dtype=torch.float32, device=dev).index_add_(0, fp, frame_desc)
        has = cnt > 0
        avg = avg / cnt.clamp(min=1.0)[:, None]
        ar, _ = engine.rank_of_target(avg, shop, target)
        ar = torch.where(has, ar, torch.full_like(ar, big))

    with engine.scorer(*aggr_last):
        rep = evaluate_aggregated(engine, seq, mask, shop_aggr, target, ks)

    def row(r, n):
        return [float((r < k).sum()) / max(1, n) for k in ks]

    n_frames = int(fr.shape[0])
    perf = torch.tensor([row(fr, n_frames), row(best, P), row(ar, P), row(rep.ranks, P)], dtype=torch.float32) * 100.0
    frf = fr.float()
    qs = torch.quantile(frf, torch.tensor([0.25, 0.5, 0.75], device=dev)) if n_frames else torch.zeros(3)
    return ProductReport(perf=perf, ret=(perf[0, 0].item() / 100.0, perf[2, 0].item() / 100.0, perf[3, 0].item() / 100.0),
                         frame_ranks=fr, product_ranks=torch.stack([best, ar, rep.ranks.to(torch.int32)]),
                         rank_median=float(qs[1]), rank_q1=float(qs[0]), rank_q3=float(qs[2]))


def evaluate_distance_fusions(engine: SeamEngine, frame_desc: torch.Tensor, frame_product: torch.Tensor,
                              shop_desc: torch.Tensor, target: torch.Tensor,
                              frame_last: Tuple[torch.Tensor, torch.Tensor],
                              k_thresholds: Sequence[int] = K_THRESHOLDS, max_pairs: Optional[int] = None):
    """The "Avg Dist" / "Max Dist" rows of the eval printout (evaluate_movingfashion.py:294-316): per product
    the (frames x gallery) matrix of class-1 probabilities is averaged / maximised over the product's frames
    and the true shop item's position in the descending order is read off.

    One fused kernel for all products (``seam_rank_fused_distances``): the (frames x gallery) matrix is never
    materialised, nothing synchronises with the host (the frames are grouped by product with a device sort, the
    hit counts are device reductions).  Returns ``(ranks (2,P) int64 [avg, max], hits (2, len(k_thresholds))
    int64)``; products without frames get rank G; ties rank by lower index first, like ``seam_rank_of_target``.
    ``max_pairs`` is accepted for compatibility and ignored."""
    dev = engine.device
    frame_desc = frame_desc.to(dev, torch.float32)
    fp = frame_product.to(dev, torch.int64)
    shop = shop_desc.to(dev, torch.float32).contiguous()
    P = int(target.shape[0])
    order = torch.argsort(fp, stable=True)
    counts = torch.bincount(fp, minlength=P)[:P]
    start = torch.zeros(P + 1, dtype=torch.int64, device=dev)
    start[1:] = torch.cumsum(counts, 0)
    frames = frame_desc.index_select(0, order).contiguous()
    with engine.scorer(*frame_last):                         # the caller's scorer is put back on exit
        ra, rm = engine.rank_fused_distances(frames, start, shop, target)
    ranks = torch.stack([ra, rm]).to(torch.int64)
    ks = torch.tensor(list(k_thresholds), device=dev)
    hits = (ranks[:, :, None] < ks[None, None, :]).sum(1)
    return ranks, hits


def self_distances(engine: SeamEngine, street_desc: torch.Tensor, frame_last: Tuple[torch.Tensor, torch.Tensor]):
    """``compute_selfdist`` of the eval script (evaluate_movingfashion.py:115-121): the street x street matrix of
    class-1 probabilities its tracker thresholds (:165-214), for the boxes of one frame group at a time
    (n <= a few hundred: a dense (n,n) fp32 matrix, fp32 values of the script's fp16 formula)."""
    x = street_desc.to(engine.device, torch.float32).contiguous()
    with engine.scorer(*frame_last):
        return engine.score_prob(x, x)
