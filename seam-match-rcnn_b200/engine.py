"""Thin torch-facing wrapper over the C ABI: one ``SeamEngine`` per CUDA device.

PyTorch is used for device memory, streams and tensor plumbing only; all arithmetic of
the hot path runs in the hand-written kernels behind ``libseam_b200.so``.
"""
from __future__ import annotations

import contextlib
import ctypes as C
from dataclasses import dataclass
from typing import Dict, Mapping, Optional, Tuple

import torch

from . import _lib
from ._lib import SeamError, SeamWeightGrads, SeamWeights, WEIGHT_KEYS

D_MODEL = 256
# shapes of the reference's hot-path parameters (TemporalAggregationNLB().state_dict(), SURVEY.md section 8(b))
WEIGHT_SHAPES = {
    "theta_w": (128, 256, 1), "theta_b": (128,), "phi_w": (128, 256, 1), "phi_b": (128,),
    "g_w": (128, 256, 1), "g_b": (128,), "W_w": (256, 128, 1), "W_b": (256,),
    "concat_w": (1, 256, 1, 1), "att_w": (1, 256), "att_b": (1,), "last_w": (2, 256), "last_b": (2,),
}
SCORE_WS_LIMIT = 2 << 30      # bytes of scorer workspace above which score_topk works through the queries in slabs
# gallery row dtype -> suffix of the C entry points that read such rows (fp16 rows are g16 itself; bf16 rows have an
# fp16 image g16 beside them and take the fp32 entries' parameters)
ROW_SUFFIX = {torch.float32: "", torch.float16: "_g16", torch.bfloat16: "_gbf16"}


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


@dataclass
class PreparedGallery:
    """A gallery shard resident on the device with its tensor-core operands.

    g    (G,256) fp32   the shop descriptors (x3_2 of models/match_head.py:131/156), or fp16 / bf16 when the
                        caller's gallery has that dtype: then it is the caller's tensor (or one contiguous copy of it)
    g16  (G,256) fp16   operand of the tcgen05 pass -- the same tensor as ``g`` for an fp16 gallery
    cg   (G)     fp32   dw . g_j^2
    gstat (4)    fp32   [max_j ||g_j||, fp16-overflow flag, max_j |dw| . g_j^2, max_j (|W0| + |W1|) . g_j^2]: the last
                        two bound the fp32 rounding of cg and of the direct form in the certificate

    Bytes per row: fp32 1,540 (g, g16, cg), fp16 516 (g16, cg), bf16 1,028 (g, g16, cg).  All three score the same:
    16-bit rows are widened exactly wherever the fp32 direct form reads them, and a bf16 gallery's g16 is the one its
    fp32 widening would get (a bf16 value need not be an fp16 one, so bf16 rows cannot be the operand themselves).
    """
    g: torch.Tensor
    g16: torch.Tensor
    cg: torch.Tensor
    gstat: torch.Tensor
    index_offset: int = 0
    scorer_epoch: int = -1      # the engine's scorer epoch cg / g16 were prepared under (cg = dw . g^2 depends on `last`)

    @property
    def G(self) -> int:
        return self.g.shape[0]

    @property
    def rows_f16(self) -> bool:
        """The gallery rows are fp16 (``g is g16``): scored through the ``_g16`` entry points."""
        return self.g.dtype == torch.float16

    @property
    def rows_bf16(self) -> bool:
        """The gallery rows are bf16 (with a separate fp16 ``g16``): scored through the ``_gbf16`` entry points."""
        return self.g.dtype == torch.bfloat16

    @property
    def row_suffix(self) -> str:
        """Suffix of the C entry points that score this gallery: ``""``, ``"_g16"`` or ``"_gbf16"``."""
        return ROW_SUFFIX[self.g.dtype]


class SeamEngine:
    """Owns a ``seam_handle`` (folded weights) for one device."""

    def __init__(self, device="cuda:0"):
        device = torch.device(device)
        if device.type != "cuda":
            raise SeamError(2, f"SeamEngine needs a CUDA device, got {device}; there is no CPU path")
        if not torch.cuda.is_available():
            raise SeamError(3, "no CUDA device is visible; the SEAM hot path has no CPU fallback")
        self.device = torch.device("cuda", device.index if device.index is not None else torch.cuda.current_device())
        self._lib = _lib.load()
        h = C.c_void_p()
        rc = self._lib.seam_create(C.byref(h), self.device.index)
        if rc != 0:
            raise SeamError(rc, self._lib.seam_last_error(None).decode())
        self._h = h
        self._ws: Dict[str, torch.Tensor] = {}
        self._weights_key = None
        self._weight_refs = None
        self._last = None            # (last.weight, last.bias) currently folded into the handle
        self.weights_epoch = 0       # bumped by every load_weights / load_scorer
        self.scorer_epoch = 0        # bumped whenever `last` is (re)loaded: prepared galleries are tied to it

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                self._lib.seam_destroy(h)
            except Exception:
                pass
            self._h = None

    # ------------------------------------------------------------------ helpers
    def _check(self, rc: int) -> None:
        if rc != 0:
            raise SeamError(rc, self._lib.seam_last_error(self._h).decode())

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _workspace(self, name: str, nbytes: int) -> torch.Tensor:
        t = self._ws.get(name)
        if t is None or t.numel() < nbytes:
            t = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=self.device)
            self._ws[name] = t
        return t

    def _f32(self, t: torch.Tensor, name: str) -> torch.Tensor:
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"{name} must be a torch.Tensor")
        if t.device != self.device or t.dtype != torch.float32 or not t.is_contiguous():
            t = t.to(device=self.device, dtype=torch.float32).contiguous()
        return t

    def device_stamp(self, stamps: torch.Tensor, index: int) -> None:
        """Enqueue a one-thread kernel that writes the device's nanosecond timer into ``stamps[index]`` (int64, on this
        device) -- graph-capturable: timing between the nodes of a replayed graph (``seam_device_stamp``)."""
        assert stamps.dtype == torch.int64 and stamps.device == self.device
        self._check(self._lib.seam_device_stamp(self._h, stamps.data_ptr() + 8 * int(index), self._stream()))

    def watchdog_records(self):
        """Records left by device-side wait watchdogs (empty in normal operation): a list of
        ``{tag, block, thread, barrier, parity}``; readable even after a failed launch."""
        buf = (C.c_uint32 * (8 * 31))()
        n = int(self._lib.seam_watchdog_read(self._h, buf, 31))
        return [dict(tag=int(buf[8 * i]), block=int(buf[8 * i + 1]), thread=int(buf[8 * i + 2]),
                     barrier=int(buf[8 * i + 3]), parity=int(buf[8 * i + 4])) for i in range(n)]

    @property
    def launch_count(self) -> int:
        return int(self._lib.seam_launch_count(self._h))

    def profile(self, enable: bool) -> None:
        """Bracket the library's kernels with CUDA events (for bench.py's roofline)."""
        self._check(self._lib.seam_profile_enable(self._h, 1 if enable else 0))

    def profile_read(self) -> Dict[str, Tuple[float, int]]:
        """{kernel: (total_ms, launches)} of everything recorded since the last read."""
        out = {}
        for name, kid in _lib.KERNELS.items():
            ms, n = C.c_double(), C.c_int()
            self._check(self._lib.seam_profile_read(self._h, kid, C.byref(ms), C.byref(n)))
            out[name] = (ms.value, n.value)
        return out

    # ------------------------------------------------------------------ weights
    def load_weights(self, state: Mapping[str, torch.Tensor], prefix: str = "") -> None:
        """Upload + fold the hot-path weights from a (possibly prefixed) state_dict.

        Accepts ``TemporalAggregationNLB().state_dict()`` keys, optionally prefixed with
        ``roi_heads.temporal_aggregator.`` as in a full checkpoint
        (models/video_matchrcnn.py:37, evaluate_movingfashion.py:502-503).
        """
        tensors = {}
        for field, key in WEIGHT_KEYS.items():
            k = prefix + key
            if k not in state:
                raise KeyError(f"state_dict is missing '{k}'")
            t = state[k].detach()
            if tuple(t.shape) != WEIGHT_SHAPES[field]:      # the fold kernels index these buffers by the reference's shapes
                raise ValueError(f"'{k}' has shape {tuple(t.shape)}, expected {WEIGHT_SHAPES[field]} "
                                 "(TemporalAggregationNLB with d_model=256, inter_channels=128)")
            tensors[field] = self._f32(t, k)
        w = SeamWeights(**{f: tensors[f].data_ptr() for f in SeamWeights.FIELDS})
        self._check(self._lib.seam_load_weights(self._h, C.byref(w), self._stream()))
        self._weight_refs = tensors   # keep alive until the fold kernels have run
        self._last = (tensors["last_w"], tensors["last_b"])
        self.weights_epoch += 1
        self.scorer_epoch += 1

    def load_scorer(self, last_w: torch.Tensor, last_b: torch.Tensor) -> None:
        """Only ``last`` (e.g. ``match_predictor.last`` for the per-frame scorers)."""
        lw, lb = self._f32(last_w.detach(), "last_w"), self._f32(last_b.detach(), "last_b")
        if lw.shape != (2, D_MODEL) or lb.shape != (2,):
            raise ValueError("last.weight must be (2,256) and last.bias (2,)")
        self._check(self._lib.seam_load_scorer(self._h, lw.data_ptr(), lb.data_ptr(), self._stream()))
        self._weight_refs = (lw, lb)
        self._last = (lw, lb)
        self.weights_epoch += 1
        self.scorer_epoch += 1

    @contextlib.contextmanager
    def scorer(self, last_w: torch.Tensor, last_b: torch.Tensor):
        """Temporarily score with another ``last`` (e.g. ``match_predictor.last`` for the per-frame rows of the
        eval script) and put the previous scorer back on exit, so that callers sharing this engine -- modules,
        ShardedRetriever, prepared galleries -- are not left with somebody else's weights."""
        prev = self._last
        self.load_scorer(last_w, last_b)
        try:
            yield self
        finally:
            if prev is not None:
                self.load_scorer(*prev)

    # ------------------------------------------------------------------ backward (SURVEY.md section 8 f4)
    def aggregate_backward(self, seq: torch.Tensor, mask, lens, params: Mapping[str, torch.Tensor], dout: torch.Tensor):
        """Vector-Jacobian product of ``aggregate``: ``dout (Q,256)`` -> ``(dseq (1+Tmax,Q,256), {field: grad})`` for
        the 11 aggregator parameters (fields of ``struct seam_weights``, un-folded fp32 tensors in ``params``)."""
        seq, m8, l32, Tmax, Q = self._tracks(seq, mask, lens, keep_16bit=False)   # the backward kernel reads fp32
        dout = self._f32(dout, "dout")
        tensors = {f: self._f32(params[f].detach(), f) for f in SeamWeightGrads.FIELDS}
        w = SeamWeights(**{f: (tensors[f].data_ptr() if f in tensors else 0) for f in SeamWeights.FIELDS})
        grads = {f: torch.zeros_like(tensors[f]) for f in SeamWeightGrads.FIELDS}
        gs = SeamWeightGrads(**{f: grads[f].data_ptr() for f in SeamWeightGrads.FIELDS})
        dseq = torch.zeros((1 + Tmax, Q, D_MODEL), dtype=torch.float32, device=self.device)
        self._check(self._lib.seam_aggregate_backward(self._h, C.byref(w), seq.data_ptr() if Q else 0, _ptr(m8), _ptr(l32),
                                                      Tmax, Q, seq.stride(0), seq.stride(1), dout.data_ptr() if Q else 0,
                                                      dseq.data_ptr(), C.byref(gs), self._stream()))
        return dseq, grads

    def score_dense_backward(self, q: torch.Tensor, g: torch.Tensor, last_w: torch.Tensor, dx5: torch.Tensor):
        """Vector-Jacobian product of ``score_dense``: ``dx5 (Q,G,2)`` -> ``(dq, dg, dlast_w, dlast_b)``."""
        q, g = self._f32(q, "queries"), self._f32(g, "gallery")
        lw, dx5 = self._f32(last_w.detach(), "last_w"), self._f32(dx5, "dx5")
        dq, dg = torch.zeros_like(q), torch.zeros_like(g)
        dw = torch.zeros((2, D_MODEL), dtype=torch.float32, device=self.device)
        db = torch.zeros((2,), dtype=torch.float32, device=self.device)
        self._check(self._lib.seam_score_dense_backward(self._h, lw.data_ptr(), q.data_ptr(), q.shape[0], g.data_ptr(),
                                                        g.shape[0], dx5.data_ptr(), dq.data_ptr(), dg.data_ptr(),
                                                        dw.data_ptr(), db.data_ptr(), self._stream()))
        return dq, dg, dw, db

    # ------------------------------------------------------------------ conv tower (SURVEY.md section 8 f3)
    TOWER_KEYS = ("conv_seq.0", "conv_seq.2", "conv_seq.4", "conv_seq.6")

    def load_tower(self, state: Mapping[str, torch.Tensor], prefix: str = "", bn_eps: float = 1e-5) -> None:
        """Upload the match head's conv tower (``conv_seq.{0,2,4,6}``, ``linear.0``, ``linear.1`` incl. running
        statistics: models/match_head.py:50-62) in the layout the tensor-core kernels read."""
        shapes = {"conv_seq.0.weight": (256, 256, 3, 3), "conv_seq.2.weight": (256, 256, 3, 3),
                  "conv_seq.4.weight": (256, 256, 3, 3), "conv_seq.6.weight": (1024, 256, 3, 3),
                  "conv_seq.0.bias": (256,), "conv_seq.2.bias": (256,), "conv_seq.4.bias": (256,), "conv_seq.6.bias": (1024,),
                  "linear.0.weight": (256, 1024), "linear.0.bias": (256,), "linear.1.weight": (256,), "linear.1.bias": (256,),
                  "linear.1.running_mean": (256,), "linear.1.running_var": (256,)}
        t = {}
        for key, shape in shapes.items():
            k = prefix + key
            if k not in state:
                raise KeyError(f"state_dict is missing '{k}'")
            if tuple(state[k].shape) != shape:
                raise ValueError(f"'{k}' has shape {tuple(state[k].shape)}, expected {shape}")
            t[key] = self._f32(state[k].detach(), k)
        cw = (C.c_void_p * 4)(*[t[f"{n}.weight"].data_ptr() for n in self.TOWER_KEYS])
        cb = (C.c_void_p * 4)(*[t[f"{n}.bias"].data_ptr() for n in self.TOWER_KEYS])
        self._check(self._lib.seam_tower_load_weights(
            self._h, cw, cb, t["linear.0.weight"].data_ptr(), t["linear.0.bias"].data_ptr(), t["linear.1.weight"].data_ptr(),
            t["linear.1.bias"].data_ptr(), t["linear.1.running_mean"].data_ptr(), t["linear.1.running_var"].data_ptr(),
            float(bn_eps), self._stream()))
        self._tower_refs = t          # keep alive until the preparation kernels have run

    def tower_forward(self, x: torch.Tensor, out: Optional[torch.Tensor] = None,
                      dst_row: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``(K,256,14,14)`` ROI features -> 256-d embeddings (eval-mode ``conv_seq`` + ``pool`` + ``linear``,
        models/match_head.py:67-69).  ``out``: fp32 rows of 256 to write into (default: a new ``(K,256)``);
        ``dst_row (K,) int64``: the row of ``out`` each ROI goes to (default: its own index)."""
        if x.dim() != 4 or tuple(x.shape[1:]) != (D_MODEL, 14, 14):
            raise ValueError(f"ROI features must be (K,256,14,14), got {tuple(x.shape)}")
        x = self._f32(x, "roi features")
        K = x.shape[0]
        if out is None:
            if dst_row is not None:
                raise ValueError("dst_row needs an explicit out")
            out = torch.empty((K, D_MODEL), dtype=torch.float32, device=self.device)
        if out.dtype != torch.float32 or out.device != self.device or not out.is_contiguous() or out.shape[-1] != D_MODEL:
            raise ValueError("out must be a contiguous fp32 tensor of rows of 256 on the engine's device")
        d64 = None
        if dst_row is not None:
            d64 = dst_row.to(device=self.device, dtype=torch.int64).contiguous()
            if d64.shape != (K,):
                raise ValueError("dst_row must hold one row index per ROI")
        nbytes = int(self._lib.seam_tower_workspace_bytes(K))
        ws = self._workspace("tower", nbytes + 1024)
        base = (ws.data_ptr() + 1023) & ~1023
        self._check(self._lib.seam_tower_forward(self._h, x.data_ptr() if K else 0, K, out.data_ptr(), _ptr(d64), base,
                                                 nbytes, self._stream()))
        return out

    # ------------------------------------------------------------------ (a) aggregation
    def _out(self, out: Optional[torch.Tensor], shape, dtype, name: str) -> torch.Tensor:
        """A caller-provided output (e.g. a slice of a peer-shared buffer) or a fresh tensor."""
        if out is None:
            return torch.empty(shape, dtype=dtype, device=self.device)
        if tuple(out.shape) != tuple(shape) or out.dtype != dtype or out.device != self.device or not out.is_contiguous():
            raise ValueError(f"{name}: out must be a contiguous {tuple(shape)} {dtype} tensor on {self.device}")
        return out

    def aggregate(self, seq: torch.Tensor, mask: Optional[torch.Tensor] = None,
                  lens: Optional[torch.Tensor] = None, getatt: bool = False, out: Optional[torch.Tensor] = None):
        """x3_1b (and attention weights) from the padded time-major track tensor.

        seq (1+Tmax, Q, 256) fp32 with dummy row 0, mask (Q, 1+Tmax) bool (True = padding):
        the arguments ``x3_1_seq`` / ``x3_1_mask`` of models/match_head.py:90, :133-154.
        An fp16 or bf16 ``seq`` on this device is read as it is (``seam_aggregate_f16`` / ``seam_aggregate_bf16``: no
        conversion pass, same results as on ``seq.float()``); other dtypes are converted to fp32.
        """
        seq, m8, l32, Tmax, Q = self._tracks(seq, mask, lens)
        out = self._out(out, (Q, D_MODEL), torch.float32, "aggregate")
        att = torch.empty((Q, Tmax), dtype=torch.float32, device=self.device) if getatt else None
        nbytes = int(self._lib.seam_aggregate_workspace_bytes(Q))
        ws = self._workspace("agg", nbytes)
        fn = self._track_entry("aggregate", seq)
        self._check(fn(self._h, seq.data_ptr(), _ptr(m8), _ptr(l32), Tmax, Q, seq.stride(0), seq.stride(1),
                       out.data_ptr(), _ptr(att), ws.data_ptr(), ws.numel(), self._stream()))
        return (out, att) if getatt else out

    # ------------------------------------------------------------------ gallery-sharded search (exchange in the kernels)
    def _tracks(self, seq, mask, lens, keep_16bit: bool = True):
        """Argument normalisation shared by aggregate / search / sharded_aggregate / aggregate_backward.  ``seq`` comes
        back fp32, or fp16 / bf16 when it has that dtype on this device and ``keep_16bit`` (the ``_f16`` / ``_bf16``
        entry points read it as it is), with 16-byte strides: copied only when its own strides do not allow that."""
        if seq.dim() != 3 or seq.shape[2] != D_MODEL:
            raise ValueError(f"x3_1_seq must be (1+Tmax, Q, 256), got {tuple(seq.shape)}")
        if not (keep_16bit and seq.dtype in (torch.float16, torch.bfloat16) and seq.device == self.device) and (
                seq.device != self.device or seq.dtype != torch.float32):
            seq = seq.to(device=self.device, dtype=torch.float32)
        per16 = 16 // seq.element_size()                 # elements per 16 bytes: 4 (fp32) / 8 (fp16, bf16)
        if seq.stride(2) != 1 or seq.stride(0) % per16 or seq.stride(1) % per16:
            seq = seq.contiguous()
        Tmax, Q = seq.shape[0] - 1, seq.shape[1]
        if Tmax > _lib.SEAM_MAX_T:
            raise SeamError(2, f"Tmax={Tmax} exceeds the supported {_lib.SEAM_MAX_T} frames per track")
        m8 = None
        if mask is not None:
            if tuple(mask.shape) != (Q, 1 + Tmax):
                raise ValueError(f"x3_1_mask must be (Q, 1+Tmax)={Q, 1 + Tmax}, got {tuple(mask.shape)}")
            m8 = mask.to(device=self.device, dtype=torch.bool).contiguous().view(torch.uint8)
        l32 = lens.to(device=self.device, dtype=torch.int32).contiguous() if lens is not None else None
        return seq, m8, l32, Tmax, Q

    _TRACK_SUFFIX = {torch.float32: "", torch.float16: "_f16", torch.bfloat16: "_bf16"}

    def _track_entry(self, op: str, seq: Optional[torch.Tensor], rows=""):
        """The C entry point of ``op`` for tracks of ``seq``'s dtype (as ``_tracks`` returns them; None for an op that
        takes no tracks) against gallery rows of the type ``rows`` names: a ``PreparedGallery.row_suffix`` (``""``,
        ``"_g16"``, ``"_gbf16"``), or a bool that says whether the rows are fp16.  E.g. ``seam_search_bf16_gbf16``,
        ``seam_score_topk_g16``, ``seam_aggregate_f16``."""
        if isinstance(rows, bool):
            rows = "_g16" if rows else ""
        return getattr(self._lib, f"seam_{op}{'' if seq is None else self._TRACK_SUFFIX[seq.dtype]}{rows}")

    def sharded_aggregate(self, x, seq: torch.Tensor, mask=None, lens=None, row0: Optional[int] = None,
                          last: bool = True, getatt: bool = False):
        """This rank's tracks (queries ``row0 .. row0+Qlocal`` of the step, default: the rows it owns) -> their
        descriptors, stored by the kernel into EVERY rank's descriptor buffer (``x``: a ``retrieval.PeerExchange``).
        ``last``: these are the rank's last tracks of the step (the other ranks are told it is complete)."""
        seq, m8, l32, Tmax, Q = self._tracks(seq, mask, lens)
        row0 = x.q_lo[x.rank] if row0 is None else int(row0)
        att = torch.empty((Q, Tmax), dtype=torch.float32, device=self.device) if getatt else None
        fn = self._track_entry("sharded_aggregate", seq)
        self._check(fn(self._h, C.byref(x.struct), seq.data_ptr() if Q else 0, _ptr(m8), _ptr(l32), Tmax, Q,
                       seq.stride(0), seq.stride(1), row0, 1 if last else 0, _ptr(att), self._stream()))
        return att

    def sharded_score_topk(self, x, gallery: PreparedGallery, return_stats: bool = False):
        """All Q queries (once every rank's descriptors have landed here) against this rank's gallery shard; each
        query's top-k row is stored into the list buffer of the rank that owns the query."""
        gallery = self._fresh(gallery)
        # the diagnostic counters cost a fill, a memset and a copy node per step: only when asked for
        stats = torch.zeros((4,), dtype=torch.int32, device=self.device) if return_stats else None
        nbytes = int(self._lib.seam_score_workspace_bytes(self._h, x.Q, gallery.G, x.k))
        ws = self._workspace("score", nbytes)
        # an fp16 gallery has no separate rows: the _g16 entry reads g16 for both the operand and the direct form
        fn = self._track_entry("sharded_score_topk", None, gallery.row_suffix)
        rows = () if gallery.rows_f16 else (gallery.g.data_ptr(),)
        self._check(fn(self._h, C.byref(x.struct), *rows, gallery.g16.data_ptr(), gallery.cg.data_ptr(),
                       gallery.gstat.data_ptr(), gallery.G, int(gallery.index_offset), _ptr(stats), ws.data_ptr(),
                       ws.numel(), self._stream()))
        return stats

    def sharded_merge(self, x):
        """Merge the per-shard lists of the queries this rank owns and end the step.  Returns
        ``(scores, margins, idx)``: the complete ``(Q,k)`` result on every rank when the exchange replicates it
        (views of its final buffers, valid until the next step's merge), else this rank's ``(own,k)`` rows."""
        if x.replicate:
            self._check(self._lib.seam_sharded_merge(self._h, C.byref(x.struct), None, None, None, self._stream()))
            return x.final
        own = x.q_lo[x.rank + 1] - x.q_lo[x.rank]
        sc = torch.empty((own, x.k), dtype=torch.float32, device=self.device)
        mg = torch.empty((own, x.k), dtype=torch.float32, device=self.device)
        ix = torch.empty((own, x.k), dtype=torch.int32, device=self.device)
        self._check(self._lib.seam_sharded_merge(self._h, C.byref(x.struct), sc.data_ptr(), mg.data_ptr(), ix.data_ptr(),
                                                 self._stream()))
        return sc, mg, ix

    def nlb_forward(self, x: torch.Tensor) -> torch.Tensor:
        """NONLocalBlock1D.forward (models/nlb.py:66-101): (B,256,T) -> (B,256,T)."""
        if x.dim() != 3 or x.shape[1] != D_MODEL:
            raise ValueError(f"x must be (B,256,T), got {tuple(x.shape)}")
        x = self._f32(x, "x")
        B, _, T = x.shape
        if T > _lib.SEAM_MAX_T:
            raise SeamError(2, f"T={T} exceeds the supported {_lib.SEAM_MAX_T}")
        z = torch.empty_like(x)
        nbytes = int(self._lib.seam_nlb_workspace_bytes(B, T))
        ws = self._workspace("nlb", nbytes)
        self._check(self._lib.seam_nlb_forward(self._h, x.data_ptr(), B, T, z.data_ptr(), ws.data_ptr(),
                                               ws.numel(), self._stream()))
        return z

    # ------------------------------------------------------------------ (b)+(c) scorer
    def prepare_gallery(self, g: torch.Tensor, index_offset: int = 0) -> PreparedGallery:
        """Device-resident gallery with its tensor-core operands.  An fp16 or bf16 ``g`` keeps its dtype: used in place
        when it is on this device, contiguous and 16-byte aligned, else copied once to a contiguous tensor here.  fp16
        rows are the tensor-core operand themselves (``seam_prepare_gallery_f16``: no fp32 copy, no second fp16
        copy); bf16 rows get an fp16 image beside them (``seam_prepare_gallery_bf16``: no fp32 copy).  Other dtypes are
        converted to fp32."""
        g = self._rows(g)
        g16 = g if g.dtype == torch.float16 else torch.empty((g.shape[0], D_MODEL), dtype=torch.float16,
                                                             device=self.device)
        G = g.shape[0]
        cg = torch.empty((max(G, 1),), dtype=torch.float32, device=self.device)
        gstat = torch.empty((4,), dtype=torch.float32, device=self.device)
        gallery = PreparedGallery(g=g, g16=g16, cg=cg, gstat=gstat, index_offset=index_offset,
                                  scorer_epoch=self.scorer_epoch)
        self._prepare(gallery)
        return gallery

    def _prepare(self, gallery: PreparedGallery) -> None:
        if gallery.rows_f16:
            self._check(self._lib.seam_prepare_gallery_f16(self._h, gallery.g16.data_ptr(), gallery.G,
                                                           gallery.cg.data_ptr(), gallery.gstat.data_ptr(),
                                                           self._stream()))
        else:       # fp32 or bf16 rows: both write g16
            fn = self._lib.seam_prepare_gallery_bf16 if gallery.rows_bf16 else self._lib.seam_prepare_gallery
            self._check(fn(self._h, gallery.g.data_ptr(), gallery.G, gallery.g16.data_ptr(), gallery.cg.data_ptr(),
                           gallery.gstat.data_ptr(), self._stream()))

    def _fresh(self, gallery: PreparedGallery) -> PreparedGallery:
        """A gallery prepared under another scorer (its cg = dw . g^2 and overflow statistics are stale after
        load_weights / load_scorer) is prepared again in place: one pass over its rows."""
        if gallery.scorer_epoch != self.scorer_epoch:
            self._prepare(gallery)
            gallery.scorer_epoch = self.scorer_epoch
        return gallery

    def score_topk(self, q: torch.Tensor, gallery: PreparedGallery, k: int,
                   return_stats: bool = False, out=None):
        """Best k gallery items per query: (scores (Q,k), margins (Q,k), idx (Q,k) int32).
        ``out``: optional (scores, margins, idx) tensors to write into."""
        if q.dim() != 2 or q.shape[1] != D_MODEL:
            raise ValueError(f"queries must be (Q,256), got {tuple(q.shape)}")
        q = self._f32(q, "queries")
        gallery = self._fresh(gallery)
        Q, G = q.shape[0], gallery.G
        k = int(k)
        o = out if out is not None else (None, None, None)
        sc = self._out(o[0], (Q, k), torch.float32, "score_topk scores")
        mg = self._out(o[1], (Q, k), torch.float32, "score_topk margins")
        ix = self._out(o[2], (Q, k), torch.int32, "score_topk idx")
        # the diagnostic counters cost a fill, a memset and a copy node per step: only when asked for
        stats = torch.zeros((4,), dtype=torch.int32, device=self.device) if return_stats else None
        # The candidate lists take 12-96 KB per query row: very large evaluations are worked through in slabs of
        # queries that reuse one bounded workspace (results do not depend on the slab size)
        slab = Q
        while slab > 1024 and int(self._lib.seam_score_workspace_bytes(self._h, slab, G, k)) > SCORE_WS_LIMIT:
            slab = (slab + 1) // 2
        for lo in range(0, max(Q, 1), max(slab, 1)):
            hi = min(Q, lo + slab)
            n = hi - lo
            nbytes = int(self._lib.seam_score_workspace_bytes(self._h, n, G, k))
            ws = self._workspace("score", nbytes)
            st = stats if (slab == Q or stats is None) else torch.zeros((4,), dtype=torch.int32, device=self.device)
            # an fp16 gallery has no separate rows: the _g16 entry reads g16 for both the operand and the direct form
            fn = self._track_entry("score_topk", None, gallery.row_suffix)
            rows = () if gallery.rows_f16 else (gallery.g.data_ptr(),)
            self._check(fn(self._h, q[lo:hi].data_ptr() if n else 0, n, *rows, gallery.g16.data_ptr(),
                           gallery.cg.data_ptr(), gallery.gstat.data_ptr(), G, int(gallery.index_offset), k,
                           sc[lo:hi].data_ptr() if n else 0, mg[lo:hi].data_ptr() if n else 0,
                           ix[lo:hi].data_ptr() if n else 0, _ptr(st), ws.data_ptr(), ws.numel(), self._stream()))
            if st is not stats:
                stats += st
        if return_stats:
            return sc, mg, ix, stats
        return sc, mg, ix

    def search(self, seq: torch.Tensor, mask, gallery: PreparedGallery, k: int, lens=None, return_stats: bool = False):
        """Tracks -> (descriptors x3_1b (Q,256), scores (Q,k), margins (Q,k), idx (Q,k) int32) in one library call
        (``seam_search``): same results as ``aggregate`` + ``score_topk``."""
        seq, m8, l32, Tmax, Q = self._tracks(seq, mask, lens)
        gallery = self._fresh(gallery)
        G, k = gallery.G, int(k)
        nbytes = int(self._lib.seam_score_workspace_bytes(self._h, Q, G, k))
        if nbytes > SCORE_WS_LIMIT:                      # very large evaluations: the slab path of score_topk
            q = self.aggregate(seq, mask, lens=lens)
            return (q,) + tuple(self.score_topk(q, gallery, k, return_stats=return_stats))
        q = torch.empty((Q, D_MODEL), dtype=torch.float32, device=self.device)
        sc = torch.empty((Q, k), dtype=torch.float32, device=self.device)
        mg = torch.empty((Q, k), dtype=torch.float32, device=self.device)
        ix = torch.empty((Q, k), dtype=torch.int32, device=self.device)
        stats = torch.zeros((4,), dtype=torch.int32, device=self.device) if return_stats else None
        ws = self._workspace("score", nbytes)
        # an fp16 gallery has no separate rows: the _g16 entry reads g16 for both the operand and the direct form
        fn = self._track_entry("search", seq, gallery.row_suffix)
        rows = () if gallery.rows_f16 else (gallery.g.data_ptr(),)
        self._check(fn(self._h, seq.data_ptr() if Q else 0, _ptr(m8), _ptr(l32), Tmax, Q, seq.stride(0), seq.stride(1),
                       q.data_ptr(), *rows, gallery.g16.data_ptr(), gallery.cg.data_ptr(),
                       gallery.gstat.data_ptr(), G, int(gallery.index_offset), k, sc.data_ptr(), mg.data_ptr(),
                       ix.data_ptr(), _ptr(stats), ws.data_ptr(), ws.numel(), self._stream()))
        return (q, sc, mg, ix, stats) if return_stats else (q, sc, mg, ix)

    def score_plan(self, Q: int, G: int) -> Dict[str, int]:
        """Work decomposition + workspace layout seam_score_topk will use for (Q,G)."""
        out = (C.c_int64 * 14)()
        self._check(self._lib.seam_score_plan(self._h, int(Q), int(G), out))
        names = ("query_tiles", "gallery_tiles", "ctas", "ctas_per_query_tile", "list_capacity", "off_a16",
                 "off_rq", "off_anorm", "off_thr", "off_rowcnt", "off_rowbuf", "off_counters", "off_rows", "bytes")
        return dict(zip(names, [int(v) for v in out]))

    def score_dense(self, q: torch.Tensor, g: torch.Tensor) -> torch.Tensor:
        """x5 (Q,G,2) = last((q-g)^2): models/match_head.py:160-162."""
        q, g = self._f32(q, "queries"), self._f32(g, "gallery")
        x5 = torch.empty((q.shape[0], g.shape[0], 2), dtype=torch.float32, device=self.device)
        self._check(self._lib.seam_score_dense(self._h, q.data_ptr(), q.shape[0], g.data_ptr(), g.shape[0],
                                               x5.data_ptr(), self._stream()))
        return x5

    def score_prob(self, q: torch.Tensor, g: torch.Tensor) -> torch.Tensor:
        """softmax(x5)[...,1] as a dense (Q,G) matrix: ``compute_distances`` of the eval script
        (evaluate_movingfashion.py:101-106); with ``g = q`` its ``compute_selfdist`` (:115-121)."""
        q, g = self._f32(q, "queries"), self._f32(g, "gallery")
        out = torch.empty((q.shape[0], g.shape[0]), dtype=torch.float32, device=self.device)
        self._check(self._lib.seam_score_prob(self._h, q.data_ptr(), q.shape[0], g.data_ptr(), g.shape[0],
                                              out.data_ptr(), self._stream()))
        return out

    def _rows(self, g: torch.Tensor) -> torch.Tensor:
        """Gallery rows for the direct-form kernels: an fp16 or bf16 ``g`` keeps its dtype (used in place when it is on
        this device, contiguous and 16-byte aligned, else copied once); other dtypes become fp32."""
        if g.dim() != 2 or g.shape[1] != D_MODEL:
            raise ValueError(f"gallery must be (G,256), got {tuple(g.shape)}")
        if g.dtype in (torch.float16, torch.bfloat16):
            g = g.to(self.device)
            if not g.is_contiguous() or g.data_ptr() % 16:
                g = g.clone(memory_format=torch.contiguous_format)
            return g
        return self._f32(g, "gallery")

    def _fused_args(self, frames: torch.Tensor, start: torch.Tensor, g: torch.Tensor, target: torch.Tensor):
        frames, g = self._f32(frames, "frames"), self._rows(g)
        s32 = start.to(device=self.device, dtype=torch.int32).contiguous()
        t32 = target.to(device=self.device, dtype=torch.int32).contiguous()
        P = int(t32.shape[0])
        if s32.shape != (P + 1,):
            raise ValueError("start must hold P+1 offsets")
        return frames, s32, g, t32, P

    def rank_fused_distances(self, frames: torch.Tensor, start: torch.Tensor, g: torch.Tensor, target: torch.Tensor):
        """Ranks of the true shop items under the per-product average / maximum of the frames' class-1
        probabilities (evaluate_movingfashion.py:294-316).  ``frames (N,256)`` sorted by product, ``start (P+1)``
        CSR offsets, ``target (P)``.  An fp16 or bf16 gallery ``g`` is read as it is (``seam_rank_fused_distances_g16``
        / ``_gbf16``: the ranks of ``g.float()``, no fp32 copy).  Returns ``(rank_avg, rank_max)`` int32 ``(P,)``; no
        host synchronisation."""
        frames, s32, g, t32, P = self._fused_args(frames, start, g, target)
        ra = torch.empty((P,), dtype=torch.int32, device=self.device)
        rm = torch.empty((P,), dtype=torch.int32, device=self.device)
        fn = self._track_entry("rank_fused_distances", None, ROW_SUFFIX[g.dtype])
        self._check(fn(self._h, frames.data_ptr() if frames.numel() else 0, s32.data_ptr(), P, g.data_ptr(), g.shape[0],
                       t32.data_ptr(), ra.data_ptr(), rm.data_ptr(), self._stream()))
        return ra, rm

    def fused_target(self, frames: torch.Tensor, start: torch.Tensor, g: torch.Tensor, index_offset: int,
                     target: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """The target item's fused average / maximum for one shard ``g`` (global rows ``[index_offset,
        index_offset + G)``) of a sharded gallery (``seam_shard_fused_target``); ``target`` holds GLOBAL rows.
        Returns ``(avg, max)`` fp32 ``(P,)``: the values ``rank_fused_distances`` compares against, bit for bit, where
        the target lies in this shard and the product has frames, ``-inf`` elsewhere, so that a MAX all-reduce over
        the shards gives every shard every target value."""
        frames, s32, g, t32, P = self._fused_args(frames, start, g, target)
        avg = torch.empty((P,), dtype=torch.float32, device=self.device)
        mx = torch.empty((P,), dtype=torch.float32, device=self.device)
        fn = self._track_entry("shard_fused_target", None, ROW_SUFFIX[g.dtype])
        self._check(fn(self._h, frames.data_ptr() if frames.numel() else 0, s32.data_ptr(), P, g.data_ptr(), g.shape[0],
                       int(index_offset), t32.data_ptr(), avg.data_ptr() if P else 0, mx.data_ptr() if P else 0,
                       self._stream()))
        return avg, mx

    def fused_rank_count(self, frames: torch.Tensor, start: torch.Tensor, g: torch.Tensor, index_offset: int,
                         target: torch.Tensor, target_avg: torch.Tensor,
                         target_max: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """This shard's counts of the rows ranking before each product's target under the two fusions, given every
        target's values (the MAX over the shards of ``fused_target``): ``seam_shard_rank_fused_distances``.  Ties
        with the target are broken by global row and a product without frames counts this shard's G, so the SUM of
        the shards' counts is ``rank_fused_distances`` on the whole gallery.  Returns ``(count_avg, count_max)``
        int32 ``(P,)``."""
        frames, s32, g, t32, P = self._fused_args(frames, start, g, target)
        ta, tm = self._f32(target_avg, "target_avg"), self._f32(target_max, "target_max")
        if ta.shape != (P,) or tm.shape != (P,):
            raise ValueError("target_avg / target_max must hold one value per product")
        ca = torch.empty((P,), dtype=torch.int32, device=self.device)
        cm = torch.empty((P,), dtype=torch.int32, device=self.device)
        fn = self._track_entry("shard_rank_fused_distances", None, ROW_SUFFIX[g.dtype])
        self._check(fn(self._h, frames.data_ptr() if frames.numel() else 0, s32.data_ptr(), P, g.data_ptr(), g.shape[0],
                       int(index_offset), t32.data_ptr(), ta.data_ptr() if P else 0, tm.data_ptr() if P else 0,
                       ca.data_ptr() if P else 0, cm.data_ptr() if P else 0, self._stream()))
        return ca, cm

    def rank_of_target(self, q: torch.Tensor, g, target: torch.Tensor, return_stats: bool = False):
        """Rank (0 = best) of gallery row target[i] for query i: evaluate_movingfashion.py:268-269.

        ``g`` is either a ``(G,256)`` tensor -- exhaustive fp32 kernel -- or a ``PreparedGallery`` -- the
        tensor-core path (count what is certainly above the target, decide the rest in fp32); both give
        the same integers.  Returns (rank int32 (Q,), target margin fp32 (Q,)[, stats])."""
        q = self._f32(q, "queries")
        prepared = isinstance(g, PreparedGallery)
        if prepared:
            g = self._fresh(g)
        gm = g.g if prepared else self._f32(g, "gallery")
        t32 = target.to(device=self.device, dtype=torch.int32).contiguous()
        Q, G = q.shape[0], gm.shape[0]
        if t32.shape != (Q,):
            raise ValueError("target must have one gallery row per query")
        if Q and (int(t32.min()) < 0 or int(t32.max()) >= G):
            raise ValueError("target index out of range")
        rank = torch.empty((Q,), dtype=torch.int32, device=self.device)
        margin = torch.empty((Q,), dtype=torch.float32, device=self.device)
        stats = torch.zeros((4,), dtype=torch.int32, device=self.device)
        if prepared and Q > 0:
            nbytes = int(self._lib.seam_rank_workspace_bytes(self._h, Q, G))
            ws = self._workspace("score", nbytes)
            fn = self._track_entry("rank_of_target_prepared", None, g.row_suffix)
            rows = () if g.rows_f16 else (gm.data_ptr(),)
            self._check(fn(self._h, q.data_ptr(), Q, *rows, g.g16.data_ptr(), g.cg.data_ptr(), g.gstat.data_ptr(), G,
                           t32.data_ptr(), rank.data_ptr(), margin.data_ptr(), stats.data_ptr(), ws.data_ptr(), ws.numel(),
                           self._stream()))
        else:
            self._check(self._lib.seam_rank_of_target(self._h, q.data_ptr(), Q, gm.data_ptr(), G,
                                                      t32.data_ptr(), rank.data_ptr(), margin.data_ptr(),
                                                      self._stream()))
        if return_stats:
            return rank, margin, stats
        return rank, margin

    def _shard_targets(self, q: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
        t32 = target.to(device=self.device, dtype=torch.int32).contiguous()
        if t32.shape != (q.shape[0],):
            raise ValueError("target must have one gallery row per query")
        return t32

    def target_margin(self, q: torch.Tensor, gallery: PreparedGallery, target: torch.Tensor) -> torch.Tensor:
        """Margin d = l1 - l0 of each query's target for one shard of a sharded gallery (``seam_shard_target_margin``).
        ``target`` holds GLOBAL gallery rows; the shard covers ``[gallery.index_offset, gallery.index_offset + G)``.
        Returns ``(Q,)`` fp32: the margin where the target lies in this shard (bit for bit the one ``rank_of_target``
        reports), ``-inf`` elsewhere, so that a MAX all-reduce over the shards gives every shard every margin."""
        q = self._f32(q, "queries")
        gallery = self._fresh(gallery)
        t32 = self._shard_targets(q, target)
        Q = q.shape[0]
        margin = torch.empty((Q,), dtype=torch.float32, device=self.device)
        fn = self._track_entry("shard_target_margin", None, gallery.row_suffix)
        self._check(fn(self._h, q.data_ptr() if Q else 0, Q, gallery.g.data_ptr(), gallery.G, int(gallery.index_offset),
                       t32.data_ptr() if Q else 0, margin.data_ptr() if Q else 0, self._stream()))
        return margin

    def rank_count(self, q: torch.Tensor, gallery: PreparedGallery, target: torch.Tensor, target_margin: torch.Tensor,
                   return_stats: bool = False):
        """This shard's count of the gallery rows ranking before each query's target, given every target's margin
        (``target_margin``: the MAX over the shards of ``target_margin``): ``seam_shard_rank_count_prepared``, the
        tensor-core path of ``rank_of_target``.  Ties with the target are broken by global row, so the SUM of the
        shards' counts is the rank over the whole gallery.  Returns ``(Q,)`` int32 [, stats (4) int32: stats[0] is the
        number of queries this shard counted exhaustively]."""
        q = self._f32(q, "queries")
        gallery = self._fresh(gallery)
        t32 = self._shard_targets(q, target)
        m = self._f32(target_margin, "target_margin")
        Q, G = q.shape[0], gallery.G
        if m.shape != (Q,):
            raise ValueError("target_margin must have one margin per query")
        count = torch.empty((Q,), dtype=torch.int32, device=self.device)
        stats = torch.zeros((4,), dtype=torch.int32, device=self.device) if return_stats else None
        if Q > 0:
            ws = self._workspace("score", int(self._lib.seam_rank_workspace_bytes(self._h, Q, G)))
            fn = self._track_entry("shard_rank_count_prepared", None, gallery.row_suffix)
            rows = () if gallery.rows_f16 else (gallery.g.data_ptr(),)
            self._check(fn(self._h, q.data_ptr(), Q, *rows, gallery.g16.data_ptr(), gallery.cg.data_ptr(),
                           gallery.gstat.data_ptr(), G, int(gallery.index_offset), t32.data_ptr(), m.data_ptr(),
                           count.data_ptr(), _ptr(stats), ws.data_ptr(), ws.numel(), self._stream()))
        return (count, stats) if return_stats else count

    def upload_tracks(self, seq_host: torch.Tensor, lo: int, hi: int) -> torch.Tensor:
        """Tracks [lo, hi) of a HOST ``x3_1_seq (1+Tmax, Q, 256)`` -> device ``(1+Tmax, hi-lo, 256)`` on the
        current stream with one pitched copy of the frame rows (row 0, the dummy frame, stays untouched).  fp32, fp16
        or bf16: the device tensor has the host tensor's dtype (16-bit tracks cross the bus at half the bytes and are
        aggregated as they are)."""
        if (seq_host.device.type != "cpu" or seq_host.dtype not in self._TRACK_SUFFIX
                or not seq_host.is_contiguous()):
            raise SeamError(2, "upload_tracks: seq_host must be a contiguous fp32, fp16 or bf16 host tensor")
        T1, Q, D = seq_host.shape
        if D != D_MODEL:
            raise SeamError(3, f"upload_tracks: feature size {D} != {D_MODEL}")
        out = torch.empty((T1, hi - lo, D), dtype=seq_host.dtype, device=self.device)
        # the _f16 entry copies any 2-byte element type
        fn = self._lib.seam_upload_tracks if seq_host.element_size() == 4 else self._lib.seam_upload_tracks_f16
        self._check(fn(self._h, seq_host.data_ptr(), T1 - 1, Q, lo, hi, out.data_ptr(), self._stream()))
        return out

    def merge_topk(self, scores: Optional[torch.Tensor], margins: torch.Tensor, idx: torch.Tensor):
        """Merge (N,Q,k) per-shard lists into (Q,k); ``scores`` may be None (recomputed from the margins)."""
        N, Q, k = margins.shape
        margins = self._f32(margins, "margins")
        scores = self._f32(scores, "scores") if scores is not None else None     # None: recomputed from the margins
        idx = idx.to(device=self.device, dtype=torch.int32).contiguous()
        sc = torch.empty((Q, k), dtype=torch.float32, device=self.device)
        mg = torch.empty((Q, k), dtype=torch.float32, device=self.device)
        ix = torch.empty((Q, k), dtype=torch.int32, device=self.device)
        self._check(self._lib.seam_merge_topk(self._h, _ptr(scores), margins.data_ptr(), idx.data_ptr(),
                                              N, Q, k, sc.data_ptr(), mg.data_ptr(), ix.data_ptr(),
                                              self._stream()))
        return sc, mg, ix


_engines: Dict[int, SeamEngine] = {}


def get_engine(device="cuda") -> SeamEngine:
    """Process-wide engine for a device (created on first use)."""
    device = torch.device(device)
    if device.type != "cuda":
        raise SeamError(2, f"the SEAM hot path runs on CUDA only (got {device}); there is no CPU fallback")
    if not torch.cuda.is_available():
        raise SeamError(3, "no CUDA device is visible; the SEAM hot path has no CPU fallback")
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _engines:
        _engines[idx] = SeamEngine(torch.device("cuda", idx))
    return _engines[idx]
