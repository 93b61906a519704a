"""Drop-in modules with the reference's constructor arguments, parameter names (state_dict
keys) and forward signatures, running the hot path on the B200 kernels.

Mirrors (signatures and return tuples, not code):
  models/nlb.py:104-109           NONLocalBlock1D
  models/match_head.py:47-76      MatchPredictor
  models/match_head.py:79-169     TemporalAggregationNLB
The conv tower (conv_seq / pool / linear) is the feature producer and stays in PyTorch, as
BASELINE.json's north_star specifies.  Inference only: the kernels do not record autograd
history (training through the hot path is SURVEY.md section 8(f4)).
"""
from __future__ import annotations

from typing import List, Optional

import torch
from torch import nn

from ._lib import SeamError
from .engine import D_MODEL, PreparedGallery, SeamEngine

DENSE_PAIR_LIMIT = 1 << 26   # x5 is (Q,G,2) fp32: 512 MiB at this many pairs
_AGG_FIELDS = ("theta_w", "theta_b", "phi_w", "phi_b", "g_w", "g_b", "W_w", "W_b", "concat_w", "att_w", "att_b")


class _AggregateFn(torch.autograd.Function):
    """x3_1b = aggregate(x3_1_seq) inside an autograd graph: forward = the fused aggregation kernel (folded
    weights), backward = seam_aggregate_backward (the same folded algebra, differentiated; tracks of up to 64 frames)."""

    @staticmethod
    def forward(ctx, eng, seq, mask, *params):
        ctx.eng, ctx.mask = eng, mask
        ctx.save_for_backward(seq, *params)
        return eng.aggregate(seq, mask)

    @staticmethod
    def backward(ctx, dout):
        seq, *params = ctx.saved_tensors
        dseq, grads = ctx.eng.aggregate_backward(seq, ctx.mask, None, dict(zip(_AGG_FIELDS, params)), dout.contiguous())
        return (None, dseq, None) + tuple(grads[f].view_as(p) for f, p in zip(_AGG_FIELDS, params))


class _PairLogitsFn(torch.autograd.Function):
    """x5 = last((q - g)^2) (models/match_head.py:160-162) inside an autograd graph."""

    @staticmethod
    def forward(ctx, eng, q, g, last_w, last_b):
        ctx.eng = eng
        ctx.save_for_backward(q, g, last_w)
        return eng.score_dense(q, g)

    @staticmethod
    def backward(ctx, dx5):
        q, g, last_w = ctx.saved_tensors
        dq, dg, dw, db = ctx.eng.score_dense_backward(q, g, last_w, dx5.contiguous())
        return None, dq, dg, dw, db


class _EngineMixin:
    """Lazily creates a SeamEngine on the module's device and keeps its folded weights in
    sync with the module's parameters."""

    _TRANSIENT = ("_seam_engine", "_seam_key", "_seam_epoch", "_gallery_cache", "_seam_tower_key", "_seam_tower_engine")

    def __getstate__(self):
        # the engine wraps a ctypes handle (not picklable, not copyable): copy.deepcopy(model), pickle and
        # torch.save(model) drop it and the copy re-creates its own on first use
        state = dict(super().__getstate__())
        for k in self._TRANSIENT:
            state.pop(k, None)
        return state

    def _engine_for(self, device: torch.device) -> SeamEngine:
        device = torch.device(device)
        if device.type != "cuda":
            raise SeamError(2, f"{type(self).__name__} runs its hot path on CUDA only (tensor on {device}); "
                               "move the module and inputs to a B200 -- there is no CPU fallback")
        eng = self.__dict__.get("_seam_engine")
        if eng is None or eng.device != device:
            eng = SeamEngine(device)
            self.__dict__["_seam_engine"] = eng
            self.__dict__["_seam_key"] = None
        return eng

    def _extra_key(self):
        return None

    def _sync_weights(self, eng: SeamEngine) -> None:
        state = self._hot_state()
        key = (tuple((k, v.data_ptr(), v._version, str(v.device)) for k, v in sorted(state.items())),
               self._extra_key())
        # re-upload when the parameters changed -- or when somebody else loaded weights into this engine
        # since (e.g. retrieval.evaluate_products switching to the per-frame scorer)
        if self.__dict__.get("_seam_key") != key or self.__dict__.get("_seam_epoch") != getattr(eng, "weights_epoch", 0):
            self._upload(eng, state)
            self.__dict__["_seam_key"] = key
            self.__dict__["_seam_epoch"] = getattr(eng, "weights_epoch", 0)


class NONLocalBlock1D(_EngineMixin, nn.Module):
    """Concatenation-form non-local block, models/nlb.py:5-101 as instantiated at
    models/match_head.py:87.  Only that instantiation is supported."""

    def __init__(self, in_channels=D_MODEL, inter_channels=None, sub_sample=False, bn_layer=False):
        super().__init__()
        if inter_channels is None:
            inter_channels = in_channels // 2
        if in_channels != D_MODEL or inter_channels != D_MODEL // 2 or sub_sample or bn_layer:
            raise NotImplementedError(
                "only NONLocalBlock1D(256, inter_channels=128, sub_sample=False, bn_layer=False) -- the "
                "configuration SEAM uses (models/match_head.py:87) -- is implemented")
        self.dimension = 1
        self.sub_sample = sub_sample
        self.in_channels = in_channels
        self.inter_channels = inter_channels
        self.g = nn.Conv1d(in_channels, inter_channels, kernel_size=1)
        self.W = nn.Conv1d(inter_channels, in_channels, kernel_size=1)
        nn.init.constant_(self.W.weight, 0)      # models/nlb.py:48-49
        nn.init.constant_(self.W.bias, 0)
        self.theta = nn.Conv1d(in_channels, inter_channels, kernel_size=1)
        self.phi = nn.Conv1d(in_channels, inter_channels, kernel_size=1)
        self.concat_project = nn.Sequential(nn.Conv2d(inter_channels * 2, 1, 1, 1, 0, bias=False), nn.ReLU())

    def _hot_state(self):
        return {"newnlb." + k: v for k, v in self.state_dict(keep_vars=True).items()}

    def _upload(self, eng, state):
        dev = eng.device
        full = dict(state)
        full["attention_scorer.weight"] = torch.zeros(1, D_MODEL, device=dev)
        full["attention_scorer.bias"] = torch.zeros(1, device=dev)
        full["last.weight"] = torch.zeros(2, D_MODEL, device=dev)
        full["last.bias"] = torch.zeros(2, device=dev)
        eng.load_weights(full)

    @torch.no_grad()
    def forward(self, x):
        eng = self._engine_for(x.device)
        self._sync_weights(eng)
        return eng.nlb_forward(x)


class MatchPredictor(_EngineMixin, nn.Module):
    """models/match_head.py:47-76."""

    def __init__(self):
        super().__init__()
        self.conv_seq = nn.Sequential(nn.Conv2d(256, 256, 3), nn.ReLU(),
                                      nn.Conv2d(256, 256, 3), nn.ReLU(),
                                      nn.Conv2d(256, 256, 3), nn.ReLU(),
                                      nn.Conv2d(256, 1024, 3), nn.ReLU())
        self.pool = nn.Sequential(nn.AvgPool2d((6, 6)), nn.ReLU())
        self.linear = nn.Sequential(nn.Linear(1024, 256), nn.BatchNorm1d(256))
        self.last = nn.Linear(256, 2)

    # ---- conv tower -> 256-d embedding (models/match_head.py:67-69 / :93-95) ---------------
    def embed_torch(self, x):
        """The PyTorch modules themselves (training, CPU, and the reference the kernels are tested against)."""
        x2 = self.pool(self.conv_seq(x))
        return self.linear(x2.view(x2.size(0), -1))

    def _tower_ready(self, x) -> bool:
        """Eval mode on a CUDA tensor: the tensor-core tower (inference kernels: BatchNorm with running statistics,
        no autograd history).  Training mode keeps the PyTorch modules (batch statistics, autograd)."""
        return (not self.training) and x.is_cuda and x.dim() == 4 and tuple(x.shape[1:]) == (256, 14, 14)

    def _sync_tower(self, eng: SeamEngine) -> None:
        names = [k for k in self.state_dict(keep_vars=True) if k.startswith(("conv_seq.", "linear."))]
        sd = self.state_dict(keep_vars=True)
        key = tuple((k, sd[k].data_ptr(), sd[k]._version) for k in names) + (self.linear[1].eps,)
        if self.__dict__.get("_seam_tower_key") != key or self.__dict__.get("_seam_tower_engine") is not eng:
            eng.load_tower(sd, bn_eps=self.linear[1].eps)
            self.__dict__["_seam_tower_key"] = key
            self.__dict__["_seam_tower_engine"] = eng

    def embed(self, x, out=None, dst_row=None):
        """conv tower -> 256-d embedding.  Eval mode on CUDA: ``seam_tower_forward`` (tcgen05 shifted-GEMM
        convolutions, fp16 operands / fp32 accumulation, fused pool + linear + BatchNorm); otherwise PyTorch."""
        if self._tower_ready(x):
            eng = self._engine_for(x.device)
            self._sync_tower(eng)
            with torch.no_grad():
                return eng.tower_forward(x, out=out, dst_row=dst_row)
        y = self.embed_torch(x)
        if out is not None:
            rows = dst_row if dst_row is not None else torch.arange(y.shape[0], device=y.device)
            out.view(-1, y.shape[1])[rows] = y
            return out
        return y

    # ---- engine plumbing --------------------------------------------------------------
    def _hot_state(self):
        return {"last.weight": self.last.weight, "last.bias": self.last.bias}

    def _upload(self, eng, state):
        eng.load_scorer(state["last.weight"], state["last.bias"])

    def _dense_logits(self, q, g):
        if q.shape[0] * g.shape[0] > DENSE_PAIR_LIMIT:
            raise SeamError(2, f"x5 for {q.shape[0]}x{g.shape[0]} pairs would materialise "
                               f"{q.shape[0] * g.shape[0] * 8 / 2**30:.1f} GiB; use score_topk() instead")
        eng = self._engine_for(q.device)
        self._sync_weights(eng)
        return eng.score_dense(q, g)

    def forward(self, x, types):
        """``(x3, x5)`` as models/match_head.py:66-76.  The conv tower runs under autograd as in the reference
        (``x3`` carries its graph); the pair scorer runs in the CUDA kernels without autograd history, so ``x5``
        is detached -- training through the scorer is SURVEY.md section 8(f4).  Raises above 64M pairs
        (``DENSE_PAIR_LIMIT``) instead of materialising x4 = (Q,G,256)."""
        x3 = self.embed(x)
        types = types.to(x3.device)
        with torch.no_grad():
            x3_1 = x3[types == 0]
            x3_2 = x3[types == 1]
            x5 = self._dense_logits(x3_1, x3_2)      # (Q,G,2): match_head.py:70-74
        return x3, x5


class TemporalAggregationNLB(MatchPredictor):
    """models/match_head.py:79-169.  Same parameters, same forward signature and return tuple;
    additionally ``score_topk`` (fused aggregation -> scorer -> top-k, no x5)."""

    def __init__(self, d_model=D_MODEL):
        super().__init__()
        if d_model != D_MODEL:
            raise NotImplementedError("d_model must be 256")
        self.n_frames = -1
        self.attention_scorer = nn.Linear(d_model, 1)
        self.newnlb = NONLocalBlock1D(in_channels=d_model, sub_sample=False, bn_layer=False)
        self.nlb = True
        self.__dict__["_gallery_cache"] = None

    def _hot_state(self):
        sd = self.state_dict(keep_vars=True)
        keys = [k for k in sd if k.startswith(("newnlb.", "attention_scorer.", "last."))]
        return {k: sd[k] for k in keys}

    def _extra_key(self):
        return bool(self.nlb)

    def _upload(self, eng, state):
        if not self.nlb:
            # the reference skips the block when self.nlb is False (match_head.py:113, :143);
            # zero output projection makes the block the identity
            state = dict(state)
            state["newnlb.W.weight"] = torch.zeros_like(state["newnlb.W.weight"])
            state["newnlb.W.bias"] = torch.zeros_like(state["newnlb.W.bias"])
        eng.load_weights(state)

    # ---- x-branch grouping: match_head.py:96-111 without the per-track host syncs --------
    @staticmethod
    def _group_layout(ids):
        """Track index and frame position of every street ROI (tracks in ascending id order, frames in arrival
        order: models/match_head.py:104-110): (inv, pos, counts, n_seqs, maxlen)."""
        uniq, inv = torch.unique(ids, sorted=True, return_inverse=True)
        n_seqs = uniq.numel()
        counts = torch.bincount(inv, minlength=n_seqs)
        maxlen = int(counts.max())
        order = torch.argsort(inv, stable=True)
        starts = torch.cumsum(counts, 0) - counts
        pos_sorted = torch.arange(inv.numel(), device=inv.device) - starts[inv[order]]
        pos = torch.empty_like(pos_sorted)
        pos[order] = pos_sorted
        return inv, pos, counts, n_seqs, maxlen

    @classmethod
    def _group_tracks(cls, x3_1, ids):
        inv, pos, counts, n_seqs, maxlen = cls._group_layout(ids)
        seq = torch.zeros((1 + maxlen, n_seqs, D_MODEL), device=x3_1.device, dtype=x3_1.dtype)
        seq[1 + pos, inv] = x3_1
        mask = torch.arange(1 + maxlen, device=x3_1.device).unsqueeze(0) > counts.unsqueeze(1)
        return seq, mask, counts

    def _att_list(self, att, mask) -> List[torch.Tensor]:
        m = mask.to(torch.bool)
        Tp1 = m.shape[1]
        first = torch.where(m.any(1), m.to(torch.int8).argmax(1), torch.full((m.shape[0],), Tp1, device=m.device))
        lens = (first - 1).clamp(min=0).tolist()
        return [att[i, :n].unsqueeze(1) for i, n in enumerate(lens)]

    def forward(self, x, types, ids, x3_1_seq=None, x3_1_mask=None, x3_2=None, getatt=False):
        """Same signature and return tuple as models/match_head.py:90-169.  Limits (errors, not fallbacks):
        tracks of at most 64 frames (``SEAM_MAX_T``), x5 for at most 64M pairs (``DENSE_PAIR_LIMIT``; use
        ``score_topk`` beyond).  The conv tower of the x-branch runs under autograd (``x3_2`` keeps its graph);
        aggregation and scorer outputs are detached (inference kernels).  In training mode with grad enabled (and
        ``getatt=False``) aggregation and scorer are differentiable, for the same tracks and both values of ``nlb``."""
        x3_1 = x3_1_ids = None
        if x3_1_seq is None and self._tower_ready(x):          # x-branch, eval: the tower writes the track layout itself
            with torch.no_grad():
                types = types.to(x.device)
                ids = ids.to(x.device)
                street = (types == 0).nonzero().flatten()
                shop = (types == 1).nonzero().flatten()
                x3_1_ids = ids[street]
                if street.numel() > 0:
                    inv, pos, counts, n_seqs, maxlen = self._group_layout(x3_1_ids)
                    base = (1 + maxlen) * n_seqs
                    buf = torch.zeros((base + shop.numel(), D_MODEL), device=x.device, dtype=torch.float32)
                    dst = torch.empty((x.shape[0],), dtype=torch.int64, device=x.device)
                    dst[street] = (1 + pos) * n_seqs + inv      # slot (1 + t, track) of the time-major x3_1_seq
                    dst[shop] = base + torch.arange(shop.numel(), device=x.device)
                    self.embed(x, out=buf, dst_row=dst)
                    x3_1_seq = buf[:base].view(1 + maxlen, n_seqs, D_MODEL)
                    x3_1_mask = torch.arange(1 + maxlen, device=x.device).unsqueeze(0) > counts.unsqueeze(1)
                    x3_2 = buf[base:]
                    return self._forward_hot(None, x3_1_ids, x3_1_seq, x3_1_mask, x3_2, getatt, from_x=True)
                x3_2 = self.embed(x)[shop]
                return self._forward_hot(None, x3_1_ids, None, None, x3_2, getatt, from_x=True)
        if x3_1_seq is None:                                   # x-branch: match_head.py:92-111
            x3 = self.embed(x)                                 # under autograd, as in the reference
            types = types.to(x3.device)
            ids = ids.to(x3.device)
            x3_1 = x3[types == 0]
            x3_1_ids = ids[types == 0]
            x3_2 = x3[types == 1]
        if torch.is_grad_enabled() and self.training and not getatt:
            return self._forward_train(x3_1, x3_1_ids, x3_1_seq, x3_1_mask, x3_2)
        with torch.no_grad():
            return self._forward_hot(x3_1, x3_1_ids, x3_1_seq, x3_1_mask, x3_2, getatt)

    def _agg_params(self):
        n = self.newnlb
        return (n.theta.weight, n.theta.bias, n.phi.weight, n.phi.bias, n.g.weight, n.g.bias, n.W.weight, n.W.bias,
                n.concat_project[0].weight, self.attention_scorer.weight, self.attention_scorer.bias)

    def _forward_train(self, x3_1, x3_1_ids, x3_1_seq, x3_1_mask, x3_2):
        """Training (models/match_head.py:339, 429 call this forward under autograd): the same kernels forward,
        ``seam_aggregate_backward`` / ``seam_score_dense_backward`` behind them, the grouping of ROI embeddings into
        tracks as differentiable index operations.  x5 carries the graph the losses differentiate.  Tracks of up to
        64 frames (``SEAM_MAX_T``), as in eval mode.  With ``nlb=False`` the block is not in the graph, as in the
        reference: the forward runs with a zero ``W`` (the eval upload), the backward gets a zero ``W`` too, and the
        ``newnlb.*`` parameters are passed detached, so their ``.grad`` stays ``None``."""
        if x3_1_seq is None:
            if x3_1_ids.numel() == 0:
                return None, x3_2, None, None, None, x3_1_ids
            x3_1_seq, x3_1_mask, _ = self._group_tracks(x3_1, x3_1_ids)      # index_put: differentiable w.r.t. x3_1
        else:
            x3_1_ids = torch.zeros((1, 2))
        eng = self._engine_for(x3_1_seq.device)
        self._sync_weights(eng)
        params = self._agg_params()
        if not self.nlb:
            params = tuple(t.detach() for t in params[:6]) + (torch.zeros_like(params[6]), torch.zeros_like(params[7]),
                                                              params[8].detach()) + params[9:]
        x3_1b = _AggregateFn.apply(eng, x3_1_seq, x3_1_mask, *params)
        g = x3_2.to(x3_1b.device).reshape(-1, D_MODEL)
        if x3_1b.shape[0] * g.shape[0] > DENSE_PAIR_LIMIT:
            raise SeamError(2, "x5 too large for the training path")
        x5 = _PairLogitsFn.apply(eng, x3_1b, g, self.last.weight, self.last.bias)
        return x3_1b, x3_2, x5, x3_1_seq, x3_1_mask, x3_1_ids

    def _forward_hot(self, x3_1, x3_1_ids, x3_1_seq, x3_1_mask, x3_2, getatt, from_x=False):
        attention_scores = None
        if from_x:
            pass                                      # x-branch with the layout already written by the tower
        elif x3_1_seq is None:
            if x3_1_ids.numel() > 0:
                x3_1_seq, x3_1_mask, _ = self._group_tracks(x3_1, x3_1_ids)
            else:
                x3_1b = None
        else:
            x3_1_ids = torch.zeros((1, 2))            # match_head.py:158
        if x3_1_seq is not None and x3_1_ids.numel() > 0:
            eng = self._engine_for(x3_1_seq.device)
            self._sync_weights(eng)
            res = eng.aggregate(x3_1_seq, x3_1_mask, getatt=getatt)
            if getatt:
                x3_1b, att = res
                attention_scores = self._att_list(att, x3_1_mask)
            else:
                x3_1b = res
            g = x3_2.to(x3_1b.device).reshape(-1, D_MODEL)
            x5 = self._dense_logits(x3_1b, g)
        else:
            x3_1b, x5 = None, None
        if getatt:
            return x3_1b, x3_2, x5, x3_1_seq, x3_1_mask, x3_1_ids, attention_scores
        return x3_1b, x3_2, x5, x3_1_seq, x3_1_mask, x3_1_ids

    # ---- fused entry (additive; SURVEY.md section 8(b)) ----------------------------------
    @torch.no_grad()
    def aggregate(self, x3_1_seq, x3_1_mask=None, lens=None, getatt=False):
        eng = self._engine_for(x3_1_seq.device)
        self._sync_weights(eng)
        return eng.aggregate(x3_1_seq, x3_1_mask, lens=lens, getatt=getatt)

    @torch.no_grad()
    def prepare_gallery(self, gallery: torch.Tensor, index_offset: int = 0) -> PreparedGallery:
        eng = self._engine_for(gallery.device)
        self._sync_weights(eng)
        return eng.prepare_gallery(gallery, index_offset)

    @torch.no_grad()
    def score_topk(self, x3_1_seq, x3_1_mask, gallery, k=20):
        """Aggregation -> pair scorer -> per-query top-k in one pass; x5 is never materialised.

        gallery: (G,256) tensor or a PreparedGallery.  Returns (scores (Q,k) = softmax(x5)[...,1],
        idx (Q,k) int64) -- the first k columns of evaluate_movingfashion.py:268's ranking."""
        eng = self._engine_for(x3_1_seq.device)
        self._sync_weights(eng)
        if not isinstance(gallery, PreparedGallery):
            gallery = eng.prepare_gallery(gallery)
        q = eng.aggregate(x3_1_seq, x3_1_mask)
        sc, _, ix = eng.score_topk(q, gallery, k)
        return sc, ix.to(torch.int64)
