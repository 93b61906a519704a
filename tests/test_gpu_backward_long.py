"""f4 for tracks of up to 64 frames: the aggregator backward in the folded algebra (seam_aggregate_backward), training
with nlb=False, and the closed form that kernel implements (checked in float64 on the CPU against autograd)."""
import ctypes as C

import pytest
import torch

import seam_match_rcnn_b200 as pkg
from seam_match_rcnn_b200._lib import SeamWeightGrads, SeamWeights
from oracle import seam_oracle as so

DEV = "cuda:0"
D, DI = so.D_MODEL, so.D_INTER
KEYS = ("newnlb.theta.weight", "newnlb.theta.bias", "newnlb.phi.weight", "newnlb.phi.bias", "newnlb.g.weight",
        "newnlb.g.bias", "newnlb.W.weight", "newnlb.W.bias", "newnlb.concat_project.0.weight",
        "attention_scorer.weight", "attention_scorer.bias", "last.weight", "last.bias")
AGG_KEYS = KEYS[:11]
FIELD_KEY = dict(zip(SeamWeightGrads.FIELDS, AGG_KEYS))      # field of struct seam_weight_grads -> state_dict key


def nlb_collapsed_pool_backward(x, o, w):
    """Vector-Jacobian product of ``so.nlb_collapsed_pool`` for ONE track, in float64: the closed form the backward
    kernel implements (DESIGN.md §4 f4).  x: (T,256), o = d loss / d pooled (256,) -> (dx (T,256), {state_dict key:
    gradient} for the 11 aggregator parameters)."""
    x, o = x.double(), o.double()
    T = x.shape[0]
    g = {k: torch.zeros(w[k].shape, dtype=torch.float64) for k in AGG_KEYS}
    if T <= 1:                                   # T == 1: the block is skipped and p = 1 (match_head.py:145-147)
        return o.expand(T, D).clone(), g
    Wt, Wp = w["newnlb.theta.weight"].double()[:, :, 0], w["newnlb.phi.weight"].double()[:, :, 0]
    Wg, WW = w["newnlb.g.weight"].double()[:, :, 0], w["newnlb.W.weight"].double()[:, :, 0]
    bt, bp = w["newnlb.theta.bias"].double(), w["newnlb.phi.bias"].double()
    bg, bW = w["newnlb.g.bias"].double(), w["newnlb.W.bias"].double()
    wc = w["newnlb.concat_project.0.weight"].double().reshape(-1)
    wt, wp = wc[:DI], wc[DI:]
    wa, ba = w["attention_scorer.weight"].double()[0], w["attention_scorer.bias"].double()[0]
    # folded vectors
    ut, ct = Wt.T @ wt, bt @ wt
    up, cp = Wp.T @ wp, bp @ wp
    nu = WW.T @ wa
    ug, cg = Wg.T @ nu, bg @ nu
    cs = bW @ wa + ba
    # per track
    mu = WW.T @ o
    m, cmu, e0 = Wg.T @ mu, bg @ mu, bW @ o
    a, b, c, d = x @ ut + ct, x @ up + cp, x @ ug + cg, x @ wa
    gam, e = x @ m + cmu, x @ o
    pre = a[:, None] + b[None, :]
    f = torch.relu(pre) / T
    p = torch.softmax(d + f @ c + cs, 0)
    h = e + f @ gam + e0
    ds = p * (h - p @ h)
    q, qp = p @ f, ds @ f
    gg = (pre > 0).double() * (p[:, None] * gam[None, :] + ds[:, None] * c[None, :]) / T
    al, be = gg.sum(1), gg.sum(0)
    dx = (p[:, None] * o + ds[:, None] * wa + al[:, None] * ut + be[:, None] * up + q[:, None] * m
          + qp[:, None] * ug)
    r, rp, A, B, E = q @ x, qp @ x, al @ x, be @ x, ds @ x
    hr, hrp = Wg @ r + q.sum() * bg, Wg @ rp + qp.sum() * bg
    S = ds.sum()
    g["newnlb.theta.weight"] = torch.outer(wt, A)[:, :, None]
    g["newnlb.theta.bias"] = al.sum() * wt
    g["newnlb.phi.weight"] = torch.outer(wp, B)[:, :, None]
    g["newnlb.phi.bias"] = be.sum() * wp
    g["newnlb.concat_project.0.weight"] = torch.cat([Wt @ A + al.sum() * bt, Wp @ B + be.sum() * bp]).view(1, 2 * DI, 1, 1)
    g["newnlb.g.weight"] = (torch.outer(mu, r) + torch.outer(nu, rp))[:, :, None]
    g["newnlb.g.bias"] = q.sum() * mu + qp.sum() * nu
    g["newnlb.W.weight"] = (torch.outer(o, hr) + torch.outer(wa, hrp))[:, :, None]
    g["newnlb.W.bias"] = o + S * wa
    g["attention_scorer.weight"] = (E + WW @ hrp + S * bW)[None, :]
    g["attention_scorer.bias"] = S.view(1)
    return dx, g


def _loss(x3_1b, x5, r1, r2):
    return (x5 * r2).sum() + (x3_1b * r1).sum() + torch.logsumexp(x5, -1).mean()


def _check(name, got, ref, rel=2e-4):
    ref = ref.float()
    tol = rel * max(1.0, float(ref.abs().max()))
    err = float((got.float().cpu() - ref).abs().max())
    assert err <= tol, f"{name}: |grad - autograd|max = {err:.3e} (scale {float(ref.abs().max()):.3e})"


def _autograd_aggregate(seq, mask, weights, dout, use_nlb=True):
    """fp64 autograd through the oracle's un-folded aggregation: (dseq, {key: grad or zeros})."""
    w64 = {k: v.double().clone().requires_grad_(True) for k, v in weights.items()}
    seq64 = seq.double().clone().requires_grad_(True)
    out, _ = so.aggregate_tracks(seq64, mask, w64, use_nlb=use_nlb)
    (out * dout.double()).sum().backward()
    grads = {k: (w64[k].grad if w64[k].grad is not None else torch.zeros_like(w64[k])) for k in AGG_KEYS}
    return seq64.grad, grads


# ------------------------------------------------------------------------------------------------ CPU: the algebra
@pytest.mark.parametrize("T", [1, 2, 17, 64])
def test_closed_form_backward_matches_autograd(weights, T):
    seq, mask, _ = so.synth_tracks(1, T, seed=70 + T)
    o = torch.randn(1, D, generator=torch.Generator().manual_seed(T))
    dseq, ref = _autograd_aggregate(seq, mask, weights, o)
    dx, got = nlb_collapsed_pool_backward(seq[1:, 0], o[0], weights)
    scale = float(dseq.abs().max())
    assert float((dx - dseq[1:, 0]).abs().max()) <= 1e-12 * scale
    for k in AGG_KEYS:
        assert got[k].shape == ref[k].shape, k
        if k == "attention_scorer.bias":            # analytically zero: compared absolutely
            assert float((got[k] - ref[k]).abs().max()) <= 1e-12, k
            continue
        scale = max(float(ref[k].abs().max()), 1e-300)
        assert float((got[k] - ref[k]).abs().max()) <= 1e-12 * scale, k


# ------------------------------------------------------------------------------------------------ GPU: the kernel
@pytest.mark.gpu
@pytest.mark.parametrize("Q,T,G,ragged", [(6, 17, 5, None), (5, 24, 4, (1, 24)), (4, 32, 3, (0, 32)),
                                          (3, 64, 4, None), (7, 50, 5, (1, 50))])
def test_long_tracks_through_the_module(weights, Q, T, G, ragged):
    seq, mask, lens = so.synth_tracks(Q, T, seed=80 + T, ragged=ragged)
    gal = so.synth_gallery(G, 80 + T, None)
    r1 = torch.randn(Q, D, generator=torch.Generator().manual_seed(1))
    r2 = torch.randn(Q, G, 2, generator=torch.Generator().manual_seed(2))
    w64 = {k: v.double().clone().requires_grad_(True) for k, v in weights.items()}
    seq64, gal64 = seq.double().clone().requires_grad_(True), gal.double().clone().requires_grad_(True)
    out = so.forward_seq_branch(seq64, mask, gal64, w64)
    _loss(out[0], out[2], r1.double(), r2.double()).backward()
    m = pkg.TemporalAggregationNLB().to(DEV).train()
    m.load_state_dict(weights, strict=False)
    seq_d, gal_d = seq.to(DEV).requires_grad_(True), gal.to(DEV).requires_grad_(True)
    x3_1b, _, x5, _, _, _ = m(None, None, None, x3_1_seq=seq_d, x3_1_mask=mask.to(DEV), x3_2=gal_d)
    _loss(x3_1b, x5, r1.to(DEV), r2.to(DEV)).backward()
    _check("x3_1_seq", seq_d.grad, seq64.grad)
    _check("x3_2", gal_d.grad, gal64.grad)
    sd = dict(m.named_parameters())
    for k in KEYS:
        _check(k, sd[k].grad, w64[k].grad if w64[k].grad is not None else torch.zeros_like(w64[k]))


def _agg_params(weights):
    return {f: weights[k].to(DEV) for f, k in FIELD_KEY.items()}


@pytest.mark.gpu
def test_many_ragged_tracks(engine, weights):
    """~600 tracks of 1-64 frames: several waves of CTAs and heavy atomic traffic on the parameter gradients."""
    Q, T = 600, 64
    seq, mask, lens = so.synth_tracks(Q, T, seed=91, ragged=(1, 64))
    dout = torch.randn(Q, D, generator=torch.Generator().manual_seed(92))
    ref_dseq, ref = _autograd_aggregate(seq, mask, weights, dout)
    params = _agg_params(weights)
    seq_d, dout_d = seq.to(DEV), dout.to(DEV)
    dseq, grads = engine.aggregate_backward(seq_d, mask.to(DEV), None, params, dout_d)
    _check("dseq", dseq, ref_dseq)
    for f, k in FIELD_KEY.items():
        _check(k, grads[f].view(ref[k].shape), ref[k])
    dseq_lens, _ = engine.aggregate_backward(seq_d, None, torch.from_numpy(lens).to(DEV), params, dout_d)
    dseq_again, _ = engine.aggregate_backward(seq_d, mask.to(DEV), None, params, dout_d)
    assert torch.equal(dseq, dseq_lens)
    assert torch.equal(dseq, dseq_again)


@pytest.mark.gpu
def test_strided_track_slice(engine, weights):
    seq, mask, _ = so.synth_tracks(40, 33, seed=93, ragged=(0, 33))
    dout = torch.randn(21, D, generator=torch.Generator().manual_seed(94)).to(DEV)
    params = _agg_params(weights)
    view = seq.to(DEV)[:, 10:31]
    assert not view.is_contiguous()
    a, ga = engine.aggregate_backward(view, mask[10:31].to(DEV), None, params, dout)
    b, gb = engine.aggregate_backward(view.contiguous(), mask[10:31].to(DEV), None, params, dout)
    assert torch.equal(a, b)
    for f in ga:
        _check(f, ga[f], gb[f].cpu(), rel=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [10, 40])
def test_training_with_nlb_false(weights, T):
    Q, G = 5, 4
    seq, mask, _ = so.synth_tracks(Q, T, seed=95 + T, ragged=(1, T))
    gal = so.synth_gallery(G, 95 + T, None)
    r1 = torch.randn(Q, D, generator=torch.Generator().manual_seed(1))
    r2 = torch.randn(Q, G, 2, generator=torch.Generator().manual_seed(2))
    w64 = {k: v.double().clone().requires_grad_(True) for k, v in weights.items()}
    seq64, gal64 = seq.double().clone().requires_grad_(True), gal.double().clone().requires_grad_(True)
    x3_1b64, _ = so.aggregate_tracks(seq64, mask, w64, use_nlb=False)
    _loss(x3_1b64, so.pair_logits(x3_1b64, gal64, w64), r1.double(), r2.double()).backward()
    m = pkg.TemporalAggregationNLB().to(DEV).train()
    m.load_state_dict(weights, strict=False)
    m.nlb = False
    seq_d, gal_d = seq.to(DEV).requires_grad_(True), gal.to(DEV).requires_grad_(True)
    x3_1b, _, x5, _, _, _ = m(None, None, None, x3_1_seq=seq_d, x3_1_mask=mask.to(DEV), x3_2=gal_d)
    _check("x3_1b", x3_1b.detach(), x3_1b64.detach(), rel=2e-5)
    _loss(x3_1b, x5, r1.to(DEV), r2.to(DEV)).backward()
    _check("x3_1_seq", seq_d.grad, seq64.grad)
    _check("x3_2", gal_d.grad, gal64.grad)
    sd = dict(m.named_parameters())
    for k in ("attention_scorer.weight", "attention_scorer.bias", "last.weight", "last.bias"):
        _check(k, sd[k].grad, w64[k].grad)
    before = {k: v.detach().clone() for k, v in sd.items() if k.startswith("newnlb.")}
    assert before and all(sd[k].grad is None for k in before)
    torch.optim.SGD(m.parameters(), lr=0.1).step()
    assert all(torch.equal(sd[k].detach(), before[k]) for k in before)


@pytest.mark.gpu
def test_x_branch_with_a_long_track(weights):
    """ids that group into one 40-frame track plus short ones: the x-branch trains, gradients reach the tower, and the
    aggregator's gradients equal those of the seq-branch call on the grouped tracks."""
    torch.manual_seed(5)
    m = pkg.TemporalAggregationNLB().to(DEV).train()
    m.load_state_dict(weights, strict=False)
    ids = torch.tensor([7] * 40 + [3, 3, 11] + [0, 1, 2])
    types = torch.tensor([0] * 43 + [1, 1, 1])
    perm = torch.randperm(ids.numel())
    ids, types = ids[perm], types[perm]
    x = torch.randn(ids.numel(), 256, 14, 14, device=DEV)
    x3_1b, x3_2, x5, seq, mask, _ = m(x, types, ids)
    assert seq.shape == (41, 3, 256)
    r1 = torch.randn(3, D, device=DEV)
    r2 = torch.randn(3, 3, 2, device=DEV)
    _loss(x3_1b, x5, r1, r2).backward()
    assert float(m.conv_seq[0].weight.grad.abs().sum()) > 0
    sd = dict(m.named_parameters())
    xb = {k: sd[k].grad.clone() for k in KEYS}
    m.zero_grad(set_to_none=True)
    y3_1b, _, y5, _, _, _ = m(None, None, None, x3_1_seq=seq.detach(), x3_1_mask=mask, x3_2=x3_2.detach())
    _loss(y3_1b, y5, r1, r2).backward()
    for k in KEYS:
        _check(k, xb[k], sd[k].grad.cpu())


@pytest.mark.gpu
def test_backward_limits(engine, weights):
    params = _agg_params(weights)
    with pytest.raises(pkg.SeamError):
        engine.aggregate_backward(torch.zeros(66, 2, D, device=DEV), None, None, params, torch.zeros(2, D, device=DEV))
    # the C entry refuses Tmax > SEAM_MAX_T on its own
    seq = torch.zeros(66, 2, D, device=DEV)
    dseq = torch.zeros(66, 2, D, device=DEV)
    dout = torch.zeros(2, D, device=DEV)
    w = SeamWeights(**{f: (params[f].data_ptr() if f in params else 0) for f in SeamWeights.FIELDS})
    grads = {f: torch.zeros_like(params[f]) for f in FIELD_KEY}
    gs = SeamWeightGrads(**{f: grads[f].data_ptr() for f in FIELD_KEY})
    st = engine._lib.seam_aggregate_backward(engine._h, C.byref(w), seq.data_ptr(), None, None, 65, 2, seq.stride(0),
                                             seq.stride(1), dout.data_ptr(), dseq.data_ptr(), C.byref(gs), None)
    assert st == 2
    for Q, T in ((0, 10), (3, 0)):
        dseq, g = engine.aggregate_backward(torch.randn(1 + T, Q, D, device=DEV), None, None, params,
                                            torch.randn(Q, D, device=DEV))
        assert dseq.shape == (1 + T, Q, D) and not dseq.any()
        assert all(not v.any() for v in g.values())
