"""The scorer's certification error model, checked on the CPU.

The tensor-core pass ranks pair (i, j) by v^_ij = fp16(a_i) . fp16(g_j) + cg_j (a_i = -2 dw (.) q_i, cg_j = dw . g_j^2,
score_tc.cuh); the re-score kernel trusts |v^ - v| <= eps_i for every pair of the row (score_exact.cuh,
rescore_kernel), and the rank-of-target path builds its band v* +- E_i on the same bound (rank_prep_kernel).  Here the
preparation kernels' fp32 arithmetic is restated (same lanes, same fma chains, same butterflies), the operands are
rounded to fp16 as the device rounds them, v^ is formed in float64 and compared with the exact v, also in float64.
The constants are read out of score_exact.cuh, so the test follows the source."""
import os
import re

import numpy as np
import pytest
import torch

from oracle import seam_oracle as so

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "seam-match-rcnn_b200", "csrc", "score_exact.cuh")
SCALES = (-24, -16, -14, -10, 0, 8, 14)
FP16_MAX = 65504.0
U32 = 2.0 ** -24                  # unit roundoff of fp32


def source_constants():
    """EPS_COEFF, SUB_COEFF, CG_COEFF, DIRECT_COEFF, EPS_ABS, TAG_REL_ERR and RANK_SLACK as score_exact.cuh defines
    them."""
    text = open(SRC).read()
    out = {}
    for name in ("EPS_COEFF", "SUB_COEFF", "CG_COEFF", "DIRECT_COEFF", "EPS_ABS", "TAG_REL_ERR", "RANK_SLACK"):
        m = re.search(r"constexpr\s+float\s+" + name + r"\s*=\s*([0-9.eE+-]+)f\s*;", text)
        assert m, f"{name} not found in score_exact.cuh"
        out[name] = float(m.group(1))
    return out


# ------------------------------------------------------------------------------------------ the kernels' fp32 sums
def _lanes(x):
    """(N,256) -> (N,32,8): lane l holds elements [4l, 4l+4) and [128+4l, 128+4l+4) (load_slice)."""
    x = x.reshape(x.shape[0], 2, 32, 4)
    return np.concatenate([x[:, 0], x[:, 1]], axis=2)


def _fma32(a, b, c):
    """fmaf: one rounding of a*b + c (the float64 product of two fp32 values is exact)."""
    return (a.astype(np.float64) * b + c).astype(np.float32)


def _warp_sum(v):
    """ptx::warp_sum over the lane axis: butterfly at distances 16, 8, 4, 2, 1 in fp32."""
    lane = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        v = (v + v[:, lane ^ o]).astype(np.float32)
    return v[:, 0]


def _wabs(W):
    """|W_0| + |W_1| as the preparation kernels form it (fp32)."""
    return (np.abs(W[0]) + np.abs(W[1])).astype(np.float32)


def prep_queries(q, W):
    """prep_queries_kernel: a = -2 dw (.) q (fp32) and its fp16 image, rq = dw . q^2, ||a||; and qw = (|W_0| + |W_1|)
    . q^2 as weighted_sq_norm forms it (rescore_kernel, rank_prep_kernel)."""
    dw = (W[1] - W[0]).astype(np.float32)                                 # fold_scorer_kernel
    x, d, wa = _lanes(q.astype(np.float32)), _lanes(dw[None]), _lanes(_wabs(W)[None])
    a = ((np.float32(-2.0) * d) * x).astype(np.float32)
    r = np.zeros(x.shape[:2], np.float32)
    qw = np.zeros(x.shape[:2], np.float32)
    n2 = np.zeros(x.shape[:2], np.float32)
    for e in range(8):
        xx = (x[:, :, e] * x[:, :, e]).astype(np.float32)
        r = _fma32(d[:, :, e], xx, r)
        qw = _fma32(wa[:, :, e], xx, qw)
        n2 = _fma32(a[:, :, e], a[:, :, e], n2)
    a_rows = np.concatenate([a[:, :, :4].reshape(-1, 128), a[:, :, 4:].reshape(-1, 128)], axis=1)
    a16 = torch.from_numpy(a_rows).half().double().numpy()
    amax = np.abs(a_rows).max(1)
    return a16, _warp_sum(r), np.sqrt(_warp_sum(n2)).astype(np.float32), _warp_sum(qw), amax


def prep_gallery(g, W):
    """prep_gallery_kernel: cg = dw . g^2 (fp32), the fp16 image of g and gstat: max_j ||g_j||, the overflow flag,
    max_j |dw| . g_j^2, max_j gw_j."""
    dw = (W[1] - W[0]).astype(np.float32)
    x, d, wa = _lanes(g.astype(np.float32)), _lanes(dw[None]), _lanes(_wabs(W)[None])
    c = np.zeros(x.shape[:2], np.float32)
    cabs = np.zeros(x.shape[:2], np.float32)
    gw = np.zeros(x.shape[:2], np.float32)
    n2 = np.zeros(x.shape[:2], np.float32)
    for e in range(8):
        xx = (x[:, :, e] * x[:, :, e]).astype(np.float32)
        c = _fma32(d[:, :, e], xx, c)
        cabs = _fma32(np.abs(d[:, :, e]), xx, cabs)
        gw = _fma32(wa[:, :, e], xx, gw)
        n2 = _fma32(x[:, :, e], x[:, :, e], n2)
    g16 = torch.from_numpy(g.astype(np.float32)).half().double().numpy()
    gstat = (np.float32(np.sqrt(_warp_sum(n2)).max()), not (np.abs(g).max() < FP16_MAX), _warp_sum(cabs).max(),
             _warp_sum(gw).max())
    return g16, _warp_sum(c), gstat


def _warp_sum_b(v):
    """ptx::warp_sum_b: butterfly at lane distances 4, 2, 1, 8, 16 (treduce<8>'s association)."""
    lane = np.arange(32)
    for o in (4, 2, 1, 8, 16):
        v = (v + v[..., lane ^ o]).astype(np.float32)
    return v[..., 0]


def direct_form(q, g, W, b):
    """The fp32 direct-form margin d~ = l1 - l0 of every pair as rescore_kernel / exact_topk_kernel /
    rank_of_target_kernel form it: per lane, even and odd channels of the slice in two chains (sub, square, mul then
    three fmas: sqdiff_dot2), their sum, the warp_sum_b butterfly, + b_c, then l1 - l0."""
    q32, g32 = _lanes(q.astype(np.float32)), _lanes(g.astype(np.float32))
    out = np.empty((q.shape[0], g.shape[0]), np.float32)
    logits = []
    for c in (0, 1):
        wl = _lanes(W[c][None].astype(np.float32))[0]                     # (32,8)
        lc = np.empty((q.shape[0], g.shape[0]), np.float32)
        for i in range(q.shape[0]):
            dd = (q32[i][None] - g32).astype(np.float32)                   # (G,32,8)
            sq = (dd * dd).astype(np.float32)
            half = []
            for par in (0, 1):                                             # lo (x, z) and hi (y, w) of each float2 pair
                es = [par, 2 + par, 4 + par, 6 + par]
                acc = (wl[:, es[0]] * sq[:, :, es[0]]).astype(np.float32)
                for e in es[1:]:
                    acc = _fma32(wl[:, e], sq[:, :, e], acc)
                half.append(acc)
            part = (half[0] + half[1]).astype(np.float32)                  # sum2
            lc[i] = (_warp_sum_b(part) + np.float32(b[c])).astype(np.float32)
        logits.append(lc)
    out[:] = (logits[1] - logits[0]).astype(np.float32)
    return out


# ------------------------------------------------------------------------------------------ the error model
def pair_errors(q, g, W, b):
    """For every pair: v^ (the tensor-core value before its column tag, rounded to fp32 as acc + cg is; the fp16
    products are summed exactly here, so the tensor core's fp32 accumulation -- covered by EPS_COEFF's slack over
    2^-10 -- is not exercised), the exact v = (W1 - W0) . ((q - g)^2 - q^2) in float64 (the margin less the row's
    constant rq + db), the exact margin d, and the preparation outputs rq, qstat and gstat.  Returns None where the
    kernel would not certify (fp16 overflow)."""
    W = W.astype(np.float32)
    a16, rq, anorm, qw, aabs = prep_queries(q, W)
    dw = (W[1] - W[0]).astype(np.float32)
    g16, cg, gstat = prep_gallery(g, W)
    if gstat[1] or not (aabs.max() < FP16_MAX):
        return None
    vhat = (a16 @ g16.T + cg.astype(np.float64)[None]).astype(np.float32).astype(np.float64)
    dwx = W[1].astype(np.float64) - W[0].astype(np.float64)
    q64, g64 = q.astype(np.float64), g.astype(np.float64)
    v = (-2.0 * (q64 * dwx) @ g64.T) + ((g64 * g64) @ dwx)[None]
    d = v + ((q64 * q64) @ dwx)[:, None] + (float(b[1]) - float(b[0]))
    assert dw.dtype == np.float32
    return dict(vhat=vhat, v=v, d=d, rq=rq, anorm=anorm.astype(np.float64), qw=qw.astype(np.float64), gstat=gstat)


def operand_bound(c, anorm, gstat):
    """operand_err_bound (score_exact.cuh): fp16 operands (relative: EPS_COEFF; subnormals, absolute 2^-25 per element:
    SUB_COEFF), the fp32 rounding of cg (CG_COEFF) and fp32 accumulation (EPS_ABS)."""
    an, gm, ca = np.float32(anorm), np.float32(gstat[0]), np.float32(gstat[2])
    return (np.float32(c["EPS_COEFF"]) * an * gm + np.float32(c["SUB_COEFF"]) * (an + gm)
            + np.float32(c["CG_COEFF"]) * ca + np.float32(c["EPS_ABS"]))


def direct_bound(c, qw, gstat, b):
    """direct_err_bound (score_exact.cuh): the fp32 direct form's rounding."""
    return np.float32(c["DIRECT_COEFF"]) * (2 * np.float32(qw) + 2 * np.float32(gstat[3])
                                            + abs(np.float32(b[0])) + abs(np.float32(b[1])))


def band_E(c, anorm, qw, gstat, b, vstar, dt):
    """rank_prep_kernel's band half-width E for a target with tensor-core image vstar and margin dt."""
    e0 = operand_bound(c, anorm, gstat) + direct_bound(c, qw, gstat, b) + np.float32(c["DIRECT_COEFF"]) * np.float32(qw)
    return (e0 + np.float32(c["TAG_REL_ERR"]) * (np.abs(vstar) + e0)
            + np.float32(c["RANK_SLACK"]) * (1.0 + np.abs(dt) + np.abs(vstar)))


def check_bound(q, g, W, b):
    """Worst ratios error / bound of the three claims the kernels rest on, for every pair:
      - |tagged v^ - v| <= the operand part of rescore_kernel's eps (+ its tag term);
      - |d~ - d| <= the direct-form part of eps (d~: the fp32 direct form, restated operation by operation);
      - the rank band: every item j taken as the target, |tagged v^_j - v*_j| <= E_j, where v*_j = d~_j - rq - db is
        formed in fp32 as rank_prep_kernel forms it (so rq's fp32 rounding is included).
    The column tag replaces 6 low mantissa bits: its error, at most 2^-17 |v^|, is added worst case; the window's amax
    is at least the pair's own |v^|."""
    m = pair_errors(q, g, W, b)
    assert m is not None, "the case overflows fp16: the kernel would not certify it"
    c = source_constants()
    vhat = m["vhat"]
    w = vhat + 2.0 ** -17 * np.abs(vhat)
    r_op = (np.abs(vhat - m["v"]) + 2.0 ** -17 * np.abs(vhat)) / (
        operand_bound(c, m["anorm"][:, None], m["gstat"]) + np.float32(c["TAG_REL_ERR"]) * np.abs(vhat))
    dt = direct_form(q, g, W, b)
    r_dir = np.abs(dt - m["d"]) / direct_bound(c, m["qw"][:, None], m["gstat"], b)
    db = np.float32(np.float32(b[1]) - np.float32(b[0]))
    vstar = ((dt - m["rq"][:, None]).astype(np.float32) - db).astype(np.float32)
    E = band_E(c, m["anorm"][:, None], m["qw"][:, None], m["gstat"], b, vstar, dt)
    r_E = (np.abs(vhat - vstar) + np.abs(w - vhat)) / E
    return float(r_op.max()), float(r_dir.max()), float(r_E.max())


# ------------------------------------------------------------------------------------------ cases
@pytest.fixture(scope="module")
def last():
    w = so.random_weights(seed=0)
    return w["last.weight"].numpy(), w["last.bias"].numpy()


def _random(Q, G, seed):
    rs = np.random.RandomState(seed)
    return rs.randn(Q, 256).astype(np.float32), rs.randn(G, 256).astype(np.float32)


def subnormal_half_step_case(W, G=4, mass=(1647.0, 4942.0, 49423.0)):
    """A query whose every a_k lies just under half the smallest fp16 subnormal (2^-25), so that fp16(a) == 0 and the
    tensor-core value of every pair is cg alone; gallery rows of L1 mass `mass` arranged so that cg = dw . g^2 is ~0
    and a . g = 0.99 * 2^-25 * ||g||_1 is entirely lost.  Returns (q (1,256), g (len(mass),256))."""
    dw = (W[1].astype(np.float32) - W[0].astype(np.float32)).astype(np.float64)
    q = (-np.sign(dw) * 0.99 * 2.0 ** -25 / (2.0 * np.abs(dw))).astype(np.float32)
    a = (np.float32(-2.0) * dw.astype(np.float32)) * q
    assert (np.abs(a) < 2.0 ** -25).all() and (a > 0).all()
    pos, neg = dw > 0, dw < 0
    sp, sn = dw[pos].sum(), -dw[neg].sum()
    rows = []
    for m1 in mass:
        shape = np.where(pos, np.sqrt(sn / sp), 1.0)                      # sum_k dw_k shape_k^2 = 0
        rows.append(shape * (m1 / shape.sum()))
    return q[None], np.stack(rows).astype(np.float32)


def test_constants_are_read_from_the_source():
    c = source_constants()
    assert 2.0 ** -10 < c["EPS_COEFF"] < 1.1 * 2.0 ** -10      # two fp16 operand roundings of 2^-11 + slack
    assert 2.0 ** -17 < c["TAG_REL_ERR"] < 1.1 * 2.0 ** -17   # six mantissa bits replaced by the column tag
    assert c["SUB_COEFF"] >= 16 * 2.0 ** -25 * 1.001         # 2^-25 per fp16 subnormal element, ||x||_1 <= 16 ||x||_2
    assert c["CG_COEFF"] >= 14 * U32                         # the 14 roundings of cg = dw . g^2
    assert c["DIRECT_COEFF"] >= 15 * U32                     # 14 roundings per logit, l1 - l0


def test_random_data(last):
    q, g = _random(64, 512, 1)
    assert max(check_bound(q, g, *last)) <= 1.0


@pytest.mark.parametrize("sq", SCALES)
@pytest.mark.parametrize("sg", SCALES)
def test_operand_scales(sq, sg, last):
    """Queries and gallery scaled independently by powers of two: the fp16 operands go subnormal, underflow to zero
    or approach the fp16 range."""
    q, g = _random(24, 160, 2)
    q, g = q * np.float32(2.0 ** sq), g * np.float32(2.0 ** sg)
    g = np.clip(g, -60000.0, 60000.0)                # 2^14 x N(0,1) tails past 65504 would only disable certification
    q = np.clip(q, -2.0 ** 14, 2.0 ** 14)
    r = check_bound(q, g, *last)
    assert max(r) <= 1.0, r


def test_all_subnormal_operands(last):
    """Every element of a (resp. g) in fp16's subnormal range."""
    W = last[0]
    dw = (W[1] - W[0]).astype(np.float32)
    q, g = _random(16, 256, 3)
    qa = (np.sign(q) * 2.0 ** -16 / (2.0 * np.abs(dw)[None]) * np.abs(q).clip(0.05, 1.0)).astype(np.float32)
    gs = (g * np.float32(2.0 ** -17)).astype(np.float32)
    for qq, gg in ((qa, g), (q, gs), (qa, gs)):
        r = check_bound(qq, gg, *last)
        assert max(r) <= 1.0, r


def test_subnormal_half_step_query(last):
    """fp16(a) == 0 while a . g is several times the absolute term of the old bound (4.8e-5 .. 1.4e-3 against 1e-5)."""
    q, g = subnormal_half_step_case(last[0])
    m = pair_errors(q, g, *last)
    assert (np.abs(m["vhat"] - m["v"]) > 4e-5).all()           # the case is what it claims to be
    r = check_bound(q, g, *last)
    assert max(r) <= 1.0, r


def test_dw_much_smaller_than_w(last):
    """W[0] ~= W[1]: dw = W[1] - W[0] is 1e-4 of W (a legitimate `last` through engine.scorer)."""
    rs = np.random.RandomState(4)
    base = last[0][0]
    W = np.stack([base, base + 1e-4 * np.abs(base).max() * rs.randn(256)]).astype(np.float32)
    q, g = _random(32, 256, 5)
    r = check_bound(q, g, W, last[1])
    assert max(r) <= 1.0, r
