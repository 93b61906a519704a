"""GPU parity tests proper: the CUDA path, called through the C ABI, against the oracle and
the committed golden vectors (which came from the unmodified reference modules)."""
import numpy as np
import pytest
import torch

from oracle import seam_oracle as so
from util import (GOLDEN_CASES, TOL_ATT, TOL_EMB, TOL_LOGIT, TOL_SCORE, assert_topk_matches, case_inputs)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


# ----------------------------------------------------------------------------- (a) aggregation
@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_aggregate_golden(name, golden, weights, engine):
    case = GOLDEN_CASES[name]
    seq, mask, lens, _ = case_inputs(case, weights)
    out, att = engine.aggregate(seq.to(DEV), mask.to(DEV), getatt=True)
    ref = torch.from_numpy(golden[f"{name}.x3_1b"])
    assert (out.cpu() - ref).abs().max() <= TOL_EMB
    assert (att.cpu() - torch.from_numpy(golden[f"{name}.att"])).abs().max() <= TOL_ATT
    # explicit lengths instead of the mask give the same result
    out2 = engine.aggregate(seq.to(DEV), None, lens=torch.as_tensor(lens))
    assert torch.equal(out, out2)


def test_aggregate_t1_is_bit_exact(weights, engine):
    """T == 1 bypasses the block and softmax of one logit is 1: out == x_0 exactly
    (models/match_head.py:145-151)."""
    seq, mask, _ = so.synth_tracks(33, 1, seed=4)
    out = engine.aggregate(seq.to(DEV), mask.to(DEV))
    assert torch.equal(out.cpu(), seq[1])


def test_aggregate_mask_semantics(weights, engine):
    """First True ends the track even when later entries are False; an all-padding track gives
    zeros (sum over an empty softmax)."""
    rs = np.random.RandomState(8)
    seq = torch.from_numpy(rs.randn(6, 4, 256).astype(np.float32))
    mask = torch.tensor([[0, 0, 0, 1, 0, 0], [0, 0, 0, 0, 0, 0], [0, 1, 0, 0, 0, 0], [1, 0, 0, 0, 0, 0]], dtype=torch.bool)
    ref, _ = so.aggregate_tracks(seq, mask, weights)
    out = engine.aggregate(seq.to(DEV), mask.to(DEV)).cpu()
    assert (out - ref).abs().max() <= TOL_EMB
    assert torch.equal(out[2], torch.zeros(256)) and torch.equal(out[3], torch.zeros(256))


def test_aggregate_strided_input(weights, engine):
    """Non-contiguous track slices (as the sharded path passes) are read through strides."""
    seq, mask, _ = so.synth_tracks(50, 7, seed=21, ragged=(1, 7))
    ref, _ = so.aggregate_tracks(seq[:, 10:31], mask[10:31], weights)
    out = engine.aggregate(seq.to(DEV)[:, 10:31], mask.to(DEV)[10:31])
    assert (out.cpu() - ref).abs().max() <= TOL_EMB


@pytest.mark.parametrize("Q,T,ragged", [(40, 17, None), (21, 32, (1, 32)), (77, 40, (0, 40)), (33, 64, (1, 64)),
                                        (12, 16, (0, 16)), (50, 11, (1, 11))])
def test_aggregate_every_kernel_variant(Q, T, ragged, weights, engine):
    """One case per aggregation kernel: warp-per-track (T <= 4 / 10 / 16 are covered by the golden cases
    and here by T = 11..16), two warps per track (17..32 frames), four warps per track (33..64),
    ragged lengths including empty and single-frame tracks; mask path and lens path."""
    seq, mask, lens = so.synth_tracks(Q, T, seed=Q + T, ragged=ragged)
    ref, att = so.aggregate_tracks(seq, mask, weights)
    out, a = engine.aggregate(seq.to(DEV), mask.to(DEV), getatt=True)
    assert (out.cpu() - ref).abs().max() <= TOL_EMB
    aref = torch.zeros(Q, T)
    for i, p in enumerate(att):
        aref[i, :p.shape[0]] = p[:, 0]
    assert (a.cpu() - aref).abs().max() <= TOL_ATT
    out2 = engine.aggregate(seq.to(DEV), None, lens=torch.as_tensor(lens))
    assert torch.equal(out2, out)
    single = torch.as_tensor(lens) == 1                      # the reference skips the block for T == 1
    if single.any():
        assert torch.equal(out.cpu()[single], seq[1][single])


@pytest.mark.parametrize("Q,T,ragged", [(7500, 4, (1, 4)), (7200, 10, None), (7300, 9, (0, 9)), (7150, 16, None),
                                        (7250, 14, (2, 14)), (7400, 32, None), (7350, 27, (17, 27)), (7104, 64, None),
                                        (7200, 50, (33, 50))])
def test_aggregate_many_tracks_per_warp(Q, T, ragged, weights, engine):
    """Every kernel variant with MORE tracks than producers (three or more iterations per producer warp: buffers are
    refilled -- by the loader warp at T <= 10, by the producers themselves otherwise) and at least three tensor-core
    batches of 16 tracks per CTA (Q >= 3 x 16 x 148 SMs of a B200: the two batch buffers are reused from the third
    batch on), against the oracle on a sample of tracks; lens and mask paths agree bit for bit."""
    seq, mask, lens = so.synth_tracks(Q, T, seed=3 * Q + T, ragged=ragged)
    out = engine.aggregate(seq.to(DEV), mask.to(DEV))
    out2 = engine.aggregate(seq.to(DEV), None, lens=torch.as_tensor(lens))
    assert torch.equal(out, out2)
    rows = torch.from_numpy(np.random.RandomState(Q).choice(Q, 160, replace=False)).sort().values
    rows = torch.cat([rows, torch.tensor([0, Q - 1])]).unique()
    ref, _ = so.aggregate_tracks(seq[:, rows], mask[rows], weights)
    assert (out.cpu()[rows] - ref).abs().max() <= TOL_EMB


def test_aggregate_empty_and_limits(engine):
    assert engine.aggregate(torch.zeros(1, 5, 256, device=DEV)).abs().sum() == 0     # Tmax == 0
    assert engine.aggregate(torch.zeros(4, 0, 256, device=DEV)).shape == (0, 256)    # Q == 0
    import seam_match_rcnn_b200 as pkg
    with pytest.raises(pkg.SeamError):
        engine.aggregate(torch.zeros(66, 2, 256, device=DEV))                        # T > 64


@pytest.mark.parametrize("t", [2, 7, 10])
def test_nlb_forward_golden(t, golden, engine):
    x = torch.from_numpy(golden[f"nlb.t{t}.x"]).to(DEV)
    z = engine.nlb_forward(x).cpu()
    assert (z - torch.from_numpy(golden[f"nlb.t{t}.z"])).abs().max() <= TOL_EMB


# ----------------------------------------------------------------------------- (b) scorer
@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_dense_logits_golden(name, golden, weights, engine):
    case = GOLDEN_CASES[name]
    seq, mask, _, gal = case_inputs(case, weights)
    q = torch.from_numpy(golden[f"{name}.x3_1b"])
    x5 = engine.score_dense(q.to(DEV), gal.to(DEV)).cpu()
    assert x5.shape == (case["Q"], case["G"], 2)
    assert (x5[:4] - torch.from_numpy(golden[f"{name}.x5_head"])).abs().max() <= TOL_LOGIT
    s = so.match_scores(x5).double().sum(1).numpy()
    np.testing.assert_allclose(s, golden[f"{name}.score_sum"], rtol=1e-5)


# ----------------------------------------------------------------------------- (c) top-k
@pytest.mark.parametrize("name", list(GOLDEN_CASES))
@pytest.mark.parametrize("k", [1, 5, 10, 20])
def test_topk_golden(name, k, golden, weights, engine):
    """End to end on the device (aggregation -> scorer -> top-k) against the reference's
    ranking stored in the goldens."""
    case = GOLDEN_CASES[name]
    seq, mask, _, gal = case_inputs(case, weights)
    q = engine.aggregate(seq.to(DEV), mask.to(DEV))
    g = engine.prepare_gallery(gal.to(DEV))
    sc, mg, ix = engine.score_topk(q, g, k)
    kk = min(k, case["G"])
    gi = torch.from_numpy(golden[f"{name}.topk_idx"])[:, :kk].long()
    gm = torch.from_numpy(golden[f"{name}.topk_margin"])[:, :kk]
    gs = torch.from_numpy(golden[f"{name}.topk_score"])[:, :kk]
    ix, mg, sc = ix.cpu().long(), mg.cpu(), sc.cpu()
    assert (ix[:, kk:] == -1).all()
    differs = ix[:, :kk] != gi
    # identical indices except ties inside the tolerance
    assert ((mg[:, :kk] - gm).abs() <= TOL_LOGIT).all()
    assert ((sc[:, :kk] - gs).abs() <= TOL_SCORE).all()
    assert not differs.any() or ((mg[:, :kk] - gm).abs()[differs] <= TOL_LOGIT).all()
    if name == "cfg1":
        assert not differs.any()


@pytest.mark.parametrize("Q,G,k", [(1, 1, 1), (3, 31, 20), (130, 257, 20), (257, 5000, 20), (64, 1000, 32),
                                   (500, 20000, 10)])
def test_topk_vs_oracle(Q, G, k, weights, engine):
    rs = np.random.RandomState(Q * 7 + G)
    q = torch.from_numpy(rs.randn(Q, 256).astype(np.float32))
    g = so.synth_gallery(G, seed=Q + G, planted=q)
    x5 = so.pair_logits(q, g, weights)
    gal = engine.prepare_gallery(g.to(DEV))
    sc, mg, ix = engine.score_topk(q.to(DEV), gal, k)
    assert_topk_matches(ix, mg, sc, so.logit_margin(x5), so.match_scores(x5), k)


def _random_shapes():
    rs = np.random.RandomState(20261017)
    shapes = []
    for _ in range(10):
        Q = int(rs.choice([1, 2, 37, 127, 128, 129, 300, 640]))
        G = int(rs.choice([1, 5, 255, 256, 257, 1023, 4097, 12000, 26000]))
        shapes.append((Q, G, int(rs.randint(1, 33))))
    return shapes + [(300, 26000, 20), (640, 12000, 32), (2, 26000, 7)]


@pytest.mark.parametrize("Q,G,k", _random_shapes())
def test_topk_random_shapes(Q, G, k, weights, engine):
    """Tile edges, single-tile and many-piece partitions, every k up to 32: the work decomposition
    (cost-balanced ranges, sweep order, sample tiles, sub-list slots) must never show in the results."""
    rs = np.random.RandomState(Q * 100003 + G * 17 + k)
    q = torch.from_numpy(rs.randn(Q, 256).astype(np.float32))
    g = so.synth_gallery(G, seed=Q + 3 * G + k, planted=q)
    x5 = so.pair_logits(q, g, weights, chunk=64)
    gal = engine.prepare_gallery(g.to(DEV))
    sc, mg, ix, stats = engine.score_topk(q.to(DEV), gal, k, return_stats=True)
    assert_topk_matches(ix, mg, sc, so.logit_margin(x5), so.match_scores(x5), k)
    if k <= 20:   # beyond ~24 the 2*eps window around the k-th value often fills the 32 nominated lanes
        assert int(stats[0]) <= max(1, Q // 20), "the candidate pass should certify nearly every row"


def test_topk_near_duplicates_take_exhaustive_path(weights, engine):
    """A gallery of near-identical items defeats the fp16 candidate pass (gaps below its error
    bound): those rows must be detected and re-ranked exhaustively, still matching the oracle."""
    rs = np.random.RandomState(3)
    q = torch.from_numpy(rs.randn(40, 256).astype(np.float32))
    base = torch.from_numpy(rs.randn(1, 256).astype(np.float32))
    g = base + 1e-4 * torch.from_numpy(rs.randn(3000, 256).astype(np.float32))
    x5 = so.pair_logits(q, g, weights)
    gal = engine.prepare_gallery(g.to(DEV))
    sc, mg, ix, stats = engine.score_topk(q.to(DEV), gal, 20, return_stats=True)
    assert int(stats[0]) > 0, "expected uncertified rows"
    assert_topk_matches(ix, mg, sc, so.logit_margin(x5), so.match_scores(x5), 20)


def test_topk_few_uncertified_rows_are_split_over_ctas(weights, engine):
    """A handful of rows with a crowd of near-ties at the top of a large gallery: the exhaustive kernel cuts each such
    row's gallery into slices (one CTA each) and merges the slice lists -- same answer as the oracle, stable over
    repeated calls (the per-row slice counters are left as found), for odd G and k up to 32."""
    rs = np.random.RandomState(11)
    Q, G = 200, 20011
    q = torch.from_numpy(rs.randn(Q, 256).astype(np.float32))
    g = torch.from_numpy(rs.randn(G, 256).astype(np.float32))
    x5 = so.pair_logits(q, g, weights, chunk=64)
    crowded = [3, 77, 199]
    for n, i in enumerate(crowded):                        # 40 near-copies of the row's best item, spread over the gallery
        best = int(so.logit_margin(x5)[i].argmax())
        rows = torch.from_numpy(rs.choice(G, 40, replace=False))
        rows = rows[rows != best]
        g[rows] = g[best] + 1e-5 * torch.from_numpy(rs.randn(len(rows), 256).astype(np.float32))
    x5 = so.pair_logits(q, g, weights, chunk=64)
    gal = engine.prepare_gallery(g.to(DEV))
    for k in (20, 32):
        first = None
        for _ in range(3):
            sc, mg, ix, stats = engine.score_topk(q.to(DEV), gal, k, return_stats=True)
            if k == 20:     # at k = 32 the window is full for every row: all rows take the exhaustive kernel, unsliced
                assert 3 <= int(stats[0]) < 148, "expected a few uncertified rows (fewer than CTAs: the sliced path)"
            assert_topk_matches(ix, mg, sc, so.logit_margin(x5), so.match_scores(x5), k)
            if first is None:
                first = (sc.clone(), mg.clone(), ix.clone())
            else:
                assert all(torch.equal(a, b) for a, b in zip(first, (sc, mg, ix)))


def test_topk_rising_gallery_overflows_candidate_lists(weights, engine):
    """A gallery whose margins rise with the row index makes nearly every new item beat the running
    bound: the per-thread candidate lists fill up, close, and the affected rows must be flagged and
    re-ranked exhaustively -- never silently truncated."""
    dw = (weights["last.weight"][1] - weights["last.weight"][0]).float()
    c = int(dw.argmax())
    assert dw[c] > 0
    rs = np.random.RandomState(8)
    Q, G, k = 96, 40000, 20
    q = torch.from_numpy(rs.randn(Q, 256).astype(np.float32))
    g = 0.05 * torch.from_numpy(rs.randn(G, 256).astype(np.float32))
    g[:, c] += torch.linspace(0.0, 40.0, G)              # dw . g^2 grows with the row index
    x5 = so.pair_logits(q, g, weights)
    gal = engine.prepare_gallery(g.to(DEV))
    sc, mg, ix, stats = engine.score_topk(q.to(DEV), gal, k, return_stats=True)
    assert int(stats[0]) > 0, "expected rows whose lists overflowed"
    assert_topk_matches(ix, mg, sc, so.logit_margin(x5), so.match_scores(x5), k, tol=2e-3)


def test_topk_fp16_overflow_is_safe(weights, engine):
    """Values beyond the fp16 range cannot go through the tensor-core pass; they are flagged and
    the exhaustive fp32 path answers."""
    rs = np.random.RandomState(5)
    q = torch.from_numpy(rs.randn(10, 256).astype(np.float32))
    g = torch.from_numpy(rs.randn(400, 256).astype(np.float32))
    g[7, 3] = 1.0e5
    x5 = so.pair_logits(q, g, weights)
    gal = engine.prepare_gallery(g.to(DEV))
    sc, mg, ix, stats = engine.score_topk(q.to(DEV), gal, 5, return_stats=True)
    assert int(stats[0]) == 10
    assert_topk_matches(ix, mg, sc, so.logit_margin(x5), so.match_scores(x5), 5, tol=2e-2)


# ----------------------------------------------------------------------------- rank of the target item
@pytest.mark.parametrize("Q,G", [(1, 1), (5, 33), (130, 257), (300, 5000), (97, 26000), (640, 12000)])
def test_rank_of_target_tensor_core_path(Q, G, weights, engine):
    """evaluate_movingfashion.py:268-269 for every query at once: the tensor-core path (count what is
    certainly above the target, decide the band in fp32) must give the integers of the exhaustive fp32
    kernel and of the oracle's argsort, for targets anywhere in the ranking."""
    rs = np.random.RandomState(Q * 31 + G)
    q = torch.from_numpy(rs.randn(Q, 256).astype(np.float32))
    g = so.synth_gallery(G, seed=Q + G, planted=q)
    target = torch.from_numpy(rs.randint(0, G, size=Q).astype(np.int64))
    target[::3] = torch.arange(Q)[::3] % G                    # planted items: ranks near the top
    gal = engine.prepare_gallery(g.to(DEV))
    r_fast, m_fast, stats = engine.rank_of_target(q.to(DEV), gal, target, return_stats=True)
    r_slow, m_slow = engine.rank_of_target(q.to(DEV), g.to(DEV), target)
    assert torch.equal(r_fast, r_slow) and torch.equal(m_fast, m_slow)
    assert int(stats[0]) <= max(1, Q // 20), "nearly every row should be certified by the tensor-core path"
    x5 = so.pair_logits(q, g, weights, chunk=64)
    ref = so.rank_of_target(x5, target)
    d = so.logit_margin(x5)
    bad = (r_fast.cpu().long() != ref).nonzero().flatten()
    for i in bad.tolist():                                     # only ties inside the stated tolerance may differ
        dt = d[i, target[i]]
        lo, hi = sorted((int(r_fast[i]), int(ref[i])))
        near = ((d[i] - dt).abs() <= TOL_LOGIT).sum()
        assert hi - lo <= int(near), (i, lo, hi, int(near))


def test_rank_of_target_crowded_band_and_overflow(weights, engine):
    """Near-identical gallery items all fall inside the error band around the target: every one of them
    is decided in exact fp32 (streamed through the resolve kernel) -- same integers as the exhaustive
    kernel; values beyond the fp16 range send every row to the exhaustive kernel."""
    rs = np.random.RandomState(12)
    q = torch.from_numpy(rs.randn(24, 256).astype(np.float32))
    base = torch.from_numpy(rs.randn(1, 256).astype(np.float32))
    g = base + 1e-4 * torch.from_numpy(rs.randn(3000, 256).astype(np.float32))
    target = torch.from_numpy(rs.randint(0, 3000, size=24).astype(np.int64))
    gal = engine.prepare_gallery(g.to(DEV))
    r_fast, _, stats = engine.rank_of_target(q.to(DEV), gal, target, return_stats=True)
    r_slow, _ = engine.rank_of_target(q.to(DEV), g.to(DEV), target)
    assert torch.equal(r_fast, r_slow)
    g[7, 3] = 1.0e5                                            # fp16 overflow: every row takes the exhaustive kernel
    gal = engine.prepare_gallery(g.to(DEV))
    r_fast, _, stats = engine.rank_of_target(q.to(DEV), gal, target, return_stats=True)
    r_slow, _ = engine.rank_of_target(q.to(DEV), g.to(DEV), target)
    assert int(stats[0]) == 24 and torch.equal(r_fast, r_slow)


def test_topk_empty(engine):
    q = torch.randn(5, 256, device=DEV)
    gal = engine.prepare_gallery(torch.zeros(0, 256, device=DEV))
    sc, mg, ix = engine.score_topk(q, gal, 3)
    assert (ix.cpu() == -1).all()
    gal = engine.prepare_gallery(torch.randn(9, 256, device=DEV))
    assert engine.score_topk(torch.zeros(0, 256, device=DEV), gal, 3)[2].shape == (0, 3)
    import seam_match_rcnn_b200 as pkg
    with pytest.raises(pkg.SeamError):
        engine.score_topk(q, gal, 33)


def test_rank_of_target_and_merge(weights, engine):
    rs = np.random.RandomState(11)
    q = torch.from_numpy(rs.randn(50, 256).astype(np.float32))
    g = torch.from_numpy(rs.randn(777, 256).astype(np.float32))
    tgt = torch.from_numpy(rs.randint(0, 777, size=50))
    x5 = so.pair_logits(q, g, weights)
    r, m = engine.rank_of_target(q.to(DEV), g.to(DEV), tgt)
    assert torch.equal(r.cpu().long(), so.rank_of_target(x5, tgt))
    # sharded search + merge == unsharded search
    bounds = [(0, 300), (300, 310), (310, 777)]
    S, M, I = [], [], []
    for a, b in bounds:
        gal = engine.prepare_gallery(g[a:b].to(DEV), index_offset=a)
        s, d, i = engine.score_topk(q.to(DEV), gal, 20)
        S.append(s), M.append(d), I.append(i)
    s, d, i = engine.merge_topk(torch.stack(S), torch.stack(M), torch.stack(I))
    s1, d1, i1 = engine.score_topk(q.to(DEV), engine.prepare_gallery(g.to(DEV)), 20)
    assert torch.equal(i, i1) and torch.equal(d, d1) and torch.equal(s, s1)
    assert_topk_matches(i, d, s, so.logit_margin(x5), so.match_scores(x5), 20)


# ----------------------------------------------------------------------------- full-size properties
def test_fullsize_cfg2_properties(weights, engine):
    """BASELINE.json configs[1]: 15k tracks x 10 frames vs 15k shop items.  Too big for the
    oracle end to end, so: (i) a 48-query sample against the oracle, (ii) planted matches are
    retrieved, (iii) permuting the gallery permutes the indices, (iv) sharding + merge is the
    identity, (v) lists are sorted."""
    Q, T, G, k = 15000, 10, 15000, 20
    gen = torch.Generator(device=DEV).manual_seed(1)
    seq = torch.zeros(1 + T, Q, 256, device=DEV)
    seq[1:] = torch.randn(T, Q, 256, device=DEV, generator=gen)
    q = engine.aggregate(seq)
    g = torch.randn(G, 256, device=DEV, generator=gen)
    g[:Q] = q + 0.1 * torch.randn(Q, 256, device=DEV, generator=gen)       # planted true match per query
    gal = engine.prepare_gallery(g)
    sc, mg, ix, stats = engine.score_topk(q, gal, k, return_stats=True)
    assert (mg[:, :-1] >= mg[:, 1:]).all()
    # (ii) the planted item ranks first for (nearly) every query: dw has mixed signs, so the
    # planted item need not maximise the margin, but it must be in the list where the oracle says so
    sample = torch.arange(0, Q, Q // 48)[:48]
    ref_q, _ = so.aggregate_tracks(seq[:, sample].cpu(), torch.zeros(len(sample), 1 + T, dtype=torch.bool), weights)
    assert (q[sample].cpu() - ref_q).abs().max() <= TOL_EMB
    x5 = so.pair_logits(q[sample].cpu(), g.cpu(), weights)
    assert_topk_matches(ix[sample], mg[sample], sc[sample], so.logit_margin(x5), so.match_scores(x5), k)
    # (iii) permutation equivariance
    perm = torch.randperm(G, device=DEV, generator=gen)
    sc2, mg2, ix2 = engine.score_topk(q, engine.prepare_gallery(g[perm]), k)
    assert torch.equal(perm[ix2.long()], ix.long()) or (mg2 - mg).abs().max() <= TOL_LOGIT
    assert (mg2 - mg).abs().max() <= TOL_LOGIT
    # (iv) shards + merge
    S, M, I = [], [], []
    for r in range(4):
        lo, hi = r * G // 4, (r + 1) * G // 4
        s, d, i = engine.score_topk(q, engine.prepare_gallery(g[lo:hi], index_offset=lo), k)
        S.append(s), M.append(d), I.append(i)
    s, d, i = engine.merge_topk(torch.stack(S), torch.stack(M), torch.stack(I))
    assert torch.equal(i, ix) and torch.equal(d, mg)


def test_fullsize_t64_aggregation(weights, engine):
    """configs[3] shape at reduced track count: T = 64, sample checked against the oracle;
    linearity-free invariants: permuting tracks permutes outputs, frame order inside a track is
    irrelevant to the pooled descriptor only through the attention weights (checked via oracle)."""
    Q, T = 4096, 64
    gen = torch.Generator(device=DEV).manual_seed(3)
    seq = torch.zeros(1 + T, Q, 256, device=DEV)
    seq[1:] = torch.randn(T, Q, 256, device=DEV, generator=gen)
    out = engine.aggregate(seq)
    sample = torch.arange(0, Q, Q // 16)[:16]
    ref, _ = so.aggregate_tracks(seq[:, sample].cpu(), torch.zeros(16, 1 + T, dtype=torch.bool), weights)
    assert (out[sample].cpu() - ref).abs().max() <= TOL_EMB
    perm = torch.randperm(Q, device=DEV, generator=gen)
    assert torch.equal(engine.aggregate(seq[:, perm].contiguous()), out[perm])


def _sample_check(engine, weights, seq, mask, lens, g, k, sample, q, sc, mg, ix):
    """`sample` queries of a full-size search against the oracle (aggregation + fp32 scorer + ranking)."""
    m_s = None if mask is None else mask[sample].cpu()
    if m_s is None:
        m_s = torch.zeros(len(sample), seq.shape[0], dtype=torch.bool)
    ref_q, _ = so.aggregate_tracks(seq[:, sample].cpu(), m_s, weights)
    assert (q[sample].cpu() - ref_q).abs().max() <= TOL_EMB
    x5 = so.pair_logits(q[sample].cpu(), g.cpu(), weights, chunk=8)
    return assert_topk_matches(ix[sample], mg[sample], sc[sample], so.logit_margin(x5), so.match_scores(x5), k)


def test_fullsize_cfg3_shape(weights, engine):
    """BASELINE.json configs[2]: 10,000 short multi-image queries (T_i in {2,3,4}, ragged mask, Tmax = 4)
    against a 50,000-item gallery with planted matches (SURVEY.md section 8(d), seed 2): a 64-query sample
    against the oracle, shards + merge = whole at the 2/4/8-GPU shard sizes, sortedness."""
    Q, T, G, k = 10000, 4, 50000, 20
    gen = torch.Generator(device=DEV).manual_seed(2)
    lens = torch.randint(2, 5, (Q,), device=DEV, generator=gen)
    seq = torch.zeros(1 + T, Q, 256, device=DEV)
    seq[1:] = torch.randn(T, Q, 256, device=DEV, generator=gen)
    mask = torch.arange(1 + T, device=DEV)[None, :] > lens[:, None]
    seq[1:] *= (~mask[:, 1:]).t()[:, :, None]
    q = engine.aggregate(seq, mask)
    assert torch.equal(q, engine.aggregate(seq, None, lens=lens))
    g = torch.randn(G, 256, device=DEV, generator=gen)
    g[:Q] = q + 0.1 * torch.randn(Q, 256, device=DEV, generator=gen)
    sc, mg, ix, stats = engine.score_topk(q, engine.prepare_gallery(g), k, return_stats=True)
    assert (mg[:, :-1] >= mg[:, 1:]).all()
    sample = torch.arange(0, Q, Q // 64)[:64]
    _sample_check(engine, weights, seq, mask, lens, g, k, sample, q, sc, mg, ix)
    for n in (2, 8):
        S, M, I = [], [], []
        for r in range(n):
            lo, hi = r * G // n, (r + 1) * G // n
            s, d, i = engine.score_topk(q, engine.prepare_gallery(g[lo:hi], index_offset=lo), k)
            S.append(s), M.append(d), I.append(i)
        s, d, i = engine.merge_topk(None, torch.stack(M), torch.stack(I))
        assert torch.equal(i, ix) and torch.equal(d, mg) and torch.equal(s, sc)


def test_fullsize_cfg5_shard_shape(weights, engine):
    """BASELINE.json configs[4] at its per-GPU shape on 8 GPUs: 10,000 queries x 10 frames against a 125,000-row
    gallery shard whose rows carry a global index offset (SURVEY.md section 8(d), seed 4).  A 64-query sample
    against the oracle; planted matches (first 10,000 rows) are found where the oracle finds them."""
    Q, T, G, k, off = 10000, 10, 125000, 20, 3 * 125000
    gen = torch.Generator(device=DEV).manual_seed(4)
    seq = torch.zeros(1 + T, Q, 256, device=DEV)
    seq[1:] = torch.randn(T, Q, 256, device=DEV, generator=gen)
    q = engine.aggregate(seq)
    g = torch.randn(G, 256, device=DEV, generator=gen)
    g[:Q] = q + 0.1 * torch.randn(Q, 256, device=DEV, generator=gen)
    sc, mg, ix = engine.score_topk(q, engine.prepare_gallery(g, index_offset=off), k)
    assert (mg[:, :-1] >= mg[:, 1:]).all() and int(ix.min()) >= off and int(ix.max()) < off + G
    sample = torch.arange(0, Q, Q // 64)[:64]
    _sample_check(engine, weights, seq, None, None, g, k, sample, q, sc, mg, ix - off)


def test_eval_script_fp16_operands(weights, engine):
    """SURVEY.md section 8 a8: the eval script scores the aggregated descriptor with an fp16-ROUNDED gallery and
    fp16-rounded `last` weights promoted to fp32 arithmetic (evaluate_movingfashion.py:82-92, 123-124, 263-267).
    Feeding the kernels the same rounded operands reproduces its scores and its ranking (argsort descending,
    :268) up to ties inside the stated tolerance."""
    import numpy as np
    Q, T, G, k = 48, 10, 3000, 20
    seq, mask, _ = so.synth_tracks(Q, T, seed=11)
    q, _ = so.aggregate_tracks(seq, mask, weights)                       # fp32 query (:262)
    gal = so.synth_gallery(G, 11, q)
    gal16 = gal.numpy().astype(np.float16)                               # shop_aggr stored as fp16 (:82-92)
    W16 = weights["last.weight"].numpy().astype(np.float16)              # :123
    B16 = weights["last.bias"].numpy().astype(np.float16)                # :124
    ref = np.concatenate([so.eval_aggr_scores_np(gal16, q[i].numpy(), W16, B16) for i in range(Q)], 0)   # (Q,G)
    assert ref.dtype == np.float32
    with engine.scorer(torch.from_numpy(W16.astype(np.float32)), torch.from_numpy(B16.astype(np.float32))):
        g = engine.prepare_gallery(torch.from_numpy(gal16.astype(np.float32)).to(DEV))
        sc, mg, ix = engine.score_topk(q.to(DEV), g, k)
        x5 = engine.score_dense(q.to(DEV), g.g).cpu()
    ref_t = torch.from_numpy(ref)
    # dense scores: softmax of the same fp32 logits
    assert (torch.softmax(x5, -1)[..., 1] - ref_t).abs().max() <= TOL_SCORE
    # ranking: the script's argsort order vs the fused top-k, ties inside the tolerance allowed
    order = torch.from_numpy(so.eval_rankings_np(ref)[:, :k].copy())
    got = ix.cpu().long()
    assert (torch.gather(ref_t, 1, got) - sc.cpu()).abs().max() <= TOL_SCORE
    differs = order != got
    d_full = so.logit_margin(x5)
    if differs.any():
        assert ((torch.gather(d_full, 1, order) - torch.gather(d_full, 1, got)).abs()[differs] <= 2 * TOL_LOGIT).all()
    # the engine's scorer is the module's again afterwards
    s2, _, i2 = engine.score_topk(q.to(DEV), engine.prepare_gallery(gal.to(DEV)), 5)
    r_s, _, r_i = so.rank_topk(so.pair_logits(q, gal, weights), 5)
    assert torch.equal(i2.cpu().long(), r_i) and (s2.cpu() - r_s).abs().max() <= TOL_SCORE


def test_prepared_gallery_follows_the_scorer(weights, engine):
    """A gallery prepared under one `last` and used after another was loaded is re-prepared (its cg = dw . g^2
    and overflow statistics belong to the old weights): results equal a fresh preparation."""
    seq, mask, _ = so.synth_tracks(40, 6, seed=31)
    q, _ = so.aggregate_tracks(seq, mask, weights)
    gal = so.synth_gallery(2000, 31, q)
    prepared = engine.prepare_gallery(gal.to(DEV))
    w2 = torch.randn(2, 256) * 0.1
    b2 = torch.randn(2) * 0.1
    with engine.scorer(w2, b2):
        a = engine.score_topk(q.to(DEV), prepared, 10)                   # stale -> re-prepared under (w2, b2)
        b = engine.score_topk(q.to(DEV), engine.prepare_gallery(gal.to(DEV)), 10)
        assert all(torch.equal(x, y) for x, y in zip(a, b))
        ra = engine.rank_of_target(q.to(DEV), prepared, torch.arange(40))
        rb = engine.rank_of_target(q.to(DEV), gal.to(DEV), torch.arange(40))
        assert torch.equal(ra[0], rb[0])
    c = engine.score_topk(q.to(DEV), prepared, 10)                       # and back under the original scorer
    r_s, r_d, r_i = so.rank_topk(so.pair_logits(q, gal, weights), 10)
    assert torch.equal(c[2].cpu().long(), r_i)


def test_load_weights_rejects_wrong_shapes(weights, engine):
    bad = {k: v.clone() for k, v in weights.items()}
    bad["newnlb.theta.weight"] = torch.zeros(64, 256, 1)
    with pytest.raises(ValueError):
        engine.load_weights({k: v.to(DEV) for k, v in bad.items()})
    engine.load_weights({k: v.to(DEV) for k, v in weights.items()})


def test_score_topk_in_query_slabs(weights, engine, monkeypatch):
    """Very large evaluations are scored in slabs of queries that share one bounded workspace; the result does not
    depend on the slab size."""
    import seam_match_rcnn_b200 as pkg
    eng_mod = __import__("sys").modules[pkg.__name__ + ".engine"]
    gen = torch.Generator(device=DEV).manual_seed(9)
    q = torch.randn(5000, 256, device=DEV, generator=gen)
    gal = engine.prepare_gallery(torch.randn(4000, 256, device=DEV, generator=gen))
    whole = engine.score_topk(q, gal, 20)
    monkeypatch.setattr(eng_mod, "SCORE_WS_LIMIT", 16 << 20)
    slabs = engine.score_topk(q, gal, 20)
    assert all(torch.equal(a, b) for a, b in zip(whole, slabs))


def test_device_stamp_between_graph_nodes(engine):
    """seam_device_stamp: the device's nanosecond timer written by a graph node -- how bench.py times a sharded step
    between the nodes of a replayed graph.  Stamps grow, and bracket the work between them."""
    st = torch.zeros(3, dtype=torch.int64, device=DEV)
    x = torch.randn(1 << 24, device=DEV)
    side = torch.cuda.Stream(device=DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(side):
        x.sum()
        engine.device_stamp(st, 0)
    torch.cuda.current_stream(DEV).wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        engine.device_stamp(st, 0)
        y = x.sum()
        engine.device_stamp(st, 1)
        z = (x * 2).sum() + y
        engine.device_stamp(st, 2)
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        a, b, c = (int(v) for v in st.cpu())
        assert 0 < a < b < c
        assert (c - a) < 50_000_000                    # two reductions over 64 MB: far below 50 ms
