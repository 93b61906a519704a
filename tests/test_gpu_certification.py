"""The certified top-k and the tensor-core rank against the exhaustive fp32 kernels, with no tolerance.

rescore_kernel, exact_topk_kernel and rank_of_target_kernel all score a pair with sqdiff_dot2 followed by treduce<8> /
warp_sum_b, which associate the same way (sm100_ptx.cuh), and 16-bit rows are widened exactly.  So for
``sc, mg, ix = score_topk(q, gal, k)`` and every position p < min(k, G):
  - the exhaustive ``rank_of_target(q, g_fp32, ix[:, p])`` is exactly p, with a margin whose bits are mg[:, p];
  - the prepared (tensor-core) rank gives the same integers and bits;
  - ix[:, p] is -1 exactly where p >= G.
This is the scorer's contract ("the index list equals the fp32 oracle's up to exact ties": ties go to the lowest
index) checked bit for bit, whichever path -- certified, sliced exhaustive, exhaustive -- answered a row.  A float64
check bounds the fp32 direct form itself.  (score_dense sums in another order and is not compared bit for bit.)"""
import numpy as np
import pytest
import torch

from oracle import seam_oracle as so
import seam_match_rcnn_b200 as pkg
from test_certification_bound import (SCALES, direct_bound, operand_bound, pair_errors, source_constants,
                                      subnormal_half_step_case)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U32 = 2.0 ** -24
# |fp32 direct-form margin - exact margin| <= C_DIRECT * u * (sum_c sum_k |W_ck| (q_k - g_k)^2 + |b0| + |b1|): along
# each logit's path a product term meets 14 roundings (q - g, the square, the product / 3 fmas of its half-lane chain,
# the pair sum, the 5-step butterfly, + b), and l1 - l0 one more.
C_DIRECT = 15.001


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _num_ctas_exact():
    return 2 * torch.cuda.get_device_properties(DEV).multi_processor_count


def assert_rank_identity(engine, q, gal, g_ref, k, mg, ix):
    """Position p of the list (global index ix - gal.index_offset in the shard g_ref) has exhaustive rank p, margin bits
    mg[:, p], and the prepared rank says the same; padding exactly where p >= G."""
    G, off = g_ref.shape[0], int(gal.index_offset)
    kk = min(k, G)
    ixc = ix.cpu()
    assert (ixc[:, kk:] == -1).all() and (ixc[:, :kk] >= off).all() and (ixc[:, :kk] < off + G).all()
    Q = q.shape[0]
    for p in range(kk):
        t = ix[:, p].long() - off
        r, m = engine.rank_of_target(q, g_ref, t)
        assert torch.equal(r, torch.full((Q,), p, dtype=torch.int32, device=DEV)), \
            f"position {p}: exhaustive ranks {r[r != p][:8].tolist()} at rows {(r != p).nonzero().flatten()[:8].tolist()}"
        assert torch.equal(_bits(m), _bits(mg[:, p].contiguous())), f"position {p}: margin bits differ"
        rf, mf = engine.rank_of_target(q, gal, t)
        assert torch.equal(rf, r) and torch.equal(_bits(mf), _bits(m)), f"position {p}: prepared rank differs"


def _d64(q, g, W, b):
    """Exact margins (float64) and the direct form's error bound for every pair."""
    q64, g64 = q.double().cpu(), g.double().cpu()
    W64, b64 = W.double().cpu(), b.double().cpu()
    d = torch.empty(q64.shape[0], g64.shape[0], dtype=torch.float64)
    s = torch.empty_like(d)
    for i in range(0, q64.shape[0], 16):
        x = (q64[i:i + 16, None] - g64[None]) ** 2
        d[i:i + 16] = x @ (W64[1] - W64[0]) + (b64[1] - b64[0])
        s[i:i + 16] = x @ (W64[0].abs() + W64[1].abs())
    return d, C_DIRECT * U32 * (s + b64.abs().sum())


def assert_float64_bounds(q, g, W, b, mg, ix):
    """The list's margins are within the bound of the exact ones, in order up to the bound, and nothing left out
    beats its last entry by more than the bound."""
    d, B = _d64(q, g, W, b)
    G = g.shape[0]
    kk = min(ix.shape[1], G)
    il = ix[:, :kk].long().cpu()
    dl, Bl = torch.gather(d, 1, il), torch.gather(B, 1, il)
    assert ((mg[:, :kk].double().cpu() - dl).abs() <= Bl).all(), "a margin lies outside the direct form's bound"
    assert (dl[:, :-1] + Bl[:, :-1] >= dl[:, 1:] - Bl[:, 1:]).all(), "list out of order beyond the bound"
    out = torch.ones_like(d, dtype=torch.bool)
    out.scatter_(1, il, False)
    worst = (dl[:, -1:] + Bl[:, -1:])
    assert ((d - B <= worst) | ~out).all(), "an item outside the list beats its last entry beyond the bound"


# ------------------------------------------------------------------------------------------------ 1. rank identity
def _planted(Q, G, seed):
    rs = np.random.RandomState(seed)
    q = torch.from_numpy(rs.randn(Q, 256).astype(np.float32))
    return q, so.synth_gallery(G, seed=seed, planted=q)


@pytest.mark.parametrize("G,Q", [(1, 37), (31, 37), (32, 129), (33, 129), (257, 128), (4097, 64), (20011, 40)])
def test_rank_identity_random_shapes(G, Q, engine):
    q, g = _planted(Q, G, seed=G * 13 + Q)
    q, g = q.to(DEV), g.to(DEV)
    gal = engine.prepare_gallery(g)
    for k in (1, 20, 24, 31, 32):
        sc, mg, ix, stats = engine.score_topk(q, gal, k, return_stats=True)
        if k <= 20 and G > 32:
            assert int(stats[0]) <= max(1, Q // 20), "expected the certified path"
        assert_rank_identity(engine, q, gal, g, k, mg, ix)


def test_rank_identity_sliced_and_exhaustive_rows(engine):
    """A few rows on the sliced exhaustive path (40 distinct rows repeated: windows full of copies), then every row
    exhaustive (queries past the fp16 range)."""
    Q, G, k = 100, 3000, 20
    q, base = _planted(Q, 40, seed=11)
    q = q.to(DEV)
    g = base.to(DEV)[torch.arange(G, device=DEV) % 40].contiguous()
    gal = engine.prepare_gallery(g)
    sc, mg, ix, stats = engine.score_topk(q, gal, k, return_stats=True)
    assert 0 < int(stats[0]) < _num_ctas_exact()
    assert_rank_identity(engine, q, gal, g, k, mg, ix)
    q2, g2 = _planted(64, 2000, seed=12)
    q2, g2 = (q2 * 1e6).to(DEV), g2.to(DEV)
    gal2 = engine.prepare_gallery(g2)
    sc, mg, ix, stats = engine.score_topk(q2, gal2, k, return_stats=True)
    assert int(stats[0]) == 64
    assert_rank_identity(engine, q2, gal2, g2, k, mg, ix)


def test_rank_identity_shard_with_offset(engine):
    Q, G, k, off = 96, 3001, 24, 70001
    q, g = _planted(Q, G, seed=21)
    q, g = q.to(DEV), g.to(DEV)
    gal = engine.prepare_gallery(g, index_offset=off)
    for kk in (20, k):
        sc, mg, ix, stats = engine.score_topk(q, gal, kk, return_stats=True)
        if kk <= 20:
            assert int(stats[0]) <= max(1, Q // 20), "expected the certified path"
        assert_rank_identity(engine, q, gal, g, kk, mg, ix)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_rank_identity_16bit_galleries(dtype, engine):
    Q, G = 64, 4097
    q, g = _planted(Q, G, seed=31)
    q, g16 = q.to(DEV), g.to(DEV).to(dtype)
    g16[100:140] = (g16[100:140].float() * 2.0 ** -18).to(dtype)       # fp16 subnormal rows
    gal = engine.prepare_gallery(g16, index_offset=5)
    for k in (1, 20, 32):
        sc, mg, ix, stats = engine.score_topk(q, gal, k, return_stats=True)
        if k <= 20:
            assert int(stats[0]) <= max(1, Q // 20), "expected the certified path"
        assert_rank_identity(engine, q, gal, g16.float(), k, mg, ix)


# ------------------------------------------------------------------------------------------------ 2. exact ties
def assert_tie_order(mg, ix, groups):
    """Equal margins come in ascending index order; of each group of bit-identical rows (groups[i]: sorted global
    indices, for query i) the list holds the lowest-indexed members, one contiguous run."""
    mb, il = _bits(mg).cpu(), ix.cpu()
    same = (mb[:, 1:] == mb[:, :-1]) & (il[:, 1:] >= 0)
    assert (il[:, 1:][same] > il[:, :-1][same]).all(), "equal margins not in ascending index order"
    for i, grp in enumerate(groups):
        row = il[i].tolist()
        pos = [p for p, j in enumerate(row) if j in set(grp)]
        assert [row[p] for p in pos] == grp[:len(pos)], (i, grp, row)
        assert pos == list(range(pos[0], pos[0] + len(pos))) if pos else True


def _groups(g, src):
    """Sorted indices of the rows bit-identical to row src[i] of g, per query."""
    return [sorted((g == g[s]).all(1).nonzero().flatten().tolist()) for s in src]


def _order64(q, g, w):
    d, _ = _d64(q, g, w["last.weight"], w["last.bias"])
    return d, torch.argsort(d, dim=1, descending=True)


@pytest.mark.parametrize("ncopy,k", [(1, 1), (1, 20), (30, 20), (31, 20), (32, 20), (31, 32), (32, 32)])
def test_ties_at_the_top(ncopy, k, weights, engine):
    """Each query's best row copied ncopy times over rows far from every query's top: 2 equal rows at rank 0, and
    31 / 32 / 33 equal rows (the 32-lane window's edge).  The list starts with the group in ascending index order."""
    Q, G = 24, 2000
    q, g = _planted(Q, G, seed=41 + ncopy)
    _, order = _order64(q, g, weights)
    rs = np.random.RandomState(ncopy)
    q_idx = torch.arange(Q)
    # every query gets its own group; copies land on rows in the bottom half of some query's ranking and in no
    # query's top 40
    bottom = torch.from_numpy(rs.permutation(order[:, G // 2:].flatten().unique().numpy()))
    used = set(order[:, :40].flatten().tolist())
    free = [int(j) for j in bottom if int(j) not in used]
    src = [int(order[i, 0]) for i in range(Q)]
    for i in range(Q):
        dst, free = free[:ncopy], free[ncopy:]
        g[dst] = g[src[i]].clone()
    groups = _groups(g, src)
    qd, gd = q.to(DEV), g.to(DEV)
    gal = engine.prepare_gallery(gd)
    sc, mg, ix, stats = engine.score_topk(qd, gal, k, return_stats=True)
    if ncopy >= 31:
        assert int(stats[0]) == Q, "a window full of equal values cannot be certified"
    assert_rank_identity(engine, qd, gal, gd, k, mg, ix)
    assert_tie_order(mg, ix, groups)
    for i in q_idx.tolist():
        n = min(k, len(groups[i]))
        assert ix[i, :n].tolist() == groups[i][:n]


def test_ties_straddling_k_and_rows_equal_to_the_query(weights, engine):
    """The item at rank k-2 copied 3 times (a group of 4 across the k boundary: the two lowest indices make the
    list), and rows equal to the query itself (q - g = 0 exactly) copied 3 times."""
    Q, G, k = 16, 1500, 20
    q, g = _planted(Q, G, seed=51)
    _, order = _order64(q, g, weights)
    used = set(order[:, :40].flatten().tolist())
    free = [int(j) for j in np.random.RandomState(5).permutation(G) if int(j) not in used]
    qd = q.to(DEV)
    for i in range(Q):                                            # one query at a time: its own gallery
        gi = g.clone()
        src = int(order[i, k - 2])
        dst = free[3 * i:3 * i + 3]
        gi[dst] = gi[src].clone()
        dq = free[100 + 3 * i:100 + 3 * i + 3]
        gi[dq] = q[i]
        gd = gi.to(DEV)
        gal = engine.prepare_gallery(gd)
        sc, mg, ix = engine.score_topk(qd[i:i + 1], gal, k)
        assert_rank_identity(engine, qd[i:i + 1], gal, gd, k, mg, ix)
        assert_tie_order(mg, ix, _groups(gd.cpu(), [src]))
        if not set(dq) & set(ix[0].tolist()):                    # the group of 4 straddles position k
            assert ix[0, k - 2:].tolist() == sorted(dst + [src])[:2]
        # the copies of the query: one contiguous, ascending run wherever they rank
        r, _ = engine.rank_of_target(qd[i:i + 1].expand(3, 256).contiguous(), gd, torch.tensor(dq, device=DEV))
        rr = sorted(r.tolist())
        assert rr == list(range(rr[0], rr[0] + 3))
        assert [dq[j] for j in torch.tensor(r.tolist()).argsort().tolist()] == sorted(dq)


def test_ties_split_across_shards_merge(weights, engine):
    """Copies of each query's best row in three shards: merge_topk's lists and the unsharded list are identical and
    the group comes first in ascending global index."""
    Q, G, k = 32, 3000, 20
    q, g = _planted(Q, G, seed=61)
    _, order = _order64(q, g, weights)
    bounds = [(0, 1100), (1100, 1101), (1101, 3000)]
    rs = np.random.RandomState(6)
    groups = []
    used = set(order[:, :40].flatten().tolist())
    for i in range(Q):
        src = int(order[i, 0])
        dst = []
        for a, b in bounds:
            cand = [j for j in rs.permutation(np.arange(a, b)).tolist() if j not in used and j != src]
            dst += cand[:1 if b - a == 1 else 2]
        used.update(dst)
        g[dst] = g[src].clone()
        groups.append(src)
    groups = _groups(g, groups)
    qd, gd = q.to(DEV), g.to(DEV)
    S, M, I = [], [], []
    for a, b in bounds:
        s, d, i = engine.score_topk(qd, engine.prepare_gallery(gd[a:b], index_offset=a), k)
        S.append(s), M.append(d), I.append(i)
    s, d, i = engine.merge_topk(None, torch.stack(M), torch.stack(I))
    gal = engine.prepare_gallery(gd)
    s1, d1, i1 = engine.score_topk(qd, gal, k)
    assert torch.equal(i, i1) and torch.equal(_bits(d), _bits(d1)) and torch.equal(_bits(s), _bits(s1))
    assert_rank_identity(engine, qd, gal, gd, k, d1, i1)
    assert_tie_order(d1, i1, groups)
    for r in range(Q):
        n = len(groups[r])
        assert i1[r, :n].tolist() == groups[r]


def test_ties_two_rank_sharded_search(weights, engine):
    """The two-rank sharded search (two engines on two streams of one GPU, test_gpu_sharded.py's set-up) over a gallery
    whose copies of rows lie in both shards: the single-GPU search's lists bit for bit, ties in ascending global index.
    A single-rank step first loads every kernel of the step: the two ranks' kernels wait for each other on the device,
    so none of them may still have to be loaded while the other rank's are running."""
    Q, T, G, k = 301, 4, 2500, 20
    seq, mask, _ = so.synth_tracks(Q, T, seed=71, ragged=(1, 4))
    seq, mask = seq.to(DEV), mask.to(DEV)
    qd = engine.aggregate(seq, mask)
    gal = torch.randn(G, 256, generator=torch.Generator().manual_seed(72)).to(DEV)
    bounds = [pkg.shard_bounds(G, 2, r) for r in range(2)]
    n = min(Q, bounds[0][1], G - bounds[1][0])
    gal[bounds[1][0]:bounds[1][0] + n] = gal[:n].clone()              # every row of the first shard's head, twice
    ref = pkg.search(engine, seq, mask, gal, k)
    warm = pkg.PeerExchange(engine, Q, k)
    pkg.ShardedRetriever(engine, gal, 0).search_peer(seq, mask, warm)
    engines = [engine, pkg.SeamEngine(DEV)]
    engines[1].load_weights({kk: v.to(DEV) for kk, v in weights.items()})
    shared = {}
    peers = [pkg.PeerExchange(engines[r], Q, k, replicate=True, local_peers={"world": 2, "rank": r, "shared": shared})
             for r in range(2)]
    for p in peers:
        p._fill_struct()
    retrs = [pkg.ShardedRetriever(engines[r], gal[bounds[r][0]:bounds[r][1]], bounds[r][0], world=2, rank=r)
             for r in range(2)]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(DEV) for _ in range(2)]
    res = [None, None]
    for r in (0, 1):
        streams[r].wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(streams[r]):
            res[r] = retrs[r].search_peer(seq, mask, peers[r])
    torch.cuda.synchronize()
    assert engines[0].watchdog_records() == []
    for r in range(2):
        sc, mg, ix = res[r]
        assert torch.equal(ix, ref[2]) and torch.equal(_bits(mg), _bits(ref[1])) and torch.equal(_bits(sc), _bits(ref[0]))
    ix = ref[2]
    groups = _groups(gal.cpu(), [row[0] for row in ix.cpu().tolist()])
    assert_tie_order(ref[1], ix, groups)
    twins = [gr for gr in groups if len(gr) > 1]
    assert twins and all(len(gr) == 2 and gr[1] - gr[0] == bounds[1][0] for gr in twins)
    assert_rank_identity(engine, qd, engine.prepare_gallery(gal), gal, k, ref[1], ix)


# ------------------------------------------------------------------------------------------------ 3. operand scale
@pytest.mark.parametrize("sq", SCALES)
def test_operand_scales(sq, weights, engine):
    """The same seeded data with queries and gallery scaled independently by 2^sq, 2^sg over the whole grid: rank
    identity, the prepared rank against the exhaustive one and the float64 bound.  Rows whose 2 eps band around the
    k-th nominated value leaves room in the 32-lane window (predicted from the CPU model of eps) are certified."""
    Q, G, k = 32, 1500, 20
    q0, g0 = _planted(Q, G, seed=81)
    W, b = weights["last.weight"], weights["last.bias"]
    target = torch.from_numpy(np.random.RandomState(82).randint(0, G, size=Q)).to(DEV)
    c = source_constants()
    for sg in SCALES:
        q, g = (q0 * 2.0 ** sq).to(DEV), (g0 * 2.0 ** sg).to(DEV)
        gal = engine.prepare_gallery(g)
        sc, mg, ix, stats = engine.score_topk(q, gal, k, return_stats=True)
        m = pair_errors(q.cpu().numpy(), g.cpu().numpy(), W.numpy(), b.numpy())
        if m is None:                                              # fp16 overflow: every row exhaustive
            assert int(stats[0]) == Q, (sq, sg)
        else:
            top = np.sort(m["vhat"], axis=1)[:, ::-1][:, :32]
            eps = (operand_bound(c, m["anorm"], m["gstat"]) + direct_bound(c, m["qw"], m["gstat"], b.numpy())
                   + np.float32(c["TAG_REL_ERR"]) * np.abs(top).max(1))
            window_full = top[:, 31] >= top[:, k - 1] - 2 * eps
            assert int(stats[0]) <= int(window_full.sum()) + max(1, Q // 20), (sq, sg, int(stats[0]))
        assert_rank_identity(engine, q, gal, g, k, mg, ix)
        r_fast, m_fast = engine.rank_of_target(q, gal, target)
        r_slow, m_slow = engine.rank_of_target(q, g, target)
        assert torch.equal(r_fast, r_slow) and torch.equal(_bits(m_fast), _bits(m_slow)), (sq, sg)
        assert_float64_bounds(q, g, W, b, mg, ix)


def _crafted_subnormal(weights, G=64):
    """One query whose fp16 operand a is all zeros (every a_k just under 2^-25) and a gallery where that matters: row T
    (L1 mass 8192, cg ~ 0) gains a . g_T = 0.99 * 2^-25 * 8192 = 2.4e-4 that the tensor-core value cannot see, row A
    has cg = 1.2e-4 on one component (and a . g_A ~ 0); every other row lies far below both.  Exact order: T, A, ...;
    nominated order: A, T, ...  Scored with `last` scaled by 2^-10 so the fp32 direct form resolves the difference."""
    W = (weights["last.weight"] * 2.0 ** -10).float()
    b = torch.zeros(2)
    q, gT = subnormal_half_step_case(W.numpy(), mass=(8192.0,))
    dw = (W[1] - W[0]).numpy()
    g = np.zeros((G, 256), np.float32)
    T, A = 37, 5
    g[T] = gT[0]
    kp, kn = int(np.argmax(dw)), int(np.argmin(dw))
    delta = 0.99 * 2.0 ** -25 * 8192.0
    g[A, kp] = np.sqrt(0.5 * delta / dw[kp])
    fill = [j for j in range(G) if j not in (A, T)]
    g[fill, kn] = np.sqrt(np.linspace(0.05, 0.5, len(fill)) / -dw[kn])
    return torch.from_numpy(q), torch.from_numpy(g), W, b, T, A


def test_crafted_subnormal_query(weights, engine):
    """The best item is nominated below the second by more than the old bound's 2 eps: a bound without the subnormal
    terms certifies the row and returns A first; with them the row is still certified and T comes first."""
    q, g, W, b, T, A = _crafted_subnormal(weights)
    with engine.scorer(W.to(DEV), b.to(DEV)):
        qd, gd = q.to(DEV), g.to(DEV)
        d, B = _d64(q, g, W, b)
        assert float(d[0, T] - d[0, A]) > 4 * float(B[0, T] + B[0, A])       # the direct form resolves T > A
        gal = engine.prepare_gallery(gd)
        for k in (1, 2, 20):
            sc, mg, ix, stats = engine.score_topk(qd, gal, k, return_stats=True)
            assert int(stats[0]) == 0, "expected the certified path"
            assert ix[0, :min(k, 2)].tolist() == [T, A][:k]
            assert_rank_identity(engine, qd, gal, gd, k, mg, ix)
            assert_float64_bounds(qd, gd, W, b, mg, ix)
        for t in (T, A):
            tgt = torch.tensor([t], device=DEV)
            r_fast, m_fast, st = engine.rank_of_target(qd, gal, tgt, return_stats=True)
            r_slow, m_slow = engine.rank_of_target(qd, gd, tgt)
            assert int(st[0]) == 0 and torch.equal(r_fast, r_slow) and torch.equal(_bits(m_fast), _bits(m_slow))
            assert int(r_slow[0]) == (0 if t == T else 1)


def test_scorer_with_dw_much_smaller_than_w(weights, engine):
    """W[0] ~= W[1] with a large W (1024 x `last`, dw = 1e-4 of max|W[0]|/1024 ... a legitimate `last` through
    engine.scorer) and a gallery of near-ties: the fp16 operands' eps shrinks with dw while the fp32 direct form's
    rounding grows with W and reorders the near-ties.  A bound without the direct form's term certifies these rows
    (the CPU model of the kernels, test_certification_bound.direct_form, then lists a wrong item first for most rows); with it they go to the exhaustive
    kernel."""
    rs = np.random.RandomState(91)
    base = weights["last.weight"][0].float()
    W0 = base * 1024.0
    W = torch.stack([W0, W0 + 1e-4 * float(base.abs().max()) * torch.from_numpy(rs.randn(256).astype(np.float32))])
    b = weights["last.bias"].float()
    Q, G = 16, 400
    q = torch.from_numpy(rs.randn(Q, 256).astype(np.float32))
    g = torch.from_numpy((rs.randn(1, 256) + 0.3 * rs.randn(G, 256)).astype(np.float32))
    with engine.scorer(W.to(DEV), b.to(DEV)):
        qd, gd = q.to(DEV), g.to(DEV)
        gal = engine.prepare_gallery(gd)
        target = torch.from_numpy(rs.randint(0, G, size=Q)).to(DEV)
        for k in (1, 5, 20):
            sc, mg, ix, stats = engine.score_topk(qd, gal, k, return_stats=True)
            assert int(stats[0]) == Q, "expected every row on the exhaustive path"
            assert_rank_identity(engine, qd, gal, gd, k, mg, ix)
            assert_float64_bounds(qd, gd, W, b, mg, ix)
        r_fast, m_fast = engine.rank_of_target(qd, gal, target)
        r_slow, m_slow = engine.rank_of_target(qd, gd, target)
        assert torch.equal(r_fast, r_slow) and torch.equal(_bits(m_fast), _bits(m_slow))
