"""Rank of the target over a sharded gallery: the gallery is split by shard_bounds into S shards on one GPU, the shard
holding each target computes its margin (seam_shard_target_margin), the MAX over the shards hands it to every shard,
every shard counts against it (seam_shard_rank_count_prepared) and the counts are summed.  The sum must be the rank
of rank_of_target on the whole gallery -- prepared and exhaustive -- integer for integer, and the margin its bits."""
import pytest
import torch

import seam_match_rcnn_b200 as pkg

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NEG_INF = float("-inf")


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _same(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(_bits(a), _bits(b))


def _data(Q, G, seed):
    """queries and a gallery whose first min(Q,G) rows are near-duplicates of the queries (a true match per query)"""
    gen = torch.Generator(device=DEV).manual_seed(seed)
    q = torch.randn(Q, 256, device=DEV, generator=gen)
    g = torch.randn(G, 256, device=DEV, generator=gen)
    n = min(Q, G)
    g[:n] = q[:n] + 0.1 * torch.randn(n, 256, device=DEV, generator=gen)
    return q, g


def _targets(engine, q, g, seed):
    """a third of the targets each query's best item (rank 0), a third in the bulk, a third the last of the ranking"""
    Q, G = q.shape[0], g.shape[0]
    gen = torch.Generator(device=DEV).manual_seed(seed)
    target = torch.randint(0, G, (Q,), device=DEV, generator=gen)
    target[0::3] = engine.score_topk(q[0::3], engine.prepare_gallery(g), 1)[2][:, 0].long()
    if Q > 2:
        x5 = engine.score_dense(q[2::3], g)
        target[2::3] = (x5[..., 1] - x5[..., 0]).argmin(1)
    return target


def _shards(engine, g, S):
    bounds = [pkg.shard_bounds(g.shape[0], S, s) for s in range(S)]
    return [engine.prepare_gallery(g[lo:hi], index_offset=lo) for lo, hi in bounds if hi > lo]


def _sharded_rank(engine, q, shards, target):
    """(sum of the shards' counts, MAX of the shards' margins, [fallback rows per shard])"""
    margins = torch.stack([engine.target_margin(q, p, target) for p in shards])
    owners = (margins != NEG_INF).sum(0)
    assert bool((owners == 1).all()), "exactly one shard holds each target"
    margin = margins.amax(0)
    rank = torch.zeros(q.shape[0], dtype=torch.int32, device=DEV)
    fallback = []
    for p in shards:
        count, stats = engine.rank_count(q, p, target, margin, return_stats=True)
        assert count.dtype == torch.int32 and count.shape == (q.shape[0],)
        rank += count
        fallback.append(int(stats[0]))
    return rank, margin, fallback


def _check(engine, q, g, target, S, shards=None):
    full = engine.prepare_gallery(g)
    r_full, m_full = engine.rank_of_target(q, full, target)
    r_slow, m_slow = engine.rank_of_target(q, g, target)
    assert _same(r_full, r_slow) and _same(m_full, m_slow)
    rank, margin, fallback = _sharded_rank(engine, q, shards or _shards(engine, g, S), target)
    assert _same(rank, r_full), (rank - r_full).abs().max()
    assert _same(margin, m_full)
    return rank, fallback


# ------------------------------------------------------------------------------------------------ sums and margins
@pytest.mark.parametrize("S", [1, 2, 3, 8])
@pytest.mark.parametrize("Q,G", [(1, 1), (5, 9), (13, 1000), (397, 2000), (1000, 30000)])
def test_shard_counts_sum_to_the_rank(engine, Q, G, S):
    """targets at the top, in the bulk and the last of the ranking; Q not a multiple of 8; with S = 8,
    G = 9 gives shards of 1 and 2 rows and G = 1000 / 2000 shards of fewer than 256 rows"""
    q, g = _data(Q, G, seed=Q * 7 + G)
    target = _targets(engine, q, g, seed=G)
    rank, _ = _check(engine, q, g, target, S)
    assert bool((rank[0::3] == 0).all())


def test_duplicates_straddling_a_shard_boundary(engine):
    """exact copies of the target on both sides of a shard boundary: ties go to the lower GLOBAL row"""
    Q, G, S = 64, 600, 3                                   # shards [0,200) [200,400) [400,600)
    q, g = _data(Q, G, seed=5)
    target = _targets(engine, q, g, seed=6)
    target[0::4] = 200                                     # copies at 199 (lower shard) and 201, 400 (same, higher)
    target[1::4] = 399                                     # copies at 199, 201 (lower), 400 (higher shard)
    g[199] = g[201] = g[400] = g[200]
    g[399] = g[200]
    target[2::4] = 400                                     # copies at 199, 200, 201, 399: every one ranks before
    rank, _ = _check(engine, q, g, target, S)
    r400 = rank[2::4]
    r200 = rank[0::4]
    assert bool((r400 >= 4).all()) and bool((r200 >= 1).all())


def test_fp16_overflow_in_one_shard_only(engine):
    """a value beyond the fp16 range in the last shard sends that shard's queries to the exhaustive kernel and
    leaves the others on the tensor-core path"""
    Q, G, S = 40, 6000, 3
    q, g = _data(Q, G, seed=8)
    target = _targets(engine, q, g, seed=9)
    g[5000, 3] = 1.0e5
    _, fallback = _check(engine, q, g, target, S)
    assert fallback[2] == Q and fallback[0] < Q and fallback[1] < Q


def test_crowded_band_takes_the_exhaustive_path(engine):
    """near-identical rows all fall inside the error band around the target: at this shape a shard's band lists hold
    fewer records than a query row's pieces produce (seam_score_partition: 94 tiles of 256 B per piece against 16 KB),
    so they close and the queries are counted exhaustively on their shard -- the sums are still the rank"""
    Q, G, S = 2048, 1 << 19, 2
    gen = torch.Generator(device=DEV).manual_seed(12)
    q = torch.randn(Q, 256, device=DEV, generator=gen)
    g = torch.randn(1, 256, device=DEV, generator=gen) + 1e-4 * torch.randn(G, 256, device=DEV, generator=gen)
    target = torch.randint(0, G, (Q,), device=DEV, generator=gen)
    _, fallback = _check(engine, q, g, target, S)
    assert sum(fallback) > 0


# ------------------------------------------------------------------------------------------------ fp16 galleries
@pytest.mark.parametrize("S", [1, 3, 8])
def test_g16_shards_match_fp32_shards(engine, S):
    Q, G = 203, 5000
    q, g = _data(Q, G, seed=14)
    g16 = g.half()
    target = _targets(engine, q, g16.float(), seed=15)
    s16, s32 = _shards(engine, g16, S), _shards(engine, g16.float(), S)
    assert all(p.rows_f16 for p in s16) and not any(p.rows_f16 for p in s32)
    for p16, p32 in zip(s16, s32):
        assert _same(engine.target_margin(q, p16, target), engine.target_margin(q, p32, target))
    r16, m16, _ = _sharded_rank(engine, q, s16, target)
    r32, m32, _ = _sharded_rank(engine, q, s32, target)
    assert _same(r16, r32) and _same(m16, m32)
    _check(engine, q, g16.float(), target, S, shards=s16)
    for p16, p32 in zip(s16, s32):                         # the exhaustive fallback of an fp16 shard
        qs = q * 1e6
        c16, st16 = engine.rank_count(qs, p16, target, torch.full((Q,), 0.5, device=DEV), return_stats=True)
        c32, st32 = engine.rank_count(qs, p32, target, torch.full((Q,), 0.5, device=DEV), return_stats=True)
        assert _same(c16, c32) and int(st16[0]) == Q == int(st32[0])


# ------------------------------------------------------------------------------------------------ scorer swap
def test_scorer_swap_between_calls(engine):
    Q, G, S = 100, 3000, 3
    q, g = _data(Q, G, seed=27)
    target = _targets(engine, q, g, seed=28)
    shards = _shards(engine, g, S)
    _check(engine, q, g, target, S, shards=shards)
    gen = torch.Generator(device=DEV).manual_seed(29)
    lw = 0.1 * torch.randn(2, 256, device=DEV, generator=gen)
    lb = 0.1 * torch.randn(2, device=DEV, generator=gen)
    with engine.scorer(lw, lb):
        _check(engine, q, g, target, S, shards=shards)     # shards re-prepared through _fresh
    _check(engine, q, g, target, S, shards=shards)


# ------------------------------------------------------------------------------------------------ ShardedRetriever
def test_sharded_retriever_world1(weights, engine):
    from oracle import seam_oracle as so
    seq, mask, _ = so.synth_tracks(150, 6, seed=31, ragged=(1, 6))
    ref_q, _ = so.aggregate_tracks(seq, mask, weights)
    g = so.synth_gallery(4000, seed=31, planted=ref_q).to(DEV)
    seq, mask = seq.to(DEV), mask.to(DEV)
    target = torch.arange(150, device=DEV) * 7 % 4000
    target[::2] = torch.arange(150, device=DEV)[::2]
    retr = pkg.ShardedRetriever(engine, g, 0)
    assert retr.world == 1
    q = engine.aggregate(seq, mask)
    rank, margin = retr.rank_of_target(q, target)
    r_ref, m_ref = engine.rank_of_target(q, engine.prepare_gallery(g), target)
    assert _same(rank, r_ref) and _same(margin, m_ref)
    rep = retr.evaluate_aggregated(seq, mask, target)
    ref = pkg.evaluate_aggregated(engine, seq, mask, g, target)
    assert _same(rep.ranks, ref.ranks) and rep.hits == ref.hits and rep.accuracies == ref.accuracies
    assert _same(rep.topk_scores, ref.topk_scores) and _same(rep.topk_idx, ref.topk_idx)
    with pytest.raises(ValueError):
        retr.rank_of_target(q[:1], torch.tensor([4000], device=DEV))
    with pytest.raises(ValueError):
        retr.rank_of_target(q[:1], torch.tensor([-1], device=DEV))


# ------------------------------------------------------------------------------------------------ C ABI arguments
def test_shard_entries_reject_bad_arguments(engine):
    lib, h = engine._lib, engine._h
    stream = torch.cuda.current_stream(DEV).cuda_stream
    Q, G = 8, 512
    q = torch.randn(Q, 256, device=DEV)
    p32 = engine.prepare_gallery(torch.randn(G, 256, device=DEV), index_offset=100)
    p16 = engine.prepare_gallery(p32.g.half(), index_offset=100)
    buf = torch.zeros(G * 256 + 8, dtype=torch.float16, device=DEV)
    bad = buf.data_ptr() + 2
    target = torch.full((Q,), 100, dtype=torch.int32, device=DEV)
    margin = torch.zeros(Q, device=DEV)
    count = torch.empty(Q, dtype=torch.int32, device=DEV)
    ws = torch.empty(lib.seam_rank_workspace_bytes(h, Q, G), dtype=torch.uint8, device=DEV)

    def check(name, rc, code):
        assert rc == code, (name, rc)
        assert name.encode() + b":" in lib.seam_last_error(h), lib.seam_last_error(h)

    def count32(off, m, g16=p32.g16.data_ptr(), n=Q):
        return lib.seam_shard_rank_count_prepared(h, q.data_ptr(), n, p32.g.data_ptr(), g16, p32.cg.data_ptr(),
                                                  p32.gstat.data_ptr(), G, off, target.data_ptr(), m, count.data_ptr(),
                                                  None, ws.data_ptr(), ws.numel(), stream)

    def count16(off, m, g16=p16.g16.data_ptr(), n=Q):
        return lib.seam_shard_rank_count_prepared_g16(h, q.data_ptr(), n, g16, p16.cg.data_ptr(), p16.gstat.data_ptr(),
                                                      G, off, target.data_ptr(), m, count.data_ptr(), None,
                                                      ws.data_ptr(), ws.numel(), stream)

    check("seam_shard_rank_count_prepared", count32(100, None), 1)
    check("seam_shard_rank_count_prepared_g16", count16(100, None), 1)
    check("seam_shard_rank_count_prepared", count32(-1, margin.data_ptr()), 1)
    check("seam_shard_rank_count_prepared_g16", count16(-1, margin.data_ptr()), 1)
    check("seam_shard_rank_count_prepared_g16", count16(100, margin.data_ptr(), g16=bad), 2)
    check("seam_shard_target_margin", lib.seam_shard_target_margin(h, q.data_ptr(), Q, p32.g.data_ptr(), G, -1,
                                                                   target.data_ptr(), margin.data_ptr(), stream), 1)
    check("seam_shard_target_margin_g16", lib.seam_shard_target_margin_g16(h, q.data_ptr(), Q, p16.g16.data_ptr(), G, -5,
                                                                           target.data_ptr(), margin.data_ptr(), stream), 1)
    check("seam_shard_target_margin_g16", lib.seam_shard_target_margin_g16(h, q.data_ptr(), Q, bad, G, 100,
                                                                           target.data_ptr(), margin.data_ptr(), stream), 2)
    check("seam_shard_target_margin", lib.seam_shard_target_margin(h, q.data_ptr(), Q, p32.g.data_ptr(), G, 100,
                                                                   target.data_ptr(), None, stream), 1)
    # Q == 0 is a no-op, and a target outside the shard gets -inf
    assert count32(100, None, n=0) == 0 and count16(100, None, n=0) == 0
    assert lib.seam_shard_target_margin(h, None, 0, p32.g.data_ptr(), G, 100, None, None, stream) == 0
    t = torch.tensor([0, 99, 100, 611, 612, 2**31 - 1], dtype=torch.int32, device=DEV)
    m = engine.target_margin(q[:6], p32, t)
    assert bool((m[[0, 1, 4, 5]] == NEG_INF).all()) and bool(torch.isfinite(m[[2, 3]]).all())
    torch.cuda.synchronize()
