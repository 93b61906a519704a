"""The "AVG & MAX DISTANCE" fusions over a sharded gallery: the gallery is split by shard_bounds into S shards on one GPU,
the shard holding each product's target computes its fused values (seam_shard_fused_target), the MAX over the shards
hands them to every shard, every shard counts against them (seam_shard_rank_fused_distances) and the counts are summed.
The sums must be the ranks of seam_rank_fused_distances on the whole gallery, integer for integer."""
import numpy as np
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


def _data(P, G, fmax, seed, empty=(1,)):
    """frames grouped by product (start: CSR offsets), a gallery in which some rows resemble their product's frames,
    targets; products in ``empty`` have no frames"""
    gen = torch.Generator(device=DEV).manual_seed(seed)
    lens = torch.randint(1, fmax + 1, (P,), device=DEV, generator=gen)
    for p in empty:
        if p < P:
            lens[p] = 0
    start = torch.zeros(P + 1, dtype=torch.int64, device=DEV)
    start[1:] = torch.cumsum(lens, 0)
    N = int(start[-1])
    frames = torch.randn(N, 256, device=DEV, generator=gen)
    g = torch.randn(G, 256, device=DEV, generator=gen)
    target = torch.randint(0, G, (P,), device=DEV, generator=gen)
    for p in range(0, P, 2):                                # half the targets resemble their product's first frame
        if lens[p] > 0:
            g[target[p]] = frames[start[p]] + 0.3 * torch.randn(256, device=DEV, generator=gen)
    return frames, start, g, target


def _shards(g, S):
    return [(lo, g[lo:hi]) for lo, hi in (pkg.shard_bounds(g.shape[0], S, s) for s in range(S)) if hi > lo]


def _sharded(engine, frames, start, shards, target):
    """(sum of the shards' counts (2,P), MAX of the shards' target values (2,P))"""
    P = target.shape[0]
    tv = torch.stack([torch.stack(engine.fused_target(frames, start, gs, lo, target)) for lo, gs in shards])
    has = (start[1:] - start[:-1]) > 0
    owners = (tv != NEG_INF).sum(0)
    assert bool((owners[:, has] == 1).all()), "exactly one shard holds each target"
    assert bool((owners[:, ~has] == 0).all()), "a product without frames has no target values"
    tv = tv.amax(0)
    ranks = torch.zeros((2, P), dtype=torch.int32, device=DEV)
    for lo, gs in shards:
        ca, cm = engine.fused_rank_count(frames, start, gs, lo, target, tv[0], tv[1])
        assert ca.dtype == torch.int32 and ca.shape == (P,)
        ranks += torch.stack([ca, cm])
    return ranks, tv


def _check(engine, frames, start, g, target, S, shards=None):
    full = torch.stack(engine.rank_fused_distances(frames, start, g, target))
    ranks, tv = _sharded(engine, frames, start, shards or _shards(g, S), target)
    assert _same(ranks, full), (ranks - full).abs().max()
    return ranks, tv


# ------------------------------------------------------------------------------------------------ sums
@pytest.mark.parametrize("S", [1, 2, 3, 8])
@pytest.mark.parametrize("P,G,fmax", [(1, 1, 1), (5, 9, 3), (17, 700, 5), (40, 2600, 40), (150, 5000, 12)])
def test_shard_counts_sum_to_the_fused_ranks(engine, P, G, fmax, S):
    """G = 9 at S = 8 gives shards of 1 and 2 rows, G = 700 shards smaller than one 1,024-row chunk; fmax = 40 gives
    products of several 16-frame chunks; product 1 has no frames (rank G)"""
    frames, start, g, target = _data(P, G, fmax, seed=P * 7 + G)
    ranks, _ = _check(engine, frames, start, g, target, S)
    if P > 1:
        assert ranks[:, 1].tolist() == [G, G]


def test_target_values_are_the_unsharded_ones(engine):
    """the owner's values are those the unsharded kernel compares against: a shard of one row (the target) counts
    nothing before it, and a full-gallery shard reproduces the unsharded ranks"""
    P, G = 30, 3000
    frames, start, g, target = _data(P, G, 20, seed=3, empty=())
    ta, tm = engine.fused_target(frames, start, g, 0, target)
    ca, cm = engine.fused_rank_count(frames, start, g, 0, target, ta, tm)
    ra, rm = engine.rank_fused_distances(frames, start, g, target)
    assert _same(ca, ra) and _same(cm, rm)
    for p in range(P):                                       # the target row on its own, as a shard at its global row
        t = int(target[p])
        a, m = engine.fused_target(frames, start, g[t:t + 1], t, target)
        assert _bits(a[p]) == _bits(ta[p]) and _bits(m[p]) == _bits(tm[p])


def test_duplicates_straddling_a_shard_boundary(engine):
    """exact copies of the target on both sides of a shard boundary: ties go to the lower GLOBAL row"""
    P, G, S = 64, 3000, 3                                   # shards [0,1000) [1000,2000) [2000,3000)
    frames, start, g, target = _data(P, G, 6, seed=5)
    target[0::4] = 1000                                     # copies at 999 (lower shard) and 1001, 2000
    target[1::4] = 1999                                     # copies at 999, 1001 (lower), 2000 (higher shard)
    g[999] = g[1001] = g[2000] = g[1000]
    g[1999] = g[1000]
    target[2::4] = 2000                                     # copies at 999, 1000, 1001, 1999: every one ranks before
    ranks, _ = _check(engine, frames, start, g, target, S)
    has = (start[1:] - start[:-1]) > 0
    assert bool((ranks[:, 2::4][:, has[2::4]] >= 4).all()) and bool((ranks[:, 0::4][:, has[0::4]] >= 1).all())


# ------------------------------------------------------------------------------------------------ fp16 galleries
@pytest.mark.parametrize("S", [1, 3, 8])
def test_g16_shards_match_fp32_shards(engine, S):
    P, G = 60, 5000
    frames, start, g, target = _data(P, G, 20, seed=14)
    g16 = g.half()
    s16, s32 = _shards(g16, S), _shards(g16.float(), S)
    r16, t16 = _sharded(engine, frames, start, s16, target)
    r32, t32 = _sharded(engine, frames, start, s32, target)
    assert _same(r16, r32) and _same(t16, t32)
    _check(engine, frames, start, g16.float(), target, S, shards=s16)


def test_g16_unsharded_entry(engine):
    """seam_rank_fused_distances_g16: the ranks of the fp32 entry on the widened gallery, without an fp32 copy; a
    misaligned or strided fp16 gallery is copied once"""
    P, G = 80, 9000
    frames, start, g, target = _data(P, G, 33, seed=21)
    g16 = g.half()
    r32 = torch.stack(engine.rank_fused_distances(frames, start, g16.float(), target))
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    r16 = torch.stack(engine.rank_fused_distances(frames, start, g16, target))
    torch.cuda.synchronize()
    assert _same(r16, r32)
    assert torch.cuda.max_memory_allocated() - base < g16.nbytes // 2
    buf = torch.empty(G * 256 + 8, dtype=torch.float16, device=DEV)
    mis = buf[1:1 + G * 256].view(G, 256)
    mis.copy_(g16)
    assert _same(torch.stack(engine.rank_fused_distances(frames, start, mis, target)), r32)
    wide = torch.empty(G, 512, dtype=torch.float16, device=DEV)
    wide[:, :256] = g16
    assert _same(torch.stack(engine.rank_fused_distances(frames, start, wide[:, :256], target)), r32)


# ------------------------------------------------------------------------------------------------ scorer swap
def test_scorer_put_back(engine):
    P, G, S = 30, 2500, 3
    frames, start, g, target = _data(P, G, 8, seed=27)
    gen = torch.Generator(device=DEV).manual_seed(29)
    lw = 0.05 * torch.randn(2, 256, device=DEV, generator=gen)
    lb = 0.05 * torch.randn(2, device=DEV, generator=gen)
    before = _check(engine, frames, start, g, target, S)[0]
    prev = engine._last
    with engine.scorer(lw, lb):
        other = _check(engine, frames, start, g, target, S)[0]
    assert engine._last[0].data_ptr() == prev[0].data_ptr()
    assert not _same(other, before)
    assert _same(_check(engine, frames, start, g, target, S)[0], before)


# ------------------------------------------------------------------------------------------------ ShardedRetriever
def _report_case(weights, P=40, G=3000, seed=31):
    from oracle import seam_oracle as so
    rs = np.random.RandomState(seed)
    seq, mask, _ = so.synth_tracks(P, 6, seed=seed, ragged=(1, 6))
    lens = rs.randint(1, 30, size=P)
    lens[3] = 0
    frame_product = torch.tensor([p for p in range(P) for _ in range(int(lens[p]))])
    frame_product = frame_product[torch.from_numpy(rs.permutation(len(frame_product)))]
    frame_desc = torch.from_numpy(rs.randn(len(frame_product), 256).astype(np.float32))
    shop_desc = torch.from_numpy(rs.randn(G, 256).astype(np.float32))
    target = torch.from_numpy(rs.permutation(G)[:P].astype(np.int64))
    shop_desc[target[frame_product[::3]]] = frame_desc[::3] + 0.3 * torch.from_numpy(
        rs.randn(len(frame_desc[::3]), 256).astype(np.float32))
    qref, _ = so.aggregate_tracks(seq, mask, weights)
    shop_aggr = so.synth_gallery(G, 4, None)
    shop_aggr[target] = qref + 0.2 * torch.from_numpy(rs.randn(P, 256).astype(np.float32))
    fw = torch.from_numpy(rs.uniform(-1 / 16, 1 / 16, (2, 256)).astype(np.float32)).to(DEV)
    fb = torch.from_numpy(rs.uniform(-1 / 16, 1 / 16, (2,)).astype(np.float32)).to(DEV)
    aw, ab = weights["last.weight"].to(DEV), weights["last.bias"].to(DEV)
    return dict(frame_desc=frame_desc.to(DEV), frame_product=frame_product.to(DEV), shop_desc=shop_desc.to(DEV),
                target=target.to(DEV), frame_last=(fw, fb), seq=seq.to(DEV), mask=mask.to(DEV),
                shop_aggr=shop_aggr.to(DEV), aggr_last=(aw, ab))


def test_sharded_retriever_world1(weights, engine):
    c = _report_case(weights)
    retr = pkg.ShardedRetriever(engine, c["shop_aggr"], 0)
    assert retr.world == 1
    for shop in (c["shop_desc"], c["shop_desc"].half()):
        ranks, hits = retr.evaluate_distance_fusions(c["frame_desc"], c["frame_product"], shop, c["target"],
                                                     c["frame_last"])
        r_ref, h_ref = pkg.evaluate_distance_fusions(engine, c["frame_desc"], c["frame_product"], shop, c["target"],
                                                     c["frame_last"])
        assert _same(ranks, r_ref) and _same(hits, h_ref)
    r16, _ = pkg.evaluate_distance_fusions(engine, c["frame_desc"], c["frame_product"], c["shop_desc"].half(),
                                           c["target"], c["frame_last"])
    r32, _ = pkg.evaluate_distance_fusions(engine, c["frame_desc"], c["frame_product"], c["shop_desc"].half().float(),
                                           c["target"], c["frame_last"])
    assert _same(r16, r32)
    with pytest.raises(ValueError):
        retr.evaluate_distance_fusions(c["frame_desc"], c["frame_product"], c["shop_desc"][1:], c["target"],
                                       c["frame_last"])

    prev = engine._last
    rep = retr.evaluate_products(c["frame_desc"], c["frame_product"], c["shop_desc"], c["target"], c["frame_last"],
                                 c["seq"], c["mask"], c["aggr_last"])
    assert engine._last[0].data_ptr() == prev[0].data_ptr()
    ref = pkg.evaluate_products(engine, c["frame_desc"], c["frame_product"], c["shop_desc"], c["target"],
                                c["frame_last"], c["seq"], c["mask"], c["shop_aggr"], c["aggr_last"])
    assert _same(rep.frame_ranks, ref.frame_ranks)
    assert _same(rep.product_ranks[[0, 2]], ref.product_ranks[[0, 2]])       # best frame, aggregated descriptor
    # the average descriptors: the sharded report sums them in a fixed order (the unsharded one with atomics)
    P = c["target"].shape[0]
    avg, has = pkg.product_means(c["frame_desc"], c["frame_product"], P)
    with engine.scorer(*c["frame_last"]):
        ar, _ = engine.rank_of_target(avg, engine.prepare_gallery(c["shop_desc"]), c["target"])
    ar = torch.where(has, ar, torch.full_like(ar, torch.iinfo(torch.int32).max))
    assert _same(rep.product_ranks[1], ar)
    assert rep.perf[[0, 1, 3]].equal(ref.perf[[0, 1, 3]]) and rep.rank_median == ref.rank_median


@pytest.mark.parametrize("S", [2, 3, 8])
def test_sharded_rows_0_to_2(weights, engine, S):
    """the S-shard composition of rows 0-2 (target margin, MAX, counts, SUM on every shard of the frame gallery)
    against the unsharded ranks on the same average descriptors"""
    c = _report_case(weights, seed=41)
    P = c["target"].shape[0]
    fp = c["frame_product"].long()
    avg, has = pkg.product_means(c["frame_desc"], fp, P)
    with engine.scorer(*c["frame_last"]):
        full = engine.prepare_gallery(c["shop_desc"])
        shards = [engine.prepare_gallery(gs, index_offset=lo) for lo, gs in _shards(c["shop_desc"], S)]
        for q, t in ((c["frame_desc"], c["target"][fp]), (avg, c["target"])):
            r_ref, m_ref = engine.rank_of_target(q, full, t)
            margin = torch.stack([engine.target_margin(q, p, t) for p in shards]).amax(0)
            rank = sum(engine.rank_count(q, p, t, margin) for p in shards)
            assert _same(rank.to(torch.int32), r_ref) and _same(margin, m_ref)


# ------------------------------------------------------------------------------------------------ C ABI arguments
def test_fused_entries_reject_bad_arguments(engine):
    lib, h = engine._lib, engine._h
    stream = torch.cuda.current_stream(DEV).cuda_stream
    P, G = 8, 512
    frames, start, g, _ = _data(P, G, 4, seed=50)
    s32 = start.to(torch.int32)
    g16 = g.half()
    buf = torch.zeros(G * 256 + 8, dtype=torch.float16, device=DEV)
    bad = buf.data_ptr() + 2
    target = torch.full((P,), 100, dtype=torch.int32, device=DEV)
    ta, tm = torch.zeros(P, device=DEV), torch.zeros(P, device=DEV)
    ra, rm = torch.empty(P, dtype=torch.int32, device=DEV), torch.empty(P, dtype=torch.int32, device=DEV)

    def check(name, rc, code):
        assert rc == code, (name, rc)
        assert name.encode() + b":" in lib.seam_last_error(h), lib.seam_last_error(h)

    def count(fn, rows, off, a, m, n=P):
        return fn(h, frames.data_ptr(), s32.data_ptr(), n, rows, G, off, target.data_ptr(), a, m, ra.data_ptr(),
                  rm.data_ptr(), stream)

    def tval(fn, rows, off, a=ta.data_ptr(), n=P):
        return fn(h, frames.data_ptr(), s32.data_ptr(), n, rows, G, off, target.data_ptr(), a, tm.data_ptr(), stream)

    c32, c16 = lib.seam_shard_rank_fused_distances, lib.seam_shard_rank_fused_distances_g16
    t32, t16 = lib.seam_shard_fused_target, lib.seam_shard_fused_target_g16
    check("seam_shard_rank_fused_distances", count(c32, g.data_ptr(), 0, None, tm.data_ptr()), 1)
    check("seam_shard_rank_fused_distances_g16", count(c16, g16.data_ptr(), 0, ta.data_ptr(), None), 1)
    check("seam_shard_rank_fused_distances", count(c32, g.data_ptr(), -1, ta.data_ptr(), tm.data_ptr()), 1)
    check("seam_shard_rank_fused_distances_g16", count(c16, g16.data_ptr(), -3, ta.data_ptr(), tm.data_ptr()), 1)
    check("seam_shard_rank_fused_distances_g16", count(c16, bad, 0, ta.data_ptr(), tm.data_ptr()), 2)
    check("seam_shard_fused_target", tval(t32, g.data_ptr(), -1), 1)
    check("seam_shard_fused_target_g16", tval(t16, g16.data_ptr(), -5), 1)
    check("seam_shard_fused_target_g16", tval(t16, bad, 0), 2)
    check("seam_shard_fused_target", tval(t32, g.data_ptr(), 0, a=None), 1)
    check("seam_rank_fused_distances_g16",
          lib.seam_rank_fused_distances_g16(h, frames.data_ptr(), s32.data_ptr(), P, bad, G, target.data_ptr(),
                                            ra.data_ptr(), rm.data_ptr(), stream), 2)
    # P == 0 is a no-op, and a target outside the shard gets -inf
    assert count(c32, g.data_ptr(), 0, None, None, n=0) == 0 and count(c16, g16.data_ptr(), 0, None, None, n=0) == 0
    assert tval(t32, g.data_ptr(), 0, a=None, n=0) == 0
    t = torch.tensor([0, 99, 100, 611, 612, 2**31 - 1, 300, 300], device=DEV)
    a, m = engine.fused_target(frames, start, g, 100, t)
    has = (start[1:] - start[:-1]) > 0
    inside = torch.tensor([False, False, True, True, False, False, True, True], device=DEV) & has
    assert bool((a[~inside] == NEG_INF).all()) and bool(torch.isfinite(a[inside]).all())
    assert bool((m[~inside] == NEG_INF).all()) and bool(torch.isfinite(m[inside]).all())
    torch.cuda.synchronize()
