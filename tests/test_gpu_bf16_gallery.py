"""bf16 galleries: a gallery given as bf16 is kept as bf16 -- the rows the fp32 direct form reads (widened exactly), with
an fp16 image g16 beside them for the tensor-core pass, through the seam_prepare_gallery_bf16 / *_gbf16 entry points --
and every result equals, bit for bit, what the fp32 path gives on the widened gallery g.float(): the prepared operand,
cg and the overflow flag, the diagnostic counters, and every score, margin, index, rank and count.  Float tensors are
compared by their bit patterns (NaN included)."""
import ctypes as C
import sys

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


def _all_same(xs, ys):
    xs, ys = list(xs), list(ys)
    assert len(xs) == len(ys)
    for i, (a, b) in enumerate(zip(xs, ys)):
        assert _same(a, b), f"output {i} differs"


def _data(Q, G, seed, planted=True, scale=1.0):
    """queries (Q,256) fp32 and a bf16 gallery (G,256) on the device whose first min(Q,G) rows are near-duplicates of
    the queries (a true match per query, as in bench.py)."""
    gen = torch.Generator(device=DEV).manual_seed(seed)
    q = torch.randn(Q, 256, device=DEV, generator=gen)
    g = torch.randn(G, 256, device=DEV, generator=gen)
    n = min(Q, G)
    if planted and n:
        g[:n] = q[:n] + 0.1 * torch.randn(n, 256, device=DEV, generator=gen)
    return q * scale, (g * scale).bfloat16()


def _tracks(Q, T, seed, dtype, ragged=None):
    g = torch.Generator(device=DEV).manual_seed(seed)
    seq = torch.randn(1 + T, Q, 256, device=DEV, generator=g).to(dtype)
    lens = (torch.full((Q,), T, dtype=torch.int64, device=DEV) if ragged is None
            else torch.randint(ragged[0], ragged[1] + 1, (Q,), device=DEV, generator=g))
    mask = torch.arange(1 + T, device=DEV).unsqueeze(0) > lens.unsqueeze(1)
    seq.masked_fill_(mask.t().unsqueeze(2), 0.0)
    seq[0] = 0.0
    return seq, mask, lens


def _topk(engine, q, gal, k):
    return engine.score_topk(q, gal, k, return_stats=True)


def _prepared_same(pb, p32):
    assert pb.rows_bf16 and not pb.rows_f16 and pb.row_suffix == "_gbf16" and pb.g16.dtype == torch.float16
    assert torch.equal(pb.g16.view(torch.int16), p32.g16.view(torch.int16))
    assert _same(pb.cg, p32.cg) and _same(pb.gstat, p32.gstat)


def _num_ctas_exact():
    return 2 * torch.cuda.get_device_properties(DEV).multi_processor_count


# ------------------------------------------------------------------------------------------------ 1. prepare
def test_prepare_bf16_matches_fp32_and_uses_the_callers_rows(engine):
    _, gb = _data(1, 5000, seed=1)
    pb = engine.prepare_gallery(gb)
    p32 = engine.prepare_gallery(gb.float())
    _prepared_same(pb, p32)
    assert pb.g.data_ptr() == gb.data_ptr() and pb.g16.data_ptr() != gb.data_ptr() and pb.G == 5000


def test_prepare_bf16_makes_no_fp32_copy(engine):
    """the prepared gallery adds g16 and cg, 516 bytes per row: an fp32 copy (1 KB per row) would show"""
    G = 200000
    _, gb = _data(1, G, seed=2, planted=False)
    engine.prepare_gallery(gb[:1000])
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(DEV)
    torch.cuda.reset_peak_memory_stats(DEV)
    p = engine.prepare_gallery(gb)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated(DEV) - base <= G * 516 + (1 << 20)
    assert p.g.data_ptr() == gb.data_ptr()


def test_prepare_bf16_copies_misaligned_strided_and_host_views(engine):
    Q, G, k = 300, 3000, 20
    q, gb = _data(Q, G, seed=3)
    p32 = engine.prepare_gallery(gb.float())
    ref = _topk(engine, q, p32, k)
    buf = torch.zeros(G * 256 + 1, dtype=torch.bfloat16, device=DEV)
    mis = buf[1:].view(G, 256)                                         # storage offset of one element
    mis.copy_(gb)
    wide = torch.zeros(G, 264, dtype=torch.bfloat16, device=DEV)
    wide[:, :256] = gb
    strided = wide[:, :256]                                            # row stride 264
    assert mis.is_contiguous() and mis.data_ptr() % 16 and not strided.is_contiguous()
    for view in (mis, strided, gb.cpu()):
        p = engine.prepare_gallery(view)
        assert p.g.is_contiguous() and p.g.data_ptr() % 16 == 0 and p.g.device == gb.device
        assert p.g.data_ptr() != view.data_ptr() and torch.equal(p.g, gb)
        _prepared_same(p, p32)
        _all_same(_topk(engine, q, p, k), ref)


def test_gbf16_entries_reject_misaligned_and_null_pointers(engine):
    lib, h = engine._lib, engine._h
    stream = torch.cuda.current_stream(DEV).cuda_stream
    Q, G, k, T, P = 8, 512, 4, 3, 4
    buf = torch.zeros(G * 256 + 8, dtype=torch.bfloat16, device=DEV)
    g16buf = torch.zeros(G * 256 + 8, dtype=torch.float16, device=DEV)
    rows, bad = buf.data_ptr(), buf.data_ptr() + 2
    g16, bad16 = g16buf.data_ptr(), g16buf.data_ptr() + 2
    q = torch.randn(Q, 256, device=DEV)
    cg = torch.empty(G, device=DEV)
    gstat = torch.zeros(4, device=DEV)
    sc, mg = torch.empty(Q, k, device=DEV), torch.empty(Q, k, device=DEV)
    ix = torch.empty(Q, k, dtype=torch.int32, device=DEV)
    target = torch.zeros(Q, dtype=torch.int32, device=DEV)
    rank, margin = torch.empty(Q, dtype=torch.int32, device=DEV), torch.zeros(Q, device=DEV)
    ws = torch.empty(max(lib.seam_score_workspace_bytes(h, Q, G, k), lib.seam_rank_workspace_bytes(h, Q, G)),
                     dtype=torch.uint8, device=DEV)
    seqs = {"": torch.zeros(1 + T, Q, 256, device=DEV)}
    seqs["_f16"], seqs["_bf16"] = seqs[""].half(), seqs[""].bfloat16()
    qo = torch.empty(Q, 256, device=DEV)
    frames = torch.randn(P * 2, 256, device=DEV)
    start = torch.arange(0, 2 * P + 1, 2, dtype=torch.int32, device=DEV)
    ftarget = torch.zeros(P, dtype=torch.int32, device=DEV)
    fa, fm = torch.zeros(P, device=DEV), torch.zeros(P, device=DEV)
    ra, rm = torch.empty(P, dtype=torch.int32, device=DEV), torch.empty(P, dtype=torch.int32, device=DEV)
    peer = pkg.PeerExchange(engine, Q, k)

    # name -> call(rows, g16): every _gbf16 entry, with everything but the gallery pointers valid
    calls = {
        "seam_prepare_gallery_bf16": lambda r, s: lib.seam_prepare_gallery_bf16(h, r, G, s, cg.data_ptr(),
                                                                               gstat.data_ptr(), stream),
        "seam_score_topk_gbf16": lambda r, s: lib.seam_score_topk_gbf16(
            h, q.data_ptr(), Q, r, s, cg.data_ptr(), gstat.data_ptr(), G, 0, k, sc.data_ptr(), mg.data_ptr(),
            ix.data_ptr(), None, ws.data_ptr(), ws.numel(), stream),
        "seam_sharded_score_topk_gbf16": lambda r, s: lib.seam_sharded_score_topk_gbf16(
            h, C.byref(peer.struct), r, s, cg.data_ptr(), gstat.data_ptr(), G, 0, None, ws.data_ptr(), ws.numel(),
            stream),
        "seam_rank_of_target_prepared_gbf16": lambda r, s: lib.seam_rank_of_target_prepared_gbf16(
            h, q.data_ptr(), Q, r, s, cg.data_ptr(), gstat.data_ptr(), G, target.data_ptr(), rank.data_ptr(),
            margin.data_ptr(), None, ws.data_ptr(), ws.numel(), stream),
        "seam_shard_rank_count_prepared_gbf16": lambda r, s: lib.seam_shard_rank_count_prepared_gbf16(
            h, q.data_ptr(), Q, r, s, cg.data_ptr(), gstat.data_ptr(), G, 0, target.data_ptr(), margin.data_ptr(),
            rank.data_ptr(), None, ws.data_ptr(), ws.numel(), stream),
        "seam_shard_target_margin_gbf16": lambda r, s: lib.seam_shard_target_margin_gbf16(
            h, q.data_ptr(), Q, r, G, 0, target.data_ptr(), margin.data_ptr(), stream),
        "seam_rank_fused_distances_gbf16": lambda r, s: lib.seam_rank_fused_distances_gbf16(
            h, frames.data_ptr(), start.data_ptr(), P, r, G, ftarget.data_ptr(), ra.data_ptr(), rm.data_ptr(), stream),
        "seam_shard_fused_target_gbf16": lambda r, s: lib.seam_shard_fused_target_gbf16(
            h, frames.data_ptr(), start.data_ptr(), P, r, G, 0, ftarget.data_ptr(), fa.data_ptr(), fm.data_ptr(),
            stream),
        "seam_shard_rank_fused_distances_gbf16": lambda r, s: lib.seam_shard_rank_fused_distances_gbf16(
            h, frames.data_ptr(), start.data_ptr(), P, r, G, 0, ftarget.data_ptr(), fa.data_ptr(), fm.data_ptr(),
            ra.data_ptr(), rm.data_ptr(), stream),
    }
    for tr, seq in seqs.items():
        calls[f"seam_search{tr}_gbf16"] = (lambda fn, seq: lambda r, s: fn(
            h, seq.data_ptr(), None, None, T, Q, Q * 256, 256, qo.data_ptr(), r, s, cg.data_ptr(), gstat.data_ptr(), G,
            0, k, sc.data_ptr(), mg.data_ptr(), ix.data_ptr(), None, ws.data_ptr(), ws.numel(), stream))(
                getattr(lib, f"seam_search{tr}_gbf16"), seq)
    takes_g16 = {n for n in calls if "fused" not in n and "target_margin" not in n}
    assert len(calls) == 12 and len(takes_g16) == 8

    def check(name, rc, code):
        assert rc == code, (name, rc)
        assert name.encode() + b":" in lib.seam_last_error(h), lib.seam_last_error(h)

    for name, call in calls.items():
        check(name, call(bad, g16), 2)                                 # SEAM_ERR_UNSUPPORTED
        check(name, call(None, g16), 1)                                # SEAM_ERR_BAD_ARG
        if name in takes_g16:
            check(name, call(rows, bad16), 2)
            check(name, call(rows, None), 1)
    # the aligned pointers are accepted
    assert calls["seam_prepare_gallery_bf16"](rows, g16) == 0
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ 2. score_topk
@pytest.mark.parametrize("G", [1, 7, 20, 255, 256, 257, 3000, 20000])
def test_score_topk_bf16_gallery_is_bit_identical(engine, G):
    for Q in (1, 130, 300):
        q, gb = _data(Q, G, seed=G * 7 + Q)
        pb = engine.prepare_gallery(gb, index_offset=1000)
        p32 = engine.prepare_gallery(gb.float(), index_offset=1000)
        _prepared_same(pb, p32)
        for k in (1, 20, 32):
            _all_same(_topk(engine, q, pb, k), _topk(engine, q, p32, k))


def test_score_topk_bf16_gallery_split_exhaustive_rows(engine):
    """40 distinct rows, each repeated 75 times: no query row can be certified, and there are fewer such rows than
    CTAs, so exact_topk_kernel<__nv_bfloat16> cuts each row's gallery into slices"""
    Q, G, k = 100, 3000, 20
    q, base = _data(Q, 40, seed=11)
    gb = base[torch.arange(G, device=DEV) % 40].contiguous()
    rb = _topk(engine, q, engine.prepare_gallery(gb, index_offset=7), k)
    r32 = _topk(engine, q, engine.prepare_gallery(gb.float(), index_offset=7), k)
    _all_same(rb, r32)
    assert 0 < int(rb[3][0]) < _num_ctas_exact()


def test_score_topk_bf16_gallery_every_row_exhaustive(engine):
    """queries scaled past the fp16 range: the query operand overflows and every row takes the exhaustive path"""
    Q, G, k = 200, 3000, 20
    q, gb = _data(Q, G, seed=13)
    q = q * 1e6
    rb = _topk(engine, q, engine.prepare_gallery(gb), k)
    _all_same(rb, _topk(engine, q, engine.prepare_gallery(gb.float()), k))
    assert int(rb[3][0]) == Q


def test_score_topk_bf16_gallery_slab_path(engine, monkeypatch):
    Q, G, k = 5000, 3000, 20
    q, gb = _data(Q, G, seed=15)
    pb, p32 = engine.prepare_gallery(gb), engine.prepare_gallery(gb.float())
    whole = _topk(engine, q, pb, k)
    monkeypatch.setattr(sys.modules[pkg.__name__ + ".engine"], "SCORE_WS_LIMIT", 16 << 20)
    assert engine._lib.seam_score_workspace_bytes(engine._h, Q, G, k) > 16 << 20
    slabs = _topk(engine, q, pb, k)
    _all_same(slabs, _topk(engine, q, p32, k))
    _all_same(slabs, whole)


# ------------------------------------------------------------------------------------------------ 3. bf16 -> fp16 inexact
@pytest.mark.parametrize("values", [(65536.0,), (65504.0, -65536.0), (float("inf"),), (float("-inf"), 1.0),
                                    (3.0e38, -3.3e38)])
def test_values_beyond_the_fp16_range(engine, values):
    """bf16 values at or above fp16's maximum, infinities and values near bf16's maximum: g16 overflows there, the
    overflow flag is set as fp32 sets it, and the outputs equal fp32's (every row exhaustive)"""
    Q, G, k = 150, 2000, 20
    q, gb = _data(Q, G, seed=14)
    for i, v in enumerate(values):
        gb[5 + 100 * i, 7 + i] = v
    pb, p32 = engine.prepare_gallery(gb), engine.prepare_gallery(gb.float())
    _prepared_same(pb, p32)
    assert float(pb.gstat[1]) != 0.0
    rb = _topk(engine, q, pb, k)
    _all_same(rb, _topk(engine, q, p32, k))
    assert int(rb[3][0]) == Q


def test_values_fp16_cannot_hold(engine):
    """rows in fp16's subnormal range, rows below 2^-25 (zero in fp16) and bf16 subnormals: g16 loses bits there, the
    same bits the fp32 path's rounding loses -- same operand, same candidates, same results"""
    Q, G, k = 300, 3000, 20
    q, gb = _data(Q, G, seed=16, scale=1e-5)                          # |g| ~ 1e-5: fp16 subnormals
    gen = torch.Generator(device=DEV).manual_seed(17)
    gb[1000:1500] = (1e-9 * torch.randn(500, 256, device=DEV, generator=gen)).bfloat16()     # below 2^-25
    sub = torch.randint(1, 0x80, (100, 256), dtype=torch.int16, device=DEV, generator=gen)   # exponent 0, mantissa != 0
    sub[:, ::2] |= -0x8000                                                                    # half of them negative
    gb[1500:1600] = sub.view(torch.bfloat16)                                                  # bf16 subnormals
    pb, p32 = engine.prepare_gallery(gb, index_offset=3), engine.prepare_gallery(gb.float(), index_offset=3)
    _prepared_same(pb, p32)
    assert float(pb.gstat[1]) == 0.0
    assert not torch.equal(pb.g16.float(), gb.float())                 # the operand is inexact here
    for qq in (q, q[:, torch.randperm(256, device=DEV, generator=gen)] * 1e-4):
        _all_same(_topk(engine, qq, pb, k), _topk(engine, qq, p32, k))
    target = torch.randint(0, G, (Q,), device=DEV, generator=gen)
    _all_same(engine.rank_of_target(q, pb, target, return_stats=True),
              engine.rank_of_target(q, p32, target, return_stats=True))


# ------------------------------------------------------------------------------------------------ 4. search
def test_search_bf16_gallery(engine, monkeypatch):
    Q, T, G, k = 700, 10, 3000, 20
    _, gb = _data(1, G, seed=18)
    pb, p32 = engine.prepare_gallery(gb), engine.prepare_gallery(gb.float())
    seqb, mask, _ = _tracks(Q, T, seed=19, dtype=torch.bfloat16, ragged=(0, 10))
    for seq in (seqb.float(), seqb.half(), seqb):                     # fp32, fp16 and bf16 tracks
        _all_same(engine.search(seq, mask, pb, k, return_stats=True), engine.search(seq, mask, p32, k, return_stats=True))
    # the large-workspace fallback (aggregate + the slab path of score_topk)
    monkeypatch.setattr(sys.modules[pkg.__name__ + ".engine"], "SCORE_WS_LIMIT", 16 << 20)
    seqb, mask, _ = _tracks(5000, 7, seed=20, dtype=torch.bfloat16, ragged=(1, 7))
    for seq in (seqb.float(), seqb.half(), seqb):
        _all_same(engine.search(seq, mask, pb, k), engine.search(seq, mask, p32, k))


# ------------------------------------------------------------------------------------------------ 5. rank of target
def test_rank_of_target_prepared_bf16_gallery(engine):
    Q, G = 400, 3000
    q, gb = _data(Q, G, seed=21)
    gen = torch.Generator(device=DEV).manual_seed(22)
    pb, p32 = engine.prepare_gallery(gb), engine.prepare_gallery(gb.float())
    ix = engine.score_topk(q, p32, 8)[2].long()
    target = torch.randint(0, G, (Q,), device=DEV, generator=gen)      # in the bulk
    target[: Q // 4] = ix[: Q // 4, 0]                                  # near the top: ranks 0 and 5
    target[Q // 4: Q // 2] = ix[Q // 4: Q // 2, 5]
    rb = engine.rank_of_target(q, pb, target, return_stats=True)
    _all_same(rb, engine.rank_of_target(q, p32, target, return_stats=True))
    _all_same(rb[:2], engine.rank_of_target(q, gb.float(), target))    # the exhaustive kernel on the widened rows
    assert bool((rb[0][: Q // 4] == 0).all()) and bool((rb[0][Q // 4: Q // 2] == 5).all())
    # every row to rank_of_target_kernel<__nv_bfloat16>: queries past the fp16 range
    qs = q * 1e6
    xb = engine.rank_of_target(qs, pb, target, return_stats=True)
    _all_same(xb, engine.rank_of_target(qs, p32, target, return_stats=True))
    _all_same(xb[:2], engine.rank_of_target(qs, gb.float(), target))
    assert int(xb[2][0]) == Q


def _shard_bounds(G, S):
    return [b for b in (pkg.shard_bounds(G, S, s) for s in range(S)) if b[1] > b[0]]


@pytest.mark.parametrize("S", [1, 2, 3, 8])
def test_sharded_rank_bf16_gallery(engine, S):
    """target margin on the owner, MAX, counts on every shard, SUM: the unsharded rank and margin, and shard for shard
    the fp32 shards' margins and counts; copies of targets straddle the boundaries of the three-shard split"""
    Q, G = 203, 6000
    q, gb = _data(Q, G, seed=23 + S)
    gen = torch.Generator(device=DEV).manual_seed(24)
    target = torch.randint(0, G, (Q,), device=DEV, generator=gen)
    target[0::5] = engine.score_topk(q[0::5], engine.prepare_gallery(gb), 1)[2][:, 0].long()
    gb[1999] = gb[2001] = gb[4000] = gb[2000]                          # boundaries of S = 3 at 2000 and 4000
    target[1::5] = 2000
    target[2::5] = 4000
    bounds = _shard_bounds(G, S)
    sb = [engine.prepare_gallery(gb[lo:hi], index_offset=lo) for lo, hi in bounds]
    s32 = [engine.prepare_gallery(gb[lo:hi].float(), index_offset=lo) for lo, hi in bounds]
    assert all(p.rows_bf16 and p.g.data_ptr() == gb[lo:].data_ptr() for p, (lo, _) in zip(sb, bounds))
    mb = torch.stack([engine.target_margin(q, p, target) for p in sb])
    m32 = torch.stack([engine.target_margin(q, p, target) for p in s32])
    assert _same(mb, m32) and bool(((mb != NEG_INF).sum(0) == 1).all())
    margin = mb.amax(0)
    rank = torch.zeros(Q, dtype=torch.int32, device=DEV)
    for pb, p32 in zip(sb, s32):
        cb = engine.rank_count(q, pb, target, margin, return_stats=True)
        _all_same(cb, engine.rank_count(q, p32, target, margin, return_stats=True))
        rank += cb[0]
    r_full, m_full = engine.rank_of_target(q, engine.prepare_gallery(gb), target)
    assert _same(rank, r_full) and _same(margin, m_full)
    assert _same(r_full, engine.rank_of_target(q, gb.float(), target)[0])
    assert bool((rank[2::5] >= 3).all())                              # the copies at 1999, 2000, 2001 rank before 4000
    for pb, p32 in zip(sb, s32):                                       # the exhaustive fallback of a bf16 shard
        qs = q * 1e6
        half = torch.full((Q,), 0.5, device=DEV)
        cb = engine.rank_count(qs, pb, target, half, return_stats=True)
        _all_same(cb, engine.rank_count(qs, p32, target, half, return_stats=True))
        assert int(cb[1][0]) == Q


# ------------------------------------------------------------------------------------------------ 6. fusions
def _fusion_data(P, G, fmax, seed):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    lens = torch.randint(1, fmax + 1, (P,), device=DEV, generator=gen)
    lens[1] = 0                                                        # a product without frames
    start = torch.zeros(P + 1, dtype=torch.int64, device=DEV)
    start[1:] = torch.cumsum(lens, 0)
    frames = torch.randn(int(start[-1]), 256, device=DEV, generator=gen)
    g = torch.randn(G, 256, device=DEV, generator=gen)
    target = torch.randint(0, G, (P,), device=DEV, generator=gen)
    for p in range(0, P, 2):
        if lens[p] > 0:
            g[target[p]] = frames[start[p]] + 0.3 * torch.randn(256, device=DEV, generator=gen)
    return frames, start, g.bfloat16(), target


@pytest.mark.parametrize("S", [1, 2, 3, 8])
def test_fusions_bf16_gallery(engine, S):
    P, G = 60, 5000
    frames, start, gb, target = _fusion_data(P, G, 20, seed=25)
    full = torch.stack(engine.rank_fused_distances(frames, start, gb, target))
    assert _same(full, torch.stack(engine.rank_fused_distances(frames, start, gb.float(), target)))
    tv = []
    for lo, hi in _shard_bounds(G, S):
        tb = torch.stack(engine.fused_target(frames, start, gb[lo:hi], lo, target))
        assert _same(tb, torch.stack(engine.fused_target(frames, start, gb[lo:hi].float(), lo, target)))
        tv.append(tb)
    tv = torch.stack(tv).amax(0)
    ranks = torch.zeros((2, P), dtype=torch.int32, device=DEV)
    for lo, hi in _shard_bounds(G, S):
        cb = torch.stack(engine.fused_rank_count(frames, start, gb[lo:hi], lo, target, tv[0], tv[1]))
        c32 = torch.stack(engine.fused_rank_count(frames, start, gb[lo:hi].float(), lo, target, tv[0], tv[1]))
        assert _same(cb, c32)
        ranks += cb
    assert _same(ranks, full) and ranks[:, 1].tolist() == [G, G]


def test_rank_fused_distances_bf16_makes_no_copy(engine):
    P, G = 80, 9000
    frames, start, gb, target = _fusion_data(P, G, 33, seed=26)
    r32 = torch.stack(engine.rank_fused_distances(frames, start, gb.float(), target))
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    rb = torch.stack(engine.rank_fused_distances(frames, start, gb, target))
    torch.cuda.synchronize()
    assert _same(rb, r32)
    assert torch.cuda.max_memory_allocated() - base < gb.nbytes // 2
    buf = torch.empty(G * 256 + 8, dtype=torch.bfloat16, device=DEV)
    mis = buf[1:1 + G * 256].view(G, 256)
    mis.copy_(gb)
    assert _same(torch.stack(engine.rank_fused_distances(frames, start, mis, target)), r32)


# ------------------------------------------------------------------------------------------------ 7. sharded search
def test_sharded_bf16_gallery_single_rank(engine):
    Q, T, G, k = 700, 10, 3000, 20
    _, gb = _data(1, G, seed=27)
    p32 = engine.prepare_gallery(gb.float())
    peer = pkg.PeerExchange(engine, Q, k)
    retr = pkg.ShardedRetriever(engine, gb, 0)
    assert retr.gallery.rows_bf16 and retr.gallery.g.data_ptr() == gb.data_ptr()
    for step in range(2):
        seqb, mask, _ = _tracks(Q, T, seed=28 + step, dtype=torch.bfloat16, ragged=(1, 10))
        _all_same(retr.search_peer(seqb, mask, peer), engine.search(seqb, mask, p32, k)[1:])
    assert peer.steps_done == 2


@pytest.mark.parametrize("replicate", [True, False])
def test_sharded_bf16_gallery_two_ranks_one_gpu(weights, engine, replicate):
    """two ranks in one process on two streams, each holding a zero-copy bf16 shard of the full bf16 gallery"""
    Q, T, G, k = 301, 4, 2500, 20
    engines = [engine, pkg.SeamEngine(DEV)]
    engines[1].load_weights({kk: v.to(DEV) for kk, v in weights.items()})
    _, gb = _data(1, G, seed=30)
    p32 = engine.prepare_gallery(gb.float())
    shared = {}
    peers = [pkg.PeerExchange(engines[r], Q, k, replicate=replicate,
                              local_peers={"world": 2, "rank": r, "shared": shared}) for r in range(2)]
    for p in peers:
        p._fill_struct()
    bounds = [pkg.shard_bounds(G, 2, r) for r in range(2)]
    retrs = [pkg.ShardedRetriever(engines[r], gb[bounds[r][0]:bounds[r][1]], bounds[r][0], world=2, rank=r)
             for r in range(2)]
    for r in range(2):
        assert retrs[r].gallery.rows_bf16 and retrs[r].gallery.g.data_ptr() == gb[bounds[r][0]:].data_ptr()
    streams = [torch.cuda.Stream(DEV) for _ in range(2)]
    for step in range(2):
        seqb, mask, _ = _tracks(Q, T, seed=31 + step, dtype=torch.bfloat16, ragged=(0, 4))
        ref = engine.search(seqb, mask, p32, k)[1:]
        torch.cuda.synchronize()
        res = [None, None]
        for r in (0, 1):
            streams[r].wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(streams[r]):
                res[r] = retrs[r].search_peer(seqb, mask, peers[r])
        torch.cuda.synchronize()
        assert engines[0].watchdog_records() == []
        for r in range(2):
            lo, hi = (0, Q) if replicate else (peers[r].q_lo[r], peers[r].q_lo[r + 1])
            _all_same(res[r], [t[lo:hi] for t in ref])
    assert peers[0].steps_done == 2 and peers[1].steps_done == 2


# ------------------------------------------------------------------------------------------------ 8. host
def test_search_host_bf16_gallery(engine, monkeypatch):
    Q, T, G, k = 403, 7, 2777, 20
    seqb, mask, _ = _tracks(Q, T, seed=33, dtype=torch.bfloat16, ragged=(1, 7))
    _, gb = _data(1, G, seed=34)
    hgb = gb.cpu().pin_memory()
    hg32 = hgb.float().pin_memory()
    hm = mask.cpu().pin_memory()
    seen = []
    prepare = engine.prepare_gallery

    def spy(g, *a, **kw):
        seen.append(g.dtype)
        return prepare(g, *a, **kw)

    monkeypatch.setattr(engine, "prepare_gallery", spy)
    stream = pkg.HostTrackStream(engine, nchunk=3)
    for hs in (seqb.cpu().float().pin_memory(), seqb.cpu().pin_memory()):   # fp32 tracks, bf16 tracks
        ob = pkg.search_host(engine, hs, hm, hgb, k, stream=stream)
        torch.cuda.synchronize()
        ob = [t.clone() for t in ob]
        o32 = pkg.search_host(engine, hs, hm, hg32, k, stream=stream)
        torch.cuda.synchronize()
        _all_same(ob, o32)
    assert seen == [torch.bfloat16, torch.float32] * 2


# ------------------------------------------------------------------------------------------------ 9. scorer swap
def test_scorer_swap_reprepares_bf16_gallery(engine):
    Q, G, k = 300, 3000, 20
    q, gb = _data(Q, G, seed=35)
    pb = engine.prepare_gallery(gb)
    g16_before = pb.g16.clone()
    gen = torch.Generator(device=DEV).manual_seed(36)
    lw = 0.1 * torch.randn(2, 256, device=DEV, generator=gen)
    lb = 0.1 * torch.randn(2, device=DEV, generator=gen)
    with engine.scorer(lw, lb):
        r = _topk(engine, q, pb, k)                                     # re-prepared through _fresh
        fresh = engine.prepare_gallery(gb)
        assert pb.g.data_ptr() == gb.data_ptr()
        assert torch.equal(pb.g16, g16_before) and torch.equal(pb.g16, fresh.g16)
        assert _same(pb.cg, fresh.cg) and _same(pb.gstat, fresh.gstat)
        _all_same(r, _topk(engine, q, fresh, k))
        _all_same(r, _topk(engine, q, engine.prepare_gallery(gb.float()), k))
    _all_same(_topk(engine, q, pb, k), _topk(engine, q, engine.prepare_gallery(gb), k))


# ------------------------------------------------------------------------------------------------ 10. module and eval
@pytest.fixture(scope="module")
def model(weights, engine):
    m = pkg.TemporalAggregationNLB().to(DEV).eval()
    missing, unexpected = m.load_state_dict(weights, strict=False)
    assert not unexpected
    return m


def test_module_score_topk_bf16_gallery(model):
    seqb, mask, _ = _tracks(37, 10, seed=37, dtype=torch.bfloat16, ragged=(0, 10))
    _, gb = _data(1, 300, seed=38)
    _all_same(model.score_topk(seqb, mask, gb, k=20), model.score_topk(seqb, mask, gb.float(), k=20))
    pb = model.prepare_gallery(gb)
    assert pb.rows_bf16 and pb.g.data_ptr() == gb.data_ptr()
    _all_same(model.score_topk(seqb, mask, pb, k=20), model.score_topk(seqb, mask, gb.float(), k=20))


def _eval_case(engine, weights, P=120, T=6, G=1500, N=400, seed=39):
    seqb, mask, _ = _tracks(P, T, seed=seed, dtype=torch.bfloat16, ragged=(1, 6))
    gen = torch.Generator(device=DEV).manual_seed(seed + 1)
    target = torch.randint(0, G, (P,), device=DEV, generator=gen)
    _, shopb = _data(1, G, seed=seed + 2)
    _, aggrb = _data(1, G, seed=seed + 3)
    frame_product = torch.randint(0, P, (N,), device=DEV, generator=gen)
    frame_desc = shopb[target[frame_product]].float() + 0.3 * torch.randn(N, 256, device=DEV, generator=gen)
    frame_last = (0.1 * torch.randn(2, 256, device=DEV, generator=gen), 0.1 * torch.randn(2, device=DEV, generator=gen))
    aggr_last = (weights["last.weight"].to(DEV), weights["last.bias"].to(DEV))
    return seqb, mask, target, shopb, aggrb, frame_product, frame_desc, frame_last, aggr_last


def test_evaluate_with_bf16_shop_descriptors(engine, weights, monkeypatch):
    seqb, mask, target, shopb, aggrb, fprod, fdesc, frame_last, aggr_last = _eval_case(engine, weights)
    seen = []
    prepare = engine.prepare_gallery

    def spy(g, *a, **kw):
        seen.append(g.dtype)
        return prepare(g, *a, **kw)

    monkeypatch.setattr(engine, "prepare_gallery", spy)
    ab = pkg.evaluate_aggregated(engine, seqb, mask, aggrb, target)
    a32 = pkg.evaluate_aggregated(engine, seqb, mask, aggrb.float(), target)
    _all_same([ab.ranks, ab.topk_scores, ab.topk_idx], [a32.ranks, a32.topk_scores, a32.topk_idx])
    assert ab.hits == a32.hits
    eb = pkg.evaluate_products(engine, fdesc, fprod, shopb, target, frame_last, seqb, mask, aggrb, aggr_last)
    e32 = pkg.evaluate_products(engine, fdesc, fprod, shopb.float(), target, frame_last, seqb, mask, aggrb.float(),
                                aggr_last)
    _all_same([eb.perf, eb.frame_ranks, eb.product_ranks], [e32.perf, e32.frame_ranks, e32.product_ranks])
    assert seen == [torch.bfloat16, torch.float32] + [torch.bfloat16] * 2 + [torch.float32] * 2
    fb = pkg.evaluate_distance_fusions(engine, fdesc, fprod, shopb, target, frame_last)
    f32 = pkg.evaluate_distance_fusions(engine, fdesc, fprod, shopb.float(), target, frame_last)
    _all_same(fb, f32)


def test_sharded_retriever_world1_bf16(engine, weights):
    seqb, mask, target, shopb, aggrb, fprod, fdesc, frame_last, aggr_last = _eval_case(engine, weights, seed=45)
    retr = pkg.ShardedRetriever(engine, aggrb, 0)
    assert retr.world == 1 and retr.gallery.rows_bf16
    ref = pkg.ShardedRetriever(engine, aggrb.float(), 0)
    fb = retr.evaluate_distance_fusions(fdesc, fprod, shopb, target, frame_last)
    _all_same(fb, ref.evaluate_distance_fusions(fdesc, fprod, shopb.float(), target, frame_last))
    eb = retr.evaluate_products(fdesc, fprod, shopb, target, frame_last, seqb, mask, aggr_last)
    e32 = ref.evaluate_products(fdesc, fprod, shopb.float(), target, frame_last, seqb, mask, aggr_last)
    _all_same([eb.perf, eb.frame_ranks, eb.product_ranks], [e32.perf, e32.frame_ranks, e32.product_ranks])
    ab = retr.evaluate_aggregated(seqb, mask, target)
    a32 = ref.evaluate_aggregated(seqb, mask, target)
    _all_same([ab.ranks, ab.topk_scores, ab.topk_idx], [a32.ranks, a32.topk_scores, a32.topk_idx])
    assert ab.hits == a32.hits
