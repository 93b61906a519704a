"""fp16 galleries: a gallery given as fp16 is kept as fp16 -- it is the tensor-core operand g16 and the rows the fp32
direct form reads (widened exactly), through the seam_prepare_gallery_f16 / *_g16 entry points -- and every result
equals, bit for bit, what the fp32 path gives on the widened gallery g16.float().  Float tensors are compared by their
bit patterns (NaN included)."""
import ctypes as C
import sys

import pytest
import torch

import seam_match_rcnn_b200 as pkg

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _same(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(_bits(a), _bits(b))


def _all_same(xs, ys):
    xs, ys = list(xs), list(ys)
    assert len(xs) == len(ys)
    for i, (a, b) in enumerate(zip(xs, ys)):
        assert _same(a, b), f"output {i} differs"


def _data(Q, G, seed, planted=True):
    """queries (Q,256) fp32 and an fp16 gallery (G,256) on the device whose first min(Q,G) rows are near-duplicates of
    the queries (a true match per query, as in bench.py)."""
    gen = torch.Generator(device=DEV).manual_seed(seed)
    q = torch.randn(Q, 256, device=DEV, generator=gen)
    g = torch.randn(G, 256, device=DEV, generator=gen)
    n = min(Q, G)
    if planted and n:
        g[:n] = q[:n] + 0.1 * torch.randn(n, 256, device=DEV, generator=gen)
    return q, g.half()


def _tracks16(Q, T, seed, ragged=None):
    g = torch.Generator(device=DEV).manual_seed(seed)
    seq = torch.randn(1 + T, Q, 256, device=DEV, generator=g).to(torch.float16)
    lens = (torch.full((Q,), T, dtype=torch.int64, device=DEV) if ragged is None
            else torch.randint(ragged[0], ragged[1] + 1, (Q,), device=DEV, generator=g))
    mask = torch.arange(1 + T, device=DEV).unsqueeze(0) > lens.unsqueeze(1)
    seq.masked_fill_(mask.t().unsqueeze(2), 0.0)
    seq[0] = 0.0
    return seq, mask, lens


def _topk(engine, q, gal, k):
    return engine.score_topk(q, gal, k, return_stats=True)


def _num_ctas_exact():
    return 2 * torch.cuda.get_device_properties(DEV).multi_processor_count


# ------------------------------------------------------------------------------------------------ 1. prepare
def test_prepare_f16_matches_fp32_and_uses_the_callers_rows(engine):
    _, g16 = _data(1, 5000, seed=1)
    p16 = engine.prepare_gallery(g16)
    p32 = engine.prepare_gallery(g16.float())
    assert p16.rows_f16 and not p32.rows_f16
    assert p16.g16.data_ptr() == g16.data_ptr() and p16.g.data_ptr() == g16.data_ptr() and p16.G == 5000
    assert _same(p16.cg, p32.cg) and _same(p16.gstat, p32.gstat)
    assert torch.equal(p32.g16, g16)                                  # round_fp16(g.float()) == g: the same operand
    with pytest.raises(AttributeError):
        p16.rows_f16 = False


def test_prepare_f16_makes_no_copy(engine):
    """cg is 4 bytes per row against 512 of g16: a fp32 copy (1 KB per row) or a second fp16 copy would show."""
    _, g16 = _data(1, 200000, seed=2, planted=False)
    engine.prepare_gallery(g16[:1000])
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(DEV)
    torch.cuda.reset_peak_memory_stats(DEV)
    p = engine.prepare_gallery(g16)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated(DEV) - base < g16.nbytes // 2
    assert p.g16.data_ptr() == g16.data_ptr()


def test_prepare_f16_copies_misaligned_strided_and_host_views(engine):
    Q, G, k = 300, 3000, 20
    q, g16 = _data(Q, G, seed=3)
    p32 = engine.prepare_gallery(g16.float())
    ref = _topk(engine, q, p32, k)
    buf = torch.zeros(G * 256 + 1, dtype=torch.float16, device=DEV)
    mis = buf[1:].view(G, 256)                                         # storage offset of one element
    mis.copy_(g16)
    wide = torch.zeros(G, 264, dtype=torch.float16, device=DEV)
    wide[:, :256] = g16
    strided = wide[:, :256]                                            # row stride 264
    assert mis.is_contiguous() and mis.data_ptr() % 16 and not strided.is_contiguous()
    for view in (mis, strided, g16.cpu()):
        p = engine.prepare_gallery(view)
        assert p.rows_f16 and p.g16.is_contiguous() and p.g16.data_ptr() % 16 == 0
        assert p.g16.data_ptr() != view.data_ptr() and torch.equal(p.g16, g16)
        assert _same(p.cg, p32.cg) and _same(p.gstat, p32.gstat)
        _all_same(_topk(engine, q, p, k), ref)


def test_g16_entries_reject_misaligned_rows(engine):
    lib, h = engine._lib, engine._h
    stream = torch.cuda.current_stream(DEV).cuda_stream
    Q, G, k, T = 8, 512, 4, 3
    buf = torch.zeros(G * 256 + 8, dtype=torch.float16, device=DEV)
    bad = buf.data_ptr() + 2
    q = torch.randn(Q, 256, device=DEV)
    cg = torch.empty(G, device=DEV)
    gstat = torch.zeros(4, device=DEV)
    sc, mg = torch.empty(Q, k, device=DEV), torch.empty(Q, k, device=DEV)
    ix = torch.empty(Q, k, dtype=torch.int32, device=DEV)
    target = torch.zeros(Q, dtype=torch.int32, device=DEV)
    rank, margin = torch.empty(Q, dtype=torch.int32, device=DEV), torch.empty(Q, device=DEV)
    ws = torch.empty(max(lib.seam_score_workspace_bytes(h, Q, G, k), lib.seam_rank_workspace_bytes(h, Q, G)),
                     dtype=torch.uint8, device=DEV)
    seq = torch.zeros(1 + T, Q, 256, device=DEV)
    seq16 = seq.half()
    qo = torch.empty(Q, 256, device=DEV)

    def check(name, rc):
        assert rc == 2, name                                            # SEAM_ERR_UNSUPPORTED
        assert name.encode() + b":" in lib.seam_last_error(h), lib.seam_last_error(h)

    check("seam_prepare_gallery_f16", lib.seam_prepare_gallery_f16(h, bad, G, cg.data_ptr(), gstat.data_ptr(), stream))
    check("seam_score_topk_g16", lib.seam_score_topk_g16(h, q.data_ptr(), Q, bad, cg.data_ptr(), gstat.data_ptr(), G, 0,
                                                         k, sc.data_ptr(), mg.data_ptr(), ix.data_ptr(), None,
                                                         ws.data_ptr(), ws.numel(), stream))
    for name, s in (("seam_search_g16", seq), ("seam_search_f16_g16", seq16)):
        check(name, getattr(lib, name)(h, s.data_ptr(), None, None, T, Q, Q * 256, 256, qo.data_ptr(), bad,
                                       cg.data_ptr(), gstat.data_ptr(), G, 0, k, sc.data_ptr(), mg.data_ptr(),
                                       ix.data_ptr(), None, ws.data_ptr(), ws.numel(), stream))
    check("seam_rank_of_target_prepared_g16",
          lib.seam_rank_of_target_prepared_g16(h, q.data_ptr(), Q, bad, cg.data_ptr(), gstat.data_ptr(), G,
                                               target.data_ptr(), rank.data_ptr(), margin.data_ptr(), None,
                                               ws.data_ptr(), ws.numel(), stream))
    peer = pkg.PeerExchange(engine, Q, k)
    check("seam_sharded_score_topk_g16",
          lib.seam_sharded_score_topk_g16(h, C.byref(peer.struct), bad, cg.data_ptr(), gstat.data_ptr(), G, 0,
                                          None, ws.data_ptr(), ws.numel(), stream))
    # the aligned pointer is accepted
    assert lib.seam_prepare_gallery_f16(h, buf.data_ptr(), G, cg.data_ptr(), gstat.data_ptr(), stream) == 0
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ 2. score_topk
@pytest.mark.parametrize("G", [1, 7, 20, 255, 256, 257, 3000, 20000])
def test_score_topk_f16_gallery_is_bit_identical(engine, G):
    for Q in (1, 130, 300):
        q, g16 = _data(Q, G, seed=G * 7 + Q)
        p16 = engine.prepare_gallery(g16, index_offset=1000)
        p32 = engine.prepare_gallery(g16.float(), index_offset=1000)
        for k in (1, 20, 32):
            _all_same(_topk(engine, q, p16, k), _topk(engine, q, p32, k))


def test_score_topk_f16_gallery_split_exhaustive_rows(engine):
    """A gallery of 40 distinct rows, each repeated 75 times: every query's window fills with copies of its best row,
    so no row can be certified -- and there are fewer such rows than CTAs, so exact_topk_kernel<__half> cuts each
    row's gallery into slices."""
    Q, G, k = 100, 3000, 20
    q, base = _data(Q, 40, seed=11)
    g16 = base[torch.arange(G, device=DEV) % 40].contiguous()
    r16 = _topk(engine, q, engine.prepare_gallery(g16, index_offset=7), k)
    r32 = _topk(engine, q, engine.prepare_gallery(g16.float(), index_offset=7), k)
    _all_same(r16, r32)
    assert 0 < int(r16[3][0]) < _num_ctas_exact()


def test_score_topk_f16_gallery_every_row_exhaustive(engine):
    """Queries scaled past the fp16 range: the query operand overflows and every row takes the exhaustive path."""
    Q, G, k = 200, 3000, 20
    q, g16 = _data(Q, G, seed=13)
    q = q * 1e6
    r16 = _topk(engine, q, engine.prepare_gallery(g16), k)
    r32 = _topk(engine, q, engine.prepare_gallery(g16.float()), k)
    _all_same(r16, r32)
    assert int(r16[3][0]) == Q


@pytest.mark.parametrize("value", [float("inf"), 65504.0])
def test_score_topk_f16_gallery_overflow_flag(engine, value):
    Q, G, k = 150, 2000, 20
    q, g16 = _data(Q, G, seed=14)
    g16[5, 7] = value
    p16, p32 = engine.prepare_gallery(g16), engine.prepare_gallery(g16.float())
    assert _same(p16.gstat, p32.gstat) and float(p16.gstat[1]) != 0.0
    r16 = _topk(engine, q, p16, k)
    _all_same(r16, _topk(engine, q, p32, k))
    assert int(r16[3][0]) == Q


def test_score_topk_f16_gallery_slab_path(engine, monkeypatch):
    Q, G, k = 5000, 3000, 20
    q, g16 = _data(Q, G, seed=15)
    p16, p32 = engine.prepare_gallery(g16), engine.prepare_gallery(g16.float())
    whole = _topk(engine, q, p16, k)
    monkeypatch.setattr(sys.modules[pkg.__name__ + ".engine"], "SCORE_WS_LIMIT", 16 << 20)
    assert engine._lib.seam_score_workspace_bytes(engine._h, Q, G, k) > 16 << 20
    slabs = _topk(engine, q, p16, k)
    _all_same(slabs, _topk(engine, q, p32, k))
    _all_same(slabs, whole)


# ------------------------------------------------------------------------------------------------ 3. search
def test_search_f16_gallery(engine, monkeypatch):
    Q, T, G, k = 700, 10, 3000, 20
    _, g16 = _data(1, G, seed=16)
    p16, p32 = engine.prepare_gallery(g16), engine.prepare_gallery(g16.float())
    seq16, mask, _ = _tracks16(Q, T, seed=17, ragged=(0, 10))
    for seq in (seq16.float(), seq16):                                  # fp32 tracks, fp16 tracks
        _all_same(engine.search(seq, mask, p16, k, return_stats=True), engine.search(seq, mask, p32, k, return_stats=True))
    # the large-workspace fallback (aggregate + the slab path of score_topk)
    monkeypatch.setattr(sys.modules[pkg.__name__ + ".engine"], "SCORE_WS_LIMIT", 16 << 20)
    seq16, mask, _ = _tracks16(5000, 7, seed=18, ragged=(1, 7))
    for seq in (seq16.float(), seq16):
        _all_same(engine.search(seq, mask, p16, k), engine.search(seq, mask, p32, k))


# ------------------------------------------------------------------------------------------------ 4. rank of target
def test_rank_of_target_prepared_f16_gallery(engine):
    Q, G = 400, 3000
    q, g16 = _data(Q, G, seed=19)
    gen = torch.Generator(device=DEV).manual_seed(20)
    p16, p32 = engine.prepare_gallery(g16), engine.prepare_gallery(g16.float())
    ix = engine.score_topk(q, p32, 8)[2].long()
    target = torch.randint(0, G, (Q,), device=DEV, generator=gen)      # in the bulk
    target[: Q // 4] = ix[: Q // 4, 0]                                  # near the top: ranks 0 and 5
    target[Q // 4: Q // 2] = ix[Q // 4: Q // 2, 5]
    r16 = engine.rank_of_target(q, p16, target, return_stats=True)
    _all_same(r16, engine.rank_of_target(q, p32, target, return_stats=True))
    _all_same(r16[:2], engine.rank_of_target(q, g16.float(), target))   # the exhaustive kernel on the widened rows
    assert bool((r16[0][: Q // 4] == 0).all()) and bool((r16[0][Q // 4: Q // 2] == 5).all())
    assert int(r16[0][Q // 2:].float().median()) > 100
    # every row to rank_of_target_kernel<__half>: queries past the fp16 range
    qs = q * 1e6
    x16 = engine.rank_of_target(qs, p16, target, return_stats=True)
    _all_same(x16, engine.rank_of_target(qs, p32, target, return_stats=True))
    _all_same(x16[:2], engine.rank_of_target(qs, g16.float(), target))
    assert int(x16[2][0]) == Q


# ------------------------------------------------------------------------------------------------ 5. sharded
def test_sharded_f16_gallery_single_rank(engine):
    Q, T, G, k = 700, 10, 3000, 20
    _, g16 = _data(1, G, seed=21)
    p32 = engine.prepare_gallery(g16.float())
    peer = pkg.PeerExchange(engine, Q, k)
    retr = pkg.ShardedRetriever(engine, g16, 0)
    assert retr.gallery.rows_f16 and retr.gallery.g16.data_ptr() == g16.data_ptr()
    for step in range(2):
        seq16, mask, _ = _tracks16(Q, T, seed=22 + step, ragged=(1, 10))
        _all_same(retr.search_peer(seq16, mask, peer), engine.search(seq16, mask, p32, k)[1:])
    assert peer.steps_done == 2


@pytest.mark.parametrize("replicate", [True, False])
def test_sharded_f16_gallery_two_ranks_one_gpu(weights, engine, replicate):
    """Two ranks in one process on two streams, each holding a zero-copy fp16 shard of the full fp16 gallery."""
    Q, T, G, k = 301, 4, 2500, 20
    engines = [engine, pkg.SeamEngine(DEV)]
    engines[1].load_weights({kk: v.to(DEV) for kk, v in weights.items()})
    _, g16 = _data(1, G, seed=23)
    p32 = engine.prepare_gallery(g16.float())
    shared = {}
    peers = [pkg.PeerExchange(engines[r], Q, k, replicate=replicate,
                              local_peers={"world": 2, "rank": r, "shared": shared}) for r in range(2)]
    for p in peers:
        p._fill_struct()
    bounds = [pkg.shard_bounds(G, 2, r) for r in range(2)]
    retrs = [pkg.ShardedRetriever(engines[r], g16[bounds[r][0]:bounds[r][1]], bounds[r][0], world=2, rank=r)
             for r in range(2)]
    for r in range(2):
        assert retrs[r].gallery.rows_f16 and retrs[r].gallery.g16.data_ptr() == g16[bounds[r][0]:].data_ptr()
    streams = [torch.cuda.Stream(DEV) for _ in range(2)]
    for step in range(2):
        seq16, mask, _ = _tracks16(Q, T, seed=24 + step, ragged=(0, 4))
        ref = engine.search(seq16, mask, p32, k)[1:]
        torch.cuda.synchronize()
        res = [None, None]
        for r in (0, 1):
            streams[r].wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(streams[r]):
                res[r] = retrs[r].search_peer(seq16, mask, peers[r])
        torch.cuda.synchronize()
        assert engines[0].watchdog_records() == []
        for r in range(2):
            lo, hi = (0, Q) if replicate else (peers[r].q_lo[r], peers[r].q_lo[r + 1])
            _all_same(res[r], [t[lo:hi] for t in ref])
    assert peers[0].steps_done == 2 and peers[1].steps_done == 2


# ------------------------------------------------------------------------------------------------ 6. host
def test_search_host_f16_gallery(engine, monkeypatch):
    Q, T, G, k = 403, 7, 2777, 20
    seq16, mask, _ = _tracks16(Q, T, seed=25, ragged=(1, 7))
    _, g16 = _data(1, G, seed=26)
    hg16 = g16.cpu().pin_memory()
    hg32 = hg16.float().pin_memory()
    hm = mask.cpu().pin_memory()
    seen = []
    prepare = engine.prepare_gallery

    def spy(g, *a, **kw):
        seen.append(g.dtype)
        return prepare(g, *a, **kw)

    monkeypatch.setattr(engine, "prepare_gallery", spy)
    stream = pkg.HostTrackStream(engine, nchunk=3)
    for hs in (seq16.cpu().float().pin_memory(), seq16.cpu().pin_memory()):   # fp32 tracks, fp16 tracks
        o16 = pkg.search_host(engine, hs, hm, hg16, k, stream=stream)
        torch.cuda.synchronize()
        o16 = [t.clone() for t in o16]
        o32 = pkg.search_host(engine, hs, hm, hg32, k, stream=stream)
        torch.cuda.synchronize()
        _all_same(o16, o32)
    assert seen == [torch.float16, torch.float32] * 2


# ------------------------------------------------------------------------------------------------ 7. scorer swap
def test_scorer_swap_reprepares_f16_gallery(engine):
    Q, G, k = 300, 3000, 20
    q, g16 = _data(Q, G, seed=27)
    p16 = engine.prepare_gallery(g16)
    gen = torch.Generator(device=DEV).manual_seed(28)
    lw = 0.1 * torch.randn(2, 256, device=DEV, generator=gen)
    lb = 0.1 * torch.randn(2, device=DEV, generator=gen)
    with engine.scorer(lw, lb):
        r = _topk(engine, q, p16, k)                                    # re-prepared through _fresh
        fresh = engine.prepare_gallery(g16)
        assert p16.g16.data_ptr() == g16.data_ptr()
        assert _same(p16.cg, fresh.cg) and _same(p16.gstat, fresh.gstat)
        _all_same(r, _topk(engine, q, fresh, k))
        _all_same(r, _topk(engine, q, engine.prepare_gallery(g16.float()), k))
    _all_same(_topk(engine, q, p16, k), _topk(engine, q, engine.prepare_gallery(g16), k))


# ------------------------------------------------------------------------------------------------ 8. module and eval
@pytest.fixture(scope="module")
def model(weights, engine):
    m = pkg.TemporalAggregationNLB().to(DEV).eval()
    missing, unexpected = m.load_state_dict(weights, strict=False)
    assert not unexpected
    return m


def test_module_score_topk_f16_gallery(model):
    seq16, mask, _ = _tracks16(37, 10, seed=29, ragged=(0, 10))
    _, g16 = _data(1, 300, seed=30)
    _all_same(model.score_topk(seq16, mask, g16, k=20), model.score_topk(seq16, mask, g16.float(), k=20))
    p16 = model.prepare_gallery(g16)
    assert p16.rows_f16 and p16.g16.data_ptr() == g16.data_ptr()
    _all_same(model.score_topk(seq16, mask, p16, k=20), model.score_topk(seq16, mask, g16.float(), k=20))


def test_evaluate_with_f16_shop_descriptors(engine, weights, monkeypatch):
    P, T, G, N = 120, 6, 1500, 400
    seq16, mask, _ = _tracks16(P, T, seed=31, ragged=(1, 6))
    gen = torch.Generator(device=DEV).manual_seed(32)
    target = torch.randint(0, G, (P,), device=DEV, generator=gen)
    _, shop16 = _data(1, G, seed=33)
    _, aggr16 = _data(1, G, seed=34)
    frame_product = torch.randint(0, P, (N,), device=DEV, generator=gen)
    frame_desc = shop16[target[frame_product]].float() + 0.3 * torch.randn(N, 256, device=DEV, generator=gen)
    frame_last = (0.1 * torch.randn(2, 256, device=DEV, generator=gen), 0.1 * torch.randn(2, device=DEV, generator=gen))
    aggr_last = (weights["last.weight"].to(DEV), weights["last.bias"].to(DEV))
    seen = []
    prepare = engine.prepare_gallery

    def spy(g, *a, **kw):
        seen.append(g.dtype)
        return prepare(g, *a, **kw)

    monkeypatch.setattr(engine, "prepare_gallery", spy)
    a16 = pkg.evaluate_aggregated(engine, seq16, mask, aggr16, target)
    a32 = pkg.evaluate_aggregated(engine, seq16, mask, aggr16.float(), target)
    _all_same([a16.ranks, a16.topk_scores, a16.topk_idx], [a32.ranks, a32.topk_scores, a32.topk_idx])
    assert a16.hits == a32.hits
    e16 = pkg.evaluate_products(engine, frame_desc, frame_product, shop16, target, frame_last, seq16, mask, aggr16,
                                aggr_last)
    e32 = pkg.evaluate_products(engine, frame_desc, frame_product, shop16.float(), target, frame_last, seq16, mask,
                                aggr16.float(), aggr_last)
    _all_same([e16.perf, e16.frame_ranks, e16.product_ranks], [e32.perf, e32.frame_ranks, e32.product_ranks])
    assert seen == [torch.float16, torch.float32] + [torch.float16] * 2 + [torch.float32] * 2
