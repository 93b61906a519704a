"""fp16 tracks: x3_1_seq given as fp16 is read as fp16 by the aggregation kernels (the seam_*_f16 entry points: half the
bytes, no conversion pass) and gives exactly what the fp32 path gives on the widened tracks.  Widening fp16 to fp32 is
exact and the kernels widen each frame as it leaves shared memory, so every comparison below is bit for bit."""
import ctypes as C
import sys

import pytest
import torch

import seam_match_rcnn_b200 as pkg

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _tracks16(Q, T, seed, ragged=None, scale=1.0):
    """(seq (1+T,Q,256) fp16 on the device with dummy row 0, mask (Q,1+T) bool, lens (Q) int64); ragged=(lo,hi) draws
    the lengths in [lo,hi] (0: empty track).  Padding frames are zero."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    seq = (torch.randn(1 + T, Q, 256, device=DEV, generator=g) * scale).to(torch.float16)
    if ragged is None:
        lens = torch.full((Q,), T, dtype=torch.int64, device=DEV)
    else:
        lens = torch.randint(ragged[0], ragged[1] + 1, (Q,), device=DEV, generator=g)
    mask = torch.arange(1 + T, device=DEV).unsqueeze(0) > lens.unsqueeze(1)
    seq.masked_fill_(mask.t().unsqueeze(2), 0.0)
    seq[0] = 0.0
    return seq, mask, lens


def _assert_same_aggregation(engine, seq16, mask, lens):
    out16, att16 = engine.aggregate(seq16, mask, getatt=True)
    out32, att32 = engine.aggregate(seq16.float(), mask, getatt=True)
    assert torch.equal(out16, out32)
    assert torch.equal(att16, att32)
    assert torch.equal(engine.aggregate(seq16, None, lens=lens), out16)          # lens path == mask path
    single = lens == 1                                                            # the block is skipped for T == 1
    if bool(single.any()):
        assert torch.equal(out16[single], seq16[1][single].float())
    return out16


# ------------------------------------------------------------------------------------------------ 1. bit identity
@pytest.mark.parametrize("Q,T,ragged", [
    (33, 1, None), (40, 3, None), (37, 4, None), (41, 7, (0, 7)),               # one warp per track, TR = 4 / 10
    (50, 10, None), (52, 10, (0, 10)),                                           # TR = 10: tensor-map path / ragged
    (30, 16, None), (45, 12, (0, 12)),                                           # TR = 16
    (40, 32, None), (21, 27, (0, 27)), (29, 17, (1, 17)),                        # two warps per track
    (33, 64, None), (77, 50, (0, 50)), (35, 48, None),                           # four warps per track
])
def test_f16_aggregate_is_bit_identical(Q, T, ragged, engine):
    seq16, mask, lens = _tracks16(Q, T, seed=Q * 100 + T, ragged=ragged)
    _assert_same_aggregation(engine, seq16, mask, lens)


@pytest.mark.parametrize("Q,T,ragged", [(7500, 4, (0, 4)), (7200, 10, None), (7300, 9, (0, 9)), (7150, 16, None),
                                        (7250, 14, (0, 14)), (7400, 32, None), (7104, 64, None), (7200, 50, (0, 50))])
def test_f16_aggregate_many_tracks_per_warp(Q, T, ragged, engine):
    """More tracks than producers and at least three tensor-core batches per CTA: buffers are refilled (by the loader
    warp at T <= 10) and the group kernel clears stale frames of a shorter block."""
    seq16, mask, lens = _tracks16(Q, T, seed=3 * Q + T, ragged=ragged)
    _assert_same_aggregation(engine, seq16, mask, lens)


def test_f16_aggregate_t1_is_exact_and_wide_range(engine):
    """T == 1: out == x_1 exactly; values across fp16's range (including subnormals) widen exactly."""
    seq16, mask, lens = _tracks16(64, 1, seed=4)
    seq16[1, :16] *= 1000.0
    seq16[1, 16:32] = (seq16[1, 16:32].float() * 1e-6).half()                    # fp16 subnormals
    out = engine.aggregate(seq16, mask)
    assert torch.equal(out, seq16[1].float())
    seq16, mask, lens = _tracks16(300, 10, seed=5, ragged=(0, 10), scale=200.0)
    _assert_same_aggregation(engine, seq16, mask, lens)


# ------------------------------------------------------------------------------------------------ 2. strided input
def test_f16_strided_input(engine):
    seq16, mask, lens = _tracks16(50, 7, seed=21, ragged=(1, 7))
    part = seq16[:, 10:31]                                                        # read through its strides
    assert not part.is_contiguous()
    assert torch.equal(engine.aggregate(part, mask[10:31]), engine.aggregate(part.float(), mask[10:31]))
    # track stride 264 halves (a multiple of 8): read in place; 260 (not a multiple of 8): copied first
    for pitch in (264, 260):
        wide = torch.zeros(1 + 7, 50, pitch, dtype=torch.float16, device=DEV)
        wide[..., :256] = seq16
        view = wide[..., :256]
        assert torch.equal(engine.aggregate(view, mask), engine.aggregate(seq16.float(), mask))


def test_f16_entry_rejects_strides_that_are_not_16_bytes(engine):
    Q, T = 4, 3
    buf = torch.zeros(((1 + T) * Q * 260,), dtype=torch.float16, device=DEV)
    out = torch.empty((Q, 256), dtype=torch.float32, device=DEV)
    ws = torch.empty((256,), dtype=torch.uint8, device=DEV)
    stream = torch.cuda.current_stream(DEV).cuda_stream
    lib = engine._lib
    rc = lib.seam_aggregate_f16(engine._h, buf.data_ptr(), None, None, T, Q, Q * 260, 260, out.data_ptr(), None,
                                ws.data_ptr(), ws.numel(), stream)
    assert rc == 2                                                                # SEAM_ERR_UNSUPPORTED
    assert b"seam_aggregate_f16" in lib.seam_last_error(engine._h)
    rc = lib.seam_aggregate_f16(engine._h, buf.data_ptr(), None, None, T, Q, Q * 264, 260, out.data_ptr(), None,
                                ws.data_ptr(), ws.numel(), stream)
    assert rc == 2
    rc = lib.seam_aggregate_f16(engine._h, buf.data_ptr() + 8, None, None, T, Q, Q * 256, 256, out.data_ptr(), None,
                                ws.data_ptr(), ws.numel(), stream)                # 8-byte aligned only
    assert rc == 2
    rc = lib.seam_aggregate_f16(engine._h, buf.data_ptr(), None, None, T, Q, Q * 256, 256, out.data_ptr(), None,
                                ws.data_ptr(), ws.numel(), stream)
    assert rc == 0


# ------------------------------------------------------------------------------------------------ 3. no conversion pass
def test_f16_aggregate_makes_no_fp32_copy(engine):
    """At T = 10 the fp32 output (1 KB per track) is under a fifth of seq16's bytes (11 x 512 B per track); the fp32
    copy a conversion pass would make is twice them.  The peak allocation must stay under half of seq16."""
    seq16, mask, _ = _tracks16(20000, 10, seed=8)
    engine.aggregate(seq16[:, :100], mask[:100])                                  # workspace and module loading
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(DEV)
    torch.cuda.reset_peak_memory_stats(DEV)
    out = engine.aggregate(seq16, mask)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated(DEV) - base < seq16.nbytes // 2
    assert torch.equal(out, engine.aggregate(seq16.float(), mask))


# ------------------------------------------------------------------------------------------------ 4. search
def test_f16_search(engine, monkeypatch):
    seq16, mask, lens = _tracks16(700, 10, seed=31, ragged=(0, 10))
    gal = engine.prepare_gallery(torch.randn(3000, 256, device=DEV, generator=torch.Generator(device=DEV).manual_seed(3)))
    r16 = engine.search(seq16, mask, gal, 20)
    r32 = engine.search(seq16.float(), mask, gal, 20)
    assert all(torch.equal(a, b) for a, b in zip(r16, r32))
    assert all(torch.equal(a, b) for a, b in zip(engine.search(seq16, None, gal, 20, lens=lens), r16))
    # the slab path (aggregate + score_topk in query slabs) keeps the tracks fp16 too
    eng_mod = sys.modules[pkg.__name__ + ".engine"]
    monkeypatch.setattr(eng_mod, "SCORE_WS_LIMIT", 16 << 20)
    seen = []
    aggregate = engine.aggregate

    def spy(seq, *a, **kw):
        seen.append(seq.dtype)
        return aggregate(seq, *a, **kw)

    monkeypatch.setattr(engine, "aggregate", spy)
    seq16, mask, _ = _tracks16(5000, 7, seed=32, ragged=(1, 7))
    s16 = engine.search(seq16, mask, gal, 20)
    assert seen == [torch.float16]
    s32 = engine.search(seq16.float(), mask, gal, 20)
    assert all(torch.equal(a, b) for a, b in zip(s16, s32))


# ------------------------------------------------------------------------------------------------ 5. host streaming
def test_f16_upload_tracks(engine):
    T, Q, lo, hi = 6, 90, 17, 60
    seq16, _, _ = _tracks16(Q, T, seed=41)
    host = seq16.cpu().pin_memory()
    host[0] = float("nan")                                                        # the dummy row is never copied
    dev = engine.upload_tracks(host, lo, hi)
    torch.cuda.synchronize()
    assert dev.dtype == torch.float16 and dev.shape == (1 + T, hi - lo, 256)
    assert torch.equal(dev[1:].cpu(), host[1:, lo:hi])
    # row 0 of the destination is left as it was
    dst = torch.full((1 + T, hi - lo, 256), 7.0, dtype=torch.float16, device=DEV)
    rc = engine._lib.seam_upload_tracks_f16(engine._h, host.data_ptr(), T, Q, lo, hi, dst.data_ptr(),
                                           torch.cuda.current_stream(DEV).cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.equal(dst[1:].cpu(), host[1:, lo:hi]) and bool((dst[0] == 7.0).all())


def test_f16_search_host(engine):
    Q, T, G, k = 403, 7, 777, 20
    seq16, mask, _ = _tracks16(Q, T, seed=11, ragged=(1, 7))
    gal = torch.randn(G, 256, generator=torch.Generator().manual_seed(12))
    h16 = seq16.cpu().pin_memory()
    h16[0] = float("nan")
    h32 = h16.float().pin_memory()
    hm, hg = mask.cpu().pin_memory(), gal.pin_memory()
    stream = pkg.HostTrackStream(engine, nchunk=3)
    o16 = pkg.search_host(engine, h16, hm, hg, k, stream=stream)
    o32 = pkg.search_host(engine, h32, hm, hg, k, stream=stream)
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(o16, o32))
    assert stream.h2d_bytes(h16, None) * 2 == stream.h2d_bytes(h32, None)


# ------------------------------------------------------------------------------------------------ 6. sharded
def test_f16_sharded_single_rank(engine):
    Q, T, G, k = 700, 10, 3000, 20
    gal = torch.randn(G, 256, generator=torch.Generator().manual_seed(5)).to(DEV)
    peer = pkg.PeerExchange(engine, Q, k)
    retr = pkg.ShardedRetriever(engine, gal, 0)
    for step in range(2):
        seq16, mask, _ = _tracks16(Q, T, seed=50 + step, ragged=(1, 10))
        r16 = [t.clone() for t in retr.search_peer(seq16, mask, peer)]
        d16 = peer.descriptors()[(2 * step + 1) & 1].clone()
        r32 = retr.search_peer(seq16.float(), mask, peer)
        d32 = peer.descriptors()[(2 * step + 2) & 1]
        assert all(torch.equal(a, b) for a, b in zip(r16, r32))
        assert torch.equal(d16, d32)
    assert peer.steps_done == 4


@pytest.mark.parametrize("replicate", [True, False])
def test_f16_sharded_two_ranks_one_gpu(weights, engine, replicate):
    """The two-ranks-in-one-process set-up of the sharded search tests: fp16 tracks give the fp32 run's results."""
    Q, T, G, k = 301, 4, 2500, 20
    engines = [engine, pkg.SeamEngine(DEV)]
    engines[1].load_weights({kk: v.to(DEV) for kk, v in weights.items()})
    gal = torch.randn(G, 256, generator=torch.Generator().manual_seed(6)).to(DEV)
    shared = {}
    peers = [pkg.PeerExchange(engines[r], Q, k, replicate=replicate,
                              local_peers={"world": 2, "rank": r, "shared": shared}) for r in range(2)]
    for p in peers:
        p._fill_struct()
    bounds = [pkg.shard_bounds(G, 2, r) for r in range(2)]
    retrs = [pkg.ShardedRetriever(engines[r], gal[bounds[r][0]:bounds[r][1]], bounds[r][0], world=2, rank=r)
             for r in range(2)]
    streams = [torch.cuda.Stream(DEV) for _ in range(2)]

    def step(seq, mask):
        torch.cuda.synchronize()
        res = [None, None]
        for r in (0, 1):
            streams[r].wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(streams[r]):
                res[r] = retrs[r].search_peer(seq, mask, peers[r])
        torch.cuda.synchronize()
        return [[t.clone() for t in rr] for rr in res]

    for s in range(2):
        seq16, mask, _ = _tracks16(Q, T, seed=60 + s, ragged=(0, 4))
        r16 = step(seq16, mask)
        r32 = step(seq16.float(), mask)
        assert engines[0].watchdog_records() == []
        for r in range(2):
            assert all(torch.equal(a, b) for a, b in zip(r16[r], r32[r]))
    assert peers[0].steps_done == 4 and peers[1].steps_done == 4


def test_f16_sharded_aggregate_in_chunks(engine):
    Q, T, G, k = 256, 10, 1500, 10
    gal = torch.randn(G, 256, generator=torch.Generator().manual_seed(7)).to(DEV)
    g = engine.prepare_gallery(gal)
    seq16, mask, _ = _tracks16(Q, T, seed=70)
    res = []
    for seq in (seq16, seq16.float()):
        peer = pkg.PeerExchange(engine, Q, k)
        for lo, hi in ((0, 100), (100, 101), (101, 256)):
            engine.sharded_aggregate(peer, seq[:, lo:hi], mask[lo:hi], row0=lo, last=hi == Q)
        engine.sharded_score_topk(peer, g)
        res.append([t.clone() for t in engine.sharded_merge(peer)] + [peer.descriptors()[1].clone()])
    assert all(torch.equal(a, b) for a, b in zip(res[0], res[1]))
    assert torch.equal(res[0][3], engine.aggregate(seq16, mask))


# ------------------------------------------------------------------------------------------------ 7. modules
@pytest.fixture(scope="module")
def model(weights):
    m = pkg.TemporalAggregationNLB().to(DEV).eval()
    missing, unexpected = m.load_state_dict(weights, strict=False)
    assert not unexpected
    return m


def test_f16_module_seq_branch(model):
    seq16, mask, _ = _tracks16(37, 10, seed=80, ragged=(0, 10))
    gal = torch.randn(300, 256, generator=torch.Generator().manual_seed(81)).to(DEV)
    o16 = model(None, None, None, x3_1_seq=seq16, x3_1_mask=mask, x3_2=gal, getatt=True)
    o32 = model(None, None, None, x3_1_seq=seq16.float(), x3_1_mask=mask, x3_2=gal, getatt=True)
    assert torch.equal(o16[0], o32[0]) and torch.equal(o16[2], o32[2])
    assert len(o16[6]) == len(o32[6]) and all(torch.equal(a, b) for a, b in zip(o16[6], o32[6]))
    assert torch.equal(model.aggregate(seq16, mask), o32[0])
    s16, i16 = model.score_topk(seq16, mask, gal, k=20)
    s32, i32 = model.score_topk(seq16.float(), mask, gal, k=20)
    assert torch.equal(s16, s32) and torch.equal(i16, i32)


def test_f16_module_training_gradients(weights):
    """Training mode: the forward reads the fp16 tracks, the backward kernel (fp32 only) gets them widened.  Gradients
    equal those of the widened fp32 input: the track and gallery gradients bit for bit (the gradient of an fp16 leaf is
    the fp32 one rounded to fp16), the parameter gradients up to the order of their atomic fp32 accumulation."""
    m = pkg.TemporalAggregationNLB().to(DEV).train()
    m.load_state_dict(weights, strict=False)
    seq16, mask, _ = _tracks16(9, 10, seed=90, ragged=(1, 10))
    gal = torch.randn(7, 256, generator=torch.Generator().manual_seed(91)).to(DEV)
    r1 = torch.randn(9, 256, generator=torch.Generator().manual_seed(1)).to(DEV)
    r2 = torch.randn(9, 7, 2, generator=torch.Generator().manual_seed(2)).to(DEV)
    grads = []
    for seq in (seq16, seq16.float()):
        m.zero_grad(set_to_none=True)
        s = seq.detach().clone().requires_grad_(True)
        g = gal.clone().requires_grad_(True)
        x3_1b, _, x5, _, _, _ = m(None, None, None, x3_1_seq=s, x3_1_mask=mask, x3_2=g)
        ((x5 * r2).sum() + (x3_1b * r1).sum()).backward()
        grads.append((x3_1b.detach(), s.grad, g.grad, {n: p.grad.clone() for n, p in m.named_parameters()
                                                       if p.grad is not None}))
    (o16, ds16, dg16, p16), (o32, ds32, dg32, p32) = grads
    assert torch.equal(o16, o32)
    assert ds16.dtype == torch.float16 and torch.equal(ds16, ds32.half())
    assert torch.equal(dg16, dg32)
    assert p16.keys() == p32.keys() and "newnlb.theta.weight" in p16
    for n in p16:
        scale = max(float(p32[n].abs().max()), 1e-30)
        assert float((p16[n] - p32[n]).abs().max()) <= 1e-5 * scale, n
