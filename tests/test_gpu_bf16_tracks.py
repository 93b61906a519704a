"""bf16 tracks: x3_1_seq given as bf16 (the dtype of torch.autocast(dtype=torch.bfloat16)) is read as bf16 by the
aggregation kernels (the seam_*_bf16 entry points: half the bytes, no conversion pass) and gives exactly what the fp32
path gives on the widened tracks.  Widening bf16 to fp32 is exact (a 16-bit shift) and the kernels widen each frame as
it leaves shared memory, so every comparison below is bit for bit, against the fp32 path run on ``seq.float()``."""
import sys

import pytest
import torch

import seam_match_rcnn_b200 as pkg

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _tracksb(Q, T, seed, ragged=None, scale=1.0):
    """(seq (1+T,Q,256) bf16 on the device with dummy row 0, mask (Q,1+T) bool, lens (Q) int64); ragged=(lo,hi) draws
    the lengths in [lo,hi] (0: empty track).  Padding frames are zero."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    seq = (torch.randn(1 + T, Q, 256, device=DEV, generator=g) * scale).to(torch.bfloat16)
    if ragged is None:
        lens = torch.full((Q,), T, dtype=torch.int64, device=DEV)
    else:
        lens = torch.randint(ragged[0], ragged[1] + 1, (Q,), device=DEV, generator=g)
    mask = torch.arange(1 + T, device=DEV).unsqueeze(0) > lens.unsqueeze(1)
    seq.masked_fill_(mask.t().unsqueeze(2), 0.0)
    seq[0] = 0.0
    return seq, mask, lens


def _assert_same_aggregation(engine, seqb, mask, lens):
    outb, attb = engine.aggregate(seqb, mask, getatt=True)
    out32, att32 = engine.aggregate(seqb.float(), mask, getatt=True)
    assert torch.equal(outb, out32)
    assert torch.equal(attb, att32)
    assert torch.equal(engine.aggregate(seqb, None, lens=lens), outb)            # lens path == mask path
    single = lens == 1                                                            # the block is skipped for T == 1
    if bool(single.any()):
        assert torch.equal(outb[single], seqb[1][single].float())
    return outb


# ------------------------------------------------------------------------------------------------ 1. bit identity
@pytest.mark.parametrize("Q,T,ragged", [
    (33, 1, None), (40, 3, None), (37, 4, None), (41, 7, (0, 7)),               # one warp per track, TR = 4 / 10
    (50, 10, None), (52, 10, (0, 10)),                                           # TR = 10: tensor-map path / ragged
    (30, 16, None), (45, 12, (0, 12)),                                           # TR = 16
    (40, 32, None), (21, 27, (0, 27)), (29, 17, (1, 17)),                        # two warps per track
    (33, 64, None), (77, 50, (0, 50)), (35, 48, None),                           # four warps per track
])
def test_bf16_aggregate_is_bit_identical(Q, T, ragged, engine):
    seqb, mask, lens = _tracksb(Q, T, seed=Q * 100 + T + 7, ragged=ragged)
    _assert_same_aggregation(engine, seqb, mask, lens)


@pytest.mark.parametrize("Q,T,ragged", [(7500, 4, (0, 4)), (7200, 10, None), (7300, 9, (0, 9)), (7150, 16, None),
                                        (7250, 14, (0, 14)), (7400, 32, None), (7104, 64, None), (7200, 50, (0, 50))])
def test_bf16_aggregate_many_tracks_per_warp(Q, T, ragged, engine):
    """More tracks than producers and at least three tensor-core batches per CTA: buffers are refilled (by the loader
    warp at T <= 10) and the group kernel clears stale frames of a shorter block."""
    seqb, mask, lens = _tracksb(Q, T, seed=5 * Q + T, ragged=ragged)
    _assert_same_aggregation(engine, seqb, mask, lens)


def test_bf16_aggregate_t1_is_exact_beyond_fp16_range(engine):
    """T == 1: out == x_1 exactly, for values fp16 cannot hold: magnitudes around 1e30 and bf16 subnormals."""
    seqb, mask, _ = _tracksb(64, 1, seed=4)
    seqb[1, :16] = (seqb[1, :16].float() * 1e30).to(torch.bfloat16)
    # bf16 subnormals (zero exponent, non-zero mantissa), built from their bit patterns: below fp32's normal range
    g = torch.Generator(device=DEV).manual_seed(44)
    bits = torch.randint(1, 128, (16, 256), dtype=torch.int32, device=DEV, generator=g) << 16
    sub = bits.view(torch.float32)
    sign = torch.randint(0, 2, (16, 256), device=DEV, generator=g).bool()
    seqb[1, 16:32] = torch.where(sign, -sub, sub).to(torch.bfloat16)             # exact: the low 16 bits are zero
    wide = seqb[1].float()
    assert bool(wide[:16].abs().max() > 1e30) and bool(wide[16:32].abs().max() < 1.1754944e-38)
    assert bool((wide[16:32] != 0).any())
    out = engine.aggregate(seqb, mask)
    assert torch.equal(out, wide)
    assert torch.equal(engine.aggregate(seqb.float(), mask), wide)


def test_bf16_aggregate_wide_range_ragged(engine):
    seqb, mask, lens = _tracksb(300, 10, seed=5, ragged=(0, 10), scale=200.0)
    out = _assert_same_aggregation(engine, seqb, mask, lens)
    assert bool(torch.isfinite(out).all())                                        # equal, and not by NaN luck


# ------------------------------------------------------------------------------------------------ 2. input layout
def test_bf16_strided_input(engine):
    seqb, mask, lens = _tracksb(50, 7, seed=21, ragged=(1, 7))
    part = seqb[:, 10:31]                                                         # read through its strides
    assert not part.is_contiguous()
    assert torch.equal(engine.aggregate(part, mask[10:31]), engine.aggregate(part.float(), mask[10:31]))
    # track stride 264 elements (a multiple of 8): read in place; 260 (not a multiple of 8): copied first
    for pitch in (264, 260):
        wide = torch.zeros(1 + 7, 50, pitch, dtype=torch.bfloat16, device=DEV)
        wide[..., :256] = seqb
        view = wide[..., :256]
        assert torch.equal(engine.aggregate(view, mask), engine.aggregate(seqb.float(), mask))


def test_bf16_entry_rejects_misaligned_input(engine):
    Q, T = 4, 3
    buf = torch.zeros(((1 + T) * Q * 264,), dtype=torch.bfloat16, device=DEV)
    out = torch.empty((Q, 256), dtype=torch.float32, device=DEV)
    ws = torch.empty((256,), dtype=torch.uint8, device=DEV)
    stream = torch.cuda.current_stream(DEV).cuda_stream
    lib = engine._lib

    def call(ptr, frame_stride, track_stride):
        return lib.seam_aggregate_bf16(engine._h, ptr, None, None, T, Q, frame_stride, track_stride, out.data_ptr(),
                                       None, ws.data_ptr(), ws.numel(), stream)

    for args in ((buf.data_ptr(), Q * 260, 260),                                  # track stride not a multiple of 8
                 (buf.data_ptr(), Q * 256 + 4, 256),                              # frame stride not a multiple of 8
                 (buf.data_ptr() + 8, Q * 256, 256)):                             # 8-byte aligned only
        assert call(*args) == 2                                                   # SEAM_ERR_UNSUPPORTED
        msg = lib.seam_last_error(engine._h)
        assert b"seam_aggregate_bf16" in msg and b"bf16" in msg.split(b":", 1)[1]
    assert call(buf.data_ptr(), Q * 264, 264) == 0
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ 3. no conversion pass
def test_bf16_aggregate_makes_no_fp32_copy(engine):
    """At T = 10 the fp32 output (1 KB per track) is under a fifth of seqb's bytes (11 x 512 B per track); the fp32
    copy a conversion pass would make is twice them.  The peak allocation must stay under half of seqb."""
    seqb, mask, _ = _tracksb(20000, 10, seed=8)
    engine.aggregate(seqb[:, :100], mask[:100])                                   # workspace and module loading
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(DEV)
    torch.cuda.reset_peak_memory_stats(DEV)
    out = engine.aggregate(seqb, mask)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated(DEV) - base < seqb.nbytes // 2
    assert torch.equal(out, engine.aggregate(seqb.float(), mask))


# ------------------------------------------------------------------------------------------------ 4. search
@pytest.mark.parametrize("gallery_dtype", [torch.float32, torch.float16])
def test_bf16_search(engine, gallery_dtype):
    """seam_search_bf16 (fp32 gallery) and seam_search_bf16_g16 (fp16 gallery) give the fp32 tracks' results."""
    seqb, mask, lens = _tracksb(700, 10, seed=31, ragged=(0, 10))
    rows = torch.randn(3000, 256, device=DEV, generator=torch.Generator(device=DEV).manual_seed(3)).to(gallery_dtype)
    gal = engine.prepare_gallery(rows)
    assert gal.rows_f16 == (gallery_dtype == torch.float16)
    name = engine._track_entry("search", seqb, gal.rows_f16).__name__
    assert name == ("seam_search_bf16_g16" if gal.rows_f16 else "seam_search_bf16")
    rb = engine.search(seqb, mask, gal, 20, return_stats=True)
    r32 = engine.search(seqb.float(), mask, gal, 20, return_stats=True)
    assert all(torch.equal(a, b) for a, b in zip(rb, r32))                        # the counters too
    assert all(torch.equal(a, b) for a, b in zip(engine.search(seqb, None, gal, 20, lens=lens), rb[:4]))


def test_bf16_search_slab_path(engine, monkeypatch):
    """The slab path (aggregate + score_topk in query slabs) keeps the tracks bf16 too."""
    gal = engine.prepare_gallery(torch.randn(3000, 256, device=DEV, generator=torch.Generator(device=DEV).manual_seed(3)))
    eng_mod = sys.modules[pkg.__name__ + ".engine"]
    monkeypatch.setattr(eng_mod, "SCORE_WS_LIMIT", 16 << 20)
    seen = []
    aggregate = engine.aggregate

    def spy(seq, *a, **kw):
        seen.append(seq.dtype)
        return aggregate(seq, *a, **kw)

    monkeypatch.setattr(engine, "aggregate", spy)
    seqb, mask, _ = _tracksb(5000, 7, seed=32, ragged=(1, 7))
    sb = engine.search(seqb, mask, gal, 20, return_stats=True)
    assert seen == [torch.bfloat16]
    s32 = engine.search(seqb.float(), mask, gal, 20, return_stats=True)
    assert all(torch.equal(a, b) for a, b in zip(sb, s32))


# ------------------------------------------------------------------------------------------------ 5. host streaming
def test_bf16_upload_tracks(engine):
    T, Q, lo, hi = 6, 90, 17, 60
    seqb, _, _ = _tracksb(Q, T, seed=41)
    host = seqb.cpu().pin_memory()
    host[0] = float("nan")                                                        # the dummy row is never copied
    dev = engine.upload_tracks(host, lo, hi)
    torch.cuda.synchronize()
    assert dev.dtype == torch.bfloat16 and dev.shape == (1 + T, hi - lo, 256)
    assert torch.equal(dev[1:], seqb[1:, lo:hi])
    # row 0 of the destination is left as it was (the _f16 entry copies any 2-byte element type)
    dst = torch.full((1 + T, hi - lo, 256), 7.0, dtype=torch.bfloat16, device=DEV)
    rc = engine._lib.seam_upload_tracks_f16(engine._h, host.data_ptr(), T, Q, lo, hi, dst.data_ptr(),
                                            torch.cuda.current_stream(DEV).cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.equal(dst[1:], seqb[1:, lo:hi]) and bool((dst[0] == 7.0).all())


def test_bf16_search_host(engine):
    Q, T, G, k = 403, 7, 777, 20
    seqb, mask, _ = _tracksb(Q, T, seed=11, ragged=(1, 7))
    gal = torch.randn(G, 256, generator=torch.Generator().manual_seed(12))
    hb = seqb.cpu().pin_memory()
    hb[0] = float("nan")
    h32 = hb.float().pin_memory()
    hm, hg = mask.cpu().pin_memory(), gal.pin_memory()
    stream = pkg.HostTrackStream(engine, nchunk=3)
    ob = pkg.search_host(engine, hb, hm, hg, k, stream=stream)
    o32 = pkg.search_host(engine, h32, hm, hg, k, stream=stream)
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(ob, o32))
    assert stream.h2d_bytes(hb, None) * 2 == stream.h2d_bytes(h32, None)


# ------------------------------------------------------------------------------------------------ 6. sharded
def test_bf16_sharded_single_rank(engine):
    Q, T, G, k = 700, 10, 3000, 20
    gal = torch.randn(G, 256, generator=torch.Generator().manual_seed(5)).to(DEV)
    peer = pkg.PeerExchange(engine, Q, k)
    retr = pkg.ShardedRetriever(engine, gal, 0)
    whole = engine.prepare_gallery(gal)
    for step in range(2):
        seqb, mask, _ = _tracksb(Q, T, seed=50 + step, ragged=(1, 10))
        rb = [t.clone() for t in retr.search_peer(seqb, mask, peer)]
        db = peer.descriptors()[(2 * step + 1) & 1].clone()
        r32 = retr.search_peer(seqb.float(), mask, peer)
        d32 = peer.descriptors()[(2 * step + 2) & 1]
        assert all(torch.equal(a, b) for a, b in zip(rb, r32))
        assert torch.equal(db, d32)
        q, sc, mg, ix = engine.search(seqb, mask, whole, k)                      # the unsharded search on the whole gallery
        assert torch.equal(db, q)
        assert all(torch.equal(a, b) for a, b in zip(rb, (sc, mg, ix)))
    assert peer.steps_done == 4


@pytest.mark.parametrize("replicate", [True, False])
def test_bf16_sharded_two_ranks_one_gpu(weights, engine, replicate):
    """The two-ranks-in-one-process set-up of the sharded search tests: bf16 tracks give the fp32 run's results, and
    those of engine.search on the whole gallery."""
    Q, T, G, k = 301, 4, 2500, 20
    engines = [engine, pkg.SeamEngine(DEV)]
    engines[1].load_weights({kk: v.to(DEV) for kk, v in weights.items()})
    gal = torch.randn(G, 256, generator=torch.Generator().manual_seed(6)).to(DEV)
    whole = engine.prepare_gallery(gal)
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
        seqb, mask, _ = _tracksb(Q, T, seed=60 + s, ragged=(0, 4))
        rb = step(seqb, mask)
        r32 = step(seqb.float(), mask)
        assert engines[0].watchdog_records() == []
        ref = engine.search(seqb, mask, whole, k)[1:]
        for r in range(2):
            assert all(torch.equal(a, b) for a, b in zip(rb[r], r32[r]))
            lo, hi = (0, Q) if replicate else (peers[r].q_lo[r], peers[r].q_lo[r + 1])
            assert all(torch.equal(a, b[lo:hi]) for a, b in zip(rb[r], ref))
    assert peers[0].steps_done == 4 and peers[1].steps_done == 4


def test_bf16_sharded_aggregate_in_chunks(engine):
    Q, T, G, k = 256, 10, 1500, 10
    gal = torch.randn(G, 256, generator=torch.Generator().manual_seed(7)).to(DEV)
    g = engine.prepare_gallery(gal)
    seqb, mask, _ = _tracksb(Q, T, seed=70)
    res = []
    for seq in (seqb, seqb.float()):
        peer = pkg.PeerExchange(engine, Q, k)
        for lo, hi in ((0, 100), (100, 101), (101, 256)):
            engine.sharded_aggregate(peer, seq[:, lo:hi], mask[lo:hi], row0=lo, last=hi == Q)
        engine.sharded_score_topk(peer, g)
        res.append([t.clone() for t in engine.sharded_merge(peer)] + [peer.descriptors()[1].clone()])
    assert all(torch.equal(a, b) for a, b in zip(res[0], res[1]))
    assert torch.equal(res[0][3], engine.aggregate(seqb, mask))


# ------------------------------------------------------------------------------------------------ 7. modules
@pytest.fixture(scope="module")
def model(weights):
    m = pkg.TemporalAggregationNLB().to(DEV).eval()
    missing, unexpected = m.load_state_dict(weights, strict=False)
    assert not unexpected
    return m


def test_bf16_module_seq_branch(model):
    seqb, mask, _ = _tracksb(37, 10, seed=80, ragged=(0, 10))
    gal = torch.randn(300, 256, generator=torch.Generator().manual_seed(81)).to(DEV)
    ob = model(None, None, None, x3_1_seq=seqb, x3_1_mask=mask, x3_2=gal, getatt=True)
    o32 = model(None, None, None, x3_1_seq=seqb.float(), x3_1_mask=mask, x3_2=gal, getatt=True)
    assert torch.equal(ob[0], o32[0]) and torch.equal(ob[2], o32[2])
    assert len(ob[6]) == len(o32[6]) and all(torch.equal(a, b) for a, b in zip(ob[6], o32[6]))
    assert torch.equal(model.aggregate(seqb, mask), o32[0])
    sb, ib = model.score_topk(seqb, mask, gal, k=20)
    s32, i32 = model.score_topk(seqb.float(), mask, gal, k=20)
    assert torch.equal(sb, s32) and torch.equal(ib, i32)


def test_bf16_module_training_gradients(weights):
    """Training mode: the forward reads the bf16 tracks, the backward kernel (fp32 only) gets them widened.  Gradients
    equal those of the widened fp32 input: the track and gallery gradients bit for bit (dseq is written without
    atomics, and the gradient of a bf16 leaf is the fp32 one rounded to bf16), the parameter gradients up to the order
    of their atomic fp32 accumulation."""
    m = pkg.TemporalAggregationNLB().to(DEV).train()
    m.load_state_dict(weights, strict=False)
    seqb, mask, _ = _tracksb(9, 10, seed=90, ragged=(1, 10))
    gal = torch.randn(7, 256, generator=torch.Generator().manual_seed(91)).to(DEV)
    r1 = torch.randn(9, 256, generator=torch.Generator().manual_seed(1)).to(DEV)
    r2 = torch.randn(9, 7, 2, generator=torch.Generator().manual_seed(2)).to(DEV)
    grads = []
    for seq in (seqb, seqb.float()):
        m.zero_grad(set_to_none=True)
        s = seq.detach().clone().requires_grad_(True)
        g = gal.clone().requires_grad_(True)
        x3_1b, _, x5, _, _, _ = m(None, None, None, x3_1_seq=s, x3_1_mask=mask, x3_2=g)
        ((x5 * r2).sum() + (x3_1b * r1).sum()).backward()
        grads.append((x3_1b.detach(), s.grad, g.grad, {n: p.grad.clone() for n, p in m.named_parameters()
                                                       if p.grad is not None}))
    (ob, dsb, dgb, pb), (o32, ds32, dg32, p32) = grads
    assert torch.equal(ob, o32)
    assert dsb.dtype == torch.bfloat16 and torch.equal(dsb, ds32.to(torch.bfloat16))
    assert torch.equal(dgb, dg32)
    assert pb.keys() == p32.keys() and "newnlb.theta.weight" in pb
    for n in pb:
        scale = max(float(p32[n].abs().max()), 1e-30)
        assert float((pb[n] - p32[n]).abs().max()) <= 1e-5 * scale, n
