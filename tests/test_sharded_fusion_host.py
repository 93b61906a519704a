"""ShardedRetriever.evaluate_distance_fusions / evaluate_products over gloo with a CPU stand-in for the engine: every
shard groups all frames, the shard holding each target computes its fused values (or margin), a MAX all-reduce, per-shard
counts with ties broken by global row, a SUM all-reduce -- equal to the unsharded report integer for integer, including
exact duplicates of a target row in lower and higher shards, products without frames, shards without rows and P = 0."""
import contextlib
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import seam_match_rcnn_b200 as pkg
from oracle import seam_oracle as so
from test_host_logic import OracleOps
from test_sharded_rank_host import OracleRankOps, _free_port


def frame_probs(frames, g, w):
    """class-1 probabilities (N, G); every logit is its own 256-long reduction, so a (frame, row) pair gets the same
    bits whichever batch it is computed in (exact ties between duplicate rows are what these tests are about)"""
    x4 = (frames[:, None, :] - g[None, :, :]) ** 2                       # (N, G, 256)
    x5 = (x4[:, :, None, :] * w["last.weight"][None, None]).sum(-1) + w["last.bias"]
    return so.match_scores(x5)


def fused_values(prob):
    """(avg, max) over the frames (rows of prob) for every column, each column reduced on its own"""
    pt = prob.t().contiguous()
    return pt.sum(1) / prob.shape[0], pt.max(1).values


class OracleReportOps(OracleRankOps, OracleOps):
    """CPU stand-in for SeamEngine's report entry points (TESTS ONLY).  A gallery shard is ``(rows, index_offset)``."""

    device = torch.device("cpu")

    @contextlib.contextmanager
    def scorer(self, last_w, last_b):
        prev = self.w
        self.w = dict(prev)
        self.w["last.weight"], self.w["last.bias"] = last_w, last_b
        try:
            yield self
        finally:
            self.w = prev

    def _fused(self, frames, start, g):
        """(avg, max, has) per product against every row of g: (P, G), (P, G), (P,)"""
        P = start.shape[0] - 1
        prob = frame_probs(frames, g, self.w)
        avg = torch.zeros(P, g.shape[0])
        mx = torch.zeros(P, g.shape[0])
        for p in range(P):
            lo, hi = int(start[p]), int(start[p + 1])
            if hi > lo:
                avg[p], mx[p] = fused_values(prob[lo:hi])
        return avg, mx, (start[1:] - start[:-1]) > 0

    def _counts(self, frames, start, g, off, target, tv):
        avg, mx, has = self._fused(frames, start, g)
        j = off + torch.arange(g.shape[0]).view(1, -1)
        t = target.long().view(-1, 1)
        out = []
        for v, vt in zip((avg, mx), tv):
            c = ((v > vt.view(-1, 1)) | ((v == vt.view(-1, 1)) & (j < t))).sum(1).int()
            out.append(torch.where(has, c, torch.full_like(c, g.shape[0])))
        return tuple(out)

    def rank_fused_distances(self, frames, start, g, target):
        avg, mx, _ = self._fused(frames, start, g)
        t = target.long()
        tv = [v.gather(1, t.view(-1, 1)).view(-1) for v in (avg, mx)]
        return self._counts(frames, start, g, 0, target, tv)

    def fused_target(self, frames, start, g, index_offset, target):
        assert g.shape[0] > 0, "the library takes no empty shard"
        avg, mx, has = self._fused(frames, start, g)
        t = target.long() - index_offset
        mine = has & (t >= 0) & (t < g.shape[0])
        out = []
        for v in (avg, mx):
            o = torch.full((target.shape[0],), -float("inf"))
            o[mine] = v[mine, t[mine]]
            out.append(o)
        return tuple(out)

    def fused_rank_count(self, frames, start, g, index_offset, target, target_avg, target_max):
        assert g.shape[0] > 0, "the library takes no empty shard"
        return self._counts(frames, start, g, index_offset, target, (target_avg, target_max))


def _case(P, G, dups, seed=11):
    """Products, frames, shop galleries, targets and tracks; ``dups`` = [(product, row)]: shop row ``row`` (of both
    galleries) is made an exact duplicate of that product's target row, so the two tie and only the global row
    decides.  Product 1 has no frames."""
    rs = np.random.RandomState(seed)
    w = so.random_weights(0)
    lens = rs.randint(1, 5, size=P)
    if P > 1:
        lens[1] = 0
    lens[::4] += 17 * (P > 2)                         # some products with more than one chunk of 16 frames
    frame_product = torch.tensor([p for p in range(P) for _ in range(int(lens[p]))], dtype=torch.int64)
    frame_product = frame_product[torch.from_numpy(rs.permutation(len(frame_product)))]
    frame_desc = torch.from_numpy(rs.randn(len(frame_product), 256).astype(np.float32))
    shop_desc = torch.from_numpy(rs.randn(G, 256).astype(np.float32))
    target = torch.from_numpy(rs.randint(0, G, size=P).astype(np.int64))
    for p, row in dups:
        assert int(target[p]) not in [r for _, r in dups] and int(target[p]) != row
    seq, mask, _ = so.synth_tracks(P, 4, seed=seed, ragged=(1, 4))
    qref = so.aggregate_tracks(seq, mask, w)[0] if P else torch.zeros(0, 256)
    shop_aggr = torch.from_numpy(rs.randn(G, 256).astype(np.float32))
    if P:
        shop_aggr[target] = qref + 0.5 * torch.from_numpy(rs.randn(P, 256).astype(np.float32))
        shop_desc[target[frame_product[::3]]] = frame_desc[::3] + 0.5 * torch.from_numpy(
            rs.randn(len(frame_desc[::3]), 256).astype(np.float32))
    for p, row in dups:
        shop_desc[row] = shop_desc[int(target[p])]
        shop_aggr[row] = shop_aggr[int(target[p])]
    fw = torch.from_numpy(rs.uniform(-1 / 16, 1 / 16, (2, 256)).astype(np.float32))
    fb = torch.from_numpy(rs.uniform(-1 / 16, 1 / 16, (2,)).astype(np.float32))
    return dict(w=w, frame_desc=frame_desc, frame_product=frame_product, shop_desc=shop_desc, target=target,
                frame_last=(fw, fb), seq=seq, mask=mask, shop_aggr=shop_aggr, aggr_last=(w["last.weight"], w["last.bias"]))


def _unsharded(c):
    ops = OracleReportOps(c["w"])
    fus = pkg.evaluate_distance_fusions(ops, c["frame_desc"], c["frame_product"], c["shop_desc"], c["target"],
                                        c["frame_last"])
    rep = pkg.evaluate_products(ops, c["frame_desc"], c["frame_product"], c["shop_desc"], c["target"],
                                c["frame_last"], c["seq"], c["mask"], c["shop_aggr"], c["aggr_last"])
    return fus, rep


def _worker(rank, world, port, P, G, dups, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.set_num_threads(1)
        c = _case(P, G, dups)
        ops = OracleReportOps(c["w"])
        r = pkg.ShardedRetriever.from_full_gallery(ops, c["shop_aggr"])
        lo, hi = pkg.shard_bounds(G, world, rank)
        fus = r.evaluate_distance_fusions(c["frame_desc"], c["frame_product"], c["shop_desc"][lo:hi], c["target"],
                                          c["frame_last"])
        rep = r.evaluate_products(c["frame_desc"], c["frame_product"], c["shop_desc"][lo:hi], c["target"],
                                  c["frame_last"], c["seq"], c["mask"], c["aggr_last"])
        with pytest.raises(ValueError):                   # not this rank's rows
            r.evaluate_distance_fusions(c["frame_desc"], c["frame_product"], torch.zeros(hi - lo + 1, 256),
                                        c["target"], c["frame_last"])
        assert ops.w is not None and ops.w["last.weight"] is c["w"]["last.weight"]    # the scorer is put back
        torch.save((fus, rep), os.path.join(out_dir, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


def _same_report(a, b):
    assert torch.equal(a.frame_ranks.long(), b.frame_ranks.long())
    assert torch.equal(a.product_ranks.long(), b.product_ranks.long())
    assert torch.equal(a.perf, b.perf) and a.ret == b.ret
    assert (a.rank_median, a.rank_q1, a.rank_q3) == (b.rank_median, b.rank_q1, b.rank_q3)


# (world, P, G, duplicates): duplicates sit in lower and in higher shards than their target; G < world leaves a shard
# without rows; P = 0 is a no-op
CASES = [
    (2, 9, 61, [(0, 3), (2, 58), (3, 30)]),
    (3, 7, 40, [(0, 0), (2, 39), (3, 14)]),
    (3, 5, 2, []),
    (2, 0, 11, []),
    (3, 0, 2, []),
]


@pytest.mark.parametrize("world,P,G,dups", CASES)
def test_sharded_report_gloo(tmp_path, world, P, G, dups):
    port = _free_port()
    mp.spawn(_worker, args=(world, port, P, G, dups, str(tmp_path)), nprocs=world, join=True)
    c = _case(P, G, dups)
    (ranks, hits), rep = _unsharded(c)
    assert ranks.shape == (2, P) and ranks.dtype == torch.int64
    if P > 1:
        assert ranks[:, 1].tolist() == [G, G]              # the product without frames
    # the unsharded stand-in agrees with the eval script's loop on the frame rows
    wf = dict(c["w"])
    wf["last.weight"], wf["last.bias"] = c["frame_last"]
    for p, row in dups:                                    # the duplicates do tie with the target
        fp = c["frame_product"] == p
        if fp.any():
            pr = frame_probs(c["frame_desc"][fp], c["shop_desc"][[int(c["target"][p]), row]], wf)
            assert torch.equal(pr[:, 0], pr[:, 1])
    if not dups:
        ref = so.eval_product_loop(c["frame_desc"], c["frame_product"], c["shop_desc"], c["target"], wf,
                                   so.aggregate_tracks(c["seq"], c["mask"], c["w"])[0] if P else torch.zeros(0, 256),
                                   c["shop_aggr"], c["w"])
        assert torch.equal(ranks, torch.stack([ref["avg_dist"], ref["max_dist"]]))
        assert torch.equal(rep.frame_ranks.long(), ref["frame_ranks"])
        big = torch.iinfo(torch.int32).max
        want = torch.stack([ref["best"], ref["avg_desc"], ref["aggr"]])
        has = torch.bincount(c["frame_product"], minlength=P)[:P] > 0
        want[:2, ~has] = big
        assert torch.equal(rep.product_ranks.long(), want)
    for rank in range(world):
        (s_ranks, s_hits), s_rep = torch.load(os.path.join(str(tmp_path), f"r{rank}.pt"), weights_only=False)
        assert torch.equal(s_ranks, ranks) and torch.equal(s_hits, hits)
        _same_report(s_rep, rep)


def test_world1_is_the_unsharded_report():
    c = _case(6, 30, [(0, 29)])
    ops = OracleReportOps(c["w"])
    r = pkg.ShardedRetriever(ops, c["shop_aggr"], 0, world=1, rank=0)
    (ranks, hits), rep = _unsharded(c)
    s_ranks, s_hits = r.evaluate_distance_fusions(c["frame_desc"], c["frame_product"], c["shop_desc"], c["target"],
                                                  c["frame_last"])
    assert torch.equal(s_ranks, ranks) and torch.equal(s_hits, hits)
    _same_report(r.evaluate_products(c["frame_desc"], c["frame_product"], c["shop_desc"], c["target"], c["frame_last"],
                                     c["seq"], c["mask"], c["aggr_last"]), rep)


def test_product_means_are_the_frame_means():
    """fixed-order sums: the k-th frame of every product is added in step k; products without frames get zeros"""
    c = _case(9, 20, [])
    P = 9
    avg, has = pkg.product_means(c["frame_desc"], c["frame_product"], P)
    for p in range(P):
        rows = c["frame_desc"][c["frame_product"] == p]
        assert bool(has[p]) == (rows.shape[0] > 0)
        want = rows.sum(0) / max(1, rows.shape[0]) if rows.shape[0] else torch.zeros(256)
        assert torch.allclose(avg[p], want, atol=1e-6)
    again, _ = pkg.product_means(c["frame_desc"], c["frame_product"], P)
    assert torch.equal(avg, again)
