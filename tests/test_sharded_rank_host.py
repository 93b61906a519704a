"""ShardedRetriever.rank_of_target over gloo with a CPU stand-in for the engine: the target's margin from the shard
that holds it, a MAX all-reduce, per-shard counts with ties broken by global row, a SUM all-reduce -- equal to the
rank over the whole gallery, including exact duplicates of the target in other shards and shards without rows."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import seam_match_rcnn_b200 as pkg
from oracle import seam_oracle as so


def pair_logits_rowwise(q, g, w):
    """so.pair_logits one gallery row at a time: CPU BLAS rounds a row's logits differently depending on where the row
    sits in the batch, and exact ties between duplicate rows are what these tests are about."""
    if g.shape[0] == 0:
        return torch.zeros(q.shape[0], 0, 2)
    return torch.cat([so.pair_logits(q, g[j:j + 1], w) for j in range(g.shape[0])], 1)


class OracleRankOps:
    """CPU stand-in for SeamEngine's rank entry points (TESTS ONLY).  A gallery shard is ``(rows, index_offset)``."""

    def __init__(self, w):
        self.w = w

    def prepare_gallery(self, g, index_offset=0):
        return (g, index_offset)

    def _margins(self, q, g):
        return so.logit_margin(pair_logits_rowwise(q, g, self.w))

    def rank_of_target(self, q, gal, target):
        g, _ = gal
        x5 = pair_logits_rowwise(q, g, self.w)
        t = target.long()
        return so.rank_of_target(x5, t).int(), so.logit_margin(x5).gather(1, t.view(-1, 1)).view(-1)

    def target_margin(self, q, gal, target):
        g, off = gal
        assert g.shape[0] > 0, "the library takes no empty shard"
        d = self._margins(q, g)
        t = target.long() - off
        mine = (t >= 0) & (t < g.shape[0])
        out = torch.full((q.shape[0],), -float("inf"))
        out[mine] = d[mine, t[mine]]
        return out

    def rank_count(self, q, gal, target, target_margin):
        g, off = gal
        assert g.shape[0] > 0, "the library takes no empty shard"
        d = self._margins(q, g)
        m = target_margin.view(-1, 1)
        j = off + torch.arange(g.shape[0]).view(1, -1)
        before = (d > m) | ((d == m) & (j < target.long().view(-1, 1)))
        return before.sum(1).int()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _case(Q, G, dups):
    """Queries, gallery and targets; ``dups`` = [(target query, copy row)]: gallery row ``copy row`` is made an exact
    duplicate of that query's target row, so the two tie and only the global row decides."""
    w = so.random_weights(0)
    q = torch.from_numpy(np.random.RandomState(7).randn(Q, 256).astype(np.float32))
    g = so.synth_gallery(G, 7, planted=q)
    gen = torch.Generator().manual_seed(3)
    target = torch.randint(0, G, (Q,), generator=gen, dtype=torch.int32)
    if Q:
        target[0] = 0                       # a planted match: near the top
        target[-1] = G - 1
    for qi, row in dups:
        assert int(target[qi]) not in [r for _, r in dups] and int(target[qi]) != row
        g[row] = g[int(target[qi])]
    return w, q, g, target


def _worker(rank, world, port, Q, G, dups, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.set_num_threads(1)
        w, q, g, target = _case(Q, G, dups)
        r = pkg.ShardedRetriever.from_full_gallery(OracleRankOps(w), g)
        lo, hi = pkg.shard_bounds(G, world, rank)
        assert r.shard_rows == hi - lo and r.shard_offset == lo
        rank_, margin = r.rank_of_target(q, target)
        assert r.gallery_rows(q.device) == G
        if Q:
            with pytest.raises(ValueError):
                r.rank_of_target(q[:1], torch.tensor([G], dtype=torch.int32))
        torch.save((rank_, margin), os.path.join(out_dir, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


# (world, Q, G, duplicates): the duplicates sit in lower and in higher shards than their target; G < world leaves a
# shard without rows; Q = 0 is a no-op
CASES = [
    (2, 9, 101, [(1, 3), (2, 97), (3, 50)]),
    (3, 7, 40, [(1, 0), (1, 39), (2, 14)]),
    (3, 5, 2, []),
    (3, 4, 3, [(2, 0)]),
    (2, 0, 11, []),
    (3, 0, 2, []),
]


@pytest.mark.parametrize("world,Q,G,dups", CASES)
def test_sharded_rank_of_target_gloo(tmp_path, world, Q, G, dups):
    port = _free_port()
    mp.spawn(_worker, args=(world, port, Q, G, dups, str(tmp_path)), nprocs=world, join=True)
    w, q, g, target = _case(Q, G, dups)
    x5 = pair_logits_rowwise(q, g, w)
    ref_rank = so.rank_of_target(x5, target.long())
    ref_margin = so.logit_margin(x5).gather(1, target.long().view(-1, 1)).view(-1)
    for qi, row in dups:                    # the duplicates do tie with the target
        assert so.logit_margin(x5)[qi, row] == ref_margin[qi]
    for rank in range(world):
        rank_, margin = torch.load(os.path.join(str(tmp_path), f"r{rank}.pt"))
        assert rank_.dtype == torch.int32 and rank_.shape == (Q,)
        assert torch.equal(rank_.long(), ref_rank)
        assert torch.equal(margin, ref_margin)


def test_world1_is_the_unsharded_rank():
    w, q, g, target = _case(6, 30, [(2, 29)])
    r = pkg.ShardedRetriever(OracleRankOps(w), g, 0, world=1, rank=0)
    rank_, margin = r.rank_of_target(q, target)
    assert torch.equal(rank_.long(), so.rank_of_target(pair_logits_rowwise(q, g, w), target.long()))
    with pytest.raises(ValueError):
        r.rank_of_target(q[:1], torch.tensor([-1], dtype=torch.int32))
