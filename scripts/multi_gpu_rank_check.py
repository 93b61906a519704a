"""N-GPU ShardedRetriever.evaluate_aggregated (sharded aggregation, search and rank of the target over NCCL) against
rank 0's single-GPU evaluate_aggregated on the whole gallery: ranks, margins, hits and top-k must be identical.
   torchrun --nproc-per-node N scripts/multi_gpu_rank_check.py"""
import os
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import seam_match_rcnn_b200 as pkg                     # noqa: E402
from bench import random_init_weights                   # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
eng = pkg.SeamEngine(dev)
eng.load_weights(random_init_weights(dev))
Q, T, G = 10000, 10, 1000000 + 13                       # G not divisible by the world size
g = torch.Generator(device="cpu").manual_seed(7)
seq = torch.zeros(1 + T, Q, 256)
seq[1:] = torch.randn(T, Q, 256, generator=g)
gal = torch.randn(G, 256, generator=g)
target = torch.randint(0, G, (Q,), generator=g)
seq, gal, target = seq.to(dev), gal.to(dev), target.to(dev)
q = eng.aggregate(seq, None)
gal[: Q // 2] = q[: Q // 2] + 0.1 * torch.randn(Q // 2, 256, device=dev)    # planted true matches: ranks near the top
target[: Q // 2] = torch.arange(Q // 2, device=dev)

r = pkg.ShardedRetriever.from_full_gallery(eng, gal)
rep = r.evaluate_aggregated(seq, None, target)
ranks, margin = r.rank_of_target(q, target)
torch.cuda.synchronize()
steps = []
for _ in range(5):
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r.rank_of_target(q, target)
    torch.cuda.synchronize()
    steps.append(time.perf_counter() - t0)
t_rank = sorted(steps)[len(steps) // 2]
dist.barrier()
t0 = time.perf_counter()
r.evaluate_aggregated(seq, None, target)
torch.cuda.synchronize()
t_eval = time.perf_counter() - t0
ok = True
if rank == 0:
    ref = pkg.evaluate_aggregated(eng, seq, None, gal, target)
    r1, m1 = eng.rank_of_target(q, eng.prepare_gallery(gal), target)
    same = {"ranks": torch.equal(rep.ranks, ref.ranks) and torch.equal(ranks, r1),
            "margins": torch.equal(margin.view(torch.int32), m1.view(torch.int32)),
            "hits": rep.hits == ref.hits,
            "topk": torch.equal(rep.topk_idx, ref.topk_idx)
            and torch.equal(rep.topk_scores.view(torch.int32), ref.topk_scores.view(torch.int32))}
    ok = all(same.values())
    print(f"world={world} Q={Q} G={G} ({torch.cuda.get_device_name(dev)}): sharded vs single-GPU identical: {same}; "
          f"hits@{list(pkg.K_THRESHOLDS)} = {rep.hits}; median rank {int(ranks.float().median())}; "
          f"sharded rank_of_target step {t_rank * 1e3:.2f} ms (median of 5, host clock), "
          f"evaluate_aggregated {t_eval * 1e3:.1f} ms", flush=True)
flag = torch.tensor([1 if ok else 0], device=dev)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
dist.destroy_process_group()
sys.exit(0 if int(flag) else 1)
