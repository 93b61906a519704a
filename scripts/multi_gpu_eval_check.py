"""N-GPU ShardedRetriever.evaluate_products / evaluate_distance_fusions (every row of the eval script's report over a
gallery sharded over NCCL) against rank 0's single-GPU report on the whole gallery: the fusion ranks and hits, the
frame, best-frame and aggregated-descriptor ranks and the report rows built from them must be identical, and the
average-descriptor ranks must equal the single-GPU ranks of the same (fixed-order) average descriptors.
   torchrun --nproc-per-node N scripts/multi_gpu_eval_check.py"""
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
P, T, G = 2000, 10, 200000 + 13                         # G not divisible by the world size
g = torch.Generator(device="cpu").manual_seed(7)
seq = torch.zeros(1 + T, P, 256)
seq[1:] = torch.randn(T, P, 256, generator=g)
frame_product = torch.randint(0, P, (P * T,), generator=g)
frame_product[frame_product == 3] = 4                   # a product without frames
frame_desc = torch.randn(P * T, 256, generator=g)
shop_desc = torch.randn(G, 256, generator=g).half()     # the eval script stores shop descriptors as fp16
shop_aggr = torch.randn(G, 256, generator=g)
target = torch.randperm(G, generator=g)[:P]
frame_last = (torch.rand(2, 256, generator=g) / 8 - 1 / 16, torch.rand(2, generator=g) / 8 - 1 / 16)
seq, frame_product, frame_desc, target = seq.to(dev), frame_product.to(dev), frame_desc.to(dev), target.to(dev)
shop_desc, shop_aggr = shop_desc.to(dev), shop_aggr.to(dev)
frame_last = tuple(t.to(dev) for t in frame_last)
aggr_last = (eng._last[0].clone(), eng._last[1].clone())
shop_desc[target[frame_product[::3]]] = (frame_desc[::3] + 0.3 * torch.randn_like(frame_desc[::3])).half()

lo, hi = pkg.shard_bounds(G, world, rank)
r = pkg.ShardedRetriever.from_full_gallery(eng, shop_aggr)
dist.barrier()
torch.cuda.synchronize()
t0 = time.perf_counter()
fus = r.evaluate_distance_fusions(frame_desc, frame_product, shop_desc[lo:hi], target, frame_last)
torch.cuda.synchronize()
t_fus = time.perf_counter() - t0
dist.barrier()
t0 = time.perf_counter()
rep = r.evaluate_products(frame_desc, frame_product, shop_desc[lo:hi], target, frame_last, seq, None, aggr_last)
torch.cuda.synchronize()
t_rep = time.perf_counter() - t0
ok = True
if rank == 0:
    ref_fus = pkg.evaluate_distance_fusions(eng, frame_desc, frame_product, shop_desc, target, frame_last)
    ref = pkg.evaluate_products(eng, frame_desc, frame_product, shop_desc, target, frame_last, seq, None, shop_aggr,
                                aggr_last)
    avg, has = pkg.product_means(frame_desc, frame_product, P)
    with eng.scorer(*frame_last):
        ar, _ = eng.rank_of_target(avg, eng.prepare_gallery(shop_desc), target)
    ar = torch.where(has, ar, torch.full_like(ar, torch.iinfo(torch.int32).max))
    same = {"fusion ranks": torch.equal(fus[0], ref_fus[0]) and torch.equal(fus[1], ref_fus[1]),
            "frame ranks": torch.equal(rep.frame_ranks, ref.frame_ranks),
            "best frame / aggregated": torch.equal(rep.product_ranks[[0, 2]], ref.product_ranks[[0, 2]]),
            "average descriptor": torch.equal(rep.product_ranks[1], ar),
            "report rows 0, 1, 3": torch.equal(rep.perf[[0, 1, 3]], ref.perf[[0, 1, 3]])}
    ok = all(same.values())
    print(f"world={world} P={P} frames={P * T} G={G} ({torch.cuda.get_device_name(dev)}): sharded vs single-GPU "
          f"identical: {same}; fusion hits {fus[1].tolist()}; evaluate_distance_fusions {t_fus * 1e3:.1f} ms, "
          f"evaluate_products {t_rep * 1e3:.1f} ms (host clock, first call)", flush=True)
flag = torch.tensor([1 if ok else 0], device=dev)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
dist.destroy_process_group()
sys.exit(0 if int(flag) else 1)
