"""fp16 against fp32 galleries (developer tool): python scripts/gpu_g16_time.py [rounds]

The same seeded data scored two ways, alternated round by round:
  fp32   the fp32 gallery g.float()  (seam_prepare_gallery, seam_score_topk, ...)
  fp16   the fp16 gallery g          (seam_prepare_gallery_f16, seam_score_topk_g16, ...)
The gallery has a planted near-duplicate of every query (as in bench.py), so the re-score and the exhaustive path see
real candidates.  Reported:
  1. per-kernel device times (SeamEngine.profile / profile_read, CUDA events) of prep_gallery, score, rescore and exact
     at cfg 2 (Q = G = 15,000, k = 20: the gallery fits in L2, 15 MB fp32 / 7.7 MB fp16) and at the cfg 5 shard
     (Q = 10,000, G = 125,000, k = 20), per call, median over the rounds;
  2. a case that sends every row to the exhaustive kernel (k = 32: the window always fills);
  3. rank_of_target on a prepared gallery at cfg 2 (CUDA events around the call);
  4. search_host end to end from a pinned fp16 and a pinned fp32 host gallery of 1,000,000 rows (host clock around
     the call and a device synchronise);
  5. the device bytes a prepared gallery holds, from its tensors' storages.
Every fp16 result is checked bit for bit against the fp32 one."""
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import seam_match_rcnn_b200 as pkg  # noqa: E402
from bench import random_init_weights  # noqa: E402

ROUNDS = int(sys.argv[1]) if len(sys.argv) > 1 else 5
CALLS = 5                       # calls per side and round
dev = torch.device("cuda:0")
smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
print(f"device: {torch.cuda.get_device_name(dev)} | nvidia-smi name, power limit: {smi}", flush=True)
e = pkg.SeamEngine(dev)
e.load_weights(random_init_weights(dev))
KERNELS = ("prep_gallery", "score", "rescore", "exact")


def data(Q, G, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    q = torch.randn(Q, 256, device=dev, generator=g)
    gal = torch.randn(G, 256, device=dev, generator=g)
    n = min(Q, G)
    gal[:n] = q[:n] + 0.1 * torch.randn(n, 256, device=dev, generator=g)
    return q, gal.half()


def same(a, b):
    return all(torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x,
                           y.view(torch.int32) if y.dtype == torch.float32 else y) for x, y in zip(a, b))


def prepared_bytes(p):
    seen, tot = set(), 0
    for t in (p.g, p.g16, p.cg, p.gstat):
        s = t.untyped_storage()
        if s.data_ptr() not in seen:
            seen.add(s.data_ptr())
            tot += s.nbytes()
    return tot


def spread(v, unit="us"):
    return f"median {statistics.median(v):9.1f} {unit} (min {min(v):9.1f}, max {max(v):9.1f})"


def kernel_times(name, Q, G, k, seed):
    q, g16 = data(Q, G, seed)
    sides = {"fp32": g16.float(), "fp16": g16}
    res = {}
    for s, g in sides.items():                                       # warm-up
        p = e.prepare_gallery(g)
        res[s] = e.score_topk(q, p, k, return_stats=True)
    torch.cuda.synchronize()
    print(f"{name} (Q={Q}, G={G}, k={k}): fp16 results == fp32 results: {same(res['fp16'], res['fp32'])}; "
          f"exhaustive rows {int(res['fp16'][3][0])}; prepared bytes fp32 {prepared_bytes(e.prepare_gallery(sides['fp32']))}"
          f", fp16 {prepared_bytes(e.prepare_gallery(sides['fp16']))}", flush=True)
    us = {s: {kk: [] for kk in KERNELS} for s in sides}
    for _ in range(ROUNDS):
        for s, g in sides.items():
            e.profile_read()
            e.profile(True)
            for _ in range(CALLS):
                p = e.prepare_gallery(g)
                e.score_topk(q, p, k)
            e.profile(False)
            r = e.profile_read()
            for kk in KERNELS:
                ms, n = r[kk]
                us[s][kk].append(ms * 1e3 / max(n, 1))
    for kk in KERNELS:
        m32, m16 = statistics.median(us["fp32"][kk]), statistics.median(us["fp16"][kk])
        print(f"  {kk:12s} fp32 {spread(us['fp32'][kk])} | fp16 {spread(us['fp16'][kk])} | fp16/fp32 "
              f"{m16 / max(m32, 1e-9):.3f}", flush=True)
    del q, g16, sides, res
    torch.cuda.empty_cache()


# ---- 1. per-kernel times, 2. the exhaustive path
kernel_times("cfg 2", 15000, 15000, 20, seed=1)
kernel_times("cfg 5 shard", 10000, 125000, 20, seed=4)
kernel_times("exhaustive (k = 32)", 2000, 125000, 32, seed=5)

# ---- 3. rank_of_target on a prepared gallery at cfg 2
Q = G = 15000
q, g16 = data(Q, G, seed=1)
target = torch.randint(0, G, (Q,), device=dev, generator=torch.Generator(device=dev).manual_seed(2))
preps = {"fp32": e.prepare_gallery(g16.float()), "fp16": e.prepare_gallery(g16)}
res = {s: e.rank_of_target(q, p, target, return_stats=True) for s, p in preps.items()}
torch.cuda.synchronize()
print(f"rank_of_target cfg 2 (Q={Q}, G={G}): fp16 == fp32: {same(res['fp16'], res['fp32'])}; "
      f"exhaustive rows {int(res['fp16'][2][0])}", flush=True)
us = {s: [] for s in preps}
for _ in range(ROUNDS):
    for s, p in preps.items():
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(CALLS):
            e.rank_of_target(q, p, target)
        b.record()
        b.synchronize()
        us[s].append(a.elapsed_time(b) * 1e3 / CALLS)
for s in preps:
    print(f"  {s}: {spread(us[s])} per call", flush=True)
del q, g16, preps, res
torch.cuda.empty_cache()

# ---- 4. search_host from a pinned host gallery of 1,000,000 rows
Q, T, G, k = 10000, 10, 1000000, 20
gen = torch.Generator().manual_seed(3)
seq_h = torch.randn(1 + T, Q, 256, generator=gen).pin_memory()
g16_h = torch.randn(G, 256, generator=gen).half().pin_memory()
hosts = {"fp32": g16_h.float().pin_memory(), "fp16": g16_h}
stream = pkg.HostTrackStream(e)
outs = {s: [torch.empty((Q, k), dtype=dt).pin_memory() for dt in (torch.float32, torch.float32, torch.int32)]
        for s in hosts}
for s, gh in hosts.items():
    pkg.search_host(e, seq_h, None, gh, k, out=outs[s], stream=stream)
torch.cuda.synchronize()
print(f"search_host (Q={Q}, T={T}, G={G}, k={k}): fp16 results == fp32 results: {same(outs['fp16'], outs['fp32'])}",
      flush=True)
ms = {s: [] for s in hosts}
for _ in range(max(3, ROUNDS // 2)):
    for s, gh in hosts.items():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pkg.search_host(e, seq_h, None, gh, k, out=outs[s], stream=stream)
        torch.cuda.synchronize()
        ms[s].append((time.perf_counter() - t0) * 1e3)
for s, gh in hosts.items():
    print(f"  {s} host gallery ({gh.numel() * gh.element_size() / 1e9:.2f} GB over PCIe): {spread(ms[s], 'ms')}",
          flush=True)

# ---- 5. device bytes of a prepared 2^26-row shard (the most one shard may hold), from the per-row sizes above
for s, dt in (("fp32", torch.float32), ("fp16", torch.float16)):
    p = e.prepare_gallery(torch.zeros(1024, 256, dtype=dt, device=dev))
    per_row = (prepared_bytes(p) - 16) / 1024
    print(f"prepared {s} gallery: {per_row:.0f} B per row, {per_row * (1 << 26) / 1e9:.1f} GB for 2^26 rows", flush=True)
