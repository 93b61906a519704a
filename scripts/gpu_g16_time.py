"""fp32, fp16 and bf16 galleries (developer tool): python scripts/gpu_g16_time.py [rounds]

One seeded fp32 gallery g scored three ways, alternated round by round:
  fp32   the fp32 gallery gb.float()       (seam_prepare_gallery, seam_score_topk, ...)
  fp16   the fp16 gallery g16 = g.half()   (seam_prepare_gallery_f16, seam_score_topk_g16, ...)
  bf16   the bf16 gallery gb = g.bfloat16() (seam_prepare_gallery_bf16, seam_score_topk_gbf16, ...)
The gallery has a planted near-duplicate of every query (as in bench.py), so the re-score and the exhaustive path see
real candidates.  Reported:
  1. per-kernel device times (SeamEngine.profile / profile_read, CUDA events) of prep_gallery, score, rescore and exact
     at cfg 2 (Q = G = 15,000, k = 20: the gallery fits in L2, 15 MB fp32 / 7.7 MB fp16) and at the cfg 5 shard
     (Q = 10,000, G = 125,000, k = 20), per call, median over the rounds; and the preparation call of each side
     against what a bf16 caller paid before bf16 galleries were kept: gb.float() and the fp32 preparation (CUDA
     events around the calls);
  2. a case that sends every row to the exhaustive kernel (k = 32: the window always fills);
  3. rank_of_target on a prepared gallery at cfg 2 (CUDA events around the call);
  4. search_host end to end from a pinned fp32, fp16 and bf16 host gallery of 1,000,000 rows (host clock around the
     call and a device synchronise);
  5. the device bytes a prepared gallery holds, from its tensors' storages.
Every bf16 result is checked bit for bit against the fp32 one (on gb.float()), every fp16 result against the fp32 path
on g16.float()."""
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
    """queries, and the three sides {fp32, fp16, bf16} of one seeded gallery (fp32 is the bf16 side widened)"""
    g = torch.Generator(device=dev).manual_seed(seed)
    q = torch.randn(Q, 256, device=dev, generator=g)
    gal = torch.randn(G, 256, device=dev, generator=g)
    n = min(Q, G)
    gal[:n] = q[:n] + 0.1 * torch.randn(n, 256, device=dev, generator=g)
    gb = gal.bfloat16()
    return q, {"fp32": gb.float(), "fp16": gal.half(), "bf16": gb}


def checks(res, ref16):
    """the bf16 side against fp32, the fp16 side against the fp32 path on its own widening"""
    return f"bf16 == fp32: {same(res['bf16'], res['fp32'])}, fp16 == fp32 on g16.float(): {same(res['fp16'], ref16)}"


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


def event_us(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(CALLS):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e3 / CALLS


def kernel_times(name, Q, G, k, seed):
    q, sides = data(Q, G, seed)
    res = {}
    for s, g in sides.items():                                       # warm-up
        p = e.prepare_gallery(g)
        res[s] = e.score_topk(q, p, k, return_stats=True)
    ref16 = e.score_topk(q, e.prepare_gallery(sides["fp16"].float()), k, return_stats=True)
    torch.cuda.synchronize()
    print(f"{name} (Q={Q}, G={G}, k={k}): {checks(res, ref16)}; exhaustive rows "
          f"{[int(res[s][3][0]) for s in sides]}; prepared bytes "
          + ", ".join(f"{s} {prepared_bytes(e.prepare_gallery(g))}" for s, g in sides.items()), flush=True)
    us = {s: {kk: [] for kk in KERNELS} for s in sides}
    prep = {s: [] for s in list(sides) + ["bf16 via .float()"]}
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
            prep[s].append(event_us(lambda: e.prepare_gallery(g)))
        prep["bf16 via .float()"].append(event_us(lambda: e.prepare_gallery(sides["bf16"].float())))
    for kk in KERNELS:
        m32 = statistics.median(us["fp32"][kk])
        print(f"  {kk:12s} " + " | ".join(f"{s} {spread(us[s][kk])}" for s in sides) + " | "
              + ", ".join(f"{s}/fp32 {statistics.median(us[s][kk]) / max(m32, 1e-9):.3f}" for s in ("fp16", "bf16")),
              flush=True)
    for s, v in prep.items():
        print(f"  prepare_gallery call, {s:17s} {spread(v)}", flush=True)
    del q, sides, res, ref16
    torch.cuda.empty_cache()


# ---- 1. per-kernel times, 2. the exhaustive path
kernel_times("cfg 2", 15000, 15000, 20, seed=1)
kernel_times("cfg 5 shard", 10000, 125000, 20, seed=4)
kernel_times("exhaustive (k = 32)", 2000, 125000, 32, seed=5)

# ---- 3. rank_of_target on a prepared gallery at cfg 2
Q = G = 15000
q, sides = data(Q, G, seed=1)
target = torch.randint(0, G, (Q,), device=dev, generator=torch.Generator(device=dev).manual_seed(2))
preps = {s: e.prepare_gallery(g) for s, g in sides.items()}
res = {s: e.rank_of_target(q, p, target, return_stats=True) for s, p in preps.items()}
ref16 = e.rank_of_target(q, e.prepare_gallery(sides["fp16"].float()), target, return_stats=True)
torch.cuda.synchronize()
print(f"rank_of_target cfg 2 (Q={Q}, G={G}): {checks(res, ref16)}; exhaustive rows "
      f"{[int(res[s][2][0]) for s in sides]}", flush=True)
us = {s: [] for s in preps}
for _ in range(ROUNDS):
    for s, p in preps.items():
        us[s].append(event_us(lambda: e.rank_of_target(q, p, target)))
for s in preps:
    print(f"  {s}: {spread(us[s])} per call", flush=True)
del q, sides, preps, res, ref16
torch.cuda.empty_cache()

# ---- 4. search_host from a pinned host gallery of 1,000,000 rows
Q, T, G, k = 10000, 10, 1000000, 20
gen = torch.Generator().manual_seed(3)
seq_h = torch.randn(1 + T, Q, 256, generator=gen).pin_memory()
g_h = torch.randn(G, 256, generator=gen)
gb_h = g_h.bfloat16().pin_memory()
hosts = {"fp32": gb_h.float().pin_memory(), "fp16": g_h.half().pin_memory(), "bf16": gb_h}
del g_h
stream = pkg.HostTrackStream(e)
outs = {s: [torch.empty((Q, k), dtype=dt).pin_memory() for dt in (torch.float32, torch.float32, torch.int32)]
        for s in list(hosts) + ["fp16 widened"]}
for s, gh in hosts.items():
    pkg.search_host(e, seq_h, None, gh, k, out=outs[s], stream=stream)
pkg.search_host(e, seq_h, None, hosts["fp16"].float(), k, out=outs["fp16 widened"], stream=stream)
torch.cuda.synchronize()
print(f"search_host (Q={Q}, T={T}, G={G}, k={k}): {checks(outs, outs['fp16 widened'])}", flush=True)
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
for s, dt in (("fp32", torch.float32), ("fp16", torch.float16), ("bf16", torch.bfloat16)):
    p = e.prepare_gallery(torch.zeros(1024, 256, dtype=dt, device=dev))
    per_row = (prepared_bytes(p) - 16) / 1024
    print(f"prepared {s} gallery: {per_row:.0f} B per row, {per_row * (1 << 26) / 1e9:.1f} GB for 2^26 rows", flush=True)
