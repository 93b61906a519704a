"""The "AVG & MAX DISTANCE" fusions over a sharded gallery, timed on one GPU.

(1) On one gallery of 125,000 items (one of the 8 shards of the 1M gallery), alternating: rank_fused_distances (the
    unsharded entry) against fused_target + fused_rank_count (the per-shard entries a sharded fusion rank runs).
(2) A 1M-item gallery split into 8 shards run back to back on this one GPU (the MAX / SUM over the shards done by torch
    on the device, standing in for the two all-reduces) against rank_fused_distances on the unsharded 1M gallery.
(3) fp16 against fp32 galleries, alternated on the same (fp16-representable) data, at 125,000 and 1M items.
Products have 10 frames each.  Every timed result is checked against the unsharded fp32 one.  Device events; medians
over alternating repetitions.
   python scripts/gpu_shard_fusion_time.py"""
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import seam_match_rcnn_b200 as pkg                     # noqa: E402
from bench import random_init_weights                   # noqa: E402

dev = torch.device("cuda:0")
e = pkg.SeamEngine(dev)
e.load_weights(random_init_weights(dev))
REPS = 5
FRAMES = 10


def card():
    name = torch.cuda.get_device_name(dev)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as ex:                             # noqa: BLE001
        out = f"unknown ({type(ex).__name__})"
    return f"{name}, power limit {out}"


def data(P, G, seed):
    """P products of FRAMES frames (grouped), an fp16-representable gallery of G items, one target per product (half of
    them resembling their product's frames)"""
    g = torch.Generator(device=dev).manual_seed(seed)
    frames = torch.randn(P * FRAMES, 256, device=dev, generator=g)
    start = torch.arange(P + 1, device=dev) * FRAMES
    gal = torch.randn(G, 256, device=dev, generator=g)
    target = torch.randint(0, G, (P,), device=dev, generator=g)
    gal[target[::2]] = frames[start[:-1:2]] + 0.3 * torch.randn(len(target[::2]), 256, device=dev, generator=g)
    return frames, start, gal.half().float(), target


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def alternate(fa, fb, reps=REPS):
    fa(), fb()                                          # warm-up (modules, allocations)
    torch.cuda.synchronize()
    ta, tb = [], []
    for _ in range(reps):
        t, ra = timed(fa)
        ta.append(t)
        t, rb = timed(fb)
        tb.append(t)
    return statistics.median(ta), statistics.median(tb), ra, rb


def sharded(frames, start, shards, target):
    tv = torch.stack([torch.stack(e.fused_target(frames, start, gs, lo, target)) for lo, gs in shards]).amax(0)
    r = torch.zeros((2, target.shape[0]), dtype=torch.int32, device=dev)
    for lo, gs in shards:
        r += torch.stack(e.fused_rank_count(frames, start, gs, lo, target, tv[0], tv[1]))
    return r


def unsharded(frames, start, gal, target):
    return torch.stack(e.rank_fused_distances(frames, start, gal, target))


def pairs(P, G):
    return f"{P * FRAMES * G / 1e9:.2f}e9 (frame, item) pairs"


print(f"[card] {card()}", flush=True)
P, G = 2000, 125000
frames, start, gal, target = data(P, G, 1)
ta, tb, ra, rb = alternate(lambda: unsharded(frames, start, gal, target),
                           lambda: sharded(frames, start, [(0, gal)], target))
print(f"(1) P={P} x {FRAMES} frames, G={G} ({pairs(P, G)}): rank_fused_distances {ta:.1f} ms, fused_target + "
      f"fused_rank_count {tb:.1f} ms, identical={torch.equal(ra, rb)}", flush=True)
g16 = gal.half()
ta, tb, ra16, rb16 = alternate(lambda: unsharded(frames, start, gal, target), lambda: unsharded(frames, start, g16, target))
print(f"(3) P={P} x {FRAMES} frames, G={G}: fp32 gallery {ta:.1f} ms, fp16 gallery {tb:.1f} ms, "
      f"identical={torch.equal(ra16, rb16)}", flush=True)
del frames, start, gal, g16

P, G, S = 1000, 1000000, 8
frames, start, gal, target = data(P, G, 2)
shards = [(lo, gal[lo:hi]) for lo, hi in (pkg.shard_bounds(G, S, s) for s in range(S))]
ta, tb, ra, rb = alternate(lambda: unsharded(frames, start, gal, target),
                           lambda: sharded(frames, start, shards, target), reps=3)
print(f"(2) P={P} x {FRAMES} frames, G={G} ({pairs(P, G)}): unsharded rank_fused_distances {ta:.1f} ms; {S} shards back "
      f"to back on this GPU {tb:.1f} ms ({tb / S:.1f} ms per shard); identical={torch.equal(ra, rb)}", flush=True)
g16 = gal.half()
ta, tb, ra16, rb16 = alternate(lambda: unsharded(frames, start, gal, target), lambda: unsharded(frames, start, g16, target),
                               reps=3)
print(f"(3) P={P} x {FRAMES} frames, G={G}: fp32 gallery {ta:.1f} ms, fp16 gallery {tb:.1f} ms, "
      f"identical={torch.equal(ra16, rb16) and torch.equal(ra16, ra)}", flush=True)
