"""Rank of the target over a sharded gallery, timed on one GPU.

(1) On one prepared gallery (index_offset 0), alternating: rank_of_target (the unsharded tensor-core entry) against
    target_margin + rank_count (the per-shard entries a sharded rank runs), at 10k x 125k (one of the 8 shards of the
    1M gallery) and 15k x 15k (the MovingFashion-scale eval).
(2) A 1M-row gallery split into 8 shards run back to back on this one GPU (the MAX / SUM over the shards done by
    torch on the device, standing in for the two all-reduces) against rank_of_target on the unsharded 1M gallery.
Every timed result is checked against the unsharded one.  Device events; medians over alternating repetitions.
   python scripts/gpu_shard_rank_time.py"""
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
REPS = 7


def card():
    name = torch.cuda.get_device_name(dev)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as ex:                             # noqa: BLE001
        out = f"unknown ({type(ex).__name__})"
    return f"{name}, power limit {out}"


def data(Q, G, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    q = torch.randn(Q, 256, device=dev, generator=g)
    gal = torch.randn(G, 256, device=dev, generator=g)
    n = min(Q, G)
    gal[:n] = q[:n] + 0.1 * torch.randn(n, 256, device=dev, generator=g)
    targets = {"planted (true match)": torch.arange(Q, device=dev) % G,
               "random item": torch.randint(0, G, (Q,), device=dev, generator=g)}
    return q, gal, targets


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def alternate(fa, fb):
    fa(), fb()                                          # warm-up (modules, workspace)
    torch.cuda.synchronize()
    ta, tb = [], []
    for _ in range(REPS):
        t, ra = timed(fa)
        ta.append(t)
        t, rb = timed(fb)
        tb.append(t)
    return statistics.median(ta), statistics.median(tb), ra, rb


def sharded(q, shards, target):
    m = torch.stack([e.target_margin(q, p, target) for p in shards]).amax(0)
    r = torch.zeros(q.shape[0], dtype=torch.int32, device=dev)
    for p in shards:
        r += e.rank_count(q, p, target, m)
    return r, m


print(f"[card] {card()}", flush=True)
for Q, G in [(10000, 125000), (15000, 15000)]:
    q, gal_t, targets = data(Q, G, 1)
    gal = e.prepare_gallery(gal_t)
    for name, target in targets.items():
        def unsharded():
            return e.rank_of_target(q, gal, target)

        def one_shard():
            m = e.target_margin(q, gal, target)
            return e.rank_count(q, gal, target, m), m

        ta, tb, ra, rb = alternate(unsharded, one_shard)
        same = torch.equal(ra[0], rb[0]) and torch.equal(ra[1].view(torch.int32), rb[1].view(torch.int32))
        print(f"Q={Q} G={G} target={name}: rank_of_target(prepared) {ta * 1e3:.0f} us, target_margin + rank_count "
              f"{tb * 1e3:.0f} us, identical={same}", flush=True)
    del gal, gal_t

Q, G, S = 10000, 1000000, 8
q, gal_t, targets = data(Q, G, 2)
full = e.prepare_gallery(gal_t)
shards = [e.prepare_gallery(gal_t[lo:hi], index_offset=lo) for lo, hi in (pkg.shard_bounds(G, S, s) for s in range(S))]
for name, target in targets.items():
    ta, tb, ra, rb = alternate(lambda: e.rank_of_target(q, full, target), lambda: sharded(q, shards, target))
    same = torch.equal(ra[0], rb[0]) and torch.equal(ra[1].view(torch.int32), rb[1].view(torch.int32))
    print(f"Q={Q} G={G} target={name}: unsharded rank_of_target(prepared) {ta:.2f} ms; {S} shards back to back on "
          f"this GPU {tb:.2f} ms ({tb / S:.2f} ms per shard); identical={same}", flush=True)
