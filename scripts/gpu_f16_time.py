"""fp16 against fp32 tracks (developer tool): python scripts/gpu_f16_time.py [iterations]

For each shape, three ways of aggregating the same tracks, alternated round by round:
  fp32   the fp32 kernel on fp32 tracks                        (seam_aggregate)
  fp16   the fp16 kernel on fp16 tracks                        (seam_aggregate_f16)
  conv   fp16 tracks converted with .float(), then the fp32 kernel (what an fp16 caller paid before the fp16 entries)
CUDA events around each call, the L2 overwritten (256 MiB written) before every timed call.  Bytes/s use the fp16
algorithmic byte count, 512 T + 1024 per track (frames read, descriptor written), for all three.  Then search_host at
cfg 2 (15,000 tracks x 10 frames vs 15,000 gallery rows, top-20) from pinned fp16 and pinned fp32 host tracks."""
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import seam_match_rcnn_b200 as pkg  # noqa: E402
from bench import random_init_weights  # noqa: E402

ITERS = int(sys.argv[1]) if len(sys.argv) > 1 else 30
SHAPES = [(15000, 10), (100000, 4), (100000, 10), (100000, 16), (100000, 32), (100000, 64)]
dev = torch.device("cuda:0")
smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
print(f"device: {torch.cuda.get_device_name(dev)} | nvidia-smi name, power limit, max SM clock: {smi}", flush=True)
e = pkg.SeamEngine(dev)
e.load_weights(random_init_weights(dev))
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def timed(fn):
    flush.fill_(1)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e3, out


def spread(v):
    return f"median {statistics.median(v):8.1f} us (min {min(v):8.1f}, max {max(v):8.1f})"


for Q, T in SHAPES:
    g = torch.Generator(device=dev).manual_seed(Q + T)
    seq16 = torch.randn(1 + T, Q, 256, device=dev, generator=g).to(torch.float16)
    seq32 = seq16.float()
    ways = {"fp32": lambda: e.aggregate(seq32), "fp16": lambda: e.aggregate(seq16),
            "conv": lambda: e.aggregate(seq16.float())}
    res = {}
    for name, fn in ways.items():
        for _ in range(3):
            res[name] = fn()
    same = torch.equal(res["fp16"], res["fp32"]) and torch.equal(res["conv"], res["fp32"])
    del res
    us = {name: [] for name in ways}
    for _ in range(ITERS):
        for name, fn in ways.items():
            t, _ = timed(fn)
            us[name].append(t)
    by16 = Q * (512 * T + 1024)
    print(f"Q={Q} T={T}: fp16 output == fp32 output: {same}; fp16 bytes {by16 / 1e6:.1f} MB", flush=True)
    for name in ways:
        m = statistics.median(us[name])
        print(f"  {name}: {spread(us[name])} = {by16 / m / 1e6:.2f} TB/s of fp16 bytes", flush=True)
    print(f"  fp16 / fp32 = {statistics.median(us['fp16']) / statistics.median(us['fp32']):.3f}, "
          f"fp16 / conv = {statistics.median(us['fp16']) / statistics.median(us['conv']):.3f}", flush=True)
    del seq16, seq32
    torch.cuda.empty_cache()

# ---- search_host at cfg 2 from pinned host memory
Q, T, G, k = 15000, 10, 15000, 20
g = torch.Generator().manual_seed(1)
h16 = torch.randn(1 + T, Q, 256, generator=g).to(torch.float16).pin_memory()
h32 = h16.float().pin_memory()
gal = torch.randn(G, 256, generator=g).pin_memory()
stream = pkg.HostTrackStream(e)
outs = {n: [torch.empty((Q, k), dtype=dt).pin_memory() for dt in (torch.float32, torch.float32, torch.int32)]
        for n in ("fp16", "fp32")}
hosts = {"fp16": h16, "fp32": h32}
ways = {n: (lambda n=n: pkg.search_host(e, hosts[n], None, gal, k, out=outs[n], stream=stream)) for n in hosts}
for _ in range(3):
    for fn in ways.values():
        fn()
torch.cuda.synchronize()
same = all(torch.equal(a, b) for a, b in zip(outs["fp16"], outs["fp32"]))
us = {n: [] for n in ways}
for _ in range(ITERS):
    for n, fn in ways.items():
        t, _ = timed(fn)
        us[n].append(t)
print(f"search_host cfg 2 (Q={Q}, T={T}, G={G}, k={k}): fp16 results == fp32 results: {same}", flush=True)
for n in ways:
    print(f"  {n} host tracks ({stream.h2d_bytes(hosts[n], None) / 1e6:.1f} MB over PCIe): {spread(us[n])}", flush=True)
