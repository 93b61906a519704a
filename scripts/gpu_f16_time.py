"""fp16 and bf16 against fp32 tracks (developer tool): python scripts/gpu_f16_time.py [iterations]

For each shape, four ways of aggregating the same tracks, alternated round by round:
  fp32   the fp32 kernel on fp32 tracks                        (seam_aggregate)
  fp16   the fp16 kernel on fp16 tracks                        (seam_aggregate_f16)
  bf16   the bf16 kernel on bf16 tracks                        (seam_aggregate_bf16)
  conv   fp16 tracks converted with .float(), then the fp32 kernel (what a 16-bit caller paid before the 16-bit entries)
The fp32 tracks are the fp16 ones widened; the bf16 tracks are drawn from the same distribution, and their output is
checked against the fp32 kernel on them widened.  CUDA events around each call, the L2 overwritten (256 MiB written)
before every timed call.
Bytes/s use the 16-bit algorithmic byte count, 512 T + 1024 per track (frames read, descriptor written), for all four.
Then search_host at cfg 2 (15,000 tracks x 10 frames vs 15,000 gallery rows, top-20) from pinned fp16, bf16 and fp32
host tracks."""
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
    seqb = torch.randn(1 + T, Q, 256, device=dev, generator=g).to(torch.bfloat16)
    ways = {"fp32": lambda: e.aggregate(seq32), "fp16": lambda: e.aggregate(seq16),
            "bf16": lambda: e.aggregate(seqb), "conv": lambda: e.aggregate(seq16.float())}
    res = {}
    for name, fn in ways.items():
        for _ in range(3):
            res[name] = fn()
    same = torch.equal(res["fp16"], res["fp32"]) and torch.equal(res["conv"], res["fp32"])
    same_b = torch.equal(res["bf16"], e.aggregate(seqb.float()))
    del res
    us = {name: [] for name in ways}
    for _ in range(ITERS):
        for name, fn in ways.items():
            t, _ = timed(fn)
            us[name].append(t)
    by16 = Q * (512 * T + 1024)
    print(f"Q={Q} T={T}: fp16 output == fp32 output: {same}; bf16 output == fp32 output on its tracks: {same_b}; "
          f"16-bit bytes {by16 / 1e6:.1f} MB", flush=True)
    for name in ways:
        m = statistics.median(us[name])
        print(f"  {name}: {spread(us[name])} = {by16 / m / 1e6:.2f} TB/s of 16-bit bytes", flush=True)
    med = {name: statistics.median(us[name]) for name in ways}
    print(f"  fp16 / fp32 = {med['fp16'] / med['fp32']:.3f}, fp16 / conv = {med['fp16'] / med['conv']:.3f}, "
          f"bf16 / fp16 = {med['bf16'] / med['fp16']:.3f}, bf16 / fp32 = {med['bf16'] / med['fp32']:.3f}", flush=True)
    del seq16, seq32, seqb
    torch.cuda.empty_cache()

# ---- search_host at cfg 2 from pinned host memory
Q, T, G, k = 15000, 10, 15000, 20
g = torch.Generator().manual_seed(1)
h16 = torch.randn(1 + T, Q, 256, generator=g).to(torch.float16).pin_memory()
h32 = h16.float().pin_memory()
hb = torch.randn(1 + T, Q, 256, generator=g).to(torch.bfloat16).pin_memory()
gal = torch.randn(G, 256, generator=g).pin_memory()
stream = pkg.HostTrackStream(e)
outs = {n: [torch.empty((Q, k), dtype=dt).pin_memory() for dt in (torch.float32, torch.float32, torch.int32)]
        for n in ("fp16", "bf16", "fp32")}
hosts = {"fp16": h16, "bf16": hb, "fp32": h32}
ways = {n: (lambda n=n: pkg.search_host(e, hosts[n], None, gal, k, out=outs[n], stream=stream)) for n in hosts}
for _ in range(3):
    for fn in ways.values():
        fn()
torch.cuda.synchronize()
same = all(torch.equal(a, b) for a, b in zip(outs["fp16"], outs["fp32"]))
ref_b = pkg.search_host(e, hb.float().pin_memory(), None, gal, k, stream=stream)
torch.cuda.synchronize()
same_b = all(torch.equal(a, b) for a, b in zip(outs["bf16"], ref_b))
us = {n: [] for n in ways}
for _ in range(ITERS):
    for n, fn in ways.items():
        t, _ = timed(fn)
        us[n].append(t)
print(f"search_host cfg 2 (Q={Q}, T={T}, G={G}, k={k}): fp16 results == fp32 results: {same}; "
      f"bf16 results == fp32 results on its tracks: {same_b}", flush=True)
for n in ways:
    print(f"  {n} host tracks ({stream.h2d_bytes(hosts[n], None) / 1e6:.1f} MB over PCIe): {spread(us[n])}", flush=True)
