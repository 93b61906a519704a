"""Aggregator backward timing (developer tool): python scripts/gpu_bwd_time.py [T ...]

Times seam_aggregate_backward alone (CUDA events around the C call, buffers allocated and zero-filled outside the
timed window) for Q in {64, 1024} tracks of T frames, median of 5 rounds of 20 calls after warm-up, and prints the
card's name and power limit with the numbers.  The inputs (Q * T * 1 KB of frames) and the parameter gradients
(0.5 MB) stay in L2 between calls: this is the time of a training step's backward on data it has just produced."""
import ctypes as C
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import seam_match_rcnn_b200 as pkg                                        # noqa: E402
from seam_match_rcnn_b200._lib import WEIGHT_KEYS, SeamWeightGrads, SeamWeights   # noqa: E402
from oracle import seam_oracle as so                                      # noqa: E402

dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
print(f"card: {card}", flush=True)
e = pkg.SeamEngine(dev)
w = {k: v.to(dev) for k, v in so.random_weights(seed=0).items()}
params = {f: w[WEIGHT_KEYS[f]].contiguous() for f in SeamWeights.FIELDS}
ws = SeamWeights(**{f: params[f].data_ptr() for f in SeamWeights.FIELDS})
grads = {f: torch.zeros_like(params[f]) for f in SeamWeightGrads.FIELDS}
gs = SeamWeightGrads(**{f: grads[f].data_ptr() for f in SeamWeightGrads.FIELDS})
Ts = [int(a) for a in sys.argv[1:]] or [10, 16, 32, 64]
for Q in (64, 1024):
    for T in Ts:
        seq = torch.randn(1 + T, Q, 256, device=dev)
        dout = torch.randn(Q, 256, device=dev)
        dseq = torch.zeros(1 + T, Q, 256, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream

        def call():
            return e._lib.seam_aggregate_backward(e._h, C.byref(ws), seq.data_ptr(), None, None, T, Q, seq.stride(0),
                                                  seq.stride(1), dout.data_ptr(), dseq.data_ptr(), C.byref(gs), stream)

        if call() != 0:
            print(f"aggregate_backward Q={Q} T={T}: refused ({e._lib.seam_last_error(e._h).decode()})", flush=True)
            continue
        for _ in range(5):
            call()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        rounds = []
        for _ in range(5):
            torch.cuda.synchronize()
            a.record()
            for _ in range(20):
                call()
            b.record()
            b.synchronize()
            rounds.append(a.elapsed_time(b) / 20 * 1e3)
        us = statistics.median(rounds)
        print(f"aggregate_backward Q={Q} T={T}: {us:.1f} us per call ({us / Q * 1e3:.0f} ns per track; "
              f"rounds {min(rounds):.1f}-{max(rounds):.1f} us)", flush=True)
