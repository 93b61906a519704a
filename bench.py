"""Benchmark of the SEAM retrieval hot path (aggregation -> pair scorer -> top-k) on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference's own CPU modules (oracle/_ref)
    python bench.py ... --dump-outputs DIR                   # also writes the last timed step's outputs as DIR/*.npy

Prints ONE JSON line (rank 0).  A "step" is one pass of the hot path over one batch of synthetic
tracks: BASELINE.json configs[1] (15,000 tracks x 10 frames vs 15,000 shop items, k=20) at N=1.
For N>1 the gallery is sharded (15,000 rows PER GPU, weak scaling), every rank aggregates the tracks
it owns and the kernels exchange descriptors / per-shard top-k lists / merged rows themselves over
NVLink peer memory (retrieval.PeerExchange; NCCL all-gathers only as a fallback).

Inputs follow SURVEY.md section 8(d): randn embeddings; gallery = randn with the first min(Q,G) rows
overwritten by agg(query_i) + 0.1 randn (a planted true match per query: non-trivial top-1, near
ties for the certified top-k, worst-case cancellation); default-init weights with newnlb.W re-drawn.

metric        pair scores/sec = Q*G / (device time of aggregation + scorer + top-k [+ exchange])
value         inputs already resident in HBM, CUDA-event timed, max over ranks
e2e           same metric through the public Python API from pinned HOST buffers: H2D of the
              tracks, mask and gallery shard, gallery preparation, the hot path, D2H of the results
roofline      dominant kernel (score_topk_kernel, tensor-bound, 512 FLOP per pair) + the whole
              scorer stage (prep + K2 + re-score + exhaustive fallback) as stage_frac;
              roofline_aggregate: the aggregation stage (ONE kernel) against HBM copy bandwidth
parity_check  a 32-query sample of the timed step's output against the CPU oracle and, for N>1,
              the sharded result against the unsharded single-GPU search (outside the timed region)
configs       the other BASELINE.json configurations, device-timed the same way: cfg3 (ragged T=2..4
              vs 50k, sharded over N), cfg4 (100k x 64 aggregation, N=1), cfg5 (10k vs 1M, N=8)
cpu_baseline  the reference's TemporalAggregationNLB.forward + softmax + top-k on the host cores
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

Q_TRACKS, T_FRAMES, G_PER_GPU, TOPK = 15000, 10, 15000, 20
FLOP_PER_PAIR = 512               # 2 * 256: single-channel dw GEMM (SURVEY.md section 8(d))
METRIC, UNIT = "pair_scores_per_sec", "pairs/s"
TOL_MARGIN = 3e-5                 # stated tolerance on margins (tests/util.py TOL_LOGIT)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "tflops": p["bf16_tflops"], "tflops_sustained": p.get("bf16_tflops_sustained"),
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops": 1590.0, "tflops_sustained": 1400.0, "source": "fallback"}


# --------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self._stop_evt.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                bits = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for b, name in self.REASONS.items():
                    if bits & b:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.0005)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join()
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# --------------------------------------------------------------------------------------
# the reference on the host cores
# --------------------------------------------------------------------------------------
def reference_step_fn(sample_q, T, G, k):
    """One step of the reference's CPU path on `sample_q` tracks x full gallery: its own modules from oracle/_ref
    (TemporalAggregationNLB.forward seq-branch, models/match_head.py:133-169, unmodified) + softmax + torch.topk
    -- kind "reference"; the bit-equal oracle port when oracle/_ref did not travel -- kind "port"."""
    from oracle import seam_oracle as so
    from oracle import build_ref
    w = so.random_weights(0)
    seq, mask, _ = so.synth_tracks(sample_q, T, seed=1)
    gal = so.synth_gallery(G, 1, None)
    mh = None
    try:
        mh = build_ref.load()
    except Exception:                                   # noqa: BLE001 -- anything wrong with _ref: use the port
        mh = None
    if mh is not None:
        model = mh.TemporalAggregationNLB().eval()
        model.load_state_dict(w, strict=False)

        def step():
            out = model(None, None, None, x3_1_seq=seq, x3_1_mask=mask, x3_2=gal)
            return torch.topk(torch.softmax(out[2], -1)[..., 1], k, dim=1)
        return step, "reference"

    def step():
        q, _ = so.aggregate_tracks(seq, mask, w)
        return so.rank_topk(so.pair_logits(q, gal, w), k)
    return step, "port"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    G = G_PER_GPU * args.gpus
    sample_q = 64
    step, kind = reference_step_fn(sample_q, T_FRAMES, G, TOPK)
    with torch.no_grad():
        for _ in range(args.warmup):
            step()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step()
        dt = (time.perf_counter() - t0) / args.steps
    value = sample_q * G / dt
    sample = f"{sample_q} tracks x {T_FRAMES} frames vs {G} shop items per step (of {Q_TRACKS} tracks)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"MovingFashion-scale eval: {Q_TRACKS} tracks x {T_FRAMES} frames vs {G} shop items, k={TOPK}",
                   "sample": sample, "threads": cores,
                   "path": "TemporalAggregationNLB.forward (seq-branch) + softmax + torch.topk, torch fp32 on the host"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "queries_per_sec": sample_q / dt,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline(budget_s=12.0):
    """The reference timed on the host cores on a bounded sample of the N=1 workload."""
    cores = os.cpu_count() or 1
    prev = torch.get_num_threads()
    torch.set_num_threads(cores)
    chunk = 64
    step, kind = reference_step_fn(chunk, T_FRAMES, G_PER_GPU, TOPK)
    with torch.no_grad():
        step()
        t0 = time.perf_counter()
        n = 0
        while True:
            step()
            n += 1
            if time.perf_counter() - t0 > budget_s or n >= 64:
                break
        dt = time.perf_counter() - t0
    torch.set_num_threads(prev)
    return {"value": n * chunk * G_PER_GPU / dt, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{n} x ({chunk} tracks x {T_FRAMES} frames vs {G_PER_GPU} shop items), {dt:.1f} s",
            "queries_per_sec": n * chunk / dt}


def random_init_weights(dev):
    """Random-init aggregator weights of the reference's architecture (default torch init
    U(+-1/sqrt(fan_in)); newnlb.W re-drawn because the reference zero-initialises it, which
    would make the block a no-op -- SURVEY.md section 0 item 2)."""
    g = torch.Generator().manual_seed(0)

    def u(shape, fan_in):
        return ((torch.rand(shape, generator=g) * 2 - 1) / fan_in ** 0.5).to(dev)

    w = {}
    for n in ("g", "theta", "phi"):
        w[f"newnlb.{n}.weight"], w[f"newnlb.{n}.bias"] = u((128, 256, 1), 256), u((128,), 256)
    w["newnlb.W.weight"], w["newnlb.W.bias"] = u((256, 128, 1), 128), u((256,), 128)
    w["newnlb.concat_project.0.weight"] = u((1, 256, 1, 1), 256)
    w["attention_scorer.weight"], w["attention_scorer.bias"] = u((1, 256), 256), u((1,), 256)
    w["last.weight"], w["last.bias"] = u((2, 256), 256), u((2,), 256)
    return w


# --------------------------------------------------------------------------------------
# workloads (SURVEY.md section 8(d))
# --------------------------------------------------------------------------------------
class Workload:
    """Synthetic tracks (all Q, identical on every rank: same seed, same device generator), this rank's gallery
    shard with the planted matches, and the step that searches them."""

    def __init__(self, pkg, eng, dev, world, rank, name, Q, T, G_total, k, seed, ragged=None):
        self.pkg, self.eng, self.dev, self.world, self.rank = pkg, eng, dev, world, rank
        self.name, self.Q, self.T, self.G, self.k = name, Q, T, G_total, k
        gen = torch.Generator(device=dev).manual_seed(seed)
        self.seq = torch.zeros(1 + T, Q, 256, device=dev)
        self.seq[1:] = torch.randn(T, Q, 256, device=dev, generator=gen)
        self.lens = self.mask = None
        self.frames = Q * T
        if ragged is not None:
            self.lens = torch.randint(ragged[0], ragged[1] + 1, (Q,), device=dev, generator=gen).int()
            self.mask = torch.arange(1 + T, device=dev)[None, :] > self.lens[:, None]
            self.seq[1:] *= (~self.mask[:, 1:]).t()[:, :, None]
            self.frames = int(self.lens.sum())
        self.qlo, self.qhi = pkg.shard_bounds(Q, world, rank)
        self.gallery = self.gal = None
        self.glo = self.ghi = 0
        if G_total > 0:
            self.glo, self.ghi = pkg.shard_bounds(G_total, world, rank)
            gg = torch.Generator(device=dev).manual_seed(seed * 7919 + 1000 + rank)
            self.gal = torch.randn(self.ghi - self.glo, 256, device=dev, generator=gg)
            n_plant = min(Q, G_total)                                  # global rows [0, n_plant) carry agg(q_i) + noise
            lo, hi = self.glo, min(self.ghi, n_plant)
            if hi > lo:
                q_rows = eng.aggregate(self.seq[:, lo:hi], None if self.mask is None else self.mask[lo:hi])
                self.gal[: hi - lo] = q_rows + 0.1 * torch.randn(hi - lo, 256, device=dev, generator=gg)
            self.gallery = eng.prepare_gallery(self.gal, index_offset=self.glo)
        self.peer = None
        self.retr = None
        self.peer_note = ""
        if world > 1 and G_total > 0 and os.environ.get("SEAM_BENCH_PEER", "1") != "0":
            try:
                self.peer = pkg.PeerExchange(eng, Q, k)
                self.retr = pkg.ShardedRetriever(eng, self.gallery, self.glo)
            except Exception as ex:                      # noqa: BLE001 -- any failure means: keep NCCL
                self.peer = None
                self.peer_note = f" (symmetric memory unavailable: {type(ex).__name__})"
        if world > 1 and G_total > 0 and self.peer is None:
            self.retr = pkg.ShardedRetriever(eng, self.gallery, self.glo)
        self.graph = None
        self.last_out = None             # what the last step returned (the graph's static outputs when replayed)
        self.stamps = None

    # one pass of the hot path, inputs resident in HBM
    def hot_path(self):
        eng = self.eng
        if self.G == 0:                                               # aggregation only (cfg 4)
            return eng.aggregate(self.seq, self.mask)
        if self.world == 1:
            return eng.search(self.seq, self.mask, self.gallery, self.k)     # one library call (seam_search)
        if self.peer is not None:
            return self.retr.search_peer(self.seq, self.mask, self.peer)
        return self.retr.search(self.seq, self.mask, self.k)        # NCCL all-gather fallback (eager)

    def capture(self):
        """The step is launch-bound (a handful of kernels of 5-500 us): replay it as ONE CUDA graph.  The NCCL
        fallback stays eager."""
        import torch.distributed as dist
        if os.environ.get("SEAM_BENCH_GRAPH", "1") == "0" or (self.world > 1 and self.peer is None):
            return
        dev = self.dev
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(3):                          # warm allocator and workspaces before capture
                self.hot_path()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, capture_error_mode="thread_local"):
            if self.world > 1:
                # N > 1: the ranks wait for each other's data inside the kernels, so a step must START at the same
                # moment on every GPU or the host's launch skew between the rank processes is measured as step time.
                # The replayed graph is [cross-rank barrier kernel, time stamp, the step, time stamp]: the barrier node
                # aligns the GPUs, the step is timed between the two stamps (%globaltimer, one-thread kernels).
                self.stamps = torch.zeros(2, dtype=torch.int64, device=dev)
                self.peer.device_barrier()
                self.eng.device_stamp(self.stamps, 0)
            self.last_out = self.hot_path()
            if self.world > 1:
                self.eng.device_stamp(self.stamps, 1)

    def step(self):
        if self.graph is not None:
            self.graph.replay()
        else:
            self.last_out = self.hot_path()
        return self.last_out

    def launch_note(self):
        if self.graph is not None:
            return "one CUDA graph replay per step"
        return "eager launches" + (" + NCCL all-gathers" if self.world > 1 else "")

    def free(self):
        self.graph = self.last_out = self.peer = self.retr = self.gallery = self.gal = self.seq = None
        torch.cuda.empty_cache()


def dump_outputs(out_dir, outputs):
    """<out_dir>/<name>.npy for each array the timed step returned to its caller: on one GPU seam_search's
    descriptors (Q,256) and the (Q,k) scores, margins and gallery indices (about 20 MB); sharded, the (Q,k) three.
    Indices are stored as float64, which holds every int32 exactly.  The inputs come from fixed seeds, so two builds
    run with the same arguments can be compared output for output."""
    import numpy as np
    names = ("descriptors", "scores", "margins", "indices")[-len(outputs):]
    os.makedirs(out_dir, exist_ok=True)
    for name, t in zip(names, outputs):
        a = t.cpu().numpy().astype(np.float64 if name == "indices" else np.float32)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def stage_record(wl, kern, ms, peaks):
    """Per-stage numbers of one configuration from the event-timed kernels (`kern`, ms) and the step time."""
    rec = {"ms_per_step": ms, "kernel_ms": kern, "launch": wl.launch_note()}
    t_agg = kern.get("aggregate")
    per_rank_frames = wl.frames if wl.world == 1 else None
    if t_agg:
        own = wl.qhi - wl.qlo
        frames = wl.frames * own / max(wl.Q, 1) if per_rank_frames is None else per_rank_frames
        agg_bytes = (frames + own) * 1024
        rec["aggregate"] = {"ms": t_agg, "GBps": agg_bytes / (t_agg * 1e-3) / 1e9,
                            "frac_of_hbm": agg_bytes / (t_agg * 1e-3) / 1e9 / peaks["hbm_gbs"],
                            "tracks_per_sec_per_gpu": own / (t_agg * 1e-3)}
    if wl.G > 0:
        pairs_gpu = wl.Q * (wl.ghi - wl.glo)
        t_stage = sum(kern.get(n) or 0.0 for n in ("prep_queries", "score", "rescore", "exact"))
        rec["scorer"] = {"k2_ms": kern.get("score"), "stage_ms": t_stage,
                         "k2_frac_of_tensor_peak": pairs_gpu * FLOP_PER_PAIR / (kern["score"] * 1e-3) / 1e12 / peaks["tflops"],
                         "stage_frac_of_tensor_peak": pairs_gpu * FLOP_PER_PAIR / (t_stage * 1e-3) / 1e12 / peaks["tflops"]}
        rec["pairs_per_sec"] = wl.Q * wl.G / (ms * 1e-3)
        rec["queries_per_sec"] = wl.Q / (ms * 1e-3)
    else:
        rec["tracks_per_sec"] = wl.Q / (ms * 1e-3)
    return rec


# --------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    import seam_match_rcnn_b200 as pkg

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # pinned host buffers (the e2e leg) should live on the NUMA node this GPU hangs off
    numa = pkg.bind_to_gpu_numa_node(dev) if os.environ.get("SEAM_BENCH_NUMA", "1") != "0" else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    eng = pkg.SeamEngine(dev)
    weights = random_init_weights(dev)
    eng.load_weights(weights)
    peaks = measured_peaks()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, stamps=None):
        """ms per step, device-timed, max over ranks: CUDA events around fn() on the launching stream -- or, with
        `stamps` (the sharded step's graph: [cross-rank barrier kernel, stamp, step, stamp]), the difference of the two
        device time stamps the graph itself wrote (events cannot be recorded between the nodes of a replayed graph)."""
        for _ in range(warmup):
            fn()
        barrier()
        total = 0.0
        for _ in range(steps):
            flush.fill_(1)                   # evict L2 between timed iterations (not timed)
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            barrier()
            total += (float(stamps[1] - stamps[0]) * 1e-6) if stamps is not None else a.elapsed_time(b)
        t = torch.tensor([total / steps], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)                      # ms per step, max over ranks

    def kernel_times(wl, steps):
        """Per-kernel durations (CUDA events inside the library, on the launching stream), eager launches (events
        cannot be recorded inside a graph replay); returns ({kernel: ms}, kernels launched per step)."""
        eng.profile(True)
        barrier()
        lc0 = eng.launch_count
        for _ in range(steps):
            flush.fill_(1)
            wl.hot_path()
        barrier()
        n_launch = (eng.launch_count - lc0) / steps
        prof = eng.profile_read()
        eng.profile(False)
        kern = {n: (tot / cnt if cnt else None) for n, (tot, cnt) in prof.items()}
        if world > 1:                        # max over ranks per kernel
            names = sorted(kern)
            t = torch.tensor([kern[n] or 0.0 for n in names], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            kern = {n: (float(v) or None) for n, v in zip(names, t)}
        return kern, n_launch

    # ================================================================= main configuration (cfg 2, weak-scaled)
    Q, T, Gs, k = Q_TRACKS, T_FRAMES, G_PER_GPU, TOPK
    G = Gs * world
    wl = Workload(pkg, eng, dev, world, rank, "cfg2", Q, T, G, k, seed=1)
    wl.capture()
    warmup = max(args.warmup, 3)
    sampler = ClockSampler(local)                             # samples through the device-timed AND the e2e timed regions
    sampler.start()
    ms = timed(wl.step, args.steps, warmup, wl.stamps if wl.graph is not None else None)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, wl.last_out)
    rank_alignment = ("the replayed graph is [cross-rank barrier kernel, device time stamp, step, device time stamp]: the GPUs "
                      "enter the step together and the step is timed between the stamps (host launch skew is not step time)"
                      if (wl.graph is not None and wl.stamps is not None) else None)

    # ---- end to end from pinned host memory through the package's host-facing entry points
    # (retrieval.search_host / HostTrackStream): the rank's tracks cross PCIe in NCHUNK slices on a copy stream;
    # slice i+1 is in flight while slice i is aggregated (and, on one GPU, scored and its results copied back).
    # Row 0 of x3_1_seq (the layout's dummy frame) is not copied.
    NCHUNK = max(1, 4 // world)          # fewer, larger slices when a rank only uploads Q/N tracks
    per = wl.qhi - wl.qlo
    seq_h = wl.seq[:, wl.qlo:wl.qhi].cpu().pin_memory()
    mask_h = torch.zeros(per, 1 + T, dtype=torch.bool).pin_memory()
    gal_h = wl.gal.cpu().pin_memory()
    out_h = [torch.empty(Q, k).pin_memory(), torch.empty(Q, k).pin_memory(), torch.empty(Q, k, dtype=torch.int32).pin_memory()]
    # every rank reads back the rows of the queries it owns (together: the whole result, once)
    d2h = sum(t[wl.qlo:wl.qhi].numel() * t.element_size() for t in out_h)
    track_stream = pkg.HostTrackStream(eng, NCHUNK)
    h2d = track_stream.h2d_bytes(seq_h, mask_h) + gal_h.numel() * 4

    def e2e_eager():
        if world == 1:
            pkg.search_host(eng, seq_h, mask_h, gal_h, k, out=out_h, stream=track_stream, index_offset=wl.glo)
            return
        main = torch.cuda.current_stream(dev)
        track_stream.copy_stream.wait_stream(main)
        with torch.cuda.stream(track_stream.copy_stream):
            g_d = gal_h.to(dev, non_blocking=True)
            ev_g = torch.cuda.Event()
            ev_g.record(track_stream.copy_stream)
        main.wait_event(ev_g)
        g_d.record_stream(main)
        g = eng.prepare_gallery(g_d, index_offset=wl.glo)
        if wl.peer is not None:
            # slices are aggregated as they land; the kernel stores each descriptor into every rank's buffer
            slices = list(track_stream.uploads(seq_h, mask_h))
            for i, (lo, hi, s_d, m_d) in enumerate(slices):
                eng.sharded_aggregate(wl.peer, s_d, m_d, row0=wl.qlo + lo, last=i == len(slices) - 1)
            eng.sharded_score_topk(wl.peer, g)
            res = eng.sharded_merge(wl.peer)
        else:
            parts = [q_c for _, _, q_c in track_stream.chunks(seq_h, mask_h)]
            q = pkg.all_gather_rows(torch.cat(parts, 0))
            keep, wl.retr.gallery = wl.retr.gallery, g
            res = wl.retr.search_descriptors(q, k)
            wl.retr.gallery = keep
        for dst, src in zip(out_h, res):
            dst[wl.qlo:wl.qhi].copy_(src[wl.qlo:wl.qhi], non_blocking=True)

    # the e2e step as ONE graph too (H2D / D2H copies from pinned memory are graph nodes): the host enqueues one
    # item per step instead of ~25
    e2e_graph = None
    if os.environ.get("SEAM_BENCH_GRAPH", "1") != "0" and (world == 1 or wl.peer is not None):
        try:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(2):
                    e2e_eager()
            torch.cuda.current_stream(dev).wait_stream(side)
            barrier()
            e2e_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(e2e_graph, capture_error_mode="thread_local"):
                e2e_eager()
        except Exception as ex:                              # noqa: BLE001 -- capture problems: stay eager
            e2e_graph = None
            print(f"[bench] e2e graph capture failed, staying eager: {type(ex).__name__}: {ex}", file=sys.stderr)
            torch.cuda.synchronize()
    ok_flag = torch.tensor([1 if e2e_graph is not None else 0], device=dev)
    if world > 1:
        dist.all_reduce(ok_flag, op=dist.ReduceOp.MIN)       # all ranks replay a graph or none does
    if int(ok_flag) == 0:
        e2e_graph = None
    if e2e_graph is not None:
        # PCIe-bound at N = 1 (eager launches hide behind the copies, and the graph's copy nodes run a little slower),
        # launch-bound at N > 1: keep whichever form is faster on this box (decided outside the timed region)
        t_graph, t_eager = timed(e2e_graph.replay, 4, 2), timed(e2e_eager, 4, 2)
        if t_eager < t_graph:
            e2e_graph = None
    e2e_step = e2e_graph.replay if e2e_graph is not None else e2e_eager
    ms_e2e = timed(e2e_step, args.steps, warmup)
    clocks = sampler.stop()
    torch.cuda.synchronize()
    e2e_idx = out_h[2].clone()

    # ---- the scorer + top-k stage by itself, as it runs in the product (descriptors resident, ONE graph replay of
    # seam_score_topk: prep_queries + score_topk + rescore + exact_topk back to back, cold L2): the event-timed
    # per-kernel durations below each carry a few microseconds of launch gap that a replayed step does not have
    stage_graph_ms = None
    if world == 1 and os.environ.get("SEAM_BENCH_GRAPH", "1") != "0":
        q_res = eng.aggregate(wl.seq, wl.mask)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(3):
                eng.score_topk(q_res, wl.gallery, k)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize()
        g_stage = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_stage):
            stage_out = eng.score_topk(q_res, wl.gallery, k)
        stage_graph_ms = timed(g_stage.replay, args.steps, 3)
        del g_stage, stage_out, q_res

    # ---- per-kernel durations of the main configuration
    kern, launches_per_step = kernel_times(wl, args.steps)
    pairs_per_gpu = Q * Gs
    t_score, t_agg = kern["score"], kern["aggregate"]
    t_stage = sum(kern.get(n) or 0.0 for n in ("prep_queries", "score", "rescore", "exact"))
    traffic = traffic_agg = tensor_pipe_pct = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath) and world == 1:
        with open(tpath) as f:
            tj = json.load(f)
        traffic = tj.get("score_topk_kernel_dram_bytes_per_launch")
        tensor_pipe_pct = tj.get("score_topk_kernel_tensor_pipe_active_pct")
        traffic_agg = tj.get("aggregate_fused_warp_kernel_dram_bytes_per_launch")
    roofline = {
        "kernel": "score_topk_kernel", "bound": "tensor",
        "achieved": pairs_per_gpu * FLOP_PER_PAIR / (t_score * 1e-3) / 1e12, "peak": peaks["tflops"],
        "unit": "TFLOP/s", "traffic": traffic, "peak_source": peaks["source"] + " cuBLAS bf16 burst",
        "avg_launch_ms": t_score,
        "stage": "prep_queries + score_topk + rescore + exact_topk (SURVEY.md section 8(d): pairs / t_score+topk)",
        "stage_ms": t_stage, "stage_achieved": pairs_per_gpu * FLOP_PER_PAIR / (t_stage * 1e-3) / 1e12,
    }
    roofline["frac"] = roofline["achieved"] / roofline["peak"]
    roofline["stage_frac"] = roofline["stage_achieved"] / roofline["peak"]
    if tensor_pipe_pct is not None:      # ncu sm__pipe_tensor_subpipe_hmma_cycles_active (profiles/r2_final_ncu_score_topk_kernel.txt)
        roofline["tensor_pipe_active_pct_ncu"] = tensor_pipe_pct
    if stage_graph_ms:
        roofline["stage_graph_ms"] = stage_graph_ms
        roofline["stage_graph_frac"] = pairs_per_gpu * FLOP_PER_PAIR / (stage_graph_ms * 1e-3) / 1e12 / roofline["peak"]
        roofline["stage_note"] = ("stage_ms / stage_frac: sum of the four kernels' event-timed durations (eager launches); "
                                  "stage_graph_ms / stage_graph_frac: the same four kernels as one CUDA graph replay")
    agg_bytes = per * 1024 * (T + 1)
    roofline_agg = {
        "kernel": "aggregate_fused_warp_kernel<10> (the whole aggregation stage is this one kernel)", "bound": "hbm",
        "achieved": agg_bytes / (t_agg * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s", "traffic": traffic_agg,
        "peak_source": peaks["source"] + " copy", "avg_launch_ms": t_agg,
    }
    roofline_agg["frac"] = roofline_agg["achieved"] / roofline_agg["peak"]

    # ---- parity of the timed step's output (outside the timed region)
    res = [t.clone() for t in wl.step()]
    torch.cuda.synchronize()
    parity = parity_check(pkg, eng, wl, res, e2e_idx, weights, world, rank, dev)

    # ================================================================= the other BASELINE.json configurations
    sub = {}
    sub_steps = max(5, args.steps // 3)
    wl.free()
    del wl
    plan = [("cfg3", dict(Q=10000, T=4, G_total=50000, k=TOPK, seed=2, ragged=(2, 4)),
             "Multi-DeepFashion2-style: 10,000 queries x T in {2,3,4} (ragged) vs 50,000 items" +
             (f", gallery sharded x{world}" if world > 1 else " on one GPU"))]
    if world == 1:
        plan.append(("cfg4", dict(Q=100000, T=64, G_total=0, k=TOPK, seed=3),
                     "long-track aggregation stress: 100,000 tracks x 64 frames, aggregation only"))
        plan.append(("cfg5_per_gpu_shape", dict(Q=10000, T=10, G_total=125000, k=TOPK, seed=4),
                     "cfg 5 at its per-GPU shape on 8 GPUs: 10,000 queries x 10 frames vs a 125,000-row shard"))
    if world == 8:
        plan.append(("cfg5", dict(Q=10000, T=10, G_total=1000000, k=TOPK, seed=4),
                     "1M-item gallery x 10,000 queries, gallery sharded x8 (125,000 rows per GPU)"))
    if os.environ.get("SEAM_BENCH_CONFIGS", "1") == "0":
        plan = []
    for name, kw, desc in plan:
        w2 = Workload(pkg, eng, dev, world, rank, name, **kw)
        w2.capture()
        ms2 = timed(w2.step, sub_steps, 3, w2.stamps if w2.graph is not None else None)
        kern2, _ = kernel_times(w2, sub_steps)
        rec = stage_record(w2, kern2, ms2, peaks)
        rec["workload"] = desc
        sub[name] = rec
        w2.free()
        del w2

    if rank == 0:
        cpu = cpu_baseline() if world == 1 else None
        line = {
            "metric": METRIC, "value": Q * G / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (fp16-operand tcgen05 pass nominates candidates, every result re-scored in f32)",
            "data": "synthetic (planted matches, SURVEY.md section 8(d))",
            "config": {"workload": f"MovingFashion-scale eval: {Q} tracks x {T} frames vs {G} shop items "
                                   f"({Gs}/GPU), k={k}; aggregation + scoring + top-k",
                       "l2": "256 MiB buffer written between timed iterations",
                       "launch": parity.pop("_launch"),
                       "e2e_launch": "one CUDA graph replay per step (H2D, kernels, D2H)" if e2e_graph is not None else "eager",
                       "host_numa_node": numa,
                       "rank_alignment": rank_alignment,
                       "parallelism": parity.pop("_parallelism")},
            "queries_per_sec": Q / (ms * 1e-3),
            "e2e": {"value": Q * G / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e, "queries_per_sec": Q / (ms_e2e * 1e-3)},
            "gpu_launches": int(round(launches_per_step * args.steps)), "gpu_launches_per_step": launches_per_step,
            "clocks": clocks, "roofline": roofline, "roofline_aggregate": roofline_agg,
            "kernel_ms": kern, "parity_check": parity, "configs": sub,
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def parity_check(pkg, eng, wl, res, e2e_idx, weights, world, rank, dev):
    """The timed step's output against (i) the CPU oracle on a 32-query sample and (ii), for N > 1, the unsharded
    single-GPU search of the whole gallery; (iii) the end-to-end leg returned the same indices.  Rank 0 does the
    checking; the other ranks only contribute their gallery shards."""
    import torch.distributed as dist
    sc, mg, ix = res[-3:]
    launch = wl.launch_note()
    par = "single GPU"
    if world > 1:
        par = (f"gallery sharded x{world}, tracks aggregated and lists merged by the rank that owns the query; exchange: " +
               ("stores from inside the kernels into peer-mapped buffers + flag words (NVLink), no collective" +
                ("; descriptors by NVSwitch multicast (one store per row reaches every rank)" if wl.peer.multicast else "")
                if wl.peer is not None else "NCCL all-gathers" + wl.peer_note))
    out = {"_launch": launch, "_parallelism": par}
    g_full = wl.gal
    if world > 1:
        shards = [torch.empty_like(wl.gal) for _ in range(world)] if wl.G % world == 0 else None
        if shards is not None:
            dist.all_gather(shards, wl.gal)
            g_full = torch.cat(shards, 0)
    if rank != 0:
        return out
    from oracle import seam_oracle as so
    w_cpu = {kk: v.cpu() for kk, v in weights.items()}
    n = 32
    sample = torch.arange(0, wl.Q, wl.Q // n)[:n]
    mask_s = torch.zeros(n, 1 + wl.T, dtype=torch.bool)
    ref_q, _ = so.aggregate_tracks(wl.seq[:, sample].cpu(), mask_s, w_cpu)
    x5 = so.pair_logits(ref_q, g_full.cpu(), w_cpu, chunk=4)
    d_full = so.logit_margin(x5)
    got = ix[sample].cpu().long()
    d_at = torch.gather(d_full, 1, got)
    err = float((mg[sample].cpu() - d_at).abs().max())
    order = torch.argsort(d_full, dim=1, descending=True, stable=True)[:, : wl.k]
    differs = order != got
    ties_ok = bool(((torch.gather(d_full, 1, order) - d_at).abs()[differs] <= 2 * TOL_MARGIN).all()) if differs.any() else True
    planted_in_topk = float((ix.cpu().long() == torch.arange(wl.Q)[:, None]).any(1).float().mean())
    out.update({"oracle_sample_queries": n, "max_abs_margin_err": err, "margin_tolerance": TOL_MARGIN,
                "topk_identical_up_to_ties": bool(err <= TOL_MARGIN and ties_ok),
                "rows_differing_from_oracle_order": int(differs.any(1).sum()),
                "planted_match_in_topk_frac": planted_in_topk,
                "planted_match_note": "random-init `last` (SURVEY 8(d): module default init): the class-1 score is not a "
                                      "similarity, so the planted rows exercise cancellation in the expanded form, not top-1",
                "e2e_indices_equal_device_run": bool(torch.equal(e2e_idx[wl.qlo:wl.qhi], ix.cpu()[wl.qlo:wl.qhi]))})
    if world > 1 and g_full is not wl.gal:
        s1, m1, i1 = pkg.search(eng, wl.seq, wl.mask, g_full, wl.k)
        out["sharded_equals_unsharded"] = bool(torch.equal(i1, ix) and torch.equal(m1, mg) and torch.equal(s1, sc))
    out["ok"] = bool(out["topk_identical_up_to_ties"] and out["e2e_indices_equal_device_run"] and
                     out.get("sharded_equals_unsharded", True))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (CUDA path)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to the CUDA path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
