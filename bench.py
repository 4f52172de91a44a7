#!/usr/bin/env python
"""Learner throughput benchmark (BASELINE.json metric: learner sequences/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--channels C] [--fast] [--impl reference] [--dump-outputs DIR]

One "step" = one learner update on one batch of 64 replay sequences (b/l/f = 40/40/5 -> 85 frames
of C x 84 x 84 u8 each):

  value  : HBM-resident pipeline   K3 sample -> K4 gather -> K1 unroll(online+target) -> K2 TD ->
           K1b BPTT -> [gradient exchange over NVLink, N > 1] -> K5 clip+Adam -> K3 priority update
           (worker.Learner.update_from_replay; the priority update and the next batch's sample + gather run on a second
           stream under the BPTT recurrence -- same operation order on the tree, bit-identical results; the strictly
           sequential loop is timed as well and reported as `sequential_sampling`)
  e2e    : the same update through the reference-facing call with HOST buffers: a 14-tuple in pinned host
           memory (worker.py:219-238) -> H2D -> update -> priorities + loss back to the host
           (worker.Learner.update_from_batch)

Prints ONE JSON line (rank 0).  DESIGN.md "Measurement" defines every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

A = 9                      # MsPacman action count (train.py:22 takes it from the env)
B = 64                     # config.batch_size
BURN, LEARN, FWD = 40, 40, 5
T = BURN + LEARN + FWD
BLOCK_LEN = 400
TREE_CAPACITY = 1 << 20    # BASELINE config #3: sum tree over 2^20 sequence slots
NUM_BLOCKS = int(os.environ.get("R2D2_BENCH_BLOCKS", "128"))   # frame store: 128 blocks x 441 frames (1.6 GB at C=4), far larger than L2


def flops_per_sequence(C: int) -> float:
    """Algorithmic FLOPs (2*MAC) of one sequence's unroll fwd (2 nets) + bwd, SURVEY.md 8(d)."""
    enc = 2 * (819_200 * C + 2_654_208 + 1_806_336 + 1_605_632)
    lstm = 2 * 4 * 512 * (512 + A + 1 + 512)
    head = 2 * (2 * 512 * 512 + 512 * A + 512)
    fwd = 2 * (T * enc + T * lstm) + 3 * LEARN * head
    enc_b = 2 * (2 * (2_654_208 + 1_806_336 + 1_605_632) + 819_200 * C)       # dgrad+wgrad, no conv1 dgrad
    bwd = (BURN + LEARN) * (enc_b + 2 * lstm) + LEARN * 2 * head
    return float(fwd + bwd)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], tflops=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, tflops=1400.0, source="fallback")


class ClockSampler(threading.Thread):
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.samples.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        ok = [s for s in self.samples if len(s) >= 6]
        sm = [float(s[0]) for s in ok if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in ok if s[1].replace(".", "").isdigit()]
        reasons = set()
        for s in ok:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- reference arm
def reference_available() -> bool:
    from oracle import ref_harness
    return ref_harness.available()


def reference_learner_times(C: int, steps: int, warmup: int, sample_B: int, device: str, thread_candidates=None, tail_1thread: int = 0):
    """Drive the UNMODIFIED reference `worker.Learner.run` (worker.py:318-381) on synthetic 14-tuples of `sample_B`
    sequences and return per-update wall times (interval between successive priority_queue.put calls, worker.py:369).

    The reference is imported from baseline/_ref (a verbatim copy of the upstream files made by __graft_entry__.build();
    /root/reference in the build container) with the two shims of SURVEY.md 8c (gym stub, int64 accumulator).  C = 4 needs
    conv1 with 4 input channels, which model.py:40 hard-codes to 1: that one layer is re-instantiated (labelled).
    device 'cpu' relies on CUDA being hidden from the process (worker.py:283 picks cuda whenever it is visible)."""
    import queue

    from oracle import ref_harness
    from r2d2_b200.synthetic import reference_tuple, synthetic_batch
    ref = ref_harness.load()
    assert (device == "cuda") == torch.cuda.is_available(), "reference device is chosen by torch.cuda.is_available() (worker.py:283)"
    torch.manual_seed(0)
    net = ref.model.Network(A, obs_shape=(C, 84, 84))
    if C != 1:
        net.feature[0] = torch.nn.Conv2d(C, 32, 8, 4)
    total = warmup + steps + tail_1thread
    ref.config.training_steps = total
    batches = [reference_tuple(synthetic_batch(sample_B, A, BURN, LEARN, FWD, channels=C, seed=s)) for s in (0, 1)]
    stamps, threads_used = [], []
    cands = list(thread_candidates or [])
    state = {"best": None, "trial": []}

    class PQ:
        def put(self, item):
            if device == "cuda":
                torch.cuda.synchronize()
            now = time.perf_counter()
            stamps.append(now)
            threads_used.append(torch.get_num_threads())
            k = len(stamps)                      # updates finished so far
            if device == "cpu" and cands:
                # warm-up updates 2.. try the candidate thread counts, the timed updates use the fastest
                if 1 <= k < warmup and k - 1 < len(cands):
                    torch.set_num_threads(cands[k - 1])
                elif k == warmup:
                    durs = np.diff(stamps)
                    tried = [(durs[i - 1], threads_used[i]) for i in range(1, k)]
                    state["best"] = min(tried)[1] if tried else torch.get_num_threads()
                    torch.set_num_threads(state["best"])
                elif k == warmup + steps and tail_1thread:
                    torch.set_num_threads(1)     # as shipped: train.py:13 pins torch to one thread

    learner = ref.worker.Learner(queue.Queue(), PQ(), net)
    learner.batched_data = [batches[i % 2] for i in range(total)]
    t0 = time.perf_counter()
    learner.run()                                # sleeps 2 s first (worker.py:321)
    durs = np.diff([t0 + 2.0] + stamps)
    return dict(timed=durs[warmup:warmup + steps], tail=durs[warmup + steps:], threads=state["best"] or torch.get_num_threads(),
                device=str(learner.device))


def port_learner_rate(C: int, steps: int, sample_B: int):
    """Fallback when the reference files are not present: the oracle port (oracle/learner.py) on the host cores."""
    import oracle.learner as ol
    from oracle import synth
    from oracle.learner import LearnerState, init_params, learner_update
    ol.LSTM_MODE = "packed"
    params = init_params(A, in_channels=C, seed=0)
    st = LearnerState(online={k: v.clone() for k, v in params.items()}, target={k: v.clone() for k, v in params.items()})
    batches = [synth.to_torch_batch(synth.synthetic_batch(sample_B, A, BURN, LEARN, FWD, channels=C, seed=s)) for s in (0, 1)]
    torch.set_num_threads(min(os.cpu_count() or 1, 16))
    learner_update(st, batches[0])
    t0 = time.perf_counter()
    for k in range(steps):
        learner_update(st, batches[k % 2])
    dt = (time.perf_counter() - t0) / steps
    return sample_B / dt, dt, torch.get_num_threads()


def reference_subprocess(device: str, steps: int, warmup: int, C: int):
    """Run `bench.py --impl reference` in a child process (CUDA hidden for the CPU arm) and return its JSON line."""
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--device", device, "--steps", str(steps),
           "--warmup", str(warmup), "--channels", str(C)]
    try:
        out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
        for ln in reversed(out.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        print(f"reference arm ({device}) printed no JSON: {out.stderr[-400:]}", file=sys.stderr)
    except Exception as e:                                           # the comparator must never take the product number down
        print(f"reference arm ({device}) failed: {e}", file=sys.stderr)
    return None


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    C = args.channels
    cores = os.cpu_count() or 1
    workload = f"configs[1]: learner update, b/l/f {BURN}/{LEARN}/{FWD} (T={T}), {C}x84x84 u8 frames, A={A}"
    if not reference_available():
        val, dt, threads = port_learner_rate(C, max(1, min(args.steps, 5)), 16)
        kind, sample, extra = "port", f"oracle port, 16-sequence sample per update, {threads} threads (reference files not found)", {}
        steps, warmup = max(1, min(args.steps, 5)), 1
    elif args.device == "cuda":
        r = reference_learner_times(C, args.steps, args.warmup, B, "cuda")
        dt = float(np.median(r["timed"]))
        val, kind, steps, warmup = B / dt, "reference", args.steps, args.warmup
        sample = f"full batch of {B} sequences per update on {r['device']} (stock PyTorch eager: cuDNN/cuBLAS), H2D of the batch inside the step as worker.py:331-334 does"
        extra = {"device": "cuda"}
    else:
        sample_B = 16
        cands = sorted({min(cores, n) for n in (8, 16, 32, 64)})
        r = reference_learner_times(C, args.steps, max(args.warmup, 2), sample_B, "cpu", cands, tail_1thread=1)
        dt = float(np.median(r["timed"]))
        val, kind, steps, warmup = sample_B / dt, "reference", args.steps, max(args.warmup, 2)
        one = sample_B / float(r["tail"][0]) if len(r["tail"]) else None
        sample = (f"each update = a {sample_B}-sequence sample of the batch-{B} workload through the unmodified reference "
                  f"worker.Learner.run (baseline/_ref) on the CPU, {r['threads']} of {cores} host threads (fastest of {cands} tried "
                  f"during warm-up); median of {args.steps} updates" + ("; conv1 re-instantiated with 4 input channels" if C != 1 else ""))
        extra = {"one_thread_value": one, "one_thread_note": "same sample, torch.set_num_threads(1) as train.py:13 ships, 1 update"}
    line = {"impl": "reference", "metric": "learner sequences/sec", "value": val, "unit": "sequences/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "channels": C},
            "cpu_baseline": {"value": val, "unit": "sequences/s", "cores": extra.get("threads", None) or (r["threads"] if kind == "reference" else 16),
                             "kind": kind, "sample": sample, **{k: v for k, v in extra.items() if k != "threads"}},
            "e2e": {"value": val, "unit": "sequences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------- our arm
def count_kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ours = other = 0
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA and "memcpy" not in ev.name.lower() and "memset" not in ev.name.lower():
            if "r2d2" in ev.name:
                ours += 1
            else:
                other += 1
    return ours, other


def kernel_times(fn, steps=3):
    """Per-kernel durations of `steps` warm learner steps (CUPTI via torch.profiler; no replay, no serialisation)."""
    import collections
    import re
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(steps):
            fn(i)
        torch.cuda.synchronize()
    agg = collections.OrderedDict()
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        name = re.sub(r"^void ", "", ev.name)
        name = re.sub(r"\(.*", "", name)[:140]
        a = agg.setdefault(name, [0, 0.0])
        a[0] += 1
        a[1] += ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
    tot = sum(a[1] for a in agg.values())
    lines = [f"{steps} steps: sum of kernel durations {tot / steps:.1f} us/step (CUPTI, warm)"]
    for k, a in sorted(agg.items(), key=lambda x: -x[1][1]):
        lines.append(f"{a[1] / steps:9.1f} us {a[0] / steps:6.1f} {100 * a[1] / tot:5.1f}%  {k}")
    return "\n".join(lines)


def kernel_timeline(fn, steps=3, profile_here=True):
    """Chronological list of the device activities of `steps` warm learner steps: start offset, duration, stream, name
    (CUPTI via torch.profiler).  Used to see which part of a data-parallel step is exposed; every rank runs the steps,
    rank 0 profiles."""
    import re
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    if not profile_here:
        if torch.distributed.is_initialized():
            torch.distributed.barrier()                   # the profiling ranks need seconds to attach CUPTI
        for i in range(steps):
            fn(i)
        torch.cuda.synchronize()
        return ""
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        if torch.distributed.is_initialized():
            torch.distributed.barrier()
        for i in range(steps):
            fn(i)
        torch.cuda.synchronize()
    evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    evs.sort(key=lambda e: e.time_range.start)
    t0 = evs[0].time_range.start
    lines = []
    for e in evs:
        name = re.sub(r"\(.*", "", re.sub(r"^void ", "", e.name))[:110]
        dur = e.device_time if hasattr(e, "device_time") else e.cuda_time
        lines.append(f"{e.time_range.start - t0:10.1f} us  +{dur:8.1f} us  {name}")
    return "\n".join(lines)


def run_ingest_mode(args, learner, replay, C, ms_step_plain):
    """BASELINE config #3: the learner + HBM replay + sum tree (2^20 slots) while `--actors` producers feed blocks through the
    pinned staging ring.  Runs the product's own Learner.run loop (prefetch thread packs blocks into pinned memory, the learner
    thread commits them: one async H2D per block on the ingest stream, priorities enter the tree at the next sample) for a
    fixed number of updates and reports learner throughput with ingest on, the achieved ingest rate and the slowdown against
    the ingest-free number.  Producers replay pre-generated synthetic actor blocks at a fixed rate (emulator and actor
    inference are outside the learner path; 8 CPU actors of the reference produce ~4 blocks/s, the default here is 50x that)."""
    import queue
    from r2d2_b200 import config
    from r2d2_b200.synthetic import synthetic_blocks
    from r2d2_b200.worker import BLOCK_MSG
    updates = max(200, 10 * args.steps)
    bq, pq = queue.Queue(256), queue.Queue()
    learner.batch_queue, learner.priority_queue = bq, pq
    learner.batched_data = []
    pool = synthetic_blocks(8, A, C, seed=4242, burn_in=BURN, learning=LEARN, forward=FWD, block_len=BLOCK_LEN)
    stop = threading.Event()
    sent = [0] * args.actors
    period = args.actors / float(args.ingest_blocks_per_s)

    def producer(i):
        k = i
        nxt = time.perf_counter() + period * i / args.actors
        while not stop.is_set():
            blk, prio = pool[k % len(pool)]
            try:
                bq.put((BLOCK_MSG, blk, prio, None), timeout=0.05)
                sent[i] += 1
                k += args.actors
            except queue.Full:
                pass
            nxt += period
            time.sleep(max(0.0, nxt - time.perf_counter()))

    def drain():
        while not stop.is_set():
            try:
                pq.get(timeout=0.05)
            except queue.Empty:
                pass

    feeding = threading.Event()
    _producer = producer

    def gated_producer(i):
        feeding.wait()
        _producer(i)

    start_updates = learner.num_updates
    warm = 30
    config.training_steps = start_updates + 2 * (warm + updates) + 10
    config.learning_starts = 0
    th = [threading.Thread(target=gated_producer, args=(i,), daemon=True) for i in range(args.actors)] + [threading.Thread(target=drain, daemon=True)]
    runner = threading.Thread(target=learner.run, daemon=True)
    for t in th:
        t.start()
    runner.start()

    def timed_window(first):
        while learner.num_updates < first + warm:
            time.sleep(0.002)
        torch.cuda.synchronize()
        u0, t0, y0 = learner.num_updates, time.perf_counter(), replay.ingested_bytes
        while learner.num_updates < first + warm + updates:
            time.sleep(0.002)
        torch.cuda.synchronize()
        u1, t1, y1 = learner.num_updates, time.perf_counter(), replay.ingested_bytes
        return (u1 - u0), (t1 - t0), (y1 - y0)

    n0, dt0, _ = timed_window(start_updates)                         # the same loop with the producers idle
    feeding.set()
    n1, dt1, nbytes = timed_window(start_updates + warm + updates)   # producers feeding
    stop.set()
    config.training_steps = 0                                         # lets Learner.run return
    runner.join(timeout=30)
    idle, fed = n0 * B / dt0, n1 * B / dt1
    return {"actors": args.actors, "updates_timed": n1, "value": fed, "unit": "sequences/s", "ms_per_step": 1e3 * dt1 / n1,
            "same_loop_without_ingest": idle, "relative_to_same_loop_without_ingest": fed / idle,
            "ingest_blocks_per_s": nbytes / replay.blob_bytes / dt1, "ingest_gb_per_s": nbytes / dt1 / 1e9, "block_bytes": replay.blob_bytes,
            "note": "worker.Learner.run loop timed by wall clock (it polls its queue and accumulates the loss between updates), first with "
                    f"idle producers, then with {args.actors} producers offering {args.ingest_blocks_per_s:g} blocks/s in total; blocks are packed "
                    "into pinned memory by the prefetch thread and copied on the ingest stream while the previous update runs"}


def last_update_outputs(learner, replay) -> dict:
    """What the replay update path leaves its caller after an update: that update's TD errors, priorities, Q values and
    loss, the online parameters after its optimizer step, and the sum tree's leaves after its priority update."""
    core, tree = learner.core, replay.tree
    torch.cuda.synchronize()
    rows = int(core.rows.item())
    leaf0 = tree.num_nodes // 2
    out = {"td": core.td[:rows], "priorities": core.prio, "q": core.q[:rows], "loss": core.loss_sum.double() / rows,
           "online_params": core.online.flat, "tree_leaves": tree.nodes_device()[leaf0:leaf0 + tree.capacity]}
    return {k: v.cpu().numpy() for k, v in out.items()}


def run_ours(args):
    import torch.distributed as dist
    from r2d2_b200 import _lib, config
    from r2d2_b200 import dist as r2dist
    from r2d2_b200.model import Network
    from r2d2_b200.replay import DeviceReplay
    from r2d2_b200.worker import Learner
    from r2d2_b200.synthetic import init_state_dict, reference_tuple, synthetic_batch, synthetic_blocks

    rank, world, local = r2dist.init_from_env("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    C = args.channels
    config.obs_shape = (C, 84, 84)
    if args.fast:
        args.precision = "fast"
    _lib.lib().r2d2_set_fast_math({"strict": 0, "fast": 1, "balanced": 2}[args.precision])

    model = Network(A, obs_shape=(C, 84, 84))
    model.load_state_dict(init_state_dict(A, in_channels=C, seed=0))
    learner = Learner(None, None, model, save_interval=10 ** 9, device=dev)
    learner._start_time = time.time()
    if world > 1:
        r2dist.broadcast_parameters(learner.core)
        exchange = None
        if os.environ.get("R2D2_DP_NCCL") != "1":                                 # our all-reduce kernels over NVLink peer memory (csrc/dp.cu)
            try:
                exchange = r2dist.PeerExchange(learner.core)
            except Exception as e:                                                # noqa: BLE001  (no symmetric memory on this box)
                print(f"[bench] rank {rank}: peer-memory exchange unavailable ({e!r}); falling back to NCCL", file=sys.stderr)
            ok = torch.tensor([1 if exchange is not None else 0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)                             # all ranks take the same path
            if int(ok.item()) == 0:
                exchange = None
        if exchange is None:                                                      # comparison arm: the same exchange on NCCL calls
            learner.is_weight_sync = r2dist.GlobalISWeights(dev, 0.6)             # importance weights of one global sampler
            learner.core.grad_hook = r2dist.make_overlapped_grad_hook(learner.core, is_sync=learner.is_weight_sync)
        else:
            learner.is_weight_sync = r2dist.PeerISWeights(exchange, 0.6)
            learner.core.pre_td_hook = learner.is_weight_sync.apply
            learner.core.grad_hook = r2dist.make_peer_grad_hook(learner.core, exchange)   # dense range overlaps the conv backward
        dp_exchange = "nccl" if exchange is None else ("peer-memory kernels, multimem" if exchange.multicast else "peer-memory kernels, p2p")
    else:
        dp_exchange = None

    # HBM replay shard of this rank: NUM_BLOCKS blocks, tree over 2^20 slots
    replay = DeviceReplay(NUM_BLOCKS * BLOCK_LEN, BLOCK_LEN, BURN, LEARN, FWD, A, (C, 84, 84), 512, 0.9, 0.6, B, device=dev,
                          seed=rank, tree_capacity=TREE_CAPACITY)
    distinct = synthetic_blocks(16, A, C, seed=1000 + rank, burn_in=BURN, learning=LEARN, forward=FWD, block_len=BLOCK_LEN)
    for i in range(NUM_BLOCKS):
        blk, prio = distinct[i % len(distinct)]
        replay.add(blk, prio, None)
    learner.replay = replay
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()                                             # ranks finish their set-up seconds apart

    tuples = [reference_tuple(synthetic_batch(B, A, BURN, LEARN, FWD, channels=C, seed=100 * rank + i), pinned=True) for i in range(3)]
    in_bytes = sum(v.numel() * v.element_size() for v in tuples[0] if isinstance(v, torch.Tensor))

    def step_resident(i):
        learner.update_from_replay()

    from collections import deque
    staged = deque([learner.prefetch(tuples[0])])

    tickets = deque()

    def step_e2e(i):
        # every step moves one full batch host -> device inside the timed region; like the reference's prefetch thread
        # (worker.py:309-316) the copy of batch i+1 is issued before batch i is trained on, on a copy stream.  As in
        # Learner.run, update i is launched before the host reads update i-1's priorities/loss (one D2H read per step):
        # enqueueing the 60 launches of an update overlaps the previous update instead of idling the GPU.
        staged.append(learner.prefetch(tuples[(i + 1) % len(tuples)]))
        tickets.append(learner.enqueue_update(staged.popleft()))
        if len(tickets) > 1:
            learner.collect(tickets.popleft())                  # priorities + loss of the previous update, host-synchronised

    def timed(fn, steps, warmup):
        for w in range(warmup):
            fn(w)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(steps):
            fn(warmup + k)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.barrier()
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / steps

    sampler = ClockSampler(local)
    sampler.start()
    ms_step_seq = None
    nccl_dp = world > 1 and dp_exchange == "nccl"                     # the NCCL hooks keep per-batch state in Python: sequential there
    learner.sample_ahead = False
    if not args.no_sample_ahead and not nccl_dp:
        learner.sample_ahead = False
        ms_step_seq = timed(step_resident, args.steps, args.warmup)   # plain sequential loop first (reported next to the headline)
        learner.sample_ahead = True                                   # priority update i / sample i+1 / gather i+1 under update i's backward
        for w in range(6):                                            # untimed: the second set of batch buffers gets its CUDA graph
            step_resident(w)                                          # (a key is captured the second time it is seen)
    ms_step = timed(step_resident, args.steps, args.warmup)
    outputs = last_update_outputs(learner, replay) if args.dump_outputs and rank == 0 else None
    ms_e2e = timed(step_e2e, args.steps, args.warmup)
    sampler.stop_flag = True

    ms_unroll = None
    if world == 1:                                 # K1 + K1b only, on the launching stream, for the roofline
        core = learner.core
        b0 = dict(replay.batch, obs=None)          # frames: whatever the last gather staged (obs=None: no u8 -> s2d conversion pass)

        def unroll_only(i):
            core.compute_forward(b0)
            core.backward(core.dq)
        for w in range(3):
            unroll_only(w)
        torch.cuda.synchronize()
        # the same launches as one CUDA graph (as the update itself runs them): no host enqueue gaps inside the timed region
        ug = None
        if core.use_graph:
            try:
                ug = torch.cuda.CUDAGraph()
                with torch.cuda.graph(ug):
                    unroll_only(0)
            except Exception as e:                 # noqa: BLE001
                print(f"[bench] unroll group not captured ({e!r}); timing eager launches", file=sys.stderr)
                ug = None
                torch.cuda.synchronize()
        if ug is not None:
            ms_unroll = timed(lambda i: ug.replay(), max(5, args.steps // 2), 3)
        else:                                      # R2D2_CUDA_GRAPH=0 (profiler runs): eager launches
            ms_unroll = timed(unroll_only, max(5, args.steps // 2), 3)

    if args.kernel_times and world == 1:
        text = kernel_times(step_resident)
        os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
        with open(os.path.join(ROOT, "gpurun_out", "kernel_times.txt"), "w") as f:
            f.write(text + "\n")
        print(text, file=sys.stderr)
    if args.timeline:
        text = kernel_timeline(step_resident, profile_here=rank < 2)
        if rank < 2:
            os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
            with open(os.path.join(ROOT, "gpurun_out", f"timeline_n{world}" + ("" if rank == 0 else f"_rank{rank}") + ".txt"), "w") as f:
                f.write(text + "\n")
    step_resident(0)                                           # (re-)primes the sample-ahead pipeline after the host-batch phase
    ours, other = count_kernels(lambda: step_resident(0))      # every rank runs it: the step contains the all-reduce
    if rank == 0:
        peaks = measured_peaks()
        value = world * B / (ms_step * 1e-3)
        e2e = world * B / (ms_e2e * 1e-3)
        line = {"metric": "learner sequences/sec", "value": value, "unit": "sequences/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": {"strict": "bf16x3 split products (fp32-equivalent), fp32 accumulate",
                          "balanced": "bf16 activations x bf16x2 weights in the encoder, bf16x3 elsewhere, fp32 accumulate",
                          "fast": "bf16 products, fp32 accumulate"}[args.precision],
                "data": "synthetic",
                "config": {"workload": f"configs[1]: 1xB200 learner per rank, batch {B}/GPU, b/l/f {BURN}/{LEARN}/{FWD} (T={T}), "
                                       f"{C}x84x84 u8 frames, A={A}, HBM replay of {NUM_BLOCKS} blocks, sum tree 2^20",
                           "channels": C, "global_batch": world * B, "parallelism": f"dp{world}", "exchange": dp_exchange, "precision": args.precision,
                           "host": f"staging copies on high-priority streams; CUDA_DEVICE_MAX_CONNECTIONS={os.environ.get('CUDA_DEVICE_MAX_CONNECTIONS')} (binding the process to the GPU's NUMA node was measured and made the copies slower on this pool: not done)",
                           "sampling": ("priority update of update i, sampling and gather of batch i+1 on a second stream while update i's "
                                        "backward pass runs (same tree operation sequence and bit-identical results as the sequential "
                                        "loop); the gather's copy CTAs are steered onto the SMs the BPTT recurrence leaves idle")
                                       if ms_step_seq is not None else "sequential: sample -> update -> priority update",
                           "l2": f"inputs larger than L2: batches are gathered from a {NUM_BLOCKS * replay.blob_bytes / 1e9:.1f} GB HBM "
                                 f"block store; ~1 GB of activations streamed per step"},
                "clocks": sampler.summary(),
                "e2e": {"value": e2e, "unit": "sequences/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": in_bytes,
                        "d2h_bytes_per_step": B * 4 + 8},
                "gpu_launches": ours, "other_launches": other}
        if ms_step_seq is not None:                # the strictly sequential loop (every sample sees the priorities of the update before it)
            line["sequential_sampling"] = {"ms_per_step": ms_step_seq, "value": world * B / (ms_step_seq * 1e-3), "unit": "sequences/s"}
        if ms_unroll is not None:
            fl = flops_per_sequence(C) * B
            ach = fl / (ms_unroll * 1e-3) / 1e12
            traffic = None
            tpath = os.path.join(ROOT, "profiles", "r02_unroll_traffic.json")
            if os.path.exists(tpath) and C == 4 and args.precision == "strict":
                with open(tpath) as f:
                    traffic = json.load(f)["bytes"]        # dram bytes of the same launches from the committed ncu pass
            line["roofline"] = {"bound": "tensor", "achieved": ach, "peak": peaks["tflops"], "unit": "TFLOP/s",
                                "frac": ach / peaks["tflops"], "traffic": traffic, "peak_source": peaks["source"],
                                "kernel": "K1+K1b unroll group (forward online+target, BPTT backward): winconv/winwgrad/umma3/umma2/rec2_fwd/rec2_bwd launches",
                                "ms": ms_unroll, "algorithmic_gflop_per_launch": fl / 1e9}
        if world == 1 and args.actors > 0:
            line["ingest"] = run_ingest_mode(args, learner, replay, C, ms_step)
        if world == 1 and not args.no_cpu_baseline:
            torch.cuda.synchronize()
            cpu = reference_subprocess("cpu", 3, 3, C)               # the reference's CPU learner on this box's host cores
            if cpu is not None:
                line["cpu_baseline"] = cpu["cpu_baseline"]
            eager = reference_subprocess("cuda", 5, 2, C)            # the reference's own learner on this GPU (stock PyTorch eager)
            if eager is not None:
                line["vs_cuda_eager"] = {"reference_value": eager["value"], "unit": "sequences/s", "ratio": value / eager["value"],
                                         "e2e_ratio": e2e / eager["value"], "sample": eager["cpu_baseline"]["sample"],
                                         "ms_per_step": eager["ms_per_step"]}
        if outputs is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in outputs.items():
                np.save(os.path.join(args.dump_outputs, f"{name}.npy"), arr)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--channels", type=int, default=4, help="frame channels: 4 = BASELINE.json shape, 1 = reference obs_shape")
    ap.add_argument("--precision", default="strict", choices=["strict", "balanced", "fast"],
                    help="strict: bf16x3 split products everywhere; balanced: hi+lo only for encoder weight operands; fast: plain bf16")
    ap.add_argument("--fast", action="store_true", help="same as --precision fast")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--device", default="cpu", choices=["cpu", "cuda"],
                    help="--impl reference only: cpu = the reference's CPU learner (the driver's reference arm), cuda = the reference's own "
                         "learner on this GPU through stock PyTorch eager (on-box comparator)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--actors", type=int, default=0,
                    help="BASELINE config #3 (N = 1 only): also run the learner with this many block producers feeding the HBM replay "
                         "through the pinned staging ring and report throughput with ingest on (adds an `ingest` object to the line)")
    ap.add_argument("--ingest-blocks-per-s", type=float, default=200.0, help="total block rate the producers offer (400-step blocks)")
    ap.add_argument("--no-sample-ahead", action="store_true",
                    help="time the strictly sequential loop only (default: batch i+1 is sampled and gathered while update i runs)")
    ap.add_argument("--timeline", action="store_true", help="also write gpurun_out/timeline_n<N>.txt (chronological device activities of 3 steps; ranks 0 and 1)")
    ap.add_argument("--kernel-times", action="store_true", help="also write gpurun_out/kernel_times.txt (per-kernel CUPTI durations)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed replay update computed (td, priorities, q, loss, online_params, tree_leaves) "
                         "as DIR/<name>.npy, float32 or float64, about 25 MB; inputs are seeded, so runs with the same arguments "
                         "can be compared output for output")
    args = ap.parse_args()
    # more hardware work queues than the default 8: the staging copies of the next batch must never share a queue with (and so
    # wait behind) the CUDA graph of the running update.  Must be set before CUDA is initialised.
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
    if args.impl == "reference":
        if args.device == "cpu":
            os.environ["CUDA_VISIBLE_DEVICES"] = ""                   # worker.py:283 takes cuda whenever it is visible
        run_reference(args)
    else:
        args.warmup = max(args.warmup, 3)
        run_ours(args)


if __name__ == "__main__":
    main()
