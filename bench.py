#!/usr/bin/env python
"""bench.py -- RNN-T loss+grad throughput on B200 (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c4|c5mb]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input: loss + dense gradient
w.r.t. log_probs for all lattices of the batch (what the reference's forward call produces,
pytorch_binding/benchmark.py:36-43), log_softmax excluded.

  value      lattices/s, inputs resident in HBM, CUDA events over exactly K steps, max over ranks.
             Buffers rotate over R input sets and R live outputs so that consecutive steps never
             touch the same lines (aggregate footprint >> 126 MB L2).
  e2e        same metric through the public Python API (warp_rnnt_b200.rnnt_loss + backward) with
             HOST (pinned) inputs: H2D copy of the step's inputs and a D2H read of the loss inside
             the timed region.
  roofline   algorithmic bytes per launch (SURVEY.md 8d: 4*N*T*U*V grad write + 8*N*T*U log-prob
             reads + 4*N*(U-1) + 12*N) / measured step time, against MEASURED_PEAKS.json hbm_gbs.
  cpu_baseline  the CPU oracle port (oracle/rnnt_oracle.c, f32 flavour, OpenMP over lattices) timed on
             this box's host cores on a bounded sample of the same workload (rank 0, N=1 only).

--dump-outputs DIR: after the timed steps, rank 0 writes what its last timed step returned to the caller as
float32 .npy files: DIR/loss.npy (the reduced loss) and DIR/grad.npy (the gradient w.r.t. the step's input); an
output of more than 8M elements is written as a fixed sample of 8M of them (flat positions drawn with seed 0,
ascending), so at most 64 MB in all.  The inputs are seeded: two builds run with the same arguments can be
compared file by file.

Multi-GPU (launched by torchrun): every rank runs the same per-GPU workload on its own shard
(weak scaling, no data-path collective) and the scalar loss is all-reduced over NCCL each step.

--impl reference: the UNMODIFIED reference kernels (oracle/_ref/warp_rnnt_ref_C.so, built from
/root/reference by oracle/build_ref.py) through the reference's own operator API on the GPU, same
harness; falls back to the CPU oracle port when that extension or a GPU is not available.
"""
import argparse
import contextlib
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

WORKLOADS = {
    # name: (N per GPU, T, U, V, API mode, ragged lengths, description)
    "c2": (128, 150, 40, 28, "dense", False, "N=128 T=150 U=40 V=28 gather=False loss+grad (BASELINE configs[1])"),
    "c2g": (128, 150, 40, 28, "gather", False, "N=128 T=150 U=40 V=28 gather=True (memory-saving mode of configs[1])"),
    "c3": (32, 150, 20, 5000, "gather", False, "N=32 T=150 U=20 V=5000 gather=True large-vocab (BASELINE configs[2])"),
    "c3d": (32, 150, 20, 5000, "dense", False, "N=32 T=150 U=20 V=5000 gather=False (dense variant of configs[2])"),
    "c4": (64, 1500, 300, 50, "compact", True,
           "N=64 T=1500 U=300 V=50 compact=True long-utterance, ragged lengths (BASELINE configs[3])"),
    "c4d": (64, 1500, 300, 50, "dense", False, "N=64 T=1500 U=300 V=50 dense layout, full lengths (variant of configs[3])"),
    "c5mb": (32, 600, 150, 1024, "dense", False,
             "N=32 T=600 U=150 V=1024 = one micro-batch of BASELINE configs[4] (256 lattices/GPU as 8 x 32)"),
    # next rows (SURVEY.md 8f): bf16 I/O and the loss straight from logits -- reported BESIDE the f32 headline
    "c2b": (128, 150, 40, 28, "bf16", False, "N=128 T=150 U=40 V=28, bfloat16 log_probs in / bfloat16 gradient out"),
    "c5mbb": (64, 600, 150, 1024, "bf16", False,
              "N=64 T=600 U=150 V=1024 bfloat16 i/o = a double-size micro-batch of BASELINE configs[4]"),
    "c2l": (128, 150, 40, 28, "logits", False,
            "N=128 T=150 U=40 V=28 from un-normalised logits (log_softmax fused; gradient w.r.t. logits)"),
    "c5mbl": (32, 600, 150, 1024, "logits", False,
              "N=32 T=600 U=150 V=1024 from un-normalised logits = one micro-batch of BASELINE configs[4], log_softmax fused"),
}
API_CALL = {"dense": "warp_rnnt_b200.rnnt_loss(x, ..., reduction='sum').backward()",
            "gather": "warp_rnnt_b200.rnnt_loss(x, ..., reduction='sum', gather=True).backward()",
            "compact": "warp_rnnt_b200.rnnt_loss(x, ..., reduction='sum', compact=True).backward() inside compact_hints(T, U)",
            "bf16": "warp_rnnt_b200.rnnt_loss(x_bf16, ..., reduction='sum').backward()",
            "logits": "warp_rnnt_b200.rnnt_loss_from_logits(logits, ..., reduction='sum').backward()"}


def b_alg(N, T, U, V, cells=None, mode="dense"):
    """SURVEY.md 8(d): dense gradient write + the two log-probs per cell + labels + lengths/costs.  Ragged layouts:
    `cells` = sum xn*(yn+1) replaces N*T*U.  bf16 i/o: 2-byte elements.  from logits: the whole tensor must be read
    (the normaliser needs every logit) and the gradient is dense: 8 bytes per element."""
    c = N * T * U if cells is None else cells
    small = 4 * N * (U - 1) + 12 * N
    if mode == "bf16":
        return 2 * c * V + 4 * c + small
    if mode == "logits":
        return 8 * c * V + small
    return 4 * c * V + 8 * c + small


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def make_host_inputs(N, T, U, V, seed, ragged=False, compact=False, dtype=None):
    """The reference's recipe (pytorch_binding/benchmark.py:11-27): randn -> log_softmax, labels in [1,V), full
    lengths; ragged = the random-length recipe of benchmark2.py:81-85 (lengths in [T/2,T] / [U/2,U), shifted so the
    maxima hit T / U-1); compact = the ragged concat of test.py:291-299.  Pinned host tensors."""
    g = torch.Generator().manual_seed(seed)
    ys = torch.randint(1, V, (N, U - 1), dtype=torch.int, generator=g)
    if ragged:
        xn = torch.randint(T // 2, T + 1, (N,), dtype=torch.int, generator=g)
        yn = torch.randint(U // 2, U, (N,), dtype=torch.int, generator=g)
        xn = xn + T - xn.max()
        yn = yn + (U - 1) - yn.max()
    else:
        xn = torch.full((N,), T, dtype=torch.int)
        yn = torch.full((N,), U - 1, dtype=torch.int)
    if compact:
        cells = int((xn.long() * (yn.long() + 1)).sum())
        xs = torch.log_softmax(torch.randn((cells, V), dtype=torch.float32, generator=g), dim=-1)
        ys = torch.cat([ys[i, :yn[i]] for i in range(N)]).contiguous()
    else:
        xs = torch.log_softmax(torch.randn((N, T, U, V), dtype=torch.float32, generator=g), dim=-1)
    if dtype is not None:
        xs = xs.to(dtype)
    pin = torch.cuda.is_available()
    return tuple(t.pin_memory() if pin else t for t in (xs, ys, xn, yn))


class ClockSampler:
    """SM clock / throttle reasons via NVML while the GPU is under load."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                 "sw_thermal_slowdown": 0x20, "hw_power_brake_slowdown": 0x80, "sync_boost": 0x10}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t is not None:
            self._t.join(timeout=1.0)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def cpu_oracle_rate(N, T, U, V, budget_s=8.0, threads=None):
    """lattices/s of the CPU oracle port (f32 flavour = the reference's arithmetic) on this box."""
    from oracle import oracle
    if threads:
        oracle.set_threads(threads)
    n_cpu = min(N, 16) if N * T * U * V > 2e8 else N             # bounded sample of the same workload
    xs, ys, xn, yn = [t.numpy() for t in make_host_inputs(n_cpu, T, U, V, seed=N)]
    oracle.dense(xs[:2], ys[:2], xn[:2], yn[:2], dtype="f32")           # warm (loads the library)
    reps, t0 = 0, time.perf_counter()
    while True:
        oracle.dense(xs, ys, xn, yn, dtype="f32")
        reps += 1
        el = time.perf_counter() - t0
        if el >= budget_s or reps >= 200:
            break
    # BASELINE configs[0]: one lattice through the numpy (awni ref_transduce style) restatement
    np_ms = None
    if T * U <= 10000:
        t1 = time.perf_counter()
        oracle.ref_transduce_np(xs[0].astype(np.float64), ys[0])
        np_ms = (time.perf_counter() - t1) * 1e3
    return {"value": n_cpu * reps / el, "unit": "lattices/s", "cores": oracle.num_threads(), "kind": "port",
            "sample": "%d x %d lattices of %s (dense layout, full lengths) through oracle/rnnt_oracle.c (f32, OpenMP over "
                      "lattices), %.1f s" % (reps, n_cpu, "T=%d U=%d V=%d" % (T, U, V), el),
            "numpy_ref_transduce_ms_per_lattice": np_ms, "host_cpus": os.cpu_count()}


def config_dict(workload, desc, N, T, U, V, world, R, footprint_mb):
    """Identical for both arms (the driver compares the dicts)."""
    return {"workload": "%s: %s" % (workload, desc), "lattices_per_gpu": N, "T": T, "U": U, "V": V,
            "global_batch": N * world, "parallelism": "batch-sharded x%d, one scalar-loss all-reduce per step" % world,
            "l2_protocol": "%d rotating input sets + %d live outputs (%.0f MB) > L2" % (R, R, footprint_mb)}


def rotation(per_set_bytes):
    return int(max(2, min(6, (700e6 // per_set_bytes) + 1))) if per_set_bytes < 4e9 else 1


def dump_outputs(dirname, outputs, max_elems=8 << 20):
    """--dump-outputs: every tensor of `outputs` as dirname/<name>.npy in float32, a fixed sample of max_elems
    elements (flat positions from seed 0, ascending) when it is larger."""
    os.makedirs(dirname, exist_ok=True)
    for name, t in outputs.items():
        a = t.detach()
        if a.numel() > max_elems:
            idx = torch.randint(a.numel(), (max_elems,), generator=torch.Generator().manual_seed(0)).sort().values
            a = a.reshape(-1)[idx.to(a.device)]
        np.save(os.path.join(dirname, name + ".npy"), a.float().cpu().numpy())


def timed(fn, steps, world, dist, dev, after=None):
    """CUDA events around exactly `steps` calls (+ `after()`, e.g. waiting for the last in-flight all-reduce), barrier +
    synchronize on both sides, max over ranks -> ms."""
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(steps):
        fn(i)
    if after is not None:
        after()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        dist.barrier()
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--lse", default="auto", choices=["auto", "fast", "exact"])
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 20)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time the eager python API instead of CUDA-graph replays")
    ap.add_argument("--no-c5", action="store_true", help="skip the cfg-5 block of multi-GPU runs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss and the gradient of the last timed step to DIR/*.npy (float32; gradients "
                         "of more than 8M elements as a fixed seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    N, T, U, V, mode, ragged, desc = WORKLOADS[args.workload]
    have_cuda = torch.cuda.is_available()

    if args.impl == "reference":
        return run_reference(args, rank, world, N, T, U, V, mode, ragged, desc, have_cuda)
    if not have_cuda:
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path (use --impl reference for the CPU oracle)")

    import torch.distributed as dist
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    import warp_rnnt_b200 as w
    from warp_rnnt_b200 import parallel
    w.set_lse_mode(args.lse)

    # R rotating input sets, R live outputs: no step re-touches lines of the previous ones
    esz = 2 if mode == "bf16" else 4
    per_set = 2 * esz * N * T * U * V
    R = rotation(per_set)
    host = [make_host_inputs(N, T, U, V, seed=1000 * rank + N + i, ragged=ragged, compact=(mode == "compact"),
                             dtype=torch.bfloat16 if mode == "bf16" else None)
            for i in range(R)]
    sets = [tuple(t.to(dev, non_blocking=True) for t in h) for h in host]
    cells = [int((h[2].long() * (h[3].long() + 1)).sum()) for h in host]
    for s in sets:
        s[0].requires_grad_(True)
    torch.cuda.synchronize()

    # ---- the step = what a user of the reference's API calls (loss + gradient w.r.t. log_probs).  N > 1: every rank
    # runs it on its own shard; the gradients need only the LOCAL loss (the weights are known up front), so the one
    # collective -- the scalar all-reduce -- is issued asynchronously after the step and overlaps the next one
    # (parallel.all_reduce_loss_async); it is waited for one step later, inside the timed region.
    def api_step(s):
        x, ys, xn, yn = s
        x.grad = None
        if mode == "compact":
            with w.compact_hints(T, U):                 # sync-free forward (no D2H shape validation)
                loss = w.rnnt_loss(x, ys, xn, yn, reduction="sum", compact=True)
        elif mode == "logits":
            loss = w.rnnt_loss_from_logits(x, ys, xn, yn, reduction="sum")
        else:
            loss = w.rnnt_loss(x, ys, xn, yn, reduction="sum", gather=(mode == "gather"))
        loss.backward()
        return loss

    pending = []

    def reduce_async(loss):
        if world > 1:
            pending.append(parallel.all_reduce_loss_async(loss.detach()))
            if len(pending) > 1:
                pending.pop(0).wait()

    def drain():
        while pending:
            pending.pop(0).wait()

    sampler = ClockSampler(local_rank)
    sampler.start()
    # eager warm-up on every set: primes the caching allocator, NCCL and the lazy per-device state
    for i in range(R + 2):
        reduce_async(api_step(sets[i % R]))
    drain()
    torch.cuda.synchronize()

    # ---- CUDA graphs of the API step, one per input set (kills the python / autograd dispatch time, which at cfg 2
    # is larger than the 45 us kernel; the reference's users do the same: "CUDA streams and graphs")
    graphs, launches_per_step, graph_note = None, None, "eager python API"
    if not args.no_graph:
        try:
            graphs = []
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for s in sets:
                    api_step(s)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            for s in sets:
                g = torch.cuda.CUDAGraph()
                s[0].grad = None
                n0 = w._C.launch_count()
                with torch.cuda.graph(g):
                    loss = api_step(s)
                launches_per_step = int(w._C.launch_count() - n0)
                graphs.append((g, loss, s))
            graph_note = "CUDA-graph replay of the python API step (one graph per input set)"
        except Exception as e:                            # capture not possible here: fall back to eager
            graphs, graph_note = None, "eager python API (graph capture failed: %s)" % (str(e).splitlines()[0][:120])
            torch.cuda.synchronize()

    if graphs is not None:
        def step(i):
            g, loss, _ = graphs[i % R]
            g.replay()
            reduce_async(loss)
    else:
        eager_loss = [None]

        def step(i):
            eager_loss[0] = api_step(sets[i % R])
            reduce_async(eager_loss[0])

    for i in range(args.warmup):
        step(i)
    drain()
    n0 = w._C.launch_count()
    ms = timed(lambda i: step(args.warmup + i), args.steps, world, dist, dev, after=drain)
    if args.dump_outputs and rank == 0:
        last = (args.warmup + args.steps - 1) % R
        dump_outputs(args.dump_outputs, {"loss": graphs[last][1] if graphs is not None else eager_loss[0],
                                         "grad": sets[last][0].grad})
    launches = (launches_per_step * args.steps) if graphs is not None else int(w._C.launch_count() - n0)
    ms_per_step = ms / args.steps
    value = N * world * args.steps / (ms * 1e-3)

    # ---- extra information (N=1): eager API, operator-level call, the opt-in short LSE chain
    extra = {}
    if world == 1:
        if graphs is not None:
            for i in range(3):
                api_step(sets[i % R])
            extra["api_eager_ms_per_step"] = timed(lambda i: api_step(sets[i % R]), min(args.steps, 30), 1, dist, dev) / min(args.steps, 30)
        if mode == "logits":
            # the same result the reference's way: torch.log_softmax, then the loss, autograd through both
            def unfused(i):
                x = sets[i % R][0]
                x.grad = None
                w.rnnt_loss(torch.log_softmax(x, -1), *sets[i % R][1:], reduction="sum").backward()
            for i in range(3):
                unfused(i)
            extra["unfused_ms_per_step"] = timed(unfused, min(args.steps, 20), 1, dist, dev) / min(args.steps, 20)
            extra["unfused_call"] = "warp_rnnt_b200.rnnt_loss(torch.log_softmax(logits, -1), ..., reduction='sum').backward(), eager"
        if mode == "dense":
            keep = [None] * R

            def op_step(i):
                s = sets[i % R]
                keep[i % R] = w._C.rnnt_loss(s[0].detach(), s[1], s[2], s[3])
            for lse in (args.lse, "fast") if args.lse == "auto" else (args.lse,):
                w.set_lse_mode(lse)
                for i in range(R + 2):
                    op_step(i)
                t = timed(op_step, args.steps, 1, dist, dev) / args.steps
                if lse == args.lse:
                    extra["operator_ms_per_step"] = t
                    extra["operator_call"] = "_C.rnnt_loss (the reference's operator boundary: costs + dense grads)"
                else:
                    extra["lse_fast"] = {"ms_per_step": t, "value": N / (t * 1e-3), "unit": "lattices/s",
                                         "roofline_frac": b_alg(N, T, U, V) / (t * 1e-3) / 1e9 / peaks()[0],
                                         "note": "opt-in RNNT_LSE_FAST through _C.rnnt_loss (fp32-noise-level deviation from the "
                                                 "reference, <= ~1e-4 on gradients); the headline uses the default mode, "
                                                 "bit-identical to the reference"}
            w.set_lse_mode(args.lse)
            del keep

    # ---- end to end: HOST (pinned) inputs, H2D copies and the D2H read of the loss inside the timed region
    ke = args.e2e_steps or min(args.steps, 20)
    hb = sum(t.numel() * t.element_size() for t in host[0])

    def e2e_step(i):
        h = host[i % R]
        if graphs is not None:
            g, loss, s = graphs[i % R]
            with torch.no_grad():
                for dst, src in zip(s, h):
                    dst.copy_(src, non_blocking=True)
            g.replay()
        else:
            s = sets[i % R]
            with torch.no_grad():
                for dst, src in zip(s, h):
                    dst.copy_(src, non_blocking=True)
            loss = api_step(s)
        if world > 1:                                   # the value is read right away: blocking all-reduce
            dist.all_reduce(loss.detach())
        return float(loss.item())                       # D2H read of the step's result

    for i in range(2):
        e2e_step(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(ke):
        e2e_step(i)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    clocks = sampler.stop()

    # ---- BASELINE configs[4] on N > 1 GPUs: 256 lattices per GPU as 8 micro-batches of 32, one all-reduce per step
    c5 = None
    if world > 1 and not args.no_c5:
        graphs = None
        del sets
        torch.cuda.empty_cache()
        c5 = run_c5(w, parallel, dist, dev, world, rank)

    if rank != 0:
        finish(world, dist)
        return
    peak, peak_src = peaks()
    balg = b_alg(N, T, U, V, cells=sum(cells) / len(cells) if mode == "compact" or ragged else None, mode=mode)
    # roofline of the DOMINANT KERNEL: on the dense f32 path that is the one kernel of the operator call (CUDA events
    # around back-to-back launches); the API step adds the rescale check + autograd's ones_like (~5 us at cfg 2)
    one_kernel = args.workload in ("c2", "c3d")           # the operator call is ONE kernel there (k_fused)
    kernel_ms = extra["operator_ms_per_step"] if one_kernel and "operator_ms_per_step" in extra else ms_per_step
    achieved = balg / (kernel_ms * 1e-3) / 1e9
    kernels = {"dense": "k_fused<exact,dense> (+ k_rescale no-op check)" if args.workload in ("c2", "c3d") else
                        "k_gather + k_wavefront + k_expand (8-group stream pipeline) + k_loss_sum + k_rescale check",
               "gather": "k_fused<exact,pairs> + k_expand<1>" if args.workload in ("c2g", "c3") else "general path + k_expand<1>",
               "compact": "k_prefix + k_gather + k_wavefront + k_grads_pairs + k_expand<2>",
               "bf16": "k_fused<exact,dense,bf16>" if args.workload == "c2b" else "k_gather<bf16> + k_wavefront + k_expand<0,bf16>",
               "logits": "k_lse_pairs + k_fused<exact,pairs> + k_expand_logits"}[mode]
    # dram__bytes_read + dram__bytes_write of the dominant kernel: from the committed ncu --set full capture of the same
    # workload (profiles/), labelled as such -- it is NOT measured in this run
    traffic, traffic_note = None, "not measured in this run; ncu dram__bytes per launch are in profiles/"
    key = {"c2": "c2", "c4d": "c4"}.get(args.workload)
    summ = os.path.join(ROOT, "profiles", "r2_summary.json")
    if key and world == 1 and os.path.exists(summ):
        try:
            ent = json.load(open(summ)).get(key)
            if ent:
                traffic = ent["dram_bytes_per_launch"]
                traffic_note = ("from the committed ncu --set full capture of this workload (profiles/r2_summary.json, kernel %s), "
                                "not measured in this run" % ent.get("kernel", "?")[:60])
        except Exception:
            pass
    out = {
        "metric": "RNN-T loss+grad lattices/sec", "value": value, "unit": "lattices/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16 i/o, f32 accumulate" if mode == "bf16" else "f32", "data": "synthetic",
        "config": config_dict(args.workload, desc, N, T, U, V, world, R, R * per_set / 1e6),
        "timed_call": API_CALL[mode] + " -- " + graph_note,
        "lse_mode": args.lse + (" (= exact: results bit-identical to the reference kernels)" if args.lse == "auto" else ""),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_note,
                     "algorithmic_bytes_per_launch": balg, "peak_source": peak_src, "kernel": kernels,
                     "kernel_ms": kernel_ms,
                     "kernel_ms_source": ("CUDA events over back-to-back operator calls (_C.rnnt_loss = the one kernel)"
                                          if one_kernel and "operator_ms_per_step" in extra else "the timed step (all its kernels)")},
        "e2e": {"value": N * world * ke / e2e_s, "unit": "lattices/s", "h2d_bytes_per_step": hb,
                "d2h_bytes_per_step": 4, "steps": ke, "ms_per_step": e2e_s / ke * 1e3,
                "call": "pinned host tensors -> device copies -> " + API_CALL[mode] + " -> loss.item()"},
        "gpu_launches": int(launches),
        "gpu_launches_note": ("kernels of this library per step, counted while the graph was captured, x steps"
                              if graphs is not None or launches_per_step else "library launch counter over the timed region"),
        "clocks": clocks,
    }
    out.update(extra)
    if c5 is not None:
        out["c5"] = c5
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_oracle_rate(N, T, U, V)
    print(json.dumps(out), flush=True)
    finish(world, dist)


def finish(world, dist):
    """Multi-rank exit: every rank has done its work and rank 0 has printed; leave without tearing NCCL down (destroying
    the communicator after CUDA graphs were captured on it hung the watchdog for minutes on this stack)."""
    if world > 1:
        torch.cuda.synchronize()
        try:
            dist.barrier()
        except Exception:
            pass
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def run_c5(w, parallel, dist, dev, world, rank, steps=4, warm=2):
    """N=2048 T=600 U=150 V=1024 over 8 GPUs = 256 lattices per GPU; log_probs + gradient of one GPU's share are
    2 x 94 GB > 180 GB, so each rank runs 8 micro-batches of 32 (the joint network upstream would be micro-batched the
    same way) and the step ends with ONE all-reduce of the scalar loss.  Synthetic log-probs are made on the device;
    one 11.8 GB input buffer serves all micro-batches (far larger than L2)."""
    N, T, U, V, MB = 32, 600, 150, 1024, 8
    g = torch.Generator(device=dev).manual_seed(5 + rank)
    x = torch.log_softmax(torch.randn((N, T, U, V), device=dev, generator=g), dim=-1)
    ys = torch.randint(1, V, (N, U - 1), dtype=torch.int, device=dev, generator=g)
    xn = torch.full((N,), T, dtype=torch.int, device=dev)
    yn = torch.full((N,), U - 1, dtype=torch.int, device=dev)
    total = N * MB * world

    x.requires_grad_(False)

    def step(i):
        # every micro-batch is its own leaf over the same 11.8 GB of synthetic log-probs (no copy): its gradient is a
        # fresh tensor, as it would be for distinct micro-batches
        return parallel.rnnt_loss_microbatches(((x.detach().requires_grad_(True), ys, xn, yn) for _ in range(MB)),
                                               global_batch=total, reduction="mean")
    for i in range(warm):
        step(i)
    ms = timed(step, steps, world, dist, dev) / steps
    peak, _ = peaks()
    balg = b_alg(N, T, U, V) * MB
    return {"workload": "c5: N=2048 T=600 U=150 V=1024 batch-sharded (BASELINE configs[4]); here %d lattices = %d GPUs x "
                        "%d micro-batches x %d" % (total, world, MB, N),
            "ms_per_step": ms, "value": total / (ms * 1e-3), "unit": "lattices/s", "steps": steps,
            "roofline_frac_per_gpu": balg / (ms * 1e-3) / 1e9 / peak,
            "call": "warp_rnnt_b200.parallel.rnnt_loss_microbatches (rnnt_loss + backward per micro-batch, one all-reduce)"}


# ---- the reference arm -------------------------------------------------------------------------------------------
class _RefRNNTLoss(torch.autograd.Function):
    """The reference's own autograd wrapper, re-stated because its module needs installed dist
    metadata (pytorch_binding/warp_rnnt/__init__.py:4-6, :9-24): grads in forward, mul_ in backward."""

    @staticmethod
    def forward(ctx, core, log_probs, labels, frames_lengths, labels_lengths, blank):
        costs, ctx.grads = core.rnnt_loss(xs=log_probs, ys=labels, xn=frames_lengths, yn=labels_lengths,
                                          blank=blank, fastemit_lambda=0.0)
        return costs

    @staticmethod
    def backward(ctx, grads_output):
        grads_output = grads_output.view(-1, 1, 1, 1).to(ctx.grads)
        return None, ctx.grads.mul_(grads_output), None, None, None, None


class _RefRNNTLossCompact(torch.autograd.Function):
    """pytorch_binding/warp_rnnt/__init__.py:26-54, re-stated for the same reason."""

    @staticmethod
    def forward(ctx, core, log_probs, labels, frames_lengths, labels_lengths):
        costs, grads, loc = core.rnnt_loss_compact(xs=log_probs, ys=labels, xn=frames_lengths, yn=labels_lengths,
                                                   blank=0, fastemit_lambda=0.0, required_grad=True)
        cumlen = torch.cumsum(frames_lengths * (labels_lengths + 1), dim=0, dtype=torch.int32)
        ctx.V = log_probs.size(-1)
        ctx.save_for_backward(grads, loc, cumlen)
        ctx.core = core
        return costs

    @staticmethod
    def backward(ctx, grads_output):
        grads, loc, cumlen = ctx.saved_tensors
        return None, ctx.core.rnnt_loss_compact_backward(grads_output.contiguous(), grads, cumlen, loc, ctx.V, 0), None, None, None


def ref_api_loss(core, x, ys, xn, yn, mode):
    """rnnt_loss(..., reduction='sum', gather=/compact=) of the reference, __init__.py:109-143."""
    if mode == "compact":
        return _RefRNNTLossCompact.apply(core, x.float(), ys, xn, yn).sum()
    blank = 0
    if mode == "gather":
        N, T, U, V = x.size()
        index = torch.full([N, T, U, 2], blank, device=ys.device, dtype=torch.long)
        index[:, :, :U - 1, 1] = ys.unsqueeze(dim=1)
        x = x.gather(dim=3, index=index)
        blank = -1
    return _RefRNNTLoss.apply(core, x, ys, xn, yn, blank).sum()


def run_reference(args, rank, world, N, T, U, V, mode, ragged, desc, have_cuda):
    if rank != 0:
        return                                          # rank 0 alone runs the reference arm
    ref = None
    if have_cuda:
        try:
            from oracle import build_ref
            ref = build_ref.load()
        except Exception:
            ref = None
    cpu = None if args.no_cpu_baseline and ref is not None else cpu_oracle_rate(N, T, U, V)
    per_set = 2 * 4 * N * T * U * V
    R = rotation(per_set)
    base = {"impl": "reference", "metric": "RNN-T loss+grad lattices/sec", "unit": "lattices/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args.workload, desc, N, T, U, V, world, R, R * per_set / 1e6),
            "reference_note": "the reference is single-GPU: rank 0 alone runs it, on %d lattices" % N}
    if cpu is not None:
        base["cpu_baseline"] = cpu
    if ref is None:
        # CPU arm: the oracle port on the host cores (no GPU or the reference extension did not travel)
        base.update({"value": cpu["value"], "ms_per_step": 1e3 * N / cpu["value"], "gpu_launches": 0,
                     "e2e": {"value": cpu["value"], "unit": "lattices/s", "h2d_bytes_per_step": 0,
                             "d2h_bytes_per_step": 0},
                     "reference_kind": "cpu oracle port (oracle/_ref not loadable)"})
        print(json.dumps(base), flush=True)
        return
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    host = [make_host_inputs(N, T, U, V, seed=N + i, ragged=ragged, compact=(mode == "compact")) for i in range(R)]
    sets = [tuple(t.to(dev) for t in h) for h in host]
    cells = [int((h[2].long() * (h[3].long() + 1)).sum()) for h in host]
    for s in sets:
        s[0].requires_grad_(True)
    steps = args.steps

    def api_step(s):                                    # the reference through its own python API, same call as ours
        s[0].grad = None
        loss = ref_api_loss(ref, s[0], s[1], s[2], s[3], mode)
        loss.backward()
        return loss

    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    for i in range(R + 2):                              # prime the caching allocator (see main())
        api_step(sets[i % R])
    for i in range(args.warmup):
        api_step(sets[i % R])
    ms = timed(lambda i: api_step(sets[(args.warmup + i) % R]), steps, 1, None, dev)
    ke = args.e2e_steps or min(steps, 20)

    def e2e_step(i):
        h, s = host[i % R], sets[i % R]
        with torch.no_grad():
            for dst, src in zip(s, h):
                dst.copy_(src, non_blocking=True)
        return float(api_step(s).item())

    for i in range(2):
        e2e_step(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(ke):
        e2e_step(i)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    hb = sum(t.numel() * t.element_size() for t in host[0])
    peak, peak_src = peaks()
    balg = b_alg(N, T, U, V, cells=sum(cells) / len(cells) if mode == "compact" or ragged else None)
    ms_per_step = ms / steps
    base.update({"value": N * steps / (ms * 1e-3), "ms_per_step": ms_per_step,
                 "timed_call": "the reference's rnnt_loss(x, ..., reduction='sum'%s).backward(), eager (its compact path "
                               "synchronises the host four times per call and cannot be graph-captured)"
                               % {"dense": "", "gather": ", gather=True", "compact": ", compact=True"}[mode],
                 "roofline": {"bound": "hbm", "achieved": balg / (ms_per_step * 1e-3) / 1e9, "peak": peak,
                              "unit": "GB/s", "frac": balg / (ms_per_step * 1e-3) / 1e9 / peak, "traffic": None,
                              "peak_source": peak_src},
                 "e2e": {"value": N * ke / e2e_s, "unit": "lattices/s", "h2d_bytes_per_step": hb,
                         "d2h_bytes_per_step": 4, "steps": ke, "ms_per_step": e2e_s / ke * 1e3},
                 "gpu_launches": None, "clocks": sampler.stop(),
                 "reference_kind": "unmodified reference kernels (oracle/_ref/warp_rnnt_ref_C.so) on the same B200"})
    print(json.dumps(base), flush=True)


if __name__ == "__main__":
    main()
