#!/usr/bin/env python
"""Benchmark of the trie-mass hot path (BASELINE.json metric: trie weight_sum/max distributions/sec at 128k vocab).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|async1024|smc4096|cfg5]
                    [--dump-outputs DIR]

Default workload (cfg2 = BASELINE.json configs[1], the one the metric is quoted on): one "step" = batch_weight_sum +
batch_weight_max over one batch of 64 synthetic Dirichlet rows on the 128,256-token synthetic byte vocabulary; a
"distribution" is one row put through both reductions.  Under torchrun every rank runs the same per-GPU workload on
its own rows (weak scaling, no collective on the data path); `value` is the whole-job rate, timed on the device, max
over ranks.

  value          device-resident: inputs in HBM, CUDA events around exactly the K steps (one CUDA graph of K steps
                 rotating over buffer sets larger than L2, replayed once untimed and, queued right behind it, once timed)
  e2e            the same step through the public, reference-shaped API: pinned HOST rows in, numpy arrays out
                 (ParallelTokenCharacterTrie.batch_weight_sum_max), H2D and D2H inside the timed region
  roofline       dominant kernel (mass_kernel): algorithmic bytes (4V + 8N per distribution) / its CUDA-event time
  cpu_baseline / --impl reference
                 the reference's CPU algorithm (oracle C restatement of the numba loops, OpenMP over rows) timed on
                 this box's host cores in 64-row steps; the reference arm never imports the product package
  reference_gpu  the reference's own GPU path restated with torch library kernels (oracle/torch_ref.py: sparse.mm +
                 scatter_reduce amax, parallel.py:92-145) on the same B200, device-resident and end to end
  sampler        the SMC row op (configs[3] per-GPU share) with `reference` = the batched torch idiom of README.md:82-87

Other workloads (BASELINE.json configs[0], [2..4]; one JSON line each, same contract):
  cfg0           weight_sum + weight_max of ONE distribution at the GPT-2-sized vocabulary (50,257 tokens): call latency of
                 both trie classes; the reference arm is the single-threaded CPU loop (what numba runs for one row)
  async1024      AsyncTokenCharacterTrie, 1,024 concurrent weight_sum requests at 128,256 tokens, requests sharded over ranks
  smc4096        fused masked logsumexp + multinomial, 4,096 particles x 128,256 tokens, particles sharded over ranks
  cfg5           batch_weight_sum + batch_weight_max at 151,665 tokens, 8,192 rows over 8 GPUs (1,024 per GPU),
                 plus (--allgather) the NCCL all-gather of the full [rows, N] node-mass slab

--dump-outputs DIR (cfg2, cfg5): after the timed steps, rank 0 writes what the last timed step computed, the [B, N]
weight_sum and weight_max results, as DIR/weight_sum.npy and DIR/weight_max.npy (float32) with DIR/node_ids.npy
(float64) naming their columns: every node when the two fit in 64 MB, otherwise a fixed seeded sample of the nodes.
The inputs depend only on the arguments, so two builds run with the same arguments can be compared file by file.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "trie weight_sum+weight_max distributions/sec at 128k vocab"
UNIT = "distributions/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg0", "async1024", "smc4096", "cfg5"])
    ap.add_argument("--vocab", type=int, default=0, help="0 = the workload's vocabulary (128256; cfg5: 151665)")
    ap.add_argument("--batch", type=int, default=0, help="rows per GPU and step; 0 = the workload's (cfg2: 64, cfg5: 1024)")
    ap.add_argument("--alpha", type=float, default=1.0)
    ap.add_argument("--sets", type=int, default=4, help="rotating buffer sets (cfg2: each 33 MB in + 176 MB out)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 10)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-gpu", action="store_true", help="skip the torch library-kernel baseline on the GPU")
    ap.add_argument("--no-sampler", action="store_true", help="skip the secondary sampler-kernel measurement")
    ap.add_argument("--allgather", action="store_true",
                    help="N > 1 only: also time the optional NCCL all-gather of the node masses (BASELINE config 5's exchange); "
                         "reported separately, never part of the timed step")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results to DIR/<name>.npy (cfg2, cfg5)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload not in ("cfg2", "cfg5")):
        ap.error("--dump-outputs covers the trie-mass workloads (cfg2, cfg5) of --impl ours")
    if not args.vocab:
        args.vocab = {"cfg5": 151665, "cfg0": 50257}.get(args.workload, 128256)
    if not args.batch:
        args.batch = {"cfg2": 64, "cfg0": 1, "cfg5": 1024, "async1024": 1024, "smc4096": 4096}[args.workload]
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def metric_name(args):
    return {"cfg5": "trie weight_sum+weight_max distributions/sec at 151,665 vocab (config 5)",
            "cfg0": "one-distribution weight_sum+weight_max calls/sec at 50,257 vocab (config 0)"}.get(args.workload, METRIC)


def workload_name(args):
    return (f"batch_weight_sum + batch_weight_max, synthetic byte vocab V={args.vocab}, batch {args.batch} "
            f"Dirichlet({args.alpha:g}) fp32 rows per GPU")


def host_threads():
    """Host threads the CPU arms use: every CPU this process may run on, whatever OMP_NUM_THREADS says (torchrun sets
    it to 1)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


# ---- the reference's CPU algorithm (oracle) -----------------------------------------------------------------
def cpu_steps(o, ws_steps, threads, steps, warmup):
    """Times `steps` steps of oracle weight_sum + weight_max (the numba loops restated in C, one thread per row, OpenMP
    over the rows of a step) over host batches of the step's shape.  Returns seconds per step (mean) and the threads used."""
    for i in range(warmup):
        o.weight_sum(ws_steps[i % len(ws_steps)], threads=threads)
        o.weight_max(ws_steps[i % len(ws_steps)], threads=threads)
    t0 = time.perf_counter()
    for i in range(steps):
        w = ws_steps[i % len(ws_steps)]
        o.weight_sum(w, threads=threads)
        o.weight_max(w, threads=threads)
    return (time.perf_counter() - t0) / steps, int(o.last_threads)


def cpu_baseline(args, o, dirichlet_rows, budget_s=12.0):
    """`cpu_baseline` object of the bench line: bounded sample of the same workload (64-row steps) on all host threads."""
    threads = host_threads()
    ws_steps = [dirichlet_rows(args.batch, args.vocab, alpha=args.alpha, seed=100 + k) for k in range(2)]
    per_step, used = cpu_steps(o, ws_steps, threads, 1, 1)
    steps = int(max(2, min(200, budget_s / max(per_step, 1e-6))))
    per_step, used = cpu_steps(o, ws_steps, threads, steps, 0)
    t0 = time.perf_counter()
    o.weight_sum(ws_steps[0][:2], threads=1)
    o.weight_max(ws_steps[0][:2], threads=1)
    single = 2 / (time.perf_counter() - t0)
    return {
        "value": args.batch / per_step, "unit": UNIT, "cores": used, "kind": "port",
        "sample": f"{steps} steps of {args.batch} rows x (sum+max), V={args.vocab}, oracle/trie_oracle.c (numba loops of "
                  f"base.py:346-393 in C, fp64), OpenMP over the rows of a step with {used} threads "
                  f"(host has {os.cpu_count()} logical cpus, OMP_NUM_THREADS ignored)",
        "single_thread_rows_per_s": single,
    }


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the path on the host cores.  Imports only numpy and
    oracle/ -- the product package (and its CUDA library) is never loaded in this process."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload not in ("cfg2", "cfg5", "cfg0"):
        print(json.dumps({"impl": "reference", "unavailable": f"the reference arm covers the trie-mass workloads (cfg2, cfg5), not {args.workload}"}), flush=True)
        return
    import oracle
    from oracle import synth

    assert "genlm_backend_b200" not in sys.modules
    t0 = time.perf_counter()
    trie = oracle.OracleTrie(synth.synth_vocab_bytes(args.vocab))  # pure-Python restatement of base.py:13-122
    build_s = time.perf_counter() - t0
    threads = host_threads()  # OpenMP over the rows of a step: a one-row step (cfg0) runs on one thread, like the numba loop
    ws_steps = [synth.dirichlet_rows(args.batch, args.vocab, alpha=args.alpha, seed=100 + k) for k in range(2)]
    # bounded: at most ~60 s of timed steps
    probe, _ = cpu_steps(trie, ws_steps, threads, 1, 1)
    K = int(max(1, min(args.steps, 60.0 / max(probe, 1e-6))))
    W = int(max(1, min(args.warmup, 5)))
    t0 = time.perf_counter()
    per_step, used = cpu_steps(trie, ws_steps, threads, K, W)
    wall = time.perf_counter() - t0
    value = args.batch / per_step
    cb = {"value": value, "unit": UNIT, "cores": used, "kind": "port",
          "sample": f"{K} steps of {args.batch} rows x (sum+max), V={args.vocab}, oracle/trie_oracle.c (numba loops of base.py:346-393 "
                    f"in C, fp64), OpenMP over the rows of a step with {used} threads (host has {os.cpu_count()} logical cpus, "
                    f"OMP_NUM_THREADS ignored); layout from oracle.OracleTrie ({build_s:.1f} s)"}
    line = {
        "impl": "reference", "metric": metric_name(args), "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": K, "warmup": W, "ms_per_step": 1e3 * per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args), "vocab": args.vocab, "nodes": trie.n_nodes, "batch_per_gpu": args.batch,
                   "note": "reference CPU algorithm (oracle port of the numba path) on host cores, rank 0 only; "
                           "a step is one batch of the workload's shape; steps bounded to about a minute"},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": wall, "product_package_loaded": "genlm_backend_b200" in sys.modules,
    }
    print(json.dumps(line), flush=True)


# ---- clocks ------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index, period=0.004):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.loaded = False
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and visible.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        while not self._stop_evt.is_set():
            try:
                if self.loaded:
                    self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                    bits = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                    for bit, name in names.items():
                        if bits & bit:
                            self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---- distributed plumbing --------------------------------------------------------------------------------------------
class Job:
    """One process per GPU (torchrun) or a single process: device selection, barrier, max over ranks."""

    def __init__(self):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            # NCCL prints its banner ("NCCL version ...") to stdout when the first communicator is created; stdout carries
            # exactly one JSON line, so file descriptor 1 points at stderr until that has happened
            sys.stdout.flush()
            saved_fd = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group("nccl", device_id=self.dev)
                dist.barrier()
                torch.cuda.synchronize()
            finally:
                sys.stdout.flush()
                os.dup2(saved_fd, 1)
                os.close(saved_fd)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def finish(self):
        if self.world > 1:
            self.dist.destroy_process_group()

    def timed(self, enqueue, clocks=None):
        """Device time of one `enqueue()` (ms, max over ranks); barrier + sync on both sides.  It is queued right behind an
        untimed `enqueue()` (a CUDA graph's first replay uploads it), so the device starts the timed work as soon as the
        start event completes instead of waiting for the host to launch it."""
        torch = self.torch
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        if clocks is not None:
            clocks.loaded = True
        enqueue()
        ev0.record()
        enqueue()
        ev1.record()
        torch.cuda.synchronize()
        if clocks is not None:
            clocks.loaded = False
        self.barrier()
        return self.max_over_ranks(ev0.elapsed_time(ev1))


# ---- secondary measurement: the SMC row op (BASELINE.json configs[3], per-GPU share) ---------------------------------
def pack_bits(keep):
    """bool [B, V] -> int32 [B, ceil(V/32)] keep-bitmask (bit i of word w = element 32 w + i)."""
    import torch

    pad = (-keep.shape[-1]) % 32
    k = torch.nn.functional.pad(keep, (0, pad)).view(keep.shape[0], -1, 32).to(torch.int64)
    w = (k << torch.arange(32, device=keep.device, dtype=torch.int64)).sum(-1)
    return torch.where(w >= 2**31, w - 2**32, w).to(torch.int32)


def graph_time(fn, n_per_graph, iters):
    """Average device seconds of one call of fn(k), replayed from a CUDA graph of n_per_graph calls."""
    import torch

    for k in range(min(3, n_per_graph)):
        fn(k)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for k in range(n_per_graph):
            fn(k)
    g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / (n_per_graph * iters) / 1e3


def sampler_metrics(dev, vocab, peak, rows=512, iters=20, with_reference=True):
    """Fused masked logsumexp + categorical draw over `rows` x `vocab` fp32 log-probabilities (one particle per row) for
    the mask kinds an SMC step uses.  Device time from a CUDA graph of 8 launches rotating over two logit buffers that
    are larger than L2 together.  `reference`: the batched torch idiom of README.md:82-87 on the same buffers."""
    import torch

    from genlm_backend_b200 import smc

    gen = torch.Generator(device=dev).manual_seed(0)
    sets = [torch.log_softmax(torch.randn(rows, vocab, device=dev, generator=gen), dim=-1) for _ in range(2)]
    masks = [torch.rand(rows, vocab, device=dev, generator=gen) < 0.5 for _ in range(2)]
    out = {}
    per_graph = 8
    shared_log = masks[0][0].float().log()           # the reference idiom ({0, -inf}): packed to a bit mask once, cached
    shared_soft = torch.where(masks[0][0], 0.0, -30.0)  # a general additive mask: stays fp32, 4V more L2-resident bytes per row
    cases = (("no_mask", lambda k: None, 0), ("shared_f32_mask", lambda k: shared_log, 0), ("shared_f32_mask_general", lambda k: shared_soft, 0),
             ("per_row_bit_mask", lambda k: pack_bits(masks[k]), 4 * ((vocab + 31) // 32)), ("per_row_bool_mask", lambda k: masks[k], vocab))
    for name, mk, mask_bytes in cases:
        ms_ = [mk(0), mk(1)]
        sec = graph_time(lambda k: smc.masked_logsumexp_sample(sets[k % 2], ms_[k % 2], seed=k), per_graph, iters)
        bytes_per_row = 4 * vocab + mask_bytes + 8
        out[name] = {"rows_per_s": rows / sec, "us_per_launch": sec * 1e6, "achieved_GBps": rows * bytes_per_row / sec / 1e9,
                     "frac_of_hbm_peak": rows * bytes_per_row / sec / 1e9 / peak}
    if with_reference:
        from oracle.torch_ref import smc_step

        shared = shared_log
        ref = {}
        for name, mask in (("no_mask", None), ("shared_f32_mask", shared)):
            for k in range(2):
                smc_step(sets[k], mask)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for k in range(10):
                smc_step(sets[k % 2], mask)
            b.record()
            torch.cuda.synchronize()
            sec = a.elapsed_time(b) / 10 / 1e3
            ref[name] = {"rows_per_s": rows / sec, "us_per_call": sec * 1e6, "speedup_of_ours": out[name]["rows_per_s"] / (rows / sec)}
        ref["what"] = ("oracle/torch_ref.smc_step on the same B200 and buffers: logps + mask, logsumexp(-1), "
                       "multinomial((masked - logZ).exp(), 1) batched over the rows (README.md:82-87; torch library kernels)")
        out["reference"] = ref
    return {"kernel": "lse_sample_kernel<float>", "rows": rows, "vocab": vocab, "bound": "hbm",
            "bytes_per_row": "4V (+ the bytes of a per-row mask: V/8 for bits, V for bools) + 8", **out}


def reference_gpu_metrics(trie, ws_dev, host_rows, ours_value, ours_e2e):
    """The reference's own GPU path (torch sparse.mm + scatter_reduce amax, parallel.py:92-145; restated in
    oracle/torch_ref.py) on this GPU and these rows: device-resident, and end to end with the .cpu().numpy() it ends on."""
    import torch

    from oracle.torch_ref import TorchReferenceTrie

    rows, cols = trie._engine.reachability()
    ref = TorchReferenceTrie(trie.idx_to_leaf, rows, cols, len(trie), ws_dev.device)
    B = ws_dev.shape[0]
    for _ in range(2):
        s = ref.batch_weight_sum_tensor(ws_dev)
        m = ref.batch_weight_max_tensor(ws_dev)
    torch.cuda.synchronize()
    # same results as the product (sanity, not the parity test): sums to fp32 summation order, maxes exactly
    hs, hm = trie.batch_weight_tensor(ws_dev, ops=("sum", "max"))
    same_max = bool(torch.equal(hm, m))
    rel = float(((hs - s).abs() / s.clamp_min(1e-30)).max())
    del hs, hm
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 5
    a.record()
    for _ in range(n):
        s = ref.batch_weight_sum_tensor(ws_dev)
        m = ref.batch_weight_max_tensor(ws_dev)
    b.record()
    torch.cuda.synchronize()
    kern_s = a.elapsed_time(b) / n / 1e3
    a.record()
    for _ in range(n):
        s = ref.batch_weight_sum_tensor(ws_dev)
    b.record()
    torch.cuda.synchronize()
    sum_s = a.elapsed_time(b) / n / 1e3
    del s, m
    ref.batch_weight_sum(host_rows)
    t0 = time.perf_counter()
    for _ in range(3):
        hs_ = ref.batch_weight_sum(host_rows)
        hm_ = ref.batch_weight_max(host_rows)
        _ = float(hs_[0, -1]) + float(hm_[-1, -1])
    e2e_s = (time.perf_counter() - t0) / 3
    return {
        "kernel": {"value": B / kern_s, "unit": UNIT, "ms_per_step": kern_s * 1e3, "sum_only_ms": sum_s * 1e3,
                   "max_only_ms": (kern_s - sum_s) * 1e3},
        "e2e": {"value": B / e2e_s, "unit": UNIT, "ms_per_step": e2e_s * 1e3},
        "speedup_of_ours": {"kernel": ours_value / (B / kern_s), "e2e": ours_e2e / (B / e2e_s)},
        "agrees_with_ours": {"max_bit_exact": same_max, "sum_max_rel_diff": rel},
        "what": "oracle/torch_ref.TorchReferenceTrie: torch.sparse.mm(ws[:, positions], M_csr) + zeros.scatter_reduce_(amax) over the "
                "(leaf, ancestor) pairs (parallel.py:92-145), fp32, same GPU and rows; e2e = pinned host rows -> .to(cuda) -> both ops -> .cpu().numpy()",
    }


DUMP_BYTES = 64_000_000


def dump_node_slabs(out_dir, slabs):
    """Writes [B, N] float32 device slabs (name -> tensor) as out_dir/<name>.npy and the node columns they hold as
    out_dir/node_ids.npy (float64): all N columns when everything fits DUMP_BYTES, otherwise a sorted sample drawn with
    a fixed seed, so that runs with the same B and N write the same elements."""
    import torch

    B, N = next(iter(slabs.values())).shape
    per_col = 4 * B * len(slabs) + 8
    S = min(N, max(1, (DUMP_BYTES - 4096) // per_col))  # 4096: room for the .npy headers
    cols = np.arange(N) if S == N else np.sort(np.random.default_rng(0).choice(N, size=S, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    idx = torch.from_numpy(cols).to(next(iter(slabs.values())).device)
    for name, slab in slabs.items():
        np.save(os.path.join(out_dir, name + ".npy"), slab[:, idx].cpu().numpy().astype(np.float32, copy=False))
    np.save(os.path.join(out_dir, "node_ids.npy"), cols.astype(np.float64))


# ---- default workload: BASELINE.json configs[1] (and cfg5's per-GPU shape) --------------------------------------------
def run_mass(args, job):
    torch = job.torch
    from genlm_backend_b200 import ParallelTokenCharacterTrie, _lib
    from genlm_backend_b200.synthetic import synth_vocab, dirichlet_rows

    rank, world, dev = job.rank, job.world, job.dev
    V, B, K, W = args.vocab, args.batch, args.steps, max(args.warmup, 3)
    cfg5 = args.workload == "cfg5"
    trie = ParallelTokenCharacterTrie(synth_vocab(V), devices=[job.local_rank])
    eng = trie._engine
    N = len(trie)
    eng.ensure_device(job.local_rank)
    info = eng.plan_info()

    base = dirichlet_rows(min(B, 64), V, alpha=args.alpha, seed=1 + rank)
    set_bytes = B * V * 4 + 2 * B * N * 4
    l2_bytes = torch.cuda.get_device_properties(dev).L2_cache_size
    nsets = max(1, args.sets) if set_bytes < 4 * l2_bytes else 1  # one set already exceeds L2 several times over (cfg5)

    def rows_for(k):
        reps = -(-B // base.shape[0])
        return torch.tensor(np.concatenate([np.roll(base, k + j, axis=0) for j in range(reps)])[:B]).to(dev)

    ws_sets = [rows_for(k) for k in range(nsets)]
    # output slabs as the engine allocates them: [B, N] views of rows padded to whole 128-byte lines
    sum_sets = [eng.alloc_out(B, torch.float32, dev) for _ in range(nsets)]
    max_sets = [eng.alloc_out(B, torch.float32, dev) for _ in range(nsets)]

    def step(k, phases=0, ops=("sum", "max"), dfs_order=False):
        eng.reduce(ws_sets[k], ops, out_sum=sum_sets[k], out_max=max_sets[k], phases=phases, dfs_order=dfs_order)

    chunks = -(-B // 64)  # the C side reduces a batch in chunks of the engine's 64 scratch rows
    launches_per_step = chunks * (2 + (1 if info["n_span"] > 0 else 0))  # permute + tile (both reductions) + span kernel

    for i in range(W):  # warm-up (also sets kernel attributes, allocates the scratch)
        step(i % nsets)
    torch.cuda.synchronize()

    # The timed loop replays ONE CUDA graph that holds exactly K consecutive steps of a stream of batches rotating over
    # the buffer sets, as a serving loop issues them.
    graph = None
    if not args.no_graph:
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for i in range(K):
                step(i % nsets)

    def run_steps():
        if graph is None:
            for i in range(K):
                step(i % nsets)
        else:
            graph.replay()

    clocks = ClockSampler(job.local_rank)
    clocks.start()
    ms_total = job.timed(run_steps, clocks)
    value = world * B * K / (ms_total / 1e3)
    if args.dump_outputs and rank == 0:  # before the per-kernel timings below overwrite the buffers
        last = (K - 1) % nsets
        dump_node_slabs(args.dump_outputs, {"weight_sum": sum_sets[last], "weight_max": max_sets[last]})

    # per-kernel timing for the roofline (one op, one phase at a time), same buffers ----------------------------------
    def time_phase(phases, ops):
        per_graph = 4 * nsets if B <= 64 else 2
        return graph_time(lambda k: step(k % nsets, phases, ops), per_graph, max(2, 400 // (per_graph * chunks))) * 1e3

    clocks.loaded = True
    ms_tile = time_phase(_lib.GT_FLAG_PHASE_TILE, ("sum",))
    ms_tile_max = time_phase(_lib.GT_FLAG_PHASE_TILE, ("max",))
    ms_tile_both = time_phase(_lib.GT_FLAG_PHASE_TILE, ("sum", "max"))
    ms_span_both = time_phase(_lib.GT_FLAG_PHASE_SPAN, ("sum", "max"))
    ms_permute = time_phase(_lib.GT_FLAG_PHASE_PERMUTE, ("sum",))
    ms_sum_op = time_phase(0, ("sum",))
    # the same step when the producer of the rows emits them in DFS leaf order (GT_FLAG_DFS_ORDER): nothing to scatter.
    # Timing only: the buffers hold the vocabulary-ordered rows (the data pattern does not change the kernels' work).
    per_graph = 4 * nsets if B <= 64 else 2
    ms_dfs_step = graph_time(lambda k: step(k % nsets, dfs_order=True), per_graph, max(2, 400 // (per_graph * chunks))) * 1e3
    ms_dfs_permute = graph_time(lambda k: step(k % nsets, _lib.GT_FLAG_PHASE_PERMUTE, ("sum",), dfs_order=True), per_graph,
                                max(2, 400 // (per_graph * chunks))) * 1e3
    clocks.loaded = False

    # end to end through the public API: pinned host rows in, numpy out -----------------------------------------------
    E = args.e2e_steps or min(K, 10 if B <= 64 else 2)
    host_sets = [ws_sets[k % nsets].cpu().pin_memory() for k in range(2)]
    sums = maxes = None
    for i in range(3):  # warm-up with the timed loop's result-retention pattern: fills the pinned-buffer pool
        sums, maxes = trie.batch_weight_sum_max(host_sets[i % 2])
    job.barrier()
    clocks.period = 0.02  # the host-side loop shares the interpreter with the sampling thread: sample it less often
    clocks.loaded = True
    t0 = time.perf_counter()
    for i in range(E):
        sums, maxes = trie.batch_weight_sum_max(host_sets[i % 2])
        _ = float(sums[0, N - 1]) + float(maxes[B - 1, N - 1])  # results are on the host
    torch.cuda.synchronize()
    e2e_s = job.max_over_ranks(time.perf_counter() - t0)
    # the same step when the caller reads K nodes per row instead of the whole slab (gt_gather_nodes): the [B, N] results
    # stay on the GPU, H2D of the rows and D2H of 2 x [B, K] values are inside the timed region
    Ks = 257  # e.g. the 256 byte children + end-of-token child of the node a particle stands on
    ids = torch.tensor(np.random.default_rng(5).integers(0, N, size=(B, Ks)), dtype=torch.int32, device=dev)
    for i in range(3):
        trie.batch_weight_sum_max_at(host_sets[i % 2], ids)
    torch.cuda.synchronize()
    job.barrier()
    t0 = time.perf_counter()
    for i in range(E):
        s_at, m_at = trie.batch_weight_sum_max_at(host_sets[i % 2], ids)
        _ = float(s_at[0, 0]) + float(m_at[B - 1, Ks - 1])
    torch.cuda.synchronize()
    sparse_s = job.max_over_ranks(time.perf_counter() - t0)
    clocks.loaded = False
    del sums, maxes
    job.barrier()
    clocks.stop()

    # optional exchange of BASELINE config 5: all-gather of the [rows, N] node masses over NVLink (not on the hot path) ----
    allgather = None
    if world > 1 and args.allgather:
        from genlm_backend_b200.sharding import all_gather_rows

        local = sum_sets[0].contiguous()  # this rank's [B, N] block (the slab's row padding is not sent)
        for _ in range(2):
            full = all_gather_rows(local, world * B)
        job.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps_ag = 5
        a.record()
        for _ in range(reps_ag):
            full = all_gather_rows(local, world * B)
        b.record()
        torch.cuda.synchronize()
        ms = job.max_over_ranks(a.elapsed_time(b) / reps_ag)
        ok = bool(torch.equal(full[rank * B:(rank + 1) * B], local))
        allgather = {"ms": ms, "rows_per_rank": B, "rows_total": world * B, "bytes_received_per_gpu": (world - 1) * B * N * 4,
                     "GBps_per_gpu_in": (world - 1) * B * N * 4 / (ms * 1e-3) / 1e9, "own_block_intact": ok,
                     "api": "genlm_backend_b200.sharding.all_gather_rows -> torch.distributed.all_gather_into_tensor (NCCL)",
                     "note": "one reduction's full [rows, N] fp32 node-mass slab; reported separately, not part of a step"}
        del full

    sampler_all = None
    if args.workload == "cfg2" and not args.no_sampler:
        peak_, _ = peaks()
        # every rank measures its own per-GPU share (512 particles); rank 0 reports its numbers and the job-wide rate
        sm = sampler_metrics(dev, V, peak_, with_reference=(rank == 0))
        if world > 1:
            sm["job_rows_per_s_no_mask"] = job.sum_over_ranks(sm["no_mask"]["rows_per_s"])
        sampler_all = sm

    job.finish()
    if rank != 0:
        return

    peak, peak_src = peaks()
    bytes_one = B * (4 * V + 4 * N)    # one reduction: rows in, one node array out
    bytes_both = B * (4 * V + 8 * N)   # both reductions from one launch (the step's mass_kernel launch)
    achieved = bytes_both / (ms_tile_both / 1e3) / 1e9
    path_achieved = bytes_both * K / (ms_total / 1e3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(tpath) and V == 128256 and B == 64:
        with open(tpath) as f:
            traffic = json.load(f)["traffic_bytes_per_launch"]
    metric = metric_name(args)
    line = {
        "metric": metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {
            "workload": workload_name(args), "vocab": V, "nodes": N, "batch_per_gpu": B, "global_batch": B * world,
            "parallelism": f"rows sharded, {world} independent GPU(s), no collective",
            "l2_policy": f"rotating {nsets} buffer set(s) of {set_bytes / 1e6:.0f} MB ({nsets * set_bytes / 1e6:.0f} MB total) "
                         f"vs L2 {l2_bytes / 1e6:.0f} MB",
            "launch": (f"one CUDA graph of the {K} steps, one timed replay ({ms_total:.1f} ms)" if graph is not None
                       else f"direct launches of the {K} steps ({ms_total:.1f} ms timed)"),
            "tile_leaves": info["tile_leaves"], "n_span": info["n_span"],
        },
        "e2e": {
            "value": world * B * E / e2e_s, "unit": UNIT, "h2d_bytes_per_step": B * V * 4,
            "d2h_bytes_per_step": 2 * B * N * 4, "steps": E,
            "host_GBps_all_ranks": world * E * (B * V * 4 + 2 * B * N * 4) / e2e_s / 1e9,
            "api": "ParallelTokenCharacterTrie.batch_weight_sum_max(pinned host tensor) -> numpy",
        },
        "e2e_sparse_readout": {
            "value": world * B * E / sparse_s, "unit": UNIT, "nodes_read_per_row": Ks, "h2d_bytes_per_step": B * V * 4,
            "d2h_bytes_per_step": 2 * B * Ks * 4, "steps": E,
            "api": "ParallelTokenCharacterTrie.batch_weight_sum_max_at(pinned host tensor, node_ids) -> numpy [B, K] x 2",
            "note": "not the headline: same kernels, results read through gt_gather_nodes instead of copying the [B, N] slabs",
        },
        "gpu_launches": launches_per_step * K,
        "roofline": {
            "bound": "hbm", "kernel": "mass_kernel<float,4> (the tile kernel: both reductions of the step in one launch)", "achieved": achieved,
            "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
            "bytes_per_launch": bytes_both, "ms_per_launch": ms_tile_both,
            "one_reduction": {"bytes_per_launch": bytes_one, "ms_per_launch": ms_tile,
                              "achieved": bytes_one / (ms_tile / 1e3) / 1e9, "frac": bytes_one / (ms_tile / 1e3) / 1e9 / peak},
            "note": "algorithmic bytes = (4V + 8N) per distribution x batch; kernel timed alone with CUDA events from a CUDA graph "
                    "rotating over the buffer sets; traffic = dram read+write of one launch from the ncu capture under profiles/",
        },
        "path_roofline": {
            "achieved": path_achieved, "peak": peak, "unit": "GB/s", "frac": path_achieved / peak,
            "note": "whole step (permute + tile kernel for both reductions + span kernel) against (4V + 8N) bytes per distribution",
        },
        "dfs_order_input": {
            "value": world * B / (ms_dfs_step / 1e3), "unit": UNIT, "ms_per_step": ms_dfs_step, "permute_ms": ms_dfs_permute,
            "path_roofline_frac": bytes_both / (ms_dfs_step / 1e3) / 1e9 / peak,
            "note": "not the headline: the same step with GT_FLAG_DFS_ORDER -- rows whose columns are already in DFS leaf order "
                    "(an LM head permuted once with ParallelTokenCharacterTrie.dfs_token_order), so the permute kernel interleaves "
                    "row groups with coalesced stores instead of scattering; per-GPU rate x ranks",
        },
        "kernel_ms": {"permute": ms_permute, "tile_sum": ms_tile, "tile_max": ms_tile_max, "tile_both": ms_tile_both,
                      "span_both": ms_span_both, "sum_op_all_phases": ms_sum_op},
        "clocks": clocks.summary(),
    }
    if allgather is not None:
        line["allgather"] = allgather
    if sampler_all is not None:
        line["sampler"] = sampler_all
    if world == 1 and not args.no_reference_gpu and B <= 256:
        try:
            line["reference_gpu"] = reference_gpu_metrics(trie, ws_sets[0], host_sets[0], value, line["e2e"]["value"])
        except Exception as e:  # the baseline must never take the bench line down with it
            line["reference_gpu"] = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    if world == 1 and not args.no_cpu_baseline:
        import oracle

        lay = trie._layout
        line["cpu_baseline"] = cpu_baseline(args, oracle.OracleLayout(trie.idx_to_leaf, lay["child_ptr"], lay["child_idx"]), dirichlet_rows,
                                            budget_s=12.0 if B <= 64 else 20.0)
    print(json.dumps(line), flush=True)


# ---- BASELINE.json configs[3]: SMC sampler, 4,096 particles x 128,256 tokens sharded over the ranks -------------------
def run_smc(args, job):
    torch = job.torch
    from genlm_backend_b200 import smc
    from genlm_backend_b200.sharding import row_block

    rank, world, dev = job.rank, job.world, job.dev
    V, total = args.vocab, args.batch
    lo, hi = row_block(total, world, rank)
    rows = hi - lo
    gen = torch.Generator(device=dev).manual_seed(rank)
    nsets = 2 if rows * V * 4 * 2 > 2 * 133e6 else 4
    sets = [torch.log_softmax(torch.randn(rows, V, device=dev, generator=gen), dim=-1) for _ in range(nsets)]
    keep = torch.rand(V, device=dev, generator=gen) < 0.5
    shared = keep.float().log()
    bits = pack_bits((torch.rand(rows, V, device=dev, generator=gen) < 0.5))
    K, W = args.steps, max(args.warmup, 3)
    cases = {"shared_f32_mask": shared, "no_mask": None, "per_row_bit_mask": bits}
    res = {}
    clocks = ClockSampler(job.local_rank)
    clocks.start()
    for name, mask in cases.items():
        for i in range(W):
            smc.masked_logsumexp_sample(sets[i % nsets], mask, seed=i)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for i in range(K):
                smc.masked_logsumexp_sample(sets[i % nsets], mask, seed=i, offset=lo)
        ms = job.timed(g.replay, clocks)
        res[name] = {"ms_per_step": ms / K, "particles_per_s": total * K / (ms / 1e3),
                     "per_gpu_GBps": rows * (4 * V + (4 * ((V + 31) // 32) if name == "per_row_bit_mask" else 0) + 8) / (ms / K / 1e3) / 1e9}
    # end to end: pinned host log-probs in, logZ + tokens out on the host
    host = sets[0].cpu().pin_memory()
    E = 3
    job.barrier()
    t0 = time.perf_counter()
    for i in range(E):
        lz, tok = smc.masked_logsumexp_sample(host.to(dev, non_blocking=True), shared, seed=i, offset=lo)
        _ = float(lz.cpu()[0]) + int(tok.cpu()[-1])
    e2e_s = job.max_over_ranks(time.perf_counter() - t0)
    ref = None
    if rank == 0:
        from oracle.torch_ref import smc_step

        for k in range(2):
            smc_step(sets[k % nsets], shared)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for k in range(5):
            smc_step(sets[k % nsets], shared)
        b.record()
        torch.cuda.synchronize()
        sec = a.elapsed_time(b) / 5 / 1e3
        ref = {"particles_per_s_per_gpu": rows / sec, "ms_per_step": sec * 1e3,
               "what": "oracle/torch_ref.smc_step (README.md:82-87 batched; torch library kernels) on rank 0's particles, shared additive mask"}
    clocks.stop()
    job.finish()
    if rank != 0:
        return
    peak, peak_src = peaks()
    head = res["shared_f32_mask"]
    line = {
        "metric": "SMC masked logsumexp + multinomial particles/sec at 128k vocab (config 4)", "value": head["particles_per_s"],
        "unit": "particles/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": head["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"fused masked logsumexp + multinomial, {total} particles x {V} fp32 log-probs sharded over {world} GPU(s) "
                               f"({rows} per GPU), shared additive fp32 mask (README.md:59-70)",
                   "l2_policy": f"rotating {nsets} logit sets of {rows * V * 4 / 1e6:.0f} MB", "launch": f"one CUDA graph of the {K} steps"},
        "e2e": {"value": total * E / e2e_s, "unit": "particles/s", "h2d_bytes_per_step": rows * V * 4, "d2h_bytes_per_step": rows * 8, "steps": E,
                "api": "smc.masked_logsumexp_sample(pinned host rows -> device) -> logZ, tokens on the host"},
        "gpu_launches": K,
        "roofline": {"bound": "hbm", "kernel": "lse_sample_kernel<float>", "achieved": head["per_gpu_GBps"], "peak": peak, "unit": "GB/s",
                     "frac": head["per_gpu_GBps"] / peak, "traffic": None, "peak_source": peak_src},
        "variants": res, "reference_gpu": ref, "clocks": clocks.summary(),
    }
    print(json.dumps(line), flush=True)


# ---- BASELINE.json configs[0]: one distribution, GPT-2-sized vocabulary ---------------------------------------------------
def run_single(args, job):
    torch = job.torch
    from genlm_backend_b200 import ParallelTokenCharacterTrie, TokenCharacterTrie
    from genlm_backend_b200.synthetic import synth_vocab, dirichlet_rows

    V, K, W = args.vocab, max(args.steps, 50), max(args.warmup, 3)
    dec = synth_vocab(V)
    row = torch.tensor(dirichlet_rows(1, V, alpha=args.alpha, seed=1)[0])
    drow = row.to(job.dev)

    def lat(fn):
        t_end = time.perf_counter() + 0.3  # call latency depends on the clocks: let them ramp before timing
        n = 0
        while n < W or time.perf_counter() < t_end:
            fn()
            n += 1
        torch.cuda.synchronize()
        ts = []
        for _ in range(K):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return float(np.median(ts)), float(np.percentile(ts, 90))

    res = {}
    for name, cls in (("parallel", ParallelTokenCharacterTrie), ("sequential", TokenCharacterTrie)):
        t0 = time.perf_counter()
        trie = cls(dec)
        build_s = time.perf_counter() - t0
        both_cuda = lat(lambda: (trie.weight_sum(drow), trie.weight_max(drow)))
        both_cpu = lat(lambda: (trie.weight_sum(row), trie.weight_max(row)))
        res[name] = {"build_s": build_s, "sum_plus_max_cuda_row_us": both_cuda[0] * 1e6, "sum_plus_max_cuda_row_p90_us": both_cuda[1] * 1e6,
                     "sum_plus_max_cpu_row_us": both_cpu[0] * 1e6, "sum_plus_max_cpu_row_p90_us": both_cpu[1] * 1e6,
                     "result_dtype": str(trie.weight_sum(row).dtype)}
        N = len(trie)
        lay = trie._layout
        idx = trie.idx_to_leaf
    job.finish()
    if job.rank != 0:
        return
    import oracle

    o = oracle.OracleLayout(idx, lay["child_ptr"], lay["child_idx"])
    w = row.numpy()[None, :]
    o.weight_sum(w, threads=1)
    ts = []
    for _ in range(20):
        t0 = time.perf_counter()
        o.weight_sum(w, threads=1)
        o.weight_max(w, threads=1)
        ts.append(time.perf_counter() - t0)
    cpu_s = float(np.median(ts))
    par = res["parallel"]
    line = {
        "metric": metric_name(args),
        "value": 1e6 / par["sum_plus_max_cuda_row_us"], "unit": UNIT, "n_gpus": 1, "steps": K, "warmup": W,
        "ms_per_step": par["sum_plus_max_cuda_row_us"] / 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"weight_sum + weight_max of one Dirichlet({args.alpha:g}) distribution, synthetic byte vocab V={V} (N={N}), "
                               "ParallelTokenCharacterTrie, numpy results; value: the row is a CUDA tensor, e2e: a CPU tensor; median wall clock of a call pair"},
        "e2e": {"value": 1e6 / par["sum_plus_max_cpu_row_us"], "unit": UNIT, "h2d_bytes_per_step": 2 * V * 4, "d2h_bytes_per_step": 2 * N * 4,
                "api": "ParallelTokenCharacterTrie.weight_sum(cpu tensor) + weight_max(cpu tensor) -> numpy"},
        "gpu_launches": 6 * K, "classes": res,
        "cpu_baseline": {"value": 1.0 / cpu_s, "unit": UNIT, "cores": 1, "kind": "port",
                         "sample": "20 x (weight_sum + weight_max) of the same row, oracle/trie_oracle.c (numba loops of base.py:346-393 in C, fp64), "
                                   "one thread: the reference processes a row on one thread"},
    }
    print(json.dumps(line), flush=True)


# ---- BASELINE.json configs[2]: AsyncTokenCharacterTrie, 1,024 concurrent requests sharded over the ranks ----------------
def run_async(args, job):
    import asyncio

    torch = job.torch
    from genlm_backend_b200 import AsyncTokenCharacterTrie
    from genlm_backend_b200.sharding import row_block
    from genlm_backend_b200.synthetic import synth_vocab, dirichlet_rows

    rank, world, dev = job.rank, job.world, job.dev
    V, total = args.vocab, args.batch
    lo, hi = row_block(total, world, rank)
    at = AsyncTokenCharacterTrie.from_vocab(synth_vocab(V), backend="parallel", devices=[job.local_rank])
    N = len(at.trie)
    base = dirichlet_rows(64, V, alpha=args.alpha, seed=1 + rank)
    cpu_rows = [torch.tensor(base[i % 64]) for i in range(hi - lo)]
    dev_rows = [r.to(dev) for r in cpu_rows]
    n_rep = max(2, min(args.steps, 4))

    async def once(reqs):
        t0 = time.perf_counter()
        out = await asyncio.gather(*[at.weight_sum(r) for r in reqs])
        dt = time.perf_counter() - t0
        assert len(out) == len(reqs) and out[0].shape == (N,)
        return dt

    async def main():
        res = {}
        for name, reqs in (("cuda_rows", dev_rows), ("cpu_rows", cpu_rows)):
            await once(reqs)
            best = 1e9
            for _ in range(n_rep):
                job.barrier()
                best = min(best, job.max_over_ranks(await once(reqs)))
            res[name] = best
        await at.cleanup()
        return res

    res = asyncio.run(main())
    job.finish()
    if rank != 0:
        return
    line = {
        "metric": "AsyncTokenCharacterTrie autobatched weight_sum requests/sec at 128k vocab (config 3)",
        "value": total / res["cuda_rows"], "unit": "requests/s", "n_gpus": world, "steps": n_rep, "warmup": 1,
        "ms_per_step": res["cuda_rows"] * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"{total} concurrent AsyncTokenCharacterTrie.weight_sum requests at V={V} (N={N}), {hi - lo} per GPU over {world} GPU(s); "
                               "every future resolves to its own float32 numpy row (the reference's contract); best wall clock of the gather, max over ranks"},
        "e2e": {"value": total / res["cpu_rows"], "unit": "requests/s", "h2d_bytes_per_step": (hi - lo) * V * 4,
                "d2h_bytes_per_step": (hi - lo) * N * 4, "api": "requests are CPU tensors (H2D inside), results numpy rows (D2H inside)"},
        "cuda_rows_ms": res["cuda_rows"] * 1e3, "cpu_rows_ms": res["cpu_rows"] * 1e3, "gpu_launches": 3 * (-(-(hi - lo) // 32) + 1),
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    job = Job()
    if args.workload in ("cfg2", "cfg5"):
        run_mass(args, job)
    elif args.workload == "cfg0":
        run_single(args, job)
    elif args.workload == "smc4096":
        run_smc(args, job)
    else:
        run_async(args, job)


if __name__ == "__main__":
    main()
