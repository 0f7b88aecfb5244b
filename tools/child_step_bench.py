"""Next-symbol step of a character-level sampler: child masses straight from the rows vs. today's slab route.

For V = 128,256 (synthetic vocabulary), log-softmax fp32 rows, B in {64, 1024}, rows in vocabulary and in DFS order, and
three node mixes -- ``root``; ``depth1`` (uniform over the root's 256 children); ``walk`` (for a uniform token t and a
uniform d in [0, len(t)], the node spelling t[:d]) -- it times with CUDA events over a CUDA graph of K steps:

  (a) ``batch_child_masses_tensor(normalize=True)``               gt_child_masses
  (b) ``sample_next_symbol``                                      gt_child_sample (+ the label gather)
  (c) ``batch_weight_sum_tensor`` + ``gather_nodes(children, normalizer=node)``   the [B, N] slab route

Step k reads buffer set k % S, with S sets covering more than three times the 126 MB L2, so rows are not L2-resident.
Algorithmic bytes (L2-resident metadata excluded, as in DESIGN section 5): (a) sum_b 4 * size(node_b) read + 4 * B * D
written; (b) the same read + 12 * B written; (c) 4 * B * V read + 4 * B * N slab written + 4 * B * D gathered.
Prints one JSON line per (B, order, mix, route); ``--out`` also writes them to a file.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from genlm_backend_b200 import ParallelTokenCharacterTrie  # noqa: E402
from genlm_backend_b200.synthetic import logsoftmax_rows, synth_vocab  # noqa: E402

L2_BYTES = 126 << 20


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
    except Exception:
        out = "unknown"
    return name, out


def node_mix(trie, mix, B, rng):
    lay = trie._layout
    if mix == "root":
        return np.full(B, trie.root, dtype=np.int32)
    if mix == "depth1":
        return rng.choice(trie.jump[trie.root], B).astype(np.int32)
    # walk: the ancestor of token t's spelling node at depth d (the leaf's parent spells t)
    toks = rng.integers(0, len(trie.decode), B)
    out = np.empty(B, dtype=np.int32)
    parent = lay["parent"]
    for b, t in enumerate(toks.tolist()):
        n = int(parent[lay["leaf_node"][t]])
        L = len(trie.decode[t].byte_string)
        for _ in range(L - int(rng.integers(0, L + 1))):
            n = int(parent[n])
        out[b] = n
    return out


def children_ids(trie, nodes, D):
    ptr, idx = trie._layout["child_ptr"], trie._layout["child_idx"]
    out = np.full((len(nodes), D), -1, dtype=np.int32)
    for b, n in enumerate(nodes.tolist()):
        k = idx[ptr[n]:ptr[n + 1]]
        out[b, :len(k)] = k
    return out


def time_graph(fn, sets, K, reps, stream):
    with torch.cuda.stream(stream):
        for s in sets:  # warm-up: workspaces of this stream, modules
            fn(*s)
    stream.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        for k in range(K):
            fn(*sets[k % len(sets)])
    g.replay()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(reps):
        t0.record()
        g.replay()
        t1.record()
        t1.synchronize()
        times.append(t0.elapsed_time(t1) * 1e3 / K)
    del g
    return float(np.median(times)), float(np.min(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="64,1024")
    ap.add_argument("--steps", type=int, default=20, help="K: steps per CUDA graph")
    ap.add_argument("--reps", type=int, default=10, help="graph replays timed (median reported)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "child_step_bench.py measures on a GPU"
    V = 128256
    trie = ParallelTokenCharacterTrie(synth_vocab(V))
    N, D = len(trie), trie.max_children
    size = (trie._layout["hi"] - trie._layout["lo"]).astype(np.int64)
    dfs_perm = trie.dfs_token_order.cuda()
    gpu, power = gpu_info()
    stream = torch.cuda.Stream()
    lines = []
    for B in [int(x) for x in args.batches.split(",")]:
        S = max(2, -(-3 * L2_BYTES // (4 * B * V)))
        base = [torch.tensor(logsoftmax_rows(B, V, seed=s)).cuda() for s in range(S)]
        for order in ("vocab", "dfs"):
            rows = base if order == "vocab" else [r[:, dfs_perm].contiguous() for r in base]
            for mix in ("root", "depth1", "walk"):
                rng = np.random.default_rng(7)
                nodes = [node_mix(trie, mix, B, rng) for _ in range(S)]
                kids = [torch.tensor(children_ids(trie, n, D)).cuda() for n in nodes]
                nt = [torch.tensor(n).cuda() for n in nodes]
                sets = list(zip(rows, nt, kids))
                dfs = order == "dfs"
                read = float(np.mean([4.0 * size[n].sum() for n in nodes]))
                routes = {
                    "a_child_masses": (lambda w, n, k: trie.batch_child_masses_tensor(w, n, log_input=True, dfs_order=dfs, normalize=True),
                                       read + 4.0 * B * D),
                    "b_sample_next_symbol": (lambda w, n, k: trie.sample_next_symbol(w, n, seed=1, log_input=True, dfs_order=dfs),
                                             read + 12.0 * B),
                    "c_slab_then_gather": (lambda w, n, k: trie.gather_nodes(
                        trie.batch_weight_tensor(w, ("sum",), log_input=True, dfs_order=dfs)[0], k, normalizer=n),
                                           4.0 * B * V + 4.0 * B * N + 4.0 * B * D),
                }
                res = {}
                for name, (fn, nbytes) in routes.items():
                    med, best = time_graph(fn, sets, args.steps, args.reps, stream)
                    res[name] = (med, best, nbytes)
                for name, (med, best, nbytes) in res.items():
                    line = {
                        "B": B, "order": order, "mix": mix, "route": name, "us_per_step": round(med, 2),
                        "us_per_step_min": round(best, 2), "bytes": int(nbytes), "GBps": round(nbytes / med / 1e3, 1),
                        "speedup_vs_c": round(res["c_slab_then_gather"][0] / med, 2), "V": V, "N": N, "D": D,
                        "buffer_sets": S, "steps_per_graph": args.steps, "gpu": gpu, "power_limit": power,
                    }
                    lines.append(line)
                    print(json.dumps(line), flush=True)
        del base
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
