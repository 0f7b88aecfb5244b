"""Next-symbol step of a constrained character-level sampler: masses by symbol and the weighted draw in one call each,
against today's composition of the child read-out with torch ops.

For V = 128,256 (synthetic vocabulary), log-softmax fp32 rows, B in {64, 1024}, rows in vocabulary and in DFS order, the
node mixes of ``child_step_bench.py`` (``root``, ``depth1``, ``walk``) and per-row symbol log-weights ``[B, S+1]``
(standard normal, about 30 % of the symbols at -inf), it times with CUDA events over a CUDA graph of K steps:

  (a) ``sample_next_symbol_weighted``                                  gt_symbol_sample
  (b) ``batch_child_masses_tensor(normalize=True)`` -> symbol gather -> ``q = p * logw.gather(1, sym).exp()``
      -> ``torch.multinomial(q, 1)``                                   today's composition of the draw
  (c) ``batch_symbol_masses_tensor(normalize=True)``                   gt_symbol_masses
  (d) ``batch_child_masses_tensor(normalize=True)`` + a torch ``scatter_add_`` into ``[B, S+1]``

Route (b) adds 1e-30 to every ``q`` so that no row is without mass (an invalid distribution for ``torch.multinomial``);
it changes no timing.  Step k reads buffer set k % sets, with sets covering more than three times the 126 MB
L2, so rows are not L2-resident.  ``bytes`` is the leaf weights read under the nodes (the same for every route).
``speedup`` is (b) / (a) for the draw and (d) / (c) for the masses.  Prints one JSON line per (B, order, mix, route);
``--out`` also writes them to a file.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from genlm_backend_b200 import ParallelTokenCharacterTrie  # noqa: E402
from genlm_backend_b200.synthetic import logsoftmax_rows, synth_vocab  # noqa: E402
from child_step_bench import L2_BYTES, gpu_info, node_mix, time_graph  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="64,1024")
    ap.add_argument("--steps", type=int, default=20, help="K: steps per CUDA graph")
    ap.add_argument("--reps", type=int, default=10, help="graph replays timed (median reported)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "symbol_step_bench.py measures on a GPU"
    V = 128256
    trie = ParallelTokenCharacterTrie(synth_vocab(V))
    N, D, S = len(trie), trie.max_children, trie.num_symbols
    size = (trie._layout["hi"] - trie._layout["lo"]).astype(np.int64)
    lab = trie.edge_labels
    node_sym = torch.tensor(np.where(lab >= 0, lab, S)).cuda()  # column of each node in the symbol read-outs
    dfs_perm = trie.dfs_token_order.cuda()
    gpu, power = gpu_info()
    stream = torch.cuda.Stream()
    lines = []
    for B in [int(x) for x in args.batches.split(",")]:
        sets = max(2, -(-3 * L2_BYTES // (4 * B * V)))
        base = [torch.tensor(logsoftmax_rows(B, V, seed=s)).cuda() for s in range(sets)]
        wrng = np.random.default_rng(11)
        logws = []
        for _ in range(sets):
            w = wrng.standard_normal((B, S + 1)).astype(np.float32)
            w[wrng.random((B, S + 1)) < 0.3] = -np.inf
            logws.append(torch.tensor(w).cuda())
        for order in ("vocab", "dfs"):
            rows = base if order == "vocab" else [r[:, dfs_perm].contiguous() for r in base]
            for mix in ("root", "depth1", "walk"):
                rng = np.random.default_rng(7)
                nodes = [node_mix(trie, mix, B, rng) for _ in range(sets)]
                nt = [torch.tensor(n).cuda() for n in nodes]
                bufs = list(zip(rows, nt, logws))
                dfs = order == "dfs"
                read = float(np.mean([4.0 * size[n].sum() for n in nodes]))

                def composed_draw(w, n, lw):
                    ids, p, _ = trie.batch_child_masses_tensor(w, n, log_input=True, dfs_order=dfs, normalize=True)
                    sym = node_sym[ids.clamp(min=0).long()]
                    q = p * lw.gather(1, sym).exp()
                    return torch.multinomial(q.add_(1e-30), 1)

                def scattered_masses(w, n, lw):
                    ids, p, _ = trie.batch_child_masses_tensor(w, n, log_input=True, dfs_order=dfs, normalize=True)
                    sym = node_sym[ids.clamp(min=0).long()]
                    return torch.zeros((B, S + 1), dtype=torch.float32, device=w.device).scatter_add_(1, sym, p)

                routes = {
                    "a_symbol_sample": lambda w, n, lw: trie.sample_next_symbol_weighted(
                        w, n, lw, seed=1, log_input=True, dfs_order=dfs),
                    "b_child_masses_then_torch_draw": composed_draw,
                    "c_symbol_masses": lambda w, n, lw: trie.batch_symbol_masses_tensor(
                        w, n, log_input=True, dfs_order=dfs, normalize=True),
                    "d_child_masses_then_scatter": scattered_masses,
                }
                res = {name: time_graph(fn, bufs, args.steps, args.reps, stream) for name, fn in routes.items()}
                vs = {"a_symbol_sample": "b_child_masses_then_torch_draw", "c_symbol_masses": "d_child_masses_then_scatter"}
                for name, (med, best) in res.items():
                    line = {
                        "B": B, "order": order, "mix": mix, "route": name, "us_per_step": round(med, 2),
                        "us_per_step_min": round(best, 2), "bytes": int(read), "GBps": round(read / med / 1e3, 1),
                        "speedup": round(res[vs[name]][0] / med, 2) if name in vs else None,
                        "V": V, "N": N, "D": D, "S": S, "buffer_sets": sets, "steps_per_graph": args.steps,
                        "gpu": gpu, "power_limit": power,
                    }
                    lines.append(line)
                    print(json.dumps(line), flush=True)
        del base, logws
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
