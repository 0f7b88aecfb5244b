"""Exact constrained byte-level step: next-symbol read-outs restricted to the tokens a keep-bitmask allows, against the
composition a caller writes without them.

For V = 128,256 (synthetic vocabulary), log-softmax fp32 rows, B in {64, 1024}, rows in vocabulary and in DFS order, the
node mixes of ``child_step_bench.py`` (``root``, ``depth1``, ``walk``) and two per-row masks in item order --

  dfa   ``dfa_token_mask`` of the UTF-8 automaton of ``dfa_step_bench.py`` at the root, random live start states
  rand  a random mask of density 0.05

-- it times with CUDA events over a CUDA graph of K steps, per-row symbol log-weights as in ``symbol_step_bench.py``:

  (a) ``batch_symbol_masses_tensor(mask=bits)`` and ``sample_next_symbol_weighted(mask=bits)``
  (b) unpack the bits, ``torch.where(keep, rows, -inf)`` into a fresh ``[B, V]`` tensor, then the unmasked call
  (u) the unmasked call on the same rows: (a) / (u) is the price of the mask lookups

Step k reads buffer set k % sets (rows, nodes, masks, log-weights), with the rows covering more than three times the
126 MB L2.  Before timing, (a) and (b) are checked to be bit-equal.  ``b_over_a`` is (b) / (a), ``a_over_u`` (a) / (u).
Prints one JSON line per (B, order, mix, mask, call); ``--out`` also writes them to a file.
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
from dfa_step_bench import utf8_dfa  # noqa: E402


def unpack(bits, V):
    """int32 keep-bitmask [B, ceil(V/32)] -> bool [B, V] (what a caller does to apply it with torch.where)."""
    shifts = torch.arange(32, device=bits.device, dtype=torch.int32)
    return ((bits[:, :, None] >> shifts) & 1).reshape(bits.shape[0], -1)[:, :V].bool()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="64,1024")
    ap.add_argument("--steps", type=int, default=20, help="K: steps per CUDA graph")
    ap.add_argument("--reps", type=int, default=10, help="graph replays timed (median reported)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "masked_step_bench.py measures on a GPU"
    V = 128256
    trie = ParallelTokenCharacterTrie(synth_vocab(V))
    N, S = len(trie), trie.num_symbols
    W = (V + 31) // 32
    dfs_perm = trie.dfs_token_order.cuda()
    delta = torch.tensor(utf8_dfa(S)).cuda()
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
        mrng = np.random.default_rng(5)
        masks = {
            "dfa": [trie.dfa_token_mask(delta, torch.tensor(mrng.integers(0, delta.shape[0], B).astype(np.int32)).cuda())
                    for _ in range(sets)],
            "rand": [trie._engine.keep_bits(torch.tensor(mrng.random((B, V)) < 0.05).cuda(), B, "cuda")[0]
                     for _ in range(sets)],
        }
        for order in ("vocab", "dfs"):
            dfs = order == "dfs"
            rows = base if not dfs else [r[:, dfs_perm].contiguous() for r in base]
            for mix in ("root", "depth1", "walk"):
                rng = np.random.default_rng(7)
                nt = [torch.tensor(node_mix(trie, mix, B, rng)).cuda() for _ in range(sets)]
                for mname, bits in masks.items():
                    density = float(np.mean([unpack(b, V).float().mean().item() for b in bits]))
                    bufs = list(zip(rows, nt, logws, bits))
                    kw = dict(log_input=True, dfs_order=dfs)

                    def zeroed(w, m):  # the caller's pass: a fresh [B, V] with the masked-out log-weights at -inf
                        keep = unpack(m, V)
                        return torch.where(keep[:, dfs_perm] if dfs else keep, w, float("-inf"))

                    calls = {
                        "symbol_masses": (
                            lambda w, n, lw, m: trie.batch_symbol_masses_tensor(w, n, normalize=True, mask=m, **kw),
                            lambda w, n, lw, m: trie.batch_symbol_masses_tensor(zeroed(w, m), n, normalize=True, **kw),
                            lambda w, n, lw, m: trie.batch_symbol_masses_tensor(w, n, normalize=True, **kw)),
                        "weighted_draw": (
                            lambda w, n, lw, m: trie.sample_next_symbol_weighted(w, n, lw, seed=1, mask=m, **kw),
                            lambda w, n, lw, m: trie.sample_next_symbol_weighted(zeroed(w, m), n, lw, seed=1, **kw),
                            lambda w, n, lw, m: trie.sample_next_symbol_weighted(w, n, lw, seed=1, **kw)),
                    }
                    for call, (a, b, u) in calls.items():
                        for s in range(min(sets, 2)):
                            for x, y in zip(a(*bufs[s]), b(*bufs[s])):
                                assert (x is None) == (y is None)
                                assert x is None or torch.equal(x.view(torch.int32), y.view(torch.int32)), (B, order, mix, mname, call)
                        ta, tb, tu = (time_graph(fn, bufs, args.steps, args.reps, stream) for fn in (a, b, u))
                        line = {
                            "B": B, "order": order, "mix": mix, "mask": mname, "call": call,
                            "a_masked_us": round(ta[0], 2), "b_where_then_unmasked_us": round(tb[0], 2),
                            "u_unmasked_us": round(tu[0], 2), "a_masked_us_min": round(ta[1], 2),
                            "b_over_a": round(tb[0] / ta[0], 2), "a_over_u": round(ta[0] / tu[0], 3),
                            "mask_density": round(density, 4), "V": V, "N": N, "S": S, "words": W,
                            "buffer_sets": sets, "steps_per_graph": args.steps, "gpu": gpu, "power_limit": power,
                        }
                        lines.append(line)
                        print(json.dumps(line), flush=True)
        del base, logws, masks
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
