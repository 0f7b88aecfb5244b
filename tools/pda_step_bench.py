"""Constrained token-level SMC step under a byte-level pushdown automaton: ``pda_token_mask`` ->
``masked_logsumexp_sample`` -> ``pda_advance``, against the DFA step on the same rows and the PDA calls on a DFA.

For two vocabularies -- the 128,256-token ``synth_vocab`` and the JSON-shaped vocabulary of ``tests/pda_oracle.py``
(1,230 items: the bytes, EOS and chunks of JSON documents) -- B in {64, 1024} root rows and two row mixes:

  depth0   half the rows at the start of a document, half inside a top-level string (empty stacks)
  depth32  half the rows after ``[{"k":`` x 16 (32 open containers), half inside a string there

it times with CUDA events over a CUDA graph of K steps:

  pda_mask        ``pda_token_mask`` under ``json_pda``                                   gt_pda_token_mask
  pda_step        pda_mask -> ``masked_logsumexp_sample`` -> ``pda_advance``
  dfa_mask        ``dfa_token_mask`` under a trimmed random DFA with json_pda's state count, random start states
  dfa_step        dfa_mask -> ``masked_logsumexp_sample`` -> ``dfa_advance``
  pdadfa_mask     ``pda_token_mask`` on that DFA with ``push`` all -1 and empty stacks (the same masks)
  pdadfa_step     pdadfa_mask -> ``masked_logsumexp_sample`` -> ``pda_advance``

(the DFA routes do not depend on the mix; they are timed again beside each mix).

``--weighted`` adds the same step under weighted automata: ``json_pda`` and the DFA get seeded log-weights (normal,
scale 0.5) on every transition, and four routes are timed on the same rows:

  pda_logw        ``pda_token_logw`` under the weighted ``json_pda``                      gt_pda_token_logw
  pda_wstep       pda_logw -> ``masked_logsumexp_sample(logps, tokw)`` -> ``pda_advance``
  dfa_logw        ``dfa_token_logw`` under the weighted DFA                               gt_dfa_token_logw
  pdadfa_logw     ``pda_token_logw`` on that DFA with ``push`` all -1 and empty stacks (the same log-weights)

with ``vs_boolean``, a route's time over its Boolean counterpart's on the same rows (pda_mask, pda_step, dfa_mask,
pdadfa_mask).  pdadfa_logw is checked bit-equal to dfa_logw before timing.  Without the flag the lines are unchanged.

The advance updates stacks and depths in place, so each PDA step first copies the rows' stacks and depths to scratch
tensors (two copies) and advances those: every replay starts from the same configurations.  The DFA step has no such
copies.  ``vs_dfa`` is a route's time over the matching DFA route's.  Step k reads buffer set k % sets of log-softmax
rows and DFA start states, with the rows of all sets covering more than three times the 126 MB L2 at V = 128,256 (at
most 64 sets: the JSON vocabulary's rows stay in L2).
Before timing, the PDA calls on the push-free table are checked to give exactly the DFA calls' masks and states.
Prints one JSON line per (vocab, B, mix, route) with the card's name and power limit; ``--out`` also writes them to a
file.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from genlm_backend_b200 import ParallelTokenCharacterTrie, pda, smc  # noqa: E402
from genlm_backend_b200.synthetic import logsoftmax_rows, synth_vocab  # noqa: E402
from child_step_bench import L2_BYTES, gpu_info, time_graph  # noqa: E402
from dfa_step_bench import random_dfa  # noqa: E402
import pda_oracle  # noqa: E402

PREFIXES = {"depth0": (b"", b'"ab'), "depth32": (b'[{"k":' * 16, b'[{"k":' * 16 + b'"ab')}


def configurations(delta, push, start, mix, B, cap):
    """(states, stack [B, cap], depth) after the two prefixes of ``mix``, alternating by row."""
    states = np.empty(B, np.int32)
    stack = np.zeros((B, cap), np.int32)
    depth = np.empty(B, np.int32)
    for b in range(B):
        q, stk = pda_oracle.walk(delta, push, start, [], list(PREFIXES[mix][b % 2]), cap)
        assert q >= 0
        states[b], depth[b] = q, len(stk)
        stack[b, :len(stk)] = stk
    return states, stack, depth


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="64,1024")
    ap.add_argument("--vocabs", default="synth128256,json")
    ap.add_argument("--steps", type=int, default=20, help="K: steps per CUDA graph")
    ap.add_argument("--reps", type=int, default=10, help="graph replays timed (median reported)")
    ap.add_argument("--weighted", action="store_true", help="also the routes under weighted automata")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "pda_step_bench.py measures on a GPU"
    gpu, power = gpu_info()
    stream = torch.cuda.Stream()
    cap = pda.GT_PDA_MAX_DEPTH
    lines = []
    for vname in args.vocabs.split(","):
        dec = synth_vocab(128256) if vname == "synth128256" else pda_oracle.json_vocab()
        trie = ParallelTokenCharacterTrie(dec)
        V, S = len(dec), trie.num_symbols
        eos = 256 if S > 256 else None
        jd, jp, start = pda.json_pda(S, eos=eos)
        Q = jd.shape[0]
        dd = random_dfa(Q, S, seed=3)
        jd_c, jp_c, dd_c = (torch.tensor(x).cuda() for x in (jd, jp, dd))
        nopush = torch.full_like(dd_c, -1)
        wrng = np.random.default_rng(5)
        jw_c, dw_c = (torch.tensor((wrng.normal(size=x.shape) * 0.5).astype(np.float32)).cuda() for x in (jd, dd))
        for B in [int(x) for x in args.batches.split(",")]:
            sets = min(64, max(2, -(-3 * L2_BYTES // (4 * B * V))))
            logps = [torch.tensor(logsoftmax_rows(B, V, seed=s)).cuda() for s in range(sets)]
            scratch_stack = torch.zeros((B, cap), dtype=torch.int32, device="cuda")
            scratch_depth = torch.zeros(B, dtype=torch.int32, device="cuda")
            for mix in PREFIXES:
                st, stk, dep = (torch.tensor(x).cuda() for x in configurations(jd, jp, start, mix, B, cap))
                rng = np.random.default_rng(7)
                dfa_states = [torch.tensor(rng.integers(0, Q, B).astype(np.int32)).cuda() for _ in range(sets)]
                zero_stack, zero_depth = torch.zeros_like(stk), torch.zeros_like(dep)

                def pda_step(d, p, lp, q, s, n):
                    bits = trie.pda_token_mask(d, p, q, s, n)
                    _, tok = smc.masked_logsumexp_sample(lp, bits, seed=1)
                    scratch_stack.copy_(s)
                    scratch_depth.copy_(n)
                    return bits, tok, trie.pda_advance(d, p, q, scratch_stack, scratch_depth, tok)

                def pda_wstep(lp, q, s, n):
                    tokw = trie.pda_token_logw(jd_c, jp_c, jw_c, q, s, n)
                    _, tok = smc.masked_logsumexp_sample(lp, tokw, seed=1)
                    scratch_stack.copy_(s)
                    scratch_depth.copy_(n)
                    return tokw, tok, trie.pda_advance(jd_c, jp_c, q, scratch_stack, scratch_depth, tok)

                def dfa_step(lp, q):
                    bits = trie.dfa_token_mask(dd_c, q)
                    _, tok = smc.masked_logsumexp_sample(lp, bits, seed=1)
                    return bits, tok, trie.dfa_advance(dd_c, q, tok)

                routes = {
                    "pda_mask": (lambda lp, q: trie.pda_token_mask(jd_c, jp_c, st, stk, dep), "dfa_mask"),
                    "pda_step": (lambda lp, q: pda_step(jd_c, jp_c, lp, st, stk, dep), "dfa_step"),
                    "dfa_mask": (lambda lp, q: trie.dfa_token_mask(dd_c, q), None),
                    "dfa_step": (dfa_step, None),
                    "pdadfa_mask": (lambda lp, q: trie.pda_token_mask(dd_c, nopush, q, zero_stack, zero_depth), "dfa_mask"),
                    "pdadfa_step": (lambda lp, q: pda_step(dd_c, nopush, lp, q, zero_stack, zero_depth), "dfa_step"),
                }
                boolean = {}
                if args.weighted:
                    routes.update({
                        "pda_logw": (lambda lp, q: trie.pda_token_logw(jd_c, jp_c, jw_c, st, stk, dep), "dfa_logw"),
                        "pda_wstep": (lambda lp, q: pda_wstep(lp, st, stk, dep), None),
                        "dfa_logw": (lambda lp, q: trie.dfa_token_logw(dd_c, dw_c, q), None),
                        "pdadfa_logw": (lambda lp, q: trie.pda_token_logw(dd_c, nopush, dw_c, q, zero_stack, zero_depth),
                                        "dfa_logw"),
                    })
                    boolean = {"pda_logw": "pda_mask", "pda_wstep": "pda_step", "dfa_logw": "dfa_mask",
                               "pdadfa_logw": "pdadfa_mask"}
                    for s in range(2):  # the PDA log-weights on the push-free table are the DFA's
                        assert torch.equal(routes["pdadfa_logw"][0](logps[s], dfa_states[s]).view(torch.int32),
                                           routes["dfa_logw"][0](logps[s], dfa_states[s]).view(torch.int32)), (vname, B)
                for s in range(2):  # the PDA calls on the push-free table give the DFA calls' results
                    for have, want in zip(routes["pdadfa_step"][0](logps[s], dfa_states[s]), dfa_step(logps[s], dfa_states[s])):
                        assert torch.equal(have, want), (vname, B)
                bufs = list(zip(logps, dfa_states))
                allowed = float(smc.masked_logsumexp_sample(logps[0], trie.pda_token_mask(jd_c, jp_c, st, stk, dep))[1]
                                .ge(0).float().mean().item())
                res = {r: time_graph(fn, bufs, args.steps, args.reps, stream) for r, (fn, _) in routes.items()}
                for r, (med, best) in res.items():
                    other = routes[r][1]
                    line = {
                        "vocab": vname, "B": B, "mix": mix, "route": r, "us_per_step": round(med, 2),
                        "us_per_step_min": round(best, 2),
                        "vs_dfa": round(med / res[other][0], 3) if other in res else None,
                        "rows_with_a_draw": round(allowed, 3), "states": Q, "stack_ld": cap,
                        "mean_depth": float(dep.float().mean().item()), "V": V, "S": S,
                        "Lmax": int(max(len(getattr(t, "byte_string", b"")) for t in dec)),
                        "buffer_sets": sets, "steps_per_graph": args.steps, "gpu": gpu, "power_limit": power,
                    }
                    if args.weighted:
                        line["vs_boolean"] = round(med / res[boolean[r]][0], 3) if r in boolean else None
                    lines.append(line)
                    print(json.dumps(line), flush=True)
            del logps
            torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
