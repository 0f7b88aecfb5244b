"""Constrained token-level SMC step under a byte DFA: the token mask and the advance computed from the trie, against the
torch composition a caller writes today.

For V = 128,256 (synthetic vocabulary), B in {64, 1024}, the node mixes ``root`` and ``depth1`` of ``child_step_bench.py``,
random live start states, and three seeded, trimmed DFAs over the 256 byte symbols:

  utf8     the 8-state UTF-8 validity automaton (character classes of lead and continuation bytes, written as a table)
  rand256  a random 256-state table (each entry live with probability 0.9)
  rand4096 a random 4096-state table (4 MB: larger than any shared-memory staging of the table)

it times with CUDA events over a CUDA graph of K steps:

  (a) ``dfa_token_mask``                                                       gt_dfa_token_mask
  (b) padded ``[V, Lmax]`` symbol matrix, ``Lmax`` steps of ``state = delta[state, sym[:, k]]`` masked by length and
      node depth, a liveness test and ``smc._pack_keep_bits``                  today's torch composition of the mask
  (c) ``dfa_token_mask`` -> ``masked_logsumexp_sample`` -> ``dfa_advance``     the whole step on the trie
  (d) (b) -> ``masked_logsumexp_sample`` -> a torch advance of ``Lmax`` gathers

``--weighted`` times the step under a weighted automaton instead: each table gets seeded log-weights (normal, scale 0.5)
on its live transitions, and the routes are

  (a) ``dfa_token_logw``                                                       gt_dfa_token_logw
  (b) the walk of (b) gathering ``delta`` and ``logw`` at each step, an fp64 sum, -inf where rejected
  (c) ``dfa_token_logw`` -> ``masked_logsumexp_sample(logps, tokw)`` (per-row fp32 additive mask) -> ``dfa_advance``
  (d) (b) -> ``masked_logsumexp_sample`` -> the torch advance
  (m) ``dfa_token_mask`` and (s) the Boolean step of (c) above, on the same rows: what the weights and the additive mask
      cost over the bits (``vs_boolean`` = (a) / (m) and (c) / (s)).

``--routes`` and ``--dfas`` time a subset (comma-separated route and table names).

Step k reads buffer set k % sets of log-softmax rows, states and nodes, with the rows of all sets covering more than three
times the 126 MB L2.  Before timing, (b) and (d) are checked to compute exactly what (a) and (c) compute (when both are timed).  ``speedup`` is
(b) / (a) for the mask and (d) / (c) for the step.  Prints one JSON line per (B, dfa, mix, route); ``--out`` also writes
them to a file.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from genlm_backend_b200 import ParallelTokenCharacterTrie, dfa, smc  # noqa: E402
from genlm_backend_b200.synthetic import logsoftmax_rows, synth_vocab  # noqa: E402
from child_step_bench import L2_BYTES, gpu_info, node_mix, time_graph  # noqa: E402


def utf8_dfa(S):
    """States: 0 boundary (accepting), 1/2/3 continuation bytes still needed, 4 after E0, 5 after ED, 6 after F0,
    7 after F4 (the lead bytes whose next byte has a narrower range)."""
    d = np.full((8, S), -1, dtype=np.int32)
    d[0, 0x00:0x80] = 0
    d[0, 0xC2:0xE0] = 1
    d[0, 0xE1:0xED] = 2
    d[0, 0xEE:0xF0] = 2
    d[0, 0xE0], d[0, 0xED] = 4, 5
    d[0, 0xF1:0xF4] = 3
    d[0, 0xF0], d[0, 0xF4] = 6, 7
    d[1, 0x80:0xC0] = 0
    d[2, 0x80:0xC0] = 1
    d[3, 0x80:0xC0] = 2
    d[4, 0xA0:0xC0] = 1
    d[5, 0x80:0xA0] = 1
    d[6, 0x90:0xC0] = 2
    d[7, 0x80:0x90] = 2
    return dfa.trim(d, [0])


def random_dfa(Q, S, seed, p_live=0.9):
    rng = np.random.default_rng(seed)
    d = np.where(rng.random((Q, S)) < p_live, rng.integers(0, Q, (Q, S)), -1)
    return dfa.trim(d, rng.choice(Q, max(1, Q // 4), replace=False))


class TorchDfa:
    """The torch composition: every token's symbols as a padded [V, Lmax] matrix, walked Lmax steps for all rows."""

    def __init__(self, trie, device):
        lay = trie._layout
        V, N = len(trie.decode), len(trie)
        syms = [list(t.byte_string) for t in trie.decode]
        self.Lmax = max(len(s) for s in syms)
        sym = np.zeros((V, self.Lmax), dtype=np.int64)
        for i, s in enumerate(syms):
            sym[i, :len(s)] = s
        depth = np.zeros(N, dtype=np.int64)
        for n in range(N - 2, -1, -1):
            depth[n] = depth[lay["parent"][n]] + (lay["edge_label"][n] >= 0)
        rank = np.empty(V, dtype=np.int64)
        rank[lay["perm"]] = np.arange(V)
        t = lambda a: torch.tensor(a, dtype=torch.int64, device=device)  # noqa: E731
        self.sym, self.lens, self.rank = t(sym), t([len(s) for s in syms]), t(rank)
        self.depth, self.lo, self.hi = t(depth), t(lay["lo"]), t(lay["hi"])
        self.V = V

    def _walk(self, delta, st, d, sym_of, lens, logw=None):
        Q, ld = delta.shape
        flat = delta.reshape(-1).long()
        wflat = None if logw is None else logw.reshape(-1)
        acc = None if logw is None else torch.zeros(st.shape, dtype=torch.float64, device=st.device)
        for k in range(self.Lmax):
            act = (st >= 0) & (k >= d) & (k < lens)
            idx = st.clamp(min=0) * ld + sym_of(k)
            nxt = flat[idx]
            if logw is not None:
                acc = torch.where(act, acc + wflat[idx].double(), acc)
            st = torch.where(act, torch.where((nxt >= 0) & (nxt < Q), nxt, -1), st)
        return st if logw is None else (st, acc)

    def _start(self, delta, states, nodes):
        Q = delta.shape[0]
        n, q = nodes.long(), states.long()
        inside = ((self.rank[None, :] - self.lo[n][:, None]) >= 0) & (self.rank[None, :] < self.hi[n][:, None])
        return torch.where(inside & ((q >= 0) & (q < Q))[:, None], q[:, None], -1), self.depth[n][:, None]

    def mask(self, delta, states, nodes):
        st, d = self._start(delta, states, nodes)
        st = self._walk(delta, st, d, lambda k: self.sym[:, k][None, :], self.lens[None, :])
        return smc._pack_keep_bits((st >= 0).reshape(-1)).view(states.shape[0], -1)  # V is a multiple of 32

    def logw(self, delta, logw, states, nodes):
        st, d = self._start(delta, states, nodes)
        st, acc = self._walk(delta, st, d, lambda k: self.sym[:, k][None, :], self.lens[None, :], logw)
        return torch.where(st >= 0, acc.float(), float("-inf"))

    def advance(self, delta, states, nodes, tok):
        Q = delta.shape[0]
        n, q = nodes.long(), states.long()
        t = tok.long().clamp(0, self.V - 1)
        ok = (tok >= 0) & (tok < self.V) & (self.rank[t] >= self.lo[n]) & (self.rank[t] < self.hi[n]) & (q >= 0) & (q < Q)
        st = self._walk(delta, torch.where(ok, q, -1), self.depth[n], lambda k: self.sym[t, k], self.lens[t])
        return st.int()


def random_logw(table, seed):
    """Seeded log-weights on the live transitions of ``table`` (normal, scale 0.5), 0 on the rejecting ones."""
    rng = np.random.default_rng(seed)
    return np.where(table >= 0, rng.normal(scale=0.5, size=table.shape), 0).astype(np.float32)


def as_tuple(x):
    return x if isinstance(x, tuple) else (x,)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="64,1024")
    ap.add_argument("--steps", type=int, default=20, help="K: steps per CUDA graph")
    ap.add_argument("--reps", type=int, default=10, help="graph replays timed (median reported)")
    ap.add_argument("--weighted", action="store_true", help="the step under a weighted automaton (legs a-d, m, s)")
    ap.add_argument("--routes", default=None, help="comma-separated subset of the routes to time")
    ap.add_argument("--dfas", default="utf8,rand256,rand4096", help="comma-separated subset of the tables")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "dfa_step_bench.py measures on a GPU"
    V = 128256
    trie = ParallelTokenCharacterTrie(synth_vocab(V))
    N, S = len(trie), trie.num_symbols
    ref = TorchDfa(trie, "cuda")
    tables = {"utf8": utf8_dfa(S), "rand256": random_dfa(256, S, seed=1), "rand4096": random_dfa(4096, S, seed=2)}
    seeds = {name: 10 + ti for ti, name in enumerate(tables)}  # the log-weights of a table do not depend on --dfas
    tables = {name: t for name, t in tables.items() if name in args.dfas.split(",")}
    gpu, power = gpu_info()
    stream = torch.cuda.Stream()
    lines = []
    for B in [int(x) for x in args.batches.split(",")]:
        sets = max(2, -(-3 * L2_BYTES // (4 * B * V)))
        logps = [torch.tensor(logsoftmax_rows(B, V, seed=s)).cuda() for s in range(sets)]
        for name, table in tables.items():
            delta = torch.tensor(table).cuda()
            logw = torch.tensor(random_logw(table, seed=seeds[name])).cuda()
            Q = table.shape[0]
            for mix in ("root", "depth1"):
                rng = np.random.default_rng(7)
                nodes = [torch.tensor(node_mix(trie, mix, B, rng)).cuda() for _ in range(sets)]
                states = [torch.tensor(rng.integers(0, Q, B).astype(np.int32)).cuda() for _ in range(sets)]
                bufs = list(zip(logps, states, nodes))

                def kernel_step(lp, st, nd):
                    bits = trie.dfa_token_mask(delta, st, nd)
                    _, tok = smc.masked_logsumexp_sample(lp, bits, seed=1)
                    return bits, tok, trie.dfa_advance(delta, st, tok, nd)

                def torch_step(lp, st, nd):
                    bits = ref.mask(delta, st, nd)
                    _, tok = smc.masked_logsumexp_sample(lp, bits, seed=1)
                    return bits, tok, ref.advance(delta, st, nd, tok)

                def kernel_logw_step(lp, st, nd):
                    tokw = trie.dfa_token_logw(delta, logw, st, nd)
                    logZ, tok = smc.masked_logsumexp_sample(lp, tokw, seed=1)
                    return tokw, logZ, tok, trie.dfa_advance(delta, st, tok, nd)

                def torch_logw_step(lp, st, nd):
                    tokw = ref.logw(delta, logw, st, nd)
                    logZ, tok = smc.masked_logsumexp_sample(lp, tokw, seed=1)
                    return tokw, logZ, tok, ref.advance(delta, st, nd, tok)

                if args.weighted:
                    routes = {
                        "a_dfa_token_logw": lambda lp, st, nd: trie.dfa_token_logw(delta, logw, st, nd),
                        "b_torch_logw": lambda lp, st, nd: ref.logw(delta, logw, st, nd),
                        "c_logw_sample_advance": kernel_logw_step,
                        "d_torch_logw_sample_advance": torch_logw_step,
                        "m_dfa_token_mask": lambda lp, st, nd: trie.dfa_token_mask(delta, st, nd),
                        "s_mask_sample_advance": kernel_step,
                    }
                    vs = {"a_dfa_token_logw": "b_torch_logw", "c_logw_sample_advance": "d_torch_logw_sample_advance"}
                    vs_bool = {"a_dfa_token_logw": "m_dfa_token_mask", "c_logw_sample_advance": "s_mask_sample_advance"}
                else:
                    routes = {
                        "a_dfa_token_mask": lambda lp, st, nd: trie.dfa_token_mask(delta, st, nd),
                        "b_torch_mask": lambda lp, st, nd: ref.mask(delta, st, nd),
                        "c_mask_sample_advance": kernel_step,
                        "d_torch_mask_sample_advance": torch_step,
                    }
                    vs, vs_bool = {"a_dfa_token_mask": "b_torch_mask", "c_mask_sample_advance": "d_torch_mask_sample_advance"}, {}
                if args.routes:
                    routes = {r: fn for r, fn in routes.items() if r in args.routes.split(",")}
                for r, other in vs.items():  # the torch composition computes exactly what the kernels compute
                    if r in routes and other in routes:
                        for s in range(min(sets, 2)):
                            for have, want in zip(as_tuple(routes[other](*bufs[s])), as_tuple(routes[r](*bufs[s]))):
                                assert torch.equal(have, want), (B, name, mix, r)
                allowed = float(np.mean([smc.masked_logsumexp_sample(lp, trie.dfa_token_mask(delta, st, nd))[1].ge(0)
                                         .float().mean().item() for lp, st, nd in bufs]))
                res = {r: time_graph(fn, bufs, args.steps, args.reps, stream) for r, fn in routes.items()}
                for r, (med, best) in res.items():
                    line = {
                        "B": B, "dfa": name, "states": Q, "mix": mix, "route": r, "us_per_step": round(med, 2),
                        "us_per_step_min": round(best, 2),
                        "speedup": round(res[vs[r]][0] / med, 2) if vs.get(r) in res else None,
                        "rows_with_a_draw": round(allowed, 3),
                        "V": V, "N": N, "S": S, "Lmax": ref.Lmax, "buffer_sets": sets, "steps_per_graph": args.steps,
                        "meta_bytes": trie._engine.plan_info()["meta_bytes"], "gpu": gpu, "power_limit": power,
                    }
                    if args.weighted:
                        line["vs_boolean"] = round(med / res[vs_bool[r]][0], 3) if vs_bool.get(r) in res else None
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
