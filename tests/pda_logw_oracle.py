"""Reference for the token log-weights under a weighted byte-level pushdown automaton (``gt_pda_token_logw``): the numpy
walk of ``pda_oracle.PdaOracle``, which copies each row's stack and pushes and pops on the copy, extended to sum the
walked transitions' log-weights.

Row ``b`` at the root in configuration ``(states[b], stack[b, :depth[b]])``: an item ``PdaOracle.mask`` allows gets the
float64 sum of ``logw[q_k, s_k]`` over all its symbols (``q_k`` the state before ``s_k``; a move, a push or a pop
alike), added in increasing ``k`` from 0.0 and cast once to float32; every other item gets ``-inf``.
"""
import numpy as np

import pda_oracle
from genlm_backend_b200.pda import GT_PDA_POP


class WeightedPdaOracle(pda_oracle.PdaOracle):
    def _weighted_walk(self, delta, push, logw, q, row_stack, cap, items):
        """Every item of ``items`` walked from ``(q, row_stack)``: the states after it (-1 once rejected) and the
        float64 sums of the walked transitions' log-weights (the rejecting transition's included: its item is -inf
        either way).  The same steps as ``PdaOracle._walk``; the row must be valid."""
        Q = delta.shape[0]
        n = len(items)
        st = np.full(n, q, dtype=np.int64)
        acc = np.zeros(n, dtype=np.float64)
        stk = np.zeros((n, cap), dtype=np.int64)
        stk[:, :len(row_stack)] = row_stack
        d = np.full(n, len(row_stack), dtype=np.int64)
        lens, sym = self.lens[items], self.sym[items]
        for k in range(int(lens.max(initial=0))):
            a = np.flatnonzero((st >= 0) & (lens > k))
            if not a.size:
                break
            cur, s, da = st[a], sym[a, k], d[a]
            acc[a] += logw[cur, s].astype(np.float64)
            nq, pu = delta[cur, s], push[cur, s]
            new = np.full(a.size, -1, dtype=np.int64)
            move = (nq >= 0) & (nq < Q)
            plain = move & (pu < 0)
            new[plain] = nq[plain]
            pushes = move & (pu >= 0) & (pu < Q) & (da < cap)
            at = a[pushes]
            stk[at, da[pushes]] = pu[pushes]
            d[at] += 1
            new[pushes] = nq[pushes]
            pops = (nq == GT_PDA_POP) & (da > 0)
            at = a[pops]
            v = stk[at, da[pops] - 1]
            d[at] -= 1
            new[pops] = np.where((v >= 0) & (v < Q), v, -1)
            st[a] = new
        return st, acc

    def logw(self, delta, push, logw, states, stack, depth):
        """float32 [B, V]: the float64 sum of logw along each allowed item's walk, cast to float32; -inf elsewhere."""
        delta, push, states, stack, depth, cap = self._rows(delta, push, states, stack, depth)
        logw = np.asarray(logw, dtype=np.float32)
        out = np.full((len(states), self.V), -np.inf, dtype=np.float32)
        items = np.arange(self.V)
        for b, (q, dep) in enumerate(zip(states.tolist(), depth.tolist())):
            if 0 <= q < delta.shape[0] and 0 <= dep <= cap:
                st, acc = self._weighted_walk(delta, push, logw, q, stack[b, :dep], cap, items)
                out[b] = np.where(st >= 0, acc, -np.inf).astype(np.float32)
        return out
