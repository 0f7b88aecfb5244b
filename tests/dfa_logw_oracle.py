"""Reference for the token log-weights under a weighted byte DFA (``gt_dfa_token_logw``): the numpy walk of
``dfa_oracle.DfaOracle`` that also sums the walked transitions' log-weights.

Row ``b`` at node ``n`` in state ``q``: an item ``DfaOracle.mask`` allows gets the float64 sum of ``logw[q_k, s_k]``
over its symbols ``k = depth(n) .. len(i)-1`` (``q_k`` the state before ``s_k``), added in increasing ``k`` from 0.0 and
cast once to float32; every other item gets ``-inf``.
"""
import numpy as np

import dfa_oracle


class WeightedDfaOracle(dfa_oracle.DfaOracle):
    def _weighted_walk(self, delta, logw, q, n, items):
        """States after items' symbols depth(n) .. end from q (-1 once rejected), and the float64 sums of the walked
        transitions' log-weights (the rejecting transition's included: its item is -inf either way)."""
        Q = delta.shape[0]
        st = np.full(len(items), q, dtype=np.int64)
        acc = np.zeros(len(items), dtype=np.float64)
        for k in range(int(self.depth[n]), self.sym.shape[1]):
            act = (st >= 0) & (self.lens[items] > k)
            src, s = np.maximum(st[act], 0), self.sym[items[act], k]
            acc[act] += logw[src, s].astype(np.float64)
            nxt = delta[src, s]
            st[act] = np.where((nxt >= 0) & (nxt < Q), nxt, -1)
        return st, acc

    def logw(self, delta, logw, states, nodes=None):
        """float32 [B, V]: the float64 sum of logw along each allowed item's walk, cast to float32; -inf elsewhere."""
        delta = np.asarray(delta, dtype=np.int64)
        logw = np.asarray(logw, dtype=np.float32)
        states = np.asarray(states, dtype=np.int64)
        nodes = np.full(len(states), self.N - 1) if nodes is None else np.asarray(nodes, dtype=np.int64)
        out = np.full((len(states), self.V), -np.inf, dtype=np.float32)
        for b, (q, n) in enumerate(zip(states.tolist(), nodes.tolist())):
            if not (0 <= n < self.N and 0 <= q < delta.shape[0]):
                continue
            items = np.flatnonzero(self._under(n))
            st, acc = self._weighted_walk(delta, logw, q, n, items)
            out[b, items] = np.where(st >= 0, acc, -np.inf).astype(np.float32)
        return out
