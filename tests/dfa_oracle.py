"""Reference for the token masks under a byte DFA and the DFA advance: a pure numpy walk over each item's symbols
(``symbol_oracle.item_symbols``), with node depths and subtrees taken from the reference layout (``oracle.OracleLayout``:
``jump`` and ``idx_to_leaf``), not from the kernels' DFS ranges.

Item ``i`` is allowed for a row at node ``n`` in state ``q`` iff ``n`` is on the path from the root to ``i``'s leaf (or
is that leaf), ``q`` is in ``[0, Q)``, and ``delta`` walked from ``q`` over symbols ``depth(n) .. len(i)-1`` stays in
``[0, Q)``.
"""
import numpy as np

import symbol_oracle


class DfaOracle:
    def __init__(self, layout, decode):
        syms, self.S = symbol_oracle.item_symbols(decode)
        V, N = layout.n_items, layout.n_nodes
        self.V, self.N = V, N
        self.lens = np.array([len(s) for s in syms], dtype=np.int64)
        L = int(self.lens.max()) if V else 0
        self.sym = np.zeros((V, max(L, 1)), dtype=np.int64)
        for i, s in enumerate(syms):
            self.sym[i, :len(s)] = s
        parent = np.full(N, -1, dtype=np.int64)
        for n in range(N):
            parent[layout.jump_idx[layout.jump_ptr[n]:layout.jump_ptr[n + 1]]] = n
        self.leaf = layout.idx_to_leaf[:, 1].astype(np.int64)
        # path[i, k]: the node at depth k on item i's path (k <= len(i)); the leaf's parent spells the whole item
        self.path = np.full((V, L + 1), -1, dtype=np.int64)
        self.path[np.arange(V), self.lens] = parent[self.leaf]
        for k in range(L, 0, -1):
            at = self.lens >= k
            self.path[at, k - 1] = parent[self.path[at, k]]
        assert (self.path[:, 0] == N - 1).all(), "every path starts at the root"
        self.depth = np.zeros(N, dtype=np.int64)
        for k in range(L + 1):
            ok = self.lens >= k
            self.depth[self.path[ok, k]] = k
        self.depth[self.leaf] = self.lens

    def _under(self, n):
        """bool [V]: items whose leaf lies under node n (n itself a leaf: that item only)."""
        d = int(self.depth[n])
        ok = self.lens >= d
        under = np.zeros(self.V, dtype=bool)
        under[ok] = self.path[ok, d] == n
        return under | (self.leaf == n)

    def _walk(self, delta, q, n, items):
        """States after items' symbols depth(n) .. end from q (-1 once rejected)."""
        Q = delta.shape[0]
        st = np.full(len(items), q, dtype=np.int64)
        for k in range(int(self.depth[n]), self.sym.shape[1]):
            act = (st >= 0) & (self.lens[items] > k)
            nxt = delta[np.maximum(st[act], 0), self.sym[items[act], k]]
            st[act] = np.where((nxt >= 0) & (nxt < Q), nxt, -1)
        return st

    def mask(self, delta, states, nodes=None):
        """bool [B, V]."""
        delta = np.asarray(delta, dtype=np.int64)
        states = np.asarray(states, dtype=np.int64)
        nodes = np.full(len(states), self.N - 1) if nodes is None else np.asarray(nodes, dtype=np.int64)
        out = np.zeros((len(states), self.V), dtype=bool)
        for b, (q, n) in enumerate(zip(states.tolist(), nodes.tolist())):
            if not (0 <= n < self.N and 0 <= q < delta.shape[0]):
                continue
            items = np.flatnonzero(self._under(n))
            out[b, items] = self._walk(delta, q, n, items) >= 0
        return out

    def advance(self, delta, states, tokens, nodes=None):
        """int64 [B]: the state after the token's remaining symbols, or -1."""
        delta = np.asarray(delta, dtype=np.int64)
        nodes = np.full(len(states), self.N - 1) if nodes is None else np.asarray(nodes, dtype=np.int64)
        out = np.full(len(states), -1, dtype=np.int64)
        for b, (q, n, t) in enumerate(zip(np.asarray(states).tolist(), nodes.tolist(), np.asarray(tokens).tolist())):
            if 0 <= t < self.V and 0 <= n < self.N and 0 <= q < delta.shape[0] and self._under(n)[t]:
                out[b] = self._walk(delta, q, n, np.array([t]))[0]
        return out


def random_dfa(rng, Q, S, p_live=0.7, n_accept=None):
    """A random table of Q states over S symbols: each entry a uniform state with probability p_live, else -1; the
    accepting states are a random subset."""
    delta = np.where(rng.random((Q, S)) < p_live, rng.integers(0, Q, (Q, S)), -1).astype(np.int32)
    acc = rng.choice(Q, n_accept or max(1, Q // 4), replace=False)
    return delta, acc
