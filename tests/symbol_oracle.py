"""Reference values of the symbol read-out and of the weighted next-symbol draw, built on ``child_oracle`` (the fp64
oracle's ``weight_sum`` / ``weight_max`` at each node's children).

Symbols are restated from the vocabulary alone: a byte is its value; any other label gets ``256, 257, ...`` in order
of first appearance; ``S = max(256, 1 + largest symbol)``, and column ``S`` stands for "the token ends here" (a leaf
child).  The symbol of each child is read off the reference layout by walking every item's path from its leaf up to
the root.  ``tests/test_symbol_masses.py`` pins these to the reference's golden sums.
"""
import numpy as np

import child_oracle


def item_symbols(decode):
    """``(list of int lists, S)``: each item's symbols and the symbol count."""
    table, out = {}, []
    for item in decode:
        word = item.byte_string if hasattr(item, "byte_string") else item
        syms = []
        for letter in word:
            if isinstance(letter, int) and 0 <= letter < 256:
                syms.append(letter)
            else:
                syms.append(table.setdefault(letter, 256 + len(table)))
        out.append(syms)
    return out, 256 + len(table)


def child_symbols(trie, decode):
    """``(sym int32[N], S)``: the symbol of the edge into each node (``S`` for a leaf, -1 for the root), from the
    reference layout ``trie`` (``jump``, ``idx_to_leaf``) and the vocabulary."""
    syms, S = item_symbols(decode)
    N = trie.n_nodes
    parent = np.full(N, -1, dtype=np.int64)
    for n in range(N):
        parent[trie.jump_idx[trie.jump_ptr[n]:trie.jump_ptr[n + 1]]] = n
    sym = np.full(N, -1, dtype=np.int64)
    for i, word in enumerate(syms):
        leaf = int(trie.idx_to_leaf[i, 1])
        sym[leaf] = S
        n = int(parent[leaf])
        for s in reversed(word):  # the node reached by the last symbol is the leaf's parent
            assert sym[n] in (-1, s), (n, sym[n], s)
            sym[n] = s
            n = int(parent[n])
        assert n == N - 1, "the path of an item ends at the root"
    return sym, S


def symbol_masses(trie, sym, S, ws, nodes, op="sum"):
    """float64 ``[B, S+1]``: column ``s < S`` the child mass (``op`` = sum or max) of the child with symbol ``s``;
    column ``S`` the fp64 sum of the leaf children's sums in child order (or the max of their maxes); 0 elsewhere."""
    ids = child_oracle.child_ids(trie, nodes)
    m = child_oracle.child_masses(trie, ws, nodes, op)
    out = np.zeros((len(ids), S + 1), dtype=np.float64)
    for b in range(len(ids)):
        end, seen = 0.0, False
        for j in np.flatnonzero(ids[b] >= 0).tolist():
            s = int(sym[ids[b, j]])
            if s < S:
                out[b, s] = m[b, j]
            elif op == "sum":
                end += m[b, j]
            else:
                end = m[b, j] if not seen else max(end, m[b, j])
            seen |= s == S
        out[b, S] = end
    return out


def weighted_child_masses(trie, sym, ws, nodes, logw):
    """``(ids int32[B, D], m float64[B, D], q float64[B, D])``: the child masses and their weights
    ``q_j = m_j * exp(logw[b, sym(c_j)])`` (0 when ``m_j = 0`` whatever the log-weight; NaN for a NaN log-weight).
    ``logw`` is ``[S+1]`` or ``[B, S+1]``."""
    ids = child_oracle.child_ids(trie, nodes)
    m = child_oracle.child_masses(trie, ws, nodes, "sum")
    logw = np.asarray(logw, dtype=np.float64)
    if logw.ndim == 1:
        logw = np.broadcast_to(logw, (len(ids), logw.shape[0]))
    w = np.take_along_axis(logw, np.where(ids >= 0, sym[np.maximum(ids, 0)], 0), axis=1)
    with np.errstate(over="ignore", invalid="ignore"):
        q = np.where(m == 0, 0.0, m * np.exp(w))
    q = np.where(np.isnan(w), np.nan, q)
    q[ids < 0] = 0.0
    return ids, m, q
