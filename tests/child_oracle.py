"""Reference values of the child read-out, built on the oracle's public API (``oracle.OracleTrie`` /
``oracle.OracleLayout`` ``weight_sum`` / ``weight_max``, the C restatement of the numba loops, fp64).

``child_masses(trie, ws, nodes, op)`` is ``weight_sum`` / ``weight_max`` of row ``ws[b]`` indexed at ``jump[nodes[b]]``
-- what a character-level sampler reads through the slab -- padded to the largest child count the way
``gt_child_masses`` pads: id -1 and mass 0 for the columns past a node's degree, and for an id outside ``[0, N)`` or
a leaf.  ``tests/test_child_masses.py`` pins it to the reference's golden sums.
"""
import numpy as np


def max_children(trie):
    return int(np.diff(trie.jump_ptr).max()) if trie.n_nodes else 0


def child_ids(trie, nodes):
    """int32 ``[B, D]``: ``jump[nodes[b]]`` padded with -1."""
    D = max_children(trie)
    out = np.full((len(nodes), D), -1, dtype=np.int32)
    for b, n in enumerate(np.asarray(nodes, dtype=np.int64).tolist()):
        if 0 <= n < trie.n_nodes:
            kids = trie.jump_idx[trie.jump_ptr[n]:trie.jump_ptr[n + 1]]
            out[b, :len(kids)] = kids
    return out


def child_masses(trie, ws, nodes, op="sum"):
    """float64 ``[B, D]``: ``weight_sum`` (``op="sum"``) or ``weight_max`` of row ``ws[b]`` at ``child_ids``, padded
    with 0.  One row at a time, so a large vocabulary needs only one ``[N]`` array in memory."""
    ws = np.atleast_2d(np.asarray(ws))
    ids = child_ids(trie, nodes)
    assert ws.shape[0] == len(ids), [ws.shape, len(ids)]
    reduce = trie.weight_sum if op == "sum" else trie.weight_max
    out = np.zeros(ids.shape, dtype=np.float64)
    for b in range(len(ids)):
        k = ids[b] >= 0
        if k.any():
            out[b, k] = reduce(ws[b])[ids[b, k]]
    return out
