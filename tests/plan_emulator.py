"""CPU emulation of the data flow of csrc/mass_kernels.cu, driven by the plan arrays the C++ planner produced
(gt_export_plan_array).  Test infrastructure: it lets the ``-m "not gpu"`` suite check the planner's metadata
(staging layout, value slots, aligned-block decomposition, spanning fix-up) against the oracle without a GPU.
Float32 arithmetic in the same association order as the kernels (pairwise pyramid, sequential term sums).
"""
import numpy as np


def swizzle_slot(s, slot_bytes):
    """Python twin of gt::swizzle_slot (csrc/trie_internal.h)."""
    cs = {4: 2, 8: 1, 16: 0}[slot_bytes]
    c = s >> cs
    return ((c ^ ((c >> 3) & (slot_bytes // 2 - 1))) << cs) | (s & ((1 << cs) - 1))


def emulate(engine, ws, op="sum"):
    """ws: float32 [B, V].  Returns float32 [B, N] computed the way mass_kernel / span_kernel do."""
    info = engine.plan_info()
    A = {name: engine.plan_array(name) for name in (
        "leaf_dest", "ell_chunk_ptr", "ell_desc", "ell_terms",
        "tile_node_lo", "node_slot", "piece_ptr", "piece_slot", "piece_idx", "span_node", "span_pp")}
    T, NT = info["tile_leaves"], info["n_tiles"]
    V, N, ZG = info["n_tokens"], info["n_nodes"], info["staged_slots"]
    assert ZG == NT * T
    phys = swizzle_slot(np.arange(2 * T), 4 * info["rows_per_item"])  # where logical slot s < 2T lives
    ws = np.asarray(ws, dtype=np.float32)
    B = ws.shape[0]
    red = np.add if op == "sum" else np.fmax
    ident = np.float32(0.0) if op == "sum" else np.float32(-np.inf)

    # permute role: every weight goes to its (tile, swizzled leaf slot) of the staging block
    z = np.full((B, ZG), np.nan, dtype=np.float32)
    dest = A["leaf_dest"].astype(np.int64)
    assert len(np.unique(dest)) == V and (V == 0 or (dest.min() >= 0 and dest.max() < ZG))
    z[:, dest] = ws

    out = np.full((B, N), np.nan, dtype=np.float32)
    part = np.full((B, max(int(A["span_pp"][-1]) if len(A["span_pp"]) else 0, 1)), np.nan, dtype=np.float32)
    if len(A["span_pp"]) == 0 or A["span_pp"][-1] == 0:
        part[:] = 0
    SV = info["max_tile_values"]
    old_err = np.seterr(invalid="ignore")
    for t in range(NT):
        # the pair's leaf block arrives by one bulk copy; leaf slots past the vocabulary hold garbage that no range reads
        vals = np.full((B, SV), np.nan, dtype=np.float32)
        vals[:, :T] = z[:, t * T:(t + 1) * T]
        nleaf = min(T, V - t * T)
        assert not np.isnan(vals[:, phys[:nleaf]]).any() or np.isnan(ws).any()
        # pyramid, level k block i at logical slot 2T - (T >> (k-1)) + i (physical: swizzled)
        prev = vals[:, phys[:T]]
        for k in range(1, info["max_levels"] + 1):  # aligned blocks stop at 2^max_levels leaves (a warp's share)
            cur = red(prev[:, 0::2], prev[:, 1::2]).astype(np.float32)
            off = 2 * T - (T >> (k - 1))
            vals[:, phys[off:off + cur.shape[1]]] = cur
            prev = cur
        # multi-term ranges, ELL chunks of 32 (padding = identity slot 2T-1)
        vals[:, phys[2 * T - 1]] = ident
        c0, c1 = A["ell_chunk_ptr"][t], A["ell_chunk_ptr"][t + 1]
        desc = A["ell_desc"].reshape(-1, 2)
        for c in range(c0, c1):
            off32, k = desc[c]
            terms = A["ell_terms"][32 * off32:32 * (off32 + k)].reshape(k, 32)
            acc = np.full((B, 32), ident, dtype=np.float32)
            for kk in range(k):
                acc = red(acc, vals[:, terms[kk]]).astype(np.float32)
            vals[:, 2 * T + 32 * (c - c0):2 * T + 32 * (c - c0 + 1)] = acc
        # emit
        n0, n1 = A["tile_node_lo"][t], A["tile_node_lo"][t + 1]
        sl = A["node_slot"][n0:n1]  # spanning nodes carry the identity slot here and are overwritten below
        out[:, n0:n1] = vals[:, sl]
        # pieces of spanning nodes
        p0, p1 = A["piece_ptr"][t], A["piece_ptr"][t + 1]
        part[:, A["piece_idx"][p0:p1]] = vals[:, A["piece_slot"][p0:p1]]
    np.seterr(**old_err)
    # span_kernel: spanning nodes from their pieces (fp64 for sums)
    assert not np.isnan(part).any() or np.isnan(ws).any()
    for i, node in enumerate(A["span_node"]):
        q0, q1 = A["span_pp"][i], A["span_pp"][i + 1]
        if q1 == q0:
            out[:, node] = 0.0
        elif op == "sum":
            out[:, node] = part[:, q0:q1].astype(np.float64).sum(axis=1).astype(np.float32)
        else:
            out[:, node] = np.fmax.reduce(part[:, q0:q1], axis=1)
    return out
