"""Next-symbol masses indexed by symbol (``gt_symbol_masses``) and the draw under per-row symbol log-weights
(``gt_symbol_sample``).

CPU part: ``gt_num_symbols`` and ``symbol_labels``, the reference values of ``symbol_oracle`` pinned to the reference's
golden sums (symbol scatter, the end-of-token column, the weighted probabilities), and the argument checks of the two
entry points.  GPU part (``-m gpu``): every node against the reference, the bit-equalities with the child read-outs and
with ``sample_next_symbol``, the weighted draw's distribution, the rows without a draw, determinism and the async
wrapper.
"""
import asyncio
import ctypes

import numpy as np
import pytest
import torch

from genlm_backend_b200 import AsyncTokenCharacterTrie, ParallelTokenCharacterTrie, _lib
from genlm_backend_b200.synthetic import dirichlet_rows, synth_vocab
import child_oracle
import symbol_oracle
from helpers import EOS, assert_within_ulp, depth1_node, golden_layout, golden_vocab, trie_layout

F32, SUM, MAX = _lib.GT_F32, _lib.GT_OP_SUM, _lib.GT_OP_MAX
NORM, LOG = _lib.GT_CHILD_NORMALIZE, _lib.GT_CHILD_LOG


def random_logw(rng, shape, frac_neginf=0.3):
    w = rng.normal(0.0, 1.0, shape).astype(np.float32)
    w[rng.random(shape) < frac_neginf] = -np.inf
    return w


# ---- CPU ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["toy", "edge", "sentinel", "synth128256"])
def test_num_symbols_and_labels_host_only(name):
    dec = golden_vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    S = int(_lib.lib.gt_num_symbols(trie._engine._handle))
    labels = trie.symbol_labels
    assert S == len(labels) == trie.num_symbols == trie.end_symbol == symbol_oracle.item_symbols(dec)[1]
    assert labels[:256] == list(range(256))
    if name == "sentinel":
        assert S == 257 and isinstance(labels[256], EOS)
    else:
        assert S == 256
    assert _lib.lib.gt_num_symbols(None) == -1


@pytest.mark.parametrize("name", ["toy", "edge", "sentinel"])
def test_symbol_reference_pinned_to_golden(name):
    lay, g = golden_layout(name)
    dec = golden_vocab(name)
    sym, S = symbol_oracle.child_symbols(lay, dec)
    N = lay.n_nodes
    if name == "sentinel":  # the reference's own edge keys: the sentinel is -1, a leaf edge -(2 + item)
        key = np.full(N, -1, dtype=np.int64)
        key[g["children_val"]] = g["children_key"]
        want = np.where(key == -1, 256, np.where(key < -1, S, key))
        want[N - 1] = -1
        assert S == 257 and np.array_equal(sym, want)
    kids = [g["jump_idx"][g["jump_ptr"][n]:g["jump_ptr"][n + 1]] for n in range(N)]
    n_end = [int((sym[k] == S).sum()) for k in kids]
    if name == "edge":  # b"ab" three times under different ids, and the empty item at the root
        assert max(n_end) == 3 and n_end[N - 1] == 1
    nodes = np.concatenate([np.arange(N), [-1, N]])
    rng = np.random.default_rng(0)
    for b in range(g["ws"].shape[0]):
        rows = np.repeat(g["ws"][b:b + 1], len(nodes), axis=0)
        ssum = symbol_oracle.symbol_masses(lay, sym, S, rows, nodes, "sum")
        smax = symbol_oracle.symbol_masses(lay, sym, S, rows, nodes, "max")
        assert ssum.shape == (len(nodes), S + 1)
        assert (ssum[N:] == 0).all() and (smax[N:] == 0).all()
        for n in range(N):
            k = kids[n]
            inner = k[sym[k] < S]
            assert np.array_equal(ssum[n, sym[inner]], g["seq_sum"][b, inner])
            assert np.array_equal(smax[n, sym[inner]], g["seq_max"][b, inner])
            leaves = k[sym[k] == S]
            end = 0.0
            for c in leaves:
                end += g["seq_sum"][b, c]
            assert ssum[n, S] == end and smax[n, S] == (g["seq_max"][b, leaves].max() if len(leaves) else 0.0)
            untouched = np.ones(S + 1, bool)
            untouched[sym[inner]] = False
            untouched[S] = len(leaves) == 0
            assert (ssum[n, untouched] == 0).all()
            if len(k):
                np.testing.assert_allclose(ssum[n].sum(), g["seq_sum"][b, n], rtol=1e-12)
        # weighted probabilities: q_j / Z from the golden child sums and the log-weights of the children's symbols
        logw = random_logw(rng, (len(nodes), S + 1))
        logw[:, S] = np.inf  # infinite weight on "ends here": only children with mass may take it
        ids, m, q = symbol_oracle.weighted_child_masses(lay, sym, rows, nodes, logw)
        for i, n in enumerate(nodes[:N].tolist()):
            for j, c in enumerate(kids[n].tolist()):
                mj = g["seq_sum"][b, c]
                want = 0.0 if mj == 0 else mj * np.exp(np.float64(logw[i, sym[c]]))
                assert m[i, j] == mj and q[i, j] == want
        assert not np.isnan(q).any()
    # a NaN log-weight counts only at a symbol the node has
    root_kids = kids[N - 1]
    logw = np.zeros(S + 1, np.float32)
    absent = np.setdiff1d(np.arange(S + 1), sym[root_kids])
    if len(absent):
        logw[absent[0]] = np.nan
        assert not np.isnan(symbol_oracle.weighted_child_masses(lay, sym, g["ws"][:1], [N - 1], logw)[2]).any()
    logw[sym[root_kids[0]]] = np.nan
    assert np.isnan(symbol_oracle.weighted_child_masses(lay, sym, g["ws"][:1], [N - 1], logw)[2]).any()


def test_symbol_entry_points_reject_bad_arguments_without_a_gpu():
    trie = ParallelTokenCharacterTrie(golden_vocab("sentinel"))
    h = trie._engine._handle
    V, S = trie._engine.V, trie.num_symbols
    lib = _lib.lib
    p = ctypes.c_void_p(1 << 20)  # stands for a device pointer: never dereferenced by the checks
    ws_bytes = lib.gt_child_workspace_bytes(h, 4)

    def masses(**kw):
        a = dict(t=h, ws=p, in_type=F32, n=4, ld_ws=V, nodes=p, s=p, m=p, ld_out=S + 1, ops=SUM | MAX, flags=0,
                 work=p, work_bytes=ws_bytes)
        a.update(kw)
        return lib.gt_symbol_masses(a["t"], a["ws"], a["in_type"], a["n"], a["ld_ws"], a["nodes"], a["s"], a["m"],
                                    a["ld_out"], a["ops"], a["flags"], a["work"], a["work_bytes"], None)

    for bad in (dict(t=None), dict(ws=None), dict(nodes=None), dict(s=None), dict(m=None), dict(ops=0), dict(ops=4),
                dict(flags=0x40), dict(in_type=7), dict(n=-1), dict(ld_ws=V - 1), dict(ld_out=S), dict(ld_out=256),
                dict(work=None), dict(work=ctypes.c_void_p((1 << 20) + 8))):
        assert masses(**bad) == 1, bad
    assert masses(ops=SUM, m=None, flags=NORM | LOG, work_bytes=16) == 3  # too small
    assert b"workspace too small" in lib.gt_last_error()
    assert masses(n=0) == 0
    # the order of the checks: scalars and strides, the early return for no rows, data pointers, the workspace
    nulls = dict(ws=None, nodes=None, s=None, m=None, work=None)
    assert masses(n=0, **nulls) == 0
    for bad in (dict(ops=0), dict(flags=0x40), dict(in_type=7), dict(ld_ws=V - 1), dict(ld_out=S)):
        assert masses(n=0, **nulls, **bad) == 1, bad
    assert masses(s=None, work=None) == 1 and b"null data pointer" in lib.gt_last_error()

    def sample(**kw):
        a = dict(t=h, ws=p, in_type=F32, n=4, ld_ws=V, nodes=p, w=p, ld_w=0, flags=0, c=p, sy=p, lp=p, lz=p, lm=p,
                 work=p, work_bytes=ws_bytes)
        a.update(kw)
        return lib.gt_symbol_sample(a["t"], a["ws"], a["in_type"], a["n"], a["ld_ws"], a["nodes"], a["w"], a["ld_w"],
                                    a["flags"], 1, 0, a["c"], a["sy"], a["lp"], a["lz"], a["lm"], a["work"],
                                    a["work_bytes"], None)

    for bad in (dict(t=None), dict(ws=None), dict(nodes=None), dict(w=None), dict(c=None), dict(sy=None), dict(lp=None),
                dict(lz=None), dict(ld_w=1), dict(ld_w=S), dict(ld_w=-1), dict(flags=NORM), dict(flags=0x40),
                dict(in_type=-1), dict(n=-1), dict(ld_ws=V - 1), dict(work=None)):
        assert sample(**bad) == 1, bad
    assert sample(work_bytes=16) == 3
    assert sample(n=0) == 0 and sample(n=0, lm=None, ld_w=S + 1) == 0
    nulls = dict(ws=None, nodes=None, w=None, c=None, sy=None, lp=None, lz=None, lm=None, work=None)
    assert sample(n=0, **nulls) == 0
    for bad in (dict(flags=NORM), dict(in_type=-1), dict(ld_ws=V - 1), dict(ld_w=S), dict(ld_w=-1)):
        assert sample(n=0, **nulls, **bad) == 1, bad
    assert sample(sy=None, work=None) == 1 and b"null data pointer" in lib.gt_last_error()


# ---- GPU ---------------------------------------------------------------------------------------------------------
def kernel_weights(x, log_input):
    """The weights the kernels reduce: the fp32 conversion of the input, exponentiated for log inputs."""
    x32 = x.float().cpu().numpy()
    return np.exp(x32.astype(np.float64)).astype(np.float32) if log_input else x32


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["toy", "edge", "sentinel", "synth3000"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64, torch.float16, torch.bfloat16])
def test_every_node_matches_reference(name, dtype):
    dec = golden_vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    lay = trie_layout(trie)
    sym, S = symbol_oracle.child_symbols(lay, dec)
    assert S == trie.num_symbols
    N, V = len(trie), len(dec)
    nodes = np.concatenate([np.arange(N), [-1, N]]).astype(np.int32)
    base = np.concatenate([dirichlet_rows(3, V, alpha=0.1, seed=11), dirichlet_rows(2, V, alpha=1.0, seed=12)])
    p = base[np.arange(len(nodes)) % len(base)]
    for log_input in (False, True):
        with np.errstate(divide="ignore"):
            x = torch.tensor(np.log(p) if log_input else p).to(dtype).cuda()
        w = kernel_weights(x, log_input)
        want = symbol_oracle.symbol_masses(lay, sym, S, w, nodes, "sum")
        want_max = symbol_oracle.symbol_masses(lay, sym, S, w, nodes, "max").astype(np.float32)
        s, m = trie.batch_symbol_masses(x, torch.tensor(nodes), ops=("sum", "max"), log_input=log_input)
        assert s.shape == m.shape == (len(nodes), S + 1)
        close = (lambda h, wt: np.testing.assert_allclose(h, wt, rtol=1e-6, atol=0)) if log_input else assert_within_ulp
        close(s, want)
        if not log_input:
            assert np.array_equal(m, want_max)
        total = child_oracle.child_masses(lay, w, nodes, "sum").sum(axis=1, keepdims=True)
        sn, _ = trie.batch_symbol_masses(x, torch.tensor(nodes), log_input=log_input, normalize=True)
        sl, ml = trie.batch_symbol_masses(x, torch.tensor(nodes), ops=("sum", "max"), log_input=log_input,
                                          normalize=True, log=True)
        # the node's own columns are divided by its mass (0 / 0 = NaN for a node without mass); the others are padding
        present = np.zeros((len(nodes), S + 1), dtype=bool)
        ids = child_oracle.child_ids(lay, nodes)
        for b in range(len(nodes)):
            present[b, sym[ids[b][ids[b] >= 0]]] = True
        with np.errstate(divide="ignore", invalid="ignore"):
            wn = np.where(present, want / total, 0.0)
            wl = np.where(present, np.log(wn), -np.inf)
        close(sn, wn)
        assert np.array_equal(np.isnan(sl), np.isnan(wl)) and np.array_equal(np.isneginf(sl), np.isneginf(wl))
        fin = np.isfinite(wl)
        err = np.abs(sl[fin] - wl[fin])
        assert (err <= np.spacing(np.abs(wl[fin]).astype(np.float32)) + (1e-6 if log_input else 1e-12)).all()
        with np.errstate(divide="ignore"):
            assert np.array_equal(ml, np.log(m.astype(np.float64)).astype(np.float32))


def child_columns(trie, ids):
    """Column of each child in the symbol read-outs (S for a leaf child), -1 for padding."""
    lab = trie.edge_labels
    return np.where(ids >= 0, np.where(lab[np.maximum(ids, 0)] >= 0, lab[np.maximum(ids, 0)], trie.end_symbol), -1)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["edge", "synth3000", "synth128256"])
def test_bit_equal_to_child_masses_and_slab_max(name):
    dec = golden_vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    N, V, S = len(trie), len(dec), trie.num_symbols
    rng = np.random.default_rng(3)
    nodes = np.concatenate([[trie.root, -1, N], rng.integers(0, N, 253)]).astype(np.int32)
    ws = torch.tensor(dirichlet_rows(len(nodes), V, alpha=0.2, seed=5)).cuda()
    nt = torch.tensor(nodes).cuda()
    mx = trie._engine.reduce(ws, ("max",))[1].cpu().numpy()
    for normalize in (False, True):
        for log in (False, True):
            ids, cs, cm = (t.cpu().numpy() for t in trie.batch_child_masses_tensor(ws, nt, ops=("sum", "max"),
                                                                                  normalize=normalize, log=log))
            ss, sm = trie.batch_symbol_masses(ws, nt, ops=("sum", "max"), normalize=normalize, log=log)
            col = child_columns(trie, ids)
            for b in range(len(nodes)):
                k = col[b] >= 0
                inner = k & (col[b] < S)
                assert np.array_equal(ss[b, col[b, inner]], cs[b, inner])
                assert np.array_equal(sm[b, col[b, inner]], cm[b, inner])
                ends = np.flatnonzero(col[b] == S)
                if len(ends) == 1:
                    assert ss[b, S] == cs[b, ends[0]] and sm[b, S] == cm[b, ends[0]]
                if len(ends):
                    assert sm[b, S] == cm[b, ends].max()
                    if not normalize and not log:
                        assert sm[b, S] == mx[b, ids[b, ends]].max()
                if not normalize and not log:
                    assert np.array_equal(sm[b, col[b, inner]], mx[b, ids[b, inner]])
    # the same bits from rows in DFS order
    dfs = ws[:, trie.dfs_token_order.cuda()].contiguous()
    a = trie.batch_symbol_masses(ws, nt, ops=("sum", "max"), normalize=True)
    d = trie.batch_symbol_masses(dfs, nt, ops=("sum", "max"), normalize=True, dfs_order=True)
    assert np.array_equal(a[0], d[0]) and np.array_equal(a[1], d[1])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["edge", "synth128256"])
def test_zero_log_weights_reproduce_sample_next_symbol(name):
    dec = golden_vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    N, V, S = len(trie), len(dec), trie.num_symbols
    B = 1024
    rng = np.random.default_rng(4)
    nodes = rng.integers(0, N, B).astype(np.int32)
    nodes[:100] = trie.root
    nodes[100:103] = (-1, N, int(trie.idx_to_leaf[0, 1]))
    ws = torch.tensor(dirichlet_rows(B, V, alpha=0.3, seed=8)).cuda()
    nt = torch.tensor(nodes).cuda()
    child, _, logp, logZ = trie.sample_next_symbol(ws, nt, seed=11, offset=5)
    for logw in (torch.zeros(S + 1), torch.zeros(B, S + 1, dtype=torch.float64)):
        c, sy, lp, lz, lm = trie.sample_next_symbol_weighted(ws, nt, logw, seed=11, offset=5)
        assert torch.equal(c, child) and torch.equal(lp, logp) and torch.equal(lz, logZ) and torch.equal(lm, logZ)
        cc = c.cpu().numpy()
        want_sym = np.where(cc >= 0, child_columns(trie, cc[None, :])[0], -1)
        assert np.array_equal(sy.cpu().numpy(), want_sym)


def _chi_square(counts, p):
    from scipy import stats

    n = counts.sum()
    exp = p * n
    big = exp >= 5  # pool the small cells
    obs_b = np.append(counts[big], counts[~big].sum())
    exp_b = np.append(exp[big], exp[~big].sum())
    keep = exp_b > 0
    return stats.chisquare(obs_b[keep], exp_b[keep] * obs_b[keep].sum() / exp_b[keep].sum()).pvalue


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["root", "depth1", "shared_end"])
def test_weighted_draw_chi_square(where):
    name = "edge" if where == "shared_end" else "synth3000"
    dec = golden_vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    lay = trie_layout(trie)
    S = trie.num_symbols
    if where == "shared_end":  # the node spelling b"ab": three leaf children (items 0, 2, 8) and the child b"c"
        node = int(trie._layout["parent"][trie.idx_to_leaf[0, 1]])
    else:
        node = trie.root if where == "root" else depth1_node(trie)
    row = dirichlet_rows(1, len(dec), alpha=1.0, seed=21)
    logw = random_logw(np.random.default_rng(9), S + 1)
    if where == "shared_end":  # the three items split in proportion to their masses; b"abc" is never drawn
        logw[S] = 0.5
        logw[[s for s in child_columns(trie, np.asarray(trie.jump[node], dtype=np.int32)[None, :])[0] if s < S]] = -np.inf
    sym = child_columns(trie, np.asarray(trie.jump[node], dtype=np.int32)[None, :])[0]
    assert (logw[sym] == -np.inf).any() and np.isfinite(logw[sym]).sum() >= 2
    n = 40000
    ws = torch.tensor(row).expand(n, -1).cuda()
    nodes = torch.full((n,), node, dtype=torch.int32)
    child, symbol, logp, logZ, logM = trie.sample_next_symbol_weighted(ws, nodes, torch.tensor(logw), seed=1234, offset=77)
    ids, m, q = symbol_oracle.weighted_child_masses(lay, child_oracle_symbols(trie), row, [node], logw)
    deg = int((ids[0] >= 0).sum())
    p = q[0, :deg] / q[0, :deg].sum()
    pos = {int(c): j for j, c in enumerate(ids[0, :deg])}
    c = child.cpu().numpy()
    assert (c >= 0).all()
    counts = np.bincount([pos[int(x)] for x in c], minlength=deg).astype(np.float64)
    assert (counts[p == 0] == 0).all()  # zero-weight children (log-weight -inf) are never drawn
    if where == "shared_end":
        ends = np.flatnonzero(sym == S)
        assert len(ends) == 3 and (counts[ends] > 0).all()
    assert _chi_square(counts, p) > 1e-4
    assert np.array_equal(symbol.cpu().numpy(), sym[[pos[int(x)] for x in c]])
    np.testing.assert_allclose(logZ.cpu().numpy(), np.log(q[0].sum()), rtol=1e-6)
    np.testing.assert_allclose(logM.cpu().numpy(), np.log(m[0].sum()), rtol=1e-6)


def child_oracle_symbols(trie):
    """Reference symbols of every node of ``trie`` (from its vocabulary and layout)."""
    return symbol_oracle.child_symbols(trie_layout(trie), trie.decode)[0]


@pytest.mark.gpu
def test_weighted_draw_outputs_against_host_values():
    dec = golden_vocab("synth3000")
    trie = ParallelTokenCharacterTrie(dec)
    lay = trie_layout(trie)
    sym = child_oracle_symbols(trie)
    N, V, S = len(trie), len(dec), trie.num_symbols
    B = 2000
    rng = np.random.default_rng(2)
    internal = np.flatnonzero(np.diff(trie._layout["child_ptr"]) > 0)
    nodes = rng.choice(internal, B).astype(np.int32)
    nodes[:50] = trie.root
    rows = dirichlet_rows(B, V, alpha=0.1, seed=9)
    logw = random_logw(rng, (B, S + 1))
    c, sy, lp, lz, lm = (t.cpu().numpy() for t in trie.sample_next_symbol_weighted(
        torch.tensor(rows).cuda(), torch.tensor(nodes), torch.tensor(logw).cuda(), seed=5, offset=10))
    ids, m, q = symbol_oracle.weighted_child_masses(lay, sym, rows, nodes, logw)
    Z = q.sum(axis=1)
    drawn = Z > 0
    assert drawn.sum() > B // 2 and (c[~drawn] == -1).all() and np.isneginf(lz[~drawn]).all()
    col = np.argmax(ids == c[:, None], axis=1)
    hm = np.flatnonzero(drawn)
    assert (ids[hm, col[hm]] == c[hm]).all() and (q[hm, col[hm]] > 0).all()
    assert np.array_equal(sy[hm], sym[c[hm]])
    np.testing.assert_allclose(lz[hm], np.log(Z[hm]), rtol=1e-6)
    np.testing.assert_allclose(lp[hm], np.log(q[hm, col[hm]] / Z[hm]), rtol=1e-6, atol=1e-6)
    with np.errstate(divide="ignore"):
        np.testing.assert_allclose(lm, np.log(m.sum(axis=1)), rtol=1e-6)


@pytest.mark.gpu
def test_rows_without_a_draw():
    dec = golden_vocab("synth3000")
    trie = ParallelTokenCharacterTrie(dec)
    V, S, N = len(dec), trie.num_symbols, len(trie)
    leaf = int(trie.idx_to_leaf[5, 1])
    root_syms = child_columns(trie, np.asarray(trie.jump[trie.root], dtype=np.int32)[None, :])[0]
    absent = int(np.setdiff1d(np.arange(S + 1), root_syms)[0])
    base = torch.tensor(dirichlet_rows(1, V, alpha=1.0, seed=1)).cuda()
    ws = base.repeat(9, 1)
    ws[3].zero_()
    ws[5, trie.dfs_token_order[0]] = float("nan")  # a NaN weight under the root
    nodes = torch.tensor([leaf, -1, N, trie.root, trie.root, trie.root, trie.root, trie.root, trie.root],
                         dtype=torch.int32)
    logw = torch.zeros(9, S + 1)
    logw[4, torch.tensor(root_syms)] = -float("inf")  # every symbol with mass at -inf
    logw[6, int(root_syms[0])] = float("nan")  # NaN at a symbol the node has
    logw[7, absent] = float("nan")  # ... and at one it does not have: ignored
    logw[8, int(root_syms[1])] = float("inf")  # an infinite weighted total
    c, sy, lp, lz, lm = (t.cpu().numpy() for t in trie.sample_next_symbol_weighted(ws, nodes, logw.cuda(), seed=1))
    ref = [t.cpu().numpy() for t in trie.sample_next_symbol_weighted(ws[7:8], nodes[7:8], torch.zeros(S + 1), seed=1, offset=7)]
    bad = [0, 1, 2, 3, 4, 5, 6, 8]
    assert (c[bad] == -1).all() and (sy[bad] == -1).all()
    assert np.isneginf(lz[:5]).all() and np.isneginf(lp[:5]).all()
    assert np.isnan(lz[5]) and np.isnan(lp[5]) and np.isnan(lm[5])
    assert np.isnan(lz[6]) and np.isnan(lp[6]) and np.isfinite(lm[6])
    assert c[7] == ref[0][0] and lp[7] == ref[2][0] and lz[7] == ref[3][0] and c[7] >= 0
    assert lz[8] == np.inf and np.isnan(lp[8])
    assert np.isneginf(lm[:4]).all() and np.isfinite(lm[4])
    with pytest.raises(RuntimeError, match="sum of probabilities"):
        trie.sample_next_symbol_weighted(ws[:5], nodes[:5], logw[:5], check_valid=True)
    for r in (5, 6, 8):
        with pytest.raises(RuntimeError, match="nan"):
            trie.sample_next_symbol_weighted(ws[r:r + 1], nodes[r:r + 1], logw[r:r + 1], check_valid=True)
    trie.sample_next_symbol_weighted(ws[7:8], nodes[7:8], logw[7:8], check_valid=True)
    s, m = trie.batch_symbol_masses(ws[:3], nodes[:3], ops=("sum", "max"))
    assert (s == 0).all() and (m == 0).all()
    sl, ml = trie.batch_symbol_masses(ws[:3], nodes[:3], ops=("sum", "max"), log=True)
    assert np.isneginf(sl).all() and np.isneginf(ml).all()
    with pytest.raises(ValueError):
        trie.sample_next_symbol_weighted(ws, nodes, torch.zeros(S))
    with pytest.raises(ValueError):
        trie.sample_next_symbol_weighted(ws, nodes, torch.zeros(8, S + 1))


@pytest.mark.gpu
def test_bit_identical_across_batches_orders_workspaces_and_graphs():
    V = 128256
    trie = ParallelTokenCharacterTrie(synth_vocab(V))
    eng = trie._engine
    S = trie.num_symbols
    rng = np.random.default_rng(8)
    B = 1024
    nodes = np.full(B, trie.root, dtype=np.int32)
    nodes[::7] = rng.integers(0, len(trie), len(nodes[::7]))
    ws = torch.tensor(dirichlet_rows(B, V, alpha=0.5, seed=6)).cuda()
    nt = torch.tensor(nodes).cuda()
    shared = torch.tensor(random_logw(rng, S + 1)).cuda()
    per_row = shared.expand(B, -1).contiguous()
    sums, maxes = trie.batch_symbol_masses_tensor(ws, nt, ops=("sum", "max"), normalize=True)
    draw = trie.sample_next_symbol_weighted(ws, nt, shared, seed=3, offset=9)
    for a, b in zip(draw, trie.sample_next_symbol_weighted(ws, nt, per_row, seed=3, offset=9)):
        assert torch.equal(a, b)
    for a, b in zip((sums, maxes), trie.batch_symbol_masses_tensor(ws, nt, ops=("sum", "max"), normalize=True)):
        assert torch.equal(a, b)
    for r in (0, 7, 517, 1023):  # a row alone (its Philox counter is offset + its position)
        one = trie.batch_symbol_masses_tensor(ws[r:r + 1], nt[r:r + 1], ops=("sum", "max"), normalize=True)
        assert torch.equal(sums[r:r + 1], one[0]) and torch.equal(maxes[r:r + 1], one[1])
        d1 = trie.sample_next_symbol_weighted(ws[r:r + 1], nt[r:r + 1], per_row[r:r + 1], seed=3, offset=9 + r)
        for a, b in zip(draw, d1):
            assert torch.equal(a[r:r + 1], b)
    # DFS-order rows
    dfs = ws[:, trie.dfs_token_order.cuda()].contiguous()
    for a, b in zip(draw, trie.sample_next_symbol_weighted(dfs, nt, shared, seed=3, offset=9, dfs_order=True)):
        assert torch.equal(a, b)
    d = trie.batch_symbol_masses_tensor(dfs, nt, ops=("sum", "max"), normalize=True, dfs_order=True)
    assert torch.equal(sums, d[0]) and torch.equal(maxes, d[1])
    # a one-row workspace through the C ABI: 64 chunks of one row
    Bs = 64
    need = _lib.lib.gt_child_workspace_bytes(eng._handle, 1)
    work = torch.empty(need, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    s1 = torch.empty((Bs, S + 1), dtype=torch.float32, device="cuda")
    m1 = torch.empty((Bs, S + 1), dtype=torch.float32, device="cuda")
    _lib.check(_lib.lib.gt_symbol_masses(eng._handle, ws.data_ptr(), F32, Bs, V, nt.data_ptr(), s1.data_ptr(),
                                         m1.data_ptr(), S + 1, SUM | MAX, NORM, work.data_ptr(), need, st),
               "gt_symbol_masses")
    assert torch.equal(sums[:Bs], s1) and torch.equal(maxes[:Bs], m1)
    outs = [torch.empty(Bs, dtype=t, device="cuda") for t in (torch.int32, torch.int32, torch.float32, torch.float32, torch.float32)]
    _lib.check(_lib.lib.gt_symbol_sample(eng._handle, ws.data_ptr(), F32, Bs, V, nt.data_ptr(), per_row.data_ptr(), S + 1,
                                         0, 3, 9, *[o.data_ptr() for o in outs], work.data_ptr(), need, st),
               "gt_symbol_sample")
    for a, b in zip(draw, outs):
        assert torch.equal(a[:Bs], b)
    # CUDA graph capture and replay == eager
    cs = torch.cuda.Stream()
    cs.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(cs):  # the workspace of this stream, before capture
        trie.batch_symbol_masses_tensor(ws, nt, ops=("sum", "max"), normalize=True)
    torch.cuda.current_stream().wait_stream(cs)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=cs):
        cap = trie.batch_symbol_masses_tensor(ws, nt, ops=("sum", "max"), normalize=True)
        cap_draw = trie.sample_next_symbol_weighted(ws, nt, shared, seed=3, offset=9)
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(sums, cap[0]) and torch.equal(maxes, cap[1])
        for a, b in zip(draw, cap_draw):
            assert torch.equal(a, b)


@pytest.mark.gpu
def test_async_symbol_masses_batch_together():
    dec = golden_vocab("synth3000")
    atrie = AsyncTokenCharacterTrie(ParallelTokenCharacterTrie(dec))
    trie = atrie.trie
    S = trie.num_symbols
    n = 64
    rows = dirichlet_rows(n, len(dec), alpha=0.3, seed=3)
    nodes = np.random.default_rng(4).integers(0, len(trie), n).astype(np.int32)
    nodes[0] = trie.root
    calls = []
    orig = trie.batch_symbol_masses

    def counting(*a, **kw):
        calls.append(len(a[1]))
        return orig(*a, **kw)

    trie.batch_symbol_masses = counting

    async def run():
        try:
            return await asyncio.gather(*[atrie.symbol_masses(torch.tensor(rows[i]), int(nodes[i]), normalize=True)
                                          for i in range(n)])
        finally:
            await atrie.cleanup()

    got = asyncio.run(run())
    assert calls == [n]
    s, _ = orig(torch.tensor(rows), nodes, normalize=True)
    for i, row in enumerate(got):
        assert row.dtype == np.float32 and row.shape == (S + 1,)
        assert np.array_equal(row, s[i])
