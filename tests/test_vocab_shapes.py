"""Every trie read-out on tokenizer-shaped vocabularies (``tests/vocab_shapes.py``), against the fp64 oracles.

CPU tier: the layout equals the reference's, the plan-emulated sum and max match the oracle wherever the tile fits,
and the preconditions that make each GPU test reach its kernel path hold (heavy spanning nodes sharing a warp of
``span_kernel``, the child and symbol counts, the depths, which tiles fit in shared memory).  GPU tier (``-m gpu``): the
mass path in both pipelines, the slab read-outs, the child and symbol read-outs, the next-symbol draws, the masked
read-outs and the DFA walks on every family, and a vocabulary whose tile node table fits no tile size: its mass calls
are refused before anything is enqueued and every tile-free read-out still works.
"""
import asyncio
import functools
import warnings

import numpy as np
import pytest
import torch

import child_oracle
import dfa_oracle
import oracle
import symbol_oracle
import vocab_shapes
from dfa_logw_oracle import WeightedDfaOracle
from genlm_backend_b200 import AsyncTokenCharacterTrie, ParallelTokenCharacterTrie, TokenCharacterTrie, _lib, dfa
from genlm_backend_b200.synthetic import dirichlet_rows
from helpers import assert_within_ulp, rel_err, trie_layout
from plan_emulator import emulate
from vocab_shapes import SMEM_LIMIT, TILE_SIZES, tile_smem_bytes

CHAINS = [f"chain{v}" for v in vocab_shapes.CHAIN_LENGTHS]
NAMES = list(vocab_shapes.FAMILIES) + CHAINS
FITS = {  # (family, tile leaves) whose tile node table fits in one CTA's shared memory: all others but these
    ("long_mixed", 2048): False, ("over_limit", 1024): False, ("over_limit", 2048): False,
}
SUM_RTOL = 2e-6  # the bar of test_gpu_trie.py


def fits(name, T):
    return FITS.get((name, T), True)


@functools.lru_cache(maxsize=None)
def vocab(name):
    return vocab_shapes.vocab(name)


def make_trie(name, T=1024, cls=ParallelTokenCharacterTrie):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        trie = cls(vocab(name))
    trie._engine.plan(T)
    return trie


def prefix_node(trie, prefix):
    """The node spelling ``prefix`` (bytes), found from the leaf of an item that starts with it."""
    parent = trie._layout["parent"]
    i = next(i for i, t in enumerate(trie.decode) if t.byte_string.startswith(prefix))
    n = int(parent[trie.idx_to_leaf[i, 1]])  # spells the whole item
    for _ in range(len(trie.decode[i].byte_string) - len(prefix)):
        n = int(parent[n])
    return n


def node_depths(trie):
    """int64 [N]: symbols on the path from the root (a leaf: its item's length + 1).  Parents have larger ids."""
    parent = trie._layout["parent"].astype(np.int64)
    depth = np.zeros(len(trie), dtype=np.int64)
    for n in range(len(trie) - 2, -1, -1):
        depth[n] = depth[parent[n]] + 1
    return depth


# ---- CPU ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", NAMES)
def test_layout_equals_reference(name):
    dec = vocab(name)
    trie = make_trie(name, cls=TokenCharacterTrie)
    ref = oracle.OracleTrie(dec)
    assert len(trie) == ref.n_nodes and trie.root == ref.root
    assert np.array_equal(trie.idx_to_leaf, ref.idx_to_leaf)
    assert np.array_equal(trie._layout["child_ptr"], ref.jump_ptr)
    assert np.array_equal(trie._layout["child_idx"], ref.jump_idx)


@pytest.mark.parametrize("T", TILE_SIZES)
@pytest.mark.parametrize("name", NAMES)
def test_plan_fits_and_emulated_kernels_match_oracle(name, T):
    trie = make_trie(name, T, cls=TokenCharacterTrie)
    smem = tile_smem_bytes(trie._engine)
    assert (smem <= SMEM_LIMIT) == fits(name, T), smem
    if smem > SMEM_LIMIT:
        return
    ws = dirichlet_rows(2, len(trie.decode), alpha=0.3, seed=1)
    o = trie_layout(trie)
    have = emulate(trie._engine, ws, "sum")
    assert not np.isnan(have).any()
    r, z = rel_err(have, o.weight_sum(ws))
    assert r <= SUM_RTOL and z == 0.0
    assert np.array_equal(emulate(trie._engine, ws, "max"), o.weight_max(ws).astype(np.float32))


def test_tile_smem_bytes_near_the_bound():
    """The families straddle the bound: the largest node tables that still fit, and the smallest that do not."""
    need = {(n, T): tile_smem_bytes(make_trie(n, T, cls=TokenCharacterTrie)._engine)
            for n in ("runs", "long_mixed", "over_limit") for T in TILE_SIZES}
    assert SMEM_LIMIT - 20 * 1024 < need["runs", 2048] <= SMEM_LIMIT
    assert SMEM_LIMIT < need["long_mixed", 2048] < SMEM_LIMIT + 32 * 1024
    assert need["over_limit", 1024] > 3 * SMEM_LIMIT


def test_heavy_spanning_nodes_share_a_warp():
    """span_kernel reduces nodes with more than kSpanInline = 8 pieces by the whole warp, one after the other: nested
    heavy prefixes put several of them in one warp (32 consecutive spanning nodes)."""
    trie = make_trie("space_heavy", 1024, cls=TokenCharacterTrie)
    eng = trie._engine
    pieces = np.diff(eng.plan_array("span_pp"))
    span_node = eng.plan_array("span_node")
    heavy = np.flatnonzero(pieces > 8)
    warps, count = np.unique(heavy // 32, return_counts=True)
    assert count.max() >= 2, (heavy, pieces[heavy])
    heavy_nodes = set(span_node[heavy].tolist())
    for p in (b" ", b" t", b" th"):
        assert prefix_node(trie, p) in heavy_nodes, p
    shared = heavy[heavy // 32 == warps[count.argmax()]]
    assert (span_node[shared] != trie.root).sum() >= 2  # not only the root
    # the b" " child of the root covers dozens of 512-rank blocks of the child read-outs
    lay = trie._layout
    sp = prefix_node(trie, b" ")
    assert (lay["hi"][sp] - 1) // 512 - lay["lo"][sp] // 512 + 1 >= 40


def test_child_symbol_and_depth_preconditions():
    # more than 256 children, most of them leaves (301 items spell b"a"), and leaf children of the root
    t = make_trie("dups", cls=TokenCharacterTrie)
    a = prefix_node(t, b"a")
    kids = t.jump[a]
    assert t._engine.max_children == len(kids) == 306
    assert (np.diff(t._layout["child_ptr"])[kids] == 0).sum() == 301
    assert (np.diff(t._layout["child_ptr"])[t.jump[t.root]] == 0).sum() == 3
    # thousands of symbols: each of 32 lanes of the finish kernel owns ~94 children of the root
    w = make_trie("wide_alphabet", cls=TokenCharacterTrie)
    assert w._engine.num_symbols == 3256 and w._engine.max_children == len(w.jump[w.root]) == 2995
    # no single-byte items: the root has no leaf child, and the first leaf in DFS order lies below depth 1
    n = make_trie("no_single_bytes", cls=TokenCharacterTrie)
    assert (np.diff(n._layout["child_ptr"])[n.jump[n.root]] > 0).all()
    assert node_depths(n)[n._layout["leaf_node"][n._layout["perm"][0]]] >= 3
    # depth: the DFA walks cover up to 299 symbols, and rows start at depth 200 and more
    for name, longest in (("runs", 256), ("long_mixed", 211), ("over_limit", 299), ("chain513", 513)):
        t = make_trie(name, cls=TokenCharacterTrie)
        assert max(len(x.byte_string) for x in t.decode) == longest, name
        assert node_depths(t).max() == longest + 1, name


# ---- GPU ---------------------------------------------------------------------------------------------------------
GPU_NAMES = ["space_heavy", "runs", "long_mixed", "dups", "no_single_bytes", "wide_alphabet", "over_limit", "chain33",
             "chain513"]


@functools.lru_cache(maxsize=None)
def gpu_trie(name):
    """The fp32 trie of ``name`` at T = 1024, with its oracles (built once per module)."""
    trie = make_trie(name)
    lay = trie_layout(trie)
    return trie, lay, WeightedDfaOracle(lay, trie.decode)


def sample_nodes(trie, o, rng, k=48):
    """The root, the nodes with the most children, the largest subtrees, the deepest internal nodes, duplicate-item
    parents, leaves, random nodes, and the invalid ids -1 and N."""
    N = len(trie)
    deg = np.diff(trie._layout["child_ptr"])
    size = trie._layout["hi"] - trie._layout["lo"]
    internal = np.flatnonzero(deg > 0)
    depth = o.depth
    leaves = trie._layout["leaf_node"]
    picks = [[trie.root] * 4, np.argsort(-deg, kind="stable")[:8], internal[np.argsort(-size[internal], kind="stable")[:8]],
             internal[np.argsort(-depth[internal], kind="stable")[:8]], leaves[rng.integers(0, len(leaves), 4)],
             rng.choice(internal, k), [-1, N]]
    return np.concatenate([np.asarray(p, dtype=np.int64) for p in picks]).astype(np.int32)


def check_mass(trie, ws, want_sum, want_max, f64):
    from test_gpu_trie import check_against

    check_against(trie, ws, want_sum, want_max, f64=f64)


@pytest.mark.gpu
@pytest.mark.parametrize("cls", [ParallelTokenCharacterTrie, TokenCharacterTrie])
@pytest.mark.parametrize("name,T", [(n, T) for n in NAMES for T in TILE_SIZES if fits(n, T)])
def test_weight_sum_and_max(name, T, cls):
    trie = make_trie(name, T, cls)
    o = trie_layout(trie)
    ws = dirichlet_rows(5, len(trie.decode), alpha=0.1, seed=2)
    check_mass(trie, ws, o.weight_sum(ws), o.weight_max(ws), f64=cls is TokenCharacterTrie)


@pytest.mark.gpu
def test_batch_of_several_chunks_near_the_bound():
    """150 rows on the node table closest to the shared-memory bound: three chunks of at most 64 rows."""
    trie = make_trie("runs", 2048)
    o = trie_layout(trie)
    ws = dirichlet_rows(150, len(trie.decode), alpha=0.3, seed=3)
    hs, hm = trie.batch_weight_tensor(torch.tensor(ws).cuda(), ops=("sum", "max"))
    r, z = rel_err(hs.cpu().numpy(), o.weight_sum(ws))
    assert r <= SUM_RTOL and z == 0.0
    assert np.array_equal(hm.cpu().numpy(), o.weight_max(ws).astype(np.float32))


@pytest.mark.gpu
@pytest.mark.parametrize("name", GPU_NAMES)
def test_slab_readouts_and_subtree_masks(name):
    trie, lay, o = gpu_trie(name)
    rng = np.random.default_rng(1)
    nodes = sample_nodes(trie, o, rng)
    B, V, N = 6, len(trie.decode), len(trie)
    ws = dirichlet_rows(B, V, alpha=0.3, seed=4)
    want_sum, want_max = lay.weight_sum(ws), lay.weight_max(ws)
    ids = np.stack([np.roll(nodes, b) for b in range(B)])
    norm = np.full(B, trie.root, dtype=np.int32)
    if fits(name, 1024):
        have = trie.batch_weight_sum_at(torch.tensor(ws), ids)
        r, z = rel_err(have, oracle.gather_nodes(want_sum, ids))
        assert r <= SUM_RTOL and z == 0.0
        have = trie.batch_weight_sum_at(torch.tensor(ws), ids, normalizer=norm)
        r, z = rel_err(have, oracle.gather_nodes(want_sum, ids, norm))
        assert r <= 2 * SUM_RTOL + 2.0 ** -24 and z == 0.0  # a ratio of two sums, rounded once more
        have = trie.batch_weight_max_at(torch.tensor(ws), ids)
        assert np.array_equal(have, oracle.gather_nodes(want_max, ids).astype(np.float32))
    # gather from a slab given directly: what it reads does not depend on the tile plan
    slab = want_sum.astype(np.float32)
    have = trie.gather_nodes(torch.tensor(slab).cuda(), torch.tensor(ids)).cpu().numpy()
    assert np.array_equal(have, oracle.gather_nodes(slab, ids).astype(np.float32))
    # subtree masks against the reachability matrix of the reference
    valid = nodes[(nodes >= 0) & (nodes < N)]
    bits = trie.subtree_token_mask(torch.tensor(valid)).cpu().numpy()
    want = oracle.OracleTrie(trie.decode).subtree_token_mask(valid)
    assert np.array_equal(oracle.unpack_bits(bits, V), want)
    assert not oracle.unpack_bits(bits, bits.shape[1] * 32)[:, V:].any()


@pytest.mark.gpu
@pytest.mark.parametrize("name", GPU_NAMES)
def test_child_and_symbol_masses(name):
    trie, lay, o = gpu_trie(name)
    rng = np.random.default_rng(2)
    nodes = sample_nodes(trie, o, rng)
    V = len(trie.decode)
    ws = dirichlet_rows(len(nodes), V, alpha=0.3, seed=5)
    x, nt = torch.tensor(ws).cuda(), torch.tensor(nodes)
    ids, s, m = trie.batch_child_masses(x, nt, ops=("sum", "max"))
    want_ids = child_oracle.child_ids(lay, nodes)
    assert ids.shape == want_ids.shape == (len(nodes), trie.max_children)
    assert np.array_equal(ids, want_ids)
    assert_within_ulp(s, child_oracle.child_masses(lay, ws, nodes, "sum"))
    assert np.array_equal(m, child_oracle.child_masses(lay, ws, nodes, "max").astype(np.float32))
    # DFS-ordered rows: the very same bits
    dfs = x[:, trie.dfs_token_order.cuda()].contiguous()
    for a, b in zip((ids, s, m), trie.batch_child_masses(dfs, nt, ops=("sum", "max"), dfs_order=True)):
        assert np.array_equal(a, b)
    sym, S = symbol_oracle.child_symbols(lay, trie.decode)
    assert S == trie.num_symbols
    ss, sm = trie.batch_symbol_masses(x, nt, ops=("sum", "max"))
    assert ss.shape == (len(nodes), S + 1)
    assert_within_ulp(ss, symbol_oracle.symbol_masses(lay, sym, S, ws, nodes, "sum"))
    assert np.array_equal(sm, symbol_oracle.symbol_masses(lay, sym, S, ws, nodes, "max").astype(np.float32))


@pytest.mark.gpu
@pytest.mark.parametrize("name", GPU_NAMES)
def test_next_symbol_draws_replay_exactly(name):
    from test_draw_replay import _child_check

    trie, lay, o = gpu_trie(name)
    rng = np.random.default_rng(3)
    internal = np.flatnonzero(np.diff(trie._layout["child_ptr"]) > 0)
    nodes = np.concatenate([sample_nodes(trie, o, rng)[:-2], np.repeat(np.argsort(-np.diff(trie._layout["child_ptr"]))[:4], 64),
                            rng.choice(internal, 256)]).astype(np.int32)
    B, V, S = len(nodes), len(trie.decode), trie.num_symbols
    sym = symbol_oracle.child_symbols(lay, trie.decode)[0]
    ws = dirichlet_rows(B, V, alpha=0.3, seed=6)
    keep = rng.random((B, V)) < 0.7
    logw = rng.normal(0.0, 1.5, (B, S + 1)).astype(np.float32)
    logw[rng.random((B, S + 1)) < 0.1] = -np.inf
    wdev, ndev, kdev = torch.tensor(ws).cuda(), torch.tensor(nodes).cuda(), torch.tensor(keep).cuda()
    ids = child_oracle.child_ids(lay, nodes)
    for masked in (False, True):
        rows = np.where(keep, ws, np.float32(0)) if masked else ws
        kw = dict(mask=kdev) if masked else {}
        m = child_oracle.child_masses(lay, rows, nodes, "sum")
        seed, offset = 9 + masked, 500 * masked
        out = trie.sample_next_symbol(wdev, ndev, seed=seed, offset=offset, **kw)
        _child_check(trie, lay, ids, m, m, out, seed, offset, (name, "masked" if masked else "plain"), False)
        out = trie.sample_next_symbol_weighted(wdev, ndev, torch.tensor(logw).cuda(), seed=seed, offset=offset + 3, **kw)
        _, m2, q = symbol_oracle.weighted_child_masses(lay, sym, rows, nodes, logw)
        _child_check(trie, lay, ids, q, m2, out, seed, offset + 3, (name, "weighted masked" if masked else "weighted"), True)


@pytest.mark.gpu
@pytest.mark.parametrize("name", GPU_NAMES)
def test_masked_readouts_equal_zeroed_rows(name):
    from test_masked_readouts import check_bit_equal

    trie, lay, o = gpu_trie(name)
    rng = np.random.default_rng(4)
    nodes = sample_nodes(trie, o, rng, k=16)
    base = dirichlet_rows(len(nodes), len(trie.decode), alpha=0.3, seed=7)
    check_bit_equal(trie, nodes, base, rng, [torch.float32], ["d0.5", "d0.02", "bool0.3"])


def dfa_tables(rng, S):
    """Accept-all (every walk goes to the end of its item), a sparse random table, and a dense one whose run symbols
    always lead on, so that walks of hundreds of symbols survive; each with random log-weights."""
    out = [np.zeros((1, S), dtype=np.int32)]
    delta, acc = dfa_oracle.random_dfa(rng, 8, S, p_live=0.5)
    out.append(dfa.trim(delta, acc))
    delta, acc = dfa_oracle.random_dfa(rng, 64, S, p_live=0.9)
    delta[:, list(vocab_shapes.RUN_CHARS)] = rng.integers(0, 64, (64, len(vocab_shapes.RUN_CHARS)))
    delta[:, 0] = rng.integers(0, 64, 64)  # the chains' symbol
    out.append(dfa.trim(delta, np.arange(64)))
    return [(d, rng.normal(0.0, 1.0, d.shape).astype(np.float32)) for d in out]


@pytest.mark.gpu
@pytest.mark.parametrize("name", GPU_NAMES)
def test_dfa_mask_logw_and_advance(name):
    trie, lay, o = gpu_trie(name)
    rng = np.random.default_rng(5)
    S, V, N = trie.num_symbols, len(trie.decode), len(trie)
    internal = np.flatnonzero(np.diff(trie._layout["child_ptr"]) > 0)
    deepest = internal[np.argsort(-o.depth[internal], kind="stable")]
    for delta, logw in dfa_tables(rng, S):
        Q = delta.shape[0]
        nodes = sample_nodes(trie, o, rng, k=8)
        # rows starting at depth 200 and more, where there is such a node
        deep = deepest[o.depth[deepest] >= 200][:: max(1, (o.depth[deepest] >= 200).sum() // 8)][:8]
        nodes = np.concatenate([nodes, deep]).astype(np.int32)
        B = len(nodes)
        states = rng.integers(0, Q, B).astype(np.int32)
        states[[1, 2]] = [-1, Q]
        d, st, nd = torch.tensor(delta).cuda(), torch.tensor(states).cuda(), torch.tensor(nodes).cuda()
        want = o.mask(delta, states, nodes)
        bits = trie.dfa_token_mask(d, st, nd).cpu().numpy()
        assert np.array_equal(oracle.unpack_bits(bits, V), want), Q
        assert not oracle.unpack_bits(bits, bits.shape[1] * 32)[:, V:].any()
        have = trie.dfa_token_logw(d, torch.tensor(logw).cuda(), st, nd).cpu().numpy()
        assert np.array_equal(have.view(np.uint32), o.logw(delta, logw, states, nodes).view(np.uint32)), Q
        toks = np.array([rng.choice(np.flatnonzero(w)) if w.any() else rng.integers(0, V) for w in want], np.int32)
        toks[3:5] = [-1, V]
        adv = trie.dfa_advance(d, st, torch.tensor(toks).cuda(), nd).cpu().numpy()
        assert np.array_equal(adv, o.advance(delta, states, toks, nodes)), Q
        if Q == 1 and len(deep):  # accept-all: every item under a deep node is walked to its end
            assert want[-len(deep):].any()


# ---- a tile node table that fits no tile size ----------------------------------------------------------------------
def refusal_message(engine):
    return f"tile plan needs {tile_smem_bytes(engine)} bytes of shared memory per CTA"


@pytest.mark.gpu
@pytest.mark.parametrize("T", TILE_SIZES)
def test_over_limit_mass_calls_are_refused(T):
    par = make_trie("over_limit", T)
    seq = make_trie("over_limit", T, TokenCharacterTrie)
    V = len(par.decode)
    ws = dirichlet_rows(20, V, alpha=0.3, seed=8)
    x = torch.tensor(ws)
    hint = "1024 leaves is already the smallest tile" if T == 1024 else "plan with 1024-leaf tiles"
    calls = [
        lambda: par.batch_weight_sum(x), lambda: par.batch_weight_max(x[:2]), lambda: par.weight_sum(x[0]),
        lambda: par.weight_max(ws[0]), lambda: par.batch_weight_sum_max(x), lambda: par.batch_weight_rows(list(x), "sum"),
        lambda: par.batch_weight_tensor(x.cuda(), ops=("sum", "max")), lambda: par.batch_weight_sum_at(x, [0, 1]),
        lambda: par.batch_weight_max_at(x, [0, 1]), lambda: par.batch_weight_sum_max_at(x, [0, 1]),
        lambda: seq.batch_weight_sum(ws.astype(np.float64)), lambda: seq.batch_weight_max(ws), lambda: seq.weight_sum(ws[0]),
    ]
    for i, call in enumerate(calls):
        with pytest.raises(_lib.GtError) as err:
            call()
        msg = str(err.value)
        for eng in (par._engine, seq._engine):
            assert refusal_message(eng) in msg, (i, msg)
        assert hint in msg and "(limit 232448)" in msg, (i, msg)
    # the same trie and stream still serve the tile-free read-outs
    torch.cuda.synchronize()
    nodes = np.array([par.root, 0, len(par) - 2], dtype=np.int32)
    lay = trie_layout(par)
    ids, s, _ = par.batch_child_masses(x[:3], nodes)
    assert np.array_equal(ids, child_oracle.child_ids(lay, nodes))
    assert_within_ulp(s, child_oracle.child_masses(lay, ws[:3], nodes, "sum"))


@pytest.mark.gpu
def test_refused_reduce_enqueues_nothing():
    """gt_weight_reduce refuses the plan before the permute of its first chunk runs: the caller's workspace and outputs
    keep what they held."""
    trie = make_trie("over_limit", 1024)
    eng = trie._engine
    B, V = 70, len(trie.decode)
    ws = torch.tensor(dirichlet_rows(B, V, alpha=0.3, seed=9), device="cuda")
    eng.ensure_device(0)
    out = torch.full((B, len(trie)), 7.0, dtype=torch.float32, device="cuda")
    need = int(_lib.lib.gt_workspace_bytes(eng._handle, B))
    work = (torch.arange(need, dtype=torch.int64, device="cuda") * 37 % 251).to(torch.uint8)
    before = work.clone()
    torch.cuda.synchronize()
    rc = _lib.lib.gt_weight_reduce(eng._handle, ws.data_ptr(), _lib.GT_F32, B, ws.stride(0), out.data_ptr(), None,
                                   _lib.GT_F32, out.stride(0), _lib.GT_OP_SUM, 0, work.data_ptr(), work.numel(),
                                   torch.cuda.current_stream().cuda_stream)
    assert rc == 4 and refusal_message(eng).encode() in _lib.lib.gt_last_error()
    torch.cuda.synchronize()
    assert torch.equal(work, before)
    assert bool((out == 7.0).all())


@pytest.mark.gpu
def test_async_worker_serves_after_a_refusal():
    trie = make_trie("over_limit", 1024)
    at = AsyncTokenCharacterTrie(trie)
    lay = trie_layout(trie)
    V = len(trie.decode)
    rows = dirichlet_rows(4, V, alpha=0.3, seed=10)
    nodes = [trie.root, int(trie.jump[trie.root][0]), trie.root, int(trie.jump[trie.root][-1])]

    async def run():
        try:
            with pytest.raises(_lib.GtError, match="bytes of shared memory"):
                await asyncio.gather(*[at.weight_sum(torch.tensor(r)) for r in rows])
            kids = await asyncio.gather(*[at.child_masses(torch.tensor(rows[i]), nodes[i]) for i in range(4)])
            syms = await asyncio.gather(*[at.symbol_masses(torch.tensor(rows[i]), nodes[i]) for i in range(4)])
            return kids, syms
        finally:
            await at.cleanup()

    kids, syms = asyncio.run(run())
    want_ids = child_oracle.child_ids(lay, nodes)
    want = child_oracle.child_masses(lay, rows, nodes, "sum")
    sym, S = symbol_oracle.child_symbols(lay, trie.decode)
    want_sym = symbol_oracle.symbol_masses(lay, sym, S, rows, nodes, "sum")
    for i, (gi, gs) in enumerate(kids):
        deg = len(gi)
        assert np.array_equal(gi, want_ids[i, :deg]) and (want_ids[i, deg:] == -1).all()
        assert_within_ulp(gs, want[i, :deg])
        assert_within_ulp(syms[i], want_sym[i])
