"""Token masks under a byte-level DFA (``gt_dfa_token_mask``) and the DFA advance over drawn tokens (``gt_dfa_advance``).

CPU part: the reference of ``dfa_oracle`` on hand-checked cases, ``dfa.trim``, ``dfa.symbol_logw`` and the argument
checks of the two entry points.  GPU part (``-m gpu``): masks and advances bit for bit against the reference on the
small vocabularies and at 128k tokens, invalid rows, padding bits, the accept-all table against the subtree mask,
stacked tables, the mask feeding the sampler, CUDA graph capture of the whole step, and the byte-level draw under
``symbol_logw``.
"""
import ctypes

import numpy as np
import pytest
import torch

import oracle
from genlm_backend_b200 import ParallelTokenCharacterTrie, _lib, dfa, smc
from genlm_backend_b200.synthetic import dirichlet_rows, logsoftmax_rows
import dfa_oracle
from helpers import golden_layout, golden_vocab, trie_layout


def golden_oracle(name):
    return dfa_oracle.DfaOracle(golden_layout(name)[0], golden_vocab(name))


def trie_oracle(trie):
    return dfa_oracle.DfaOracle(trie_layout(trie), trie.decode)


def a_then_b(S):
    """The language "a" or "ab": 0 -a-> 1 -b-> 2, accepting {1, 2}."""
    delta = np.full((3, S), -1, dtype=np.int32)
    delta[0, ord("a")] = 1
    delta[1, ord("b")] = 2
    return delta


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_oracle_hand_checked_on_toy():
    o = golden_oracle("toy")  # items: b"a", b"b", b"ab", b"<eos>"
    delta = a_then_b(256)
    node_a = int(o.path[2, 1])  # the node spelling "a"
    leaf_ab = int(o.leaf[2])
    have = o.mask(delta, [0, 1, 2, -1, 3, 1, 2, 0, 0], [o.N - 1, o.N - 1, o.N - 1, o.N - 1, o.N - 1, node_a, leaf_ab, -1, o.N])
    want = np.array([
        [1, 0, 1, 0],  # state 0 at the root: "a" and "ab"
        [0, 1, 0, 0],  # state 1 (after "a"): "b"
        [0, 0, 0, 0],  # state 2 accepts only the empty continuation; no item is empty
        [0, 0, 0, 0],  # dead state
        [0, 0, 0, 0],  # state outside [0, Q)
        [1, 0, 1, 0],  # at node "a" in state 1: "a" (nothing left) and "ab" (then "b")
        [0, 0, 1, 0],  # at the leaf of "ab" in state 2: that item only, with nothing left
        [0, 0, 0, 0],  # invalid nodes
        [0, 0, 0, 0],
    ], dtype=bool)
    assert np.array_equal(have, want)
    assert o.mask(delta, [0]).tolist() == [[True, False, True, False]]  # nodes None: the root
    adv = o.advance(delta, [0, 0, 0, 1, 1, 0], [2, 0, 1, 2, -1, 4], [o.N - 1, o.N - 1, o.N - 1, node_a, o.N - 1, o.N - 1])
    assert adv.tolist() == [2, 1, -1, 2, -1, -1]


def test_oracle_eos_recipe_on_sentinel():
    o = golden_oracle("sentinel")  # items: b"ab", b"", b"ab", b"a", EOS, b"plain"
    assert o.S == 257
    delta = a_then_b(o.S)
    delta[[1, 2], 256] = [1, 2]  # EOS from an accepting state keeps it; from any other state it rejects
    have = o.mask(delta, [0, 1, 2])
    assert have.astype(int).tolist() == [[1, 1, 1, 1, 0, 0], [0, 1, 0, 0, 1, 0], [0, 1, 0, 0, 1, 0]]


def test_trim_dead_ends_and_unreachable_states():
    a, b, c = 0, 1, 2
    delta = np.full((6, 3), -1, dtype=np.int32)
    delta[0, a] = 1      # 1 accepts
    delta[0, b] = 2      # 2 is a dead end: no way to an accepting state
    delta[2, a] = 2
    delta[1, c] = 5      # 5 loops on itself without accepting
    delta[5, c] = 5
    delta[3, a] = 1      # 3 is unreachable but can still accept: kept
    delta[4, a] = 4      # 4 is unreachable and cannot accept
    delta[1, a] = 7      # out of range: a reject
    want = np.full((6, 3), -1, dtype=np.int32)
    want[0, a] = 1
    want[3, a] = 1
    have = dfa.trim(delta, [1])
    assert have.dtype == np.int32 and np.array_equal(have, want)
    assert np.array_equal(dfa.trim(delta, np.arange(6) == 1), want)
    # trimming is idempotent and keeps a fully co-reachable table as it is
    assert np.array_equal(dfa.trim(have, [1]), have)
    full = np.array([[1, 0], [1, 0]], dtype=np.int32)
    assert np.array_equal(dfa.trim(full, [0]), full)


def test_symbol_logw_matches_reference():
    rng = np.random.default_rng(0)
    delta, acc = dfa_oracle.random_dfa(rng, 16, 257, p_live=0.3)
    delta = dfa.trim(delta, acc)
    states = np.array([0, 3, 15, -1, 16, 7, 7], dtype=np.int32)
    w = dfa.symbol_logw(torch.tensor(delta), torch.tensor(states)).numpy()
    assert w.dtype == np.float32 and w.shape == (len(states), 258)
    for b, q in enumerate(states.tolist()):
        for s in range(258):
            if s < 257:
                ok = 0 <= q < 16 and 0 <= delta[q, s] < 16
            else:
                ok = 0 <= q < 16
            assert w[b, s] == (0.0 if ok else -np.inf), (b, s)
    # with a padded row stride the symbol count is explicit
    wide = np.concatenate([delta, np.zeros((16, 7), np.int32)], axis=1)
    assert np.array_equal(dfa.symbol_logw(wide, states, num_symbols=257).numpy(), w)


def test_dfa_entry_points_reject_bad_arguments_without_a_gpu():
    trie = ParallelTokenCharacterTrie(golden_vocab("sentinel"))
    h = trie._engine._handle
    V, S = trie._engine.V, trie.num_symbols
    W = (V + 31) // 32
    lib = _lib.lib
    p = ctypes.c_void_p(1 << 20)  # stands for a device pointer: never dereferenced by the checks

    def mask(**kw):
        a = dict(t=h, delta=p, Q=4, ld=S, states=p, nodes=p, n=4, bits=p, ld_bits=W)
        a.update(kw)
        return lib.gt_dfa_token_mask(a["t"], a["delta"], a["Q"], a["ld"], a["states"], a["nodes"], a["n"], a["bits"],
                                     a["ld_bits"], None)

    def advance(**kw):
        a = dict(t=h, delta=p, Q=4, ld=S, states=p, nodes=p, tokens=p, n=4, out=p)
        a.update(kw)
        return lib.gt_dfa_advance(a["t"], a["delta"], a["Q"], a["ld"], a["states"], a["nodes"], a["tokens"], a["n"],
                                  a["out"], None)

    for bad in (dict(t=None), dict(delta=None), dict(states=None), dict(bits=None), dict(Q=0), dict(Q=-1),
                dict(ld=S - 1), dict(ld=0), dict(n=-1), dict(ld_bits=W - 1), dict(ld_bits=0)):
        assert mask(**bad) == 1, bad
    for bad in (dict(t=None), dict(delta=None), dict(states=None), dict(tokens=None), dict(out=None), dict(Q=0),
                dict(ld=S - 1), dict(n=-1)):
        assert advance(**bad) == 1, bad
    assert b"gt_dfa_advance" in lib.gt_last_error()
    # a table of 2^31 entries or more cannot be indexed with 32-bit offsets
    for fn in (mask, advance):
        assert fn(Q=(1 << 31) // S + 1) == 4
        assert fn(Q=1 << 40, ld=S) == 4
        assert fn(n=0) == 0 and fn(n=0, nodes=None) == 0


# ---- GPU ---------------------------------------------------------------------------------------------------------
def random_tables(rng, S):
    """Seeded, trimmed random tables: 1 state (accept-all), 8, 256 and 4096 states."""
    out = [np.zeros((1, S), dtype=np.int32)]
    for Q, p_live in ((8, 0.5), (256, 0.8), (4096, 0.9)):
        delta, acc = dfa_oracle.random_dfa(rng, Q, S, p_live=p_live)
        out.append(dfa.trim(delta, acc))
    return out


def row_inputs(rng, trie, Q, B):
    """Node ids (the root, random internal nodes, leaves, -1 and N) and states (random live ones, -1 and Q)."""
    N = len(trie)
    leaves = trie._layout["leaf_node"]
    nodes = rng.integers(0, N, B).astype(np.int32)
    nodes[: B // 4] = N - 1
    nodes[B // 4: B // 4 + 4] = leaves[rng.integers(0, len(leaves), 4)]
    nodes[-2:] = [-1, N]
    states = rng.integers(0, Q, B).astype(np.int32)
    states[1] = -1
    states[2] = Q
    return nodes, states


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["toy", "edge", "sentinel", "synth128256"])
def test_mask_and_advance_match_oracle(name):
    dec = golden_vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    o = trie_oracle(trie)
    S, V = trie.num_symbols, len(dec)
    assert o.S == S
    rng = np.random.default_rng(1)
    B = 64
    for delta in random_tables(rng, S):
        Q = delta.shape[0]
        nodes, states = row_inputs(rng, trie, Q, B)
        d = torch.tensor(delta).cuda()
        for nd in (nodes, None):
            bits = trie.dfa_token_mask(d, torch.tensor(states).cuda(), None if nd is None else torch.tensor(nd).cuda())
            assert bits.dtype == torch.int32 and bits.shape == (B, (V + 31) // 32)
            hb = bits.cpu().numpy()
            want = o.mask(delta, states, nd)
            assert np.array_equal(oracle.unpack_bits(hb, V), want), (Q, nd is None)
            assert not oracle.unpack_bits(hb, hb.shape[1] * 32)[:, V:].any()
            # advance: every allowed token to its oracle state, anything else to -1
            toks = np.array([rng.choice(np.flatnonzero(m)) if m.any() else rng.integers(0, V) for m in want], np.int32)
            toks[3:6] = [-1, V, rng.integers(0, V)]
            adv = trie.dfa_advance(d, torch.tensor(states).cuda(), torch.tensor(toks).cuda(),
                                   None if nd is None else torch.tensor(nd).cuda()).cpu().numpy()
            assert np.array_equal(adv, o.advance(delta, states, toks, nd)), (Q, nd is None)
            ok = (toks >= 0) & (toks < V)
            allowed = np.zeros(B, bool)
            allowed[ok] = want[np.flatnonzero(ok), toks[ok]]
            assert np.array_equal(adv >= 0, allowed)
            assert (adv[3:5] == -1).all()


@pytest.mark.gpu
def test_eos_recipe_and_literal_rows_on_sentinel():
    trie = ParallelTokenCharacterTrie(golden_vocab("sentinel"))
    delta = a_then_b(trie.num_symbols)
    delta[[1, 2], trie.num_symbols - 1] = [1, 2]
    bits = trie.dfa_token_mask(torch.tensor(delta).cuda(), torch.tensor([0, 1, 2, -1, 3], dtype=torch.int32).cuda())
    have = oracle.unpack_bits(bits.cpu().numpy(), 6).astype(int).tolist()
    assert have == [[1, 1, 1, 1, 0, 0], [0, 1, 0, 0, 1, 0], [0, 1, 0, 0, 1, 0], [0] * 6, [0] * 6]
    adv = trie.dfa_advance(torch.tensor(delta).cuda(), torch.tensor([0, 0, 1, 1, 2]).cuda(), torch.tensor([0, 1, 4, 0, 4]).cuda())
    assert adv.cpu().tolist() == [2, 0, 1, -1, 2]


@pytest.mark.gpu
def test_padding_words_and_row_stride():
    dec = golden_vocab("synth3000")
    trie = ParallelTokenCharacterTrie(dec)
    V, S, W = len(dec), trie.num_symbols, (len(dec) + 31) // 32
    rng = np.random.default_rng(2)
    delta = torch.tensor(random_tables(rng, S)[2]).cuda()
    B, ld = 37, W + 5
    nodes, states = row_inputs(rng, trie, delta.shape[0], B)
    st, nd = torch.tensor(states).cuda(), torch.tensor(nodes).cuda()
    buf = torch.full((B, ld), 0x55555555, dtype=torch.int32, device="cuda")
    trie._engine.ensure_device(torch.cuda.current_device())  # the raw entry point needs the metadata resident
    _lib.check(_lib.lib.gt_dfa_token_mask(trie._engine._handle, delta.data_ptr(), delta.shape[0], S, st.data_ptr(),
                                          nd.data_ptr(), B, buf.data_ptr(), ld, torch.cuda.current_stream().cuda_stream),
               "gt_dfa_token_mask")
    have = buf.cpu().numpy()
    assert np.array_equal(have[:, :W], trie.dfa_token_mask(delta, st, nd).cpu().numpy())
    assert not oracle.unpack_bits(have[:, :W], W * 32)[:, V:].any()
    assert (have[:, W:] == 0x55555555).all()  # words past ceil(V/32) are not touched


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["edge", "synth3000"])
def test_accept_all_equals_subtree_mask(name):
    dec = golden_vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    V, N = len(dec), len(trie)
    delta = torch.zeros((1, trie.num_symbols), dtype=torch.int32, device="cuda")
    nodes = torch.tensor(np.concatenate([np.arange(min(N, 500)), [N - 1, -1, N]]), dtype=torch.int32).cuda()
    zeros = torch.zeros(nodes.shape[0], dtype=torch.int32, device="cuda")
    assert torch.equal(trie.dfa_token_mask(delta, zeros, nodes), trie.subtree_token_mask(nodes))
    allb = trie.dfa_token_mask(delta, zeros[:3])
    assert oracle.unpack_bits(allb.cpu().numpy(), V).all()
    assert not oracle.unpack_bits(allb.cpu().numpy(), allb.shape[1] * 32)[:, V:].any()


@pytest.mark.gpu
def test_stacked_tables_equal_separate_calls():
    dec = golden_vocab("synth3000")
    trie = ParallelTokenCharacterTrie(dec)
    S = trie.num_symbols
    rng = np.random.default_rng(4)
    _, t8, t256, _ = random_tables(rng, S)
    stacked = np.concatenate([t8, np.where(t256 >= 0, t256 + t8.shape[0], -1)]).astype(np.int32)
    B = 48
    nodes, s8 = row_inputs(rng, trie, 8, B)
    s256 = rng.integers(0, 256, B).astype(np.int32)
    which = rng.random(B) < 0.5
    nd = torch.tensor(nodes).cuda()
    sep = torch.where(torch.tensor(which).cuda()[:, None],
                      trie.dfa_token_mask(torch.tensor(t8).cuda(), torch.tensor(s8).cuda(), nd),
                      trie.dfa_token_mask(torch.tensor(t256).cuda(), torch.tensor(s256).cuda(), nd))
    st = np.where(which, s8, np.where(s256 >= 0, s256 + 8, s256)).astype(np.int32)
    st[1] = -1  # still dead in the stacked table
    st[2] = 8 + 256
    sep[1:3] = 0
    assert torch.equal(trie.dfa_token_mask(torch.tensor(stacked).cuda(), torch.tensor(st).cuda(), nd), sep)


def constrained_step(trie, delta, states, nodes, logp, seed):
    bits = trie.dfa_token_mask(delta, states, nodes)
    logZ, tok = smc.masked_logsumexp_sample(logp, bits, seed=seed)
    return bits, logZ, tok, trie.dfa_advance(delta, states, tok, nodes)


@pytest.mark.gpu
def test_mask_feeds_sampler_and_advance():
    """exp(logZ) of the masked draw is the probability of the allowed tokens, every draw is allowed and advances to a live
    state equal to the reference's, and a row without allowed tokens draws -1 and advances to -1."""
    dec = golden_vocab("synth3000")
    trie = ParallelTokenCharacterTrie(dec)
    o = trie_oracle(trie)
    V, S, B = len(dec), trie.num_symbols, 64
    rng = np.random.default_rng(5)
    delta = random_tables(rng, S)[2]
    nodes, states = row_inputs(rng, trie, delta.shape[0], B)
    p = dirichlet_rows(B, V, alpha=1.0, seed=5)
    logp = torch.tensor(np.log(p)).cuda()
    d, st, nd = torch.tensor(delta).cuda(), torch.tensor(states).cuda(), torch.tensor(nodes).cuda()
    bits, logZ, tok, adv = constrained_step(trie, d, st, nd, logp, seed=7)
    want = o.mask(delta, states, nodes)
    mass = (p * want).sum(axis=1)
    nz = mass > 0
    assert nz.sum() > B // 2
    np.testing.assert_allclose(np.exp(logZ.cpu().numpy()[nz].astype(np.float64)), mass[nz], rtol=2e-5)
    t, a = tok.cpu().numpy(), adv.cpu().numpy()
    assert (t[nz] >= 0).all() and want[np.flatnonzero(nz), t[nz]].all()
    assert (t[~nz] == -1).all() and (a[~nz] == -1).all()
    assert ((a[nz] >= 0) & (a[nz] < delta.shape[0])).all()
    assert np.array_equal(a, o.advance(delta, states, t, nodes))


@pytest.mark.gpu
def test_step_in_cuda_graph_matches_eager():
    dec = golden_vocab("synth3000")
    trie = ParallelTokenCharacterTrie(dec)
    V, S, B = len(dec), trie.num_symbols, 64
    rng = np.random.default_rng(6)
    delta = torch.tensor(random_tables(rng, S)[1]).cuda()
    nodes, states = row_inputs(rng, trie, delta.shape[0], B)
    st, nd = torch.tensor(states).cuda(), torch.tensor(nodes).cuda()
    logp = torch.tensor(logsoftmax_rows(B, V, seed=3)).cuda()
    eager = constrained_step(trie, delta, st, nd, logp, seed=11)
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        constrained_step(trie, delta, st, nd, logp, seed=11)  # warm-up on the capturing stream
    stream.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        out = constrained_step(trie, delta, st, nd, logp, seed=11)
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        for have, want in zip(out, eager):
            assert torch.equal(have, want)


@pytest.mark.gpu
def test_symbol_draw_under_symbol_logw_never_rejects():
    dec = golden_vocab("sentinel")
    trie = ParallelTokenCharacterTrie(dec)
    S = trie.num_symbols
    delta = a_then_b(S)
    delta[[1, 2], S - 1] = [1, 2]
    B = 256
    states = np.tile(np.array([0, 1, 2, -1], np.int32), B // 4)
    ws = torch.tensor(dirichlet_rows(B, len(dec), alpha=1.0, seed=9)).cuda()
    root = torch.full((B,), len(trie) - 1, dtype=torch.int32, device="cuda")
    logw = dfa.symbol_logw(torch.tensor(delta).cuda(), torch.tensor(states).cuda())
    assert logw.is_cuda and logw.shape == (B, S + 1)
    for seed in range(8):
        child, sym, _, logZ, _ = trie.sample_next_symbol_weighted(ws, root, logw, seed=seed)
        sym, st = sym.cpu().numpy(), states
        drew = sym >= 0
        assert (drew == (st >= 0)).all()  # every live state has a symbol (or the end of the token) to go to
        for q, s in zip(st[drew].tolist(), sym[drew].tolist()):
            assert s == S or 0 <= delta[q, s] < 3, (q, s)
