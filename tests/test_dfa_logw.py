"""Token log-weights under a weighted byte automaton (``gt_dfa_token_logw``).

CPU part: the reference of ``dfa_logw_oracle`` on hand-checked cases (an EOS final weight included), ``dfa.symbol_logw`` with
a weighted table, and the argument checks of the entry point and their order.  GPU part (``-m gpu``): the kernel bit for
bit against the reference on the small vocabularies and at 128k tokens, special values, the all-zero table against the
Boolean mask, stacked tables, a padded row stride, the weighted step through the sampler and the advance, the
composition with the masked next-symbol draw, and CUDA graph capture of the whole step.
"""
import ctypes

import numpy as np
import pytest
import torch

import oracle
from genlm_backend_b200 import ParallelTokenCharacterTrie, _lib, dfa, smc
from genlm_backend_b200.synthetic import logsoftmax_rows
import dfa_oracle
from dfa_logw_oracle import WeightedDfaOracle
from helpers import golden_layout, golden_vocab, trie_layout
from test_dfa_mask import a_then_b, random_tables, row_inputs

NINF = -np.inf


def golden_oracle(name):
    return WeightedDfaOracle(golden_layout(name)[0], golden_vocab(name))


def trie_oracle(trie):
    return WeightedDfaOracle(trie_layout(trie), trie.decode)


def a_then_b_weights(S):
    """Log-weights for ``a_then_b``: 0.5 on "a", -1.25 on "b", and 7 on every transition the table rejects."""
    logw = np.full((3, S), 7.0, dtype=np.float32)
    logw[0, ord("a")] = 0.5
    logw[1, ord("b")] = -1.25
    return logw


def ieee_oracle(o, delta, logw, states, nodes=None):
    with np.errstate(invalid="ignore", over="ignore"):  # inf - inf and sums past the float32 range are the point here
        return o.logw(delta, logw, states, nodes)


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_oracle_hand_checked_on_toy():
    o = golden_oracle("toy")  # items: b"a", b"b", b"ab", b"<eos>"
    delta, logw = a_then_b(256), a_then_b_weights(256)
    node_a = int(o.path[2, 1])  # the node spelling "a"
    have = o.logw(delta, logw, [0, 1, 2, -1, 3, 1, 0], [o.N - 1, o.N - 1, o.N - 1, o.N - 1, o.N - 1, node_a, -1])
    want = np.array([
        [0.5, NINF, -0.75, NINF],  # state 0 at the root: "a", and "ab" = 0.5 - 1.25
        [NINF, -1.25, NINF, NINF],  # state 1 (after "a"): "b"
        [NINF] * 4,  # state 2 accepts only the empty continuation; no item is empty
        [NINF] * 4,  # dead state
        [NINF] * 4,  # state outside [0, Q)
        [0.0, NINF, -1.25, NINF],  # at node "a" in state 1: "a" (nothing left) and "ab" (then "b")
        [NINF] * 4,  # invalid node
    ], dtype=np.float32)
    assert have.dtype == np.float32 and np.array_equal(have, want)
    assert np.array_equal(o.logw(delta, np.zeros_like(logw), [0, 1]), np.where(o.mask(delta, [0, 1]), 0, NINF))


def test_oracle_eos_final_weight_on_sentinel():
    o = golden_oracle("sentinel")  # items: b"ab", b"", b"ab", b"a", EOS, b"plain"
    delta, logw = a_then_b(o.S), a_then_b_weights(o.S)
    delta[[1, 2], 256] = [1, 2]  # EOS from an accepting state keeps it
    logw[[1, 2], 256] = [-0.5, -2.0]  # ... with that state's final weight
    have = o.logw(delta, logw, [0, 1, 2])
    want = np.array([
        [-0.75, 0.0, -0.75, 0.5, NINF, NINF],
        [NINF, 0.0, NINF, NINF, -0.5, NINF],
        [NINF, 0.0, NINF, NINF, -2.0, NINF],
    ], dtype=np.float32)
    assert np.array_equal(have, want)


def test_symbol_logw_with_weights_matches_a_direct_loop():
    rng = np.random.default_rng(0)
    delta, acc = dfa_oracle.random_dfa(rng, 16, 257, p_live=0.3)
    delta = dfa.trim(delta, acc)
    logw = rng.normal(size=delta.shape).astype(np.float32)
    states = np.array([0, 3, 15, -1, 16, 7, 7], dtype=np.int32)
    w = dfa.symbol_logw(torch.tensor(delta), torch.tensor(states), logw=torch.tensor(logw)).numpy()
    assert w.dtype == np.float32 and w.shape == (len(states), 258)
    for b, q in enumerate(states.tolist()):
        live = 0 <= q < 16
        for s in range(257):
            assert w[b, s] == (logw[q, s] if live and 0 <= delta[q, s] < 16 else NINF), (b, s)
        assert w[b, 257] == (0.0 if live else NINF)
    # float64 tables are converted to float32; a padded row stride needs the symbol count
    assert np.array_equal(dfa.symbol_logw(delta, states, logw=logw.astype(np.float64)).numpy(), w)
    pad = lambda t, v: np.concatenate([t, np.full((16, 7), v, t.dtype)], axis=1)  # noqa: E731
    assert np.array_equal(dfa.symbol_logw(pad(delta, 0), states, num_symbols=257, logw=pad(logw, 9.0)).numpy(), w)
    # without weights the result is that of the Boolean table, and a zero table gives the same bits
    plain = dfa.symbol_logw(torch.tensor(delta), torch.tensor(states)).numpy()
    zeros = dfa.symbol_logw(torch.tensor(delta), torch.tensor(states), logw=torch.zeros(delta.shape)).numpy()
    assert np.array_equal(plain.view(np.uint32), zeros.view(np.uint32))
    assert np.array_equal(np.isfinite(plain), np.isfinite(w))
    for bad in (logw[:, :-1], logw[:-1], delta):
        with pytest.raises(ValueError):
            dfa.symbol_logw(delta, states, logw=bad)


def test_logw_entry_point_rejects_bad_arguments_in_order_without_a_gpu():
    trie = ParallelTokenCharacterTrie(golden_vocab("sentinel"))
    h = trie._engine._handle
    V, S = trie._engine.V, trie.num_symbols
    lib = _lib.lib
    p = ctypes.c_void_p(1 << 20)  # stands for a device pointer: never dereferenced by the checks

    def call(**kw):
        a = dict(t=h, delta=p, logw=p, Q=4, ld=S, states=p, nodes=p, n=4, out=p, ld_out=V)
        a.update(kw)
        rc = lib.gt_dfa_token_logw(a["t"], a["delta"], a["logw"], a["Q"], a["ld"], a["states"], a["nodes"], a["n"],
                                   a["out"], a["ld_out"], None)
        return rc, lib.gt_last_error().decode() if rc else ""

    for bad in (dict(t=None), dict(delta=None), dict(logw=None), dict(states=None), dict(out=None), dict(ld_out=V - 1),
                dict(ld_out=0), dict(Q=0), dict(Q=-1), dict(ld=S - 1), dict(ld=0), dict(n=-1)):
        rc, msg = call(**bad)
        assert rc == 1 and "gt_dfa_token_logw" in msg, bad
    # the order: null trie, null pointers, ld_out, the table and row counts, the table's size, no rows, the grid
    assert "null trie" in call(t=None, logw=None, ld_out=0, Q=0)[1]
    assert "null data pointer" in call(logw=None, ld_out=0, Q=0)[1]
    assert "ld_out" in call(ld_out=V - 1, Q=0, n=-1)[1]
    assert "bad n_states" in call(Q=0, n=0)[1]
    assert call(Q=(1 << 31) // S + 1, n=0)[0] == 4
    assert call(Q=1 << 40)[0] == 4
    assert call(n=0)[0] == 0 and call(n=0, nodes=None)[0] == 0
    rc, msg = call(n=65535 * 8 + 1, nodes=None)
    assert rc == 4 and "too many rows" in msg


# ---- GPU ---------------------------------------------------------------------------------------------------------
def cuda(*xs):
    return [None if x is None else torch.tensor(x).cuda() for x in xs]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["toy", "edge", "sentinel", "synth128256"])
def test_logw_matches_oracle(name):
    dec = golden_vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    o = trie_oracle(trie)
    S, V = trie.num_symbols, len(dec)
    rng = np.random.default_rng(11)
    B = 64
    for delta in random_tables(rng, S):
        Q = delta.shape[0]
        logw = (rng.normal(size=delta.shape) * 2).astype(np.float32)
        nodes, states = row_inputs(rng, trie, Q, B)
        d, w, st = cuda(delta, logw, states)
        for nd in (nodes, None):
            out = trie.dfa_token_logw(d, w, st, None if nd is None else torch.tensor(nd).cuda())
            assert out.dtype == torch.float32 and out.shape == (B, V) and out.device == d.device
            have = out.cpu().numpy()
            want = o.logw(delta, logw, states, nd)
            assert np.array_equal(have.view(np.uint32), want.view(np.uint32)), (Q, nd is None)
            assert np.array_equal(np.isfinite(have), o.mask(delta, states, nd))


@pytest.mark.gpu
def test_hand_checked_rows_on_sentinel():
    trie = ParallelTokenCharacterTrie(golden_vocab("sentinel"))
    S = trie.num_symbols
    delta, logw = a_then_b(S), a_then_b_weights(S)
    delta[[1, 2], S - 1] = [1, 2]
    logw[[1, 2], S - 1] = [-0.5, -2.0]
    have = trie.dfa_token_logw(*cuda(delta, logw, np.array([0, 1, 2, -1, 3], np.int32))).cpu().numpy()
    want = [[-0.75, 0.0, -0.75, 0.5, NINF, NINF], [NINF, 0.0, NINF, NINF, -0.5, NINF],
            [NINF, 0.0, NINF, NINF, -2.0, NINF], [NINF] * 6, [NINF] * 6]
    assert np.array_equal(have, np.array(want, np.float32))


@pytest.mark.gpu
def test_special_values_follow_ieee():
    dec = golden_vocab("synth3000")
    trie = ParallelTokenCharacterTrie(dec)
    o = trie_oracle(trie)
    S = trie.num_symbols
    rng = np.random.default_rng(12)
    B = 64
    seen = {"nan": 0, "pinf": 0, "ninf_allowed": 0}
    for delta in random_tables(rng, S)[1:3]:
        Q = delta.shape[0]
        nodes, states = row_inputs(rng, trie, Q, B)
        for frac in (0.002, 0.02):
            logw = rng.normal(size=delta.shape).astype(np.float32)
            u = rng.random(delta.shape)
            logw[u < frac] = np.inf
            logw[(u >= frac) & (u < 2 * frac)] = -np.inf
            logw[(u >= 2 * frac) & (u < 3 * frac)] = np.nan
            logw[delta < 0] = np.nan  # a rejecting transition's weight never shows: the token is -inf
            for nd in (nodes, None):
                have = trie.dfa_token_logw(*cuda(delta, logw, states, nd)).cpu().numpy()
                want = ieee_oracle(o, delta, logw, states, nd)
                assert np.array_equal(have, want, equal_nan=True), (Q, frac, nd is None)
                allowed = o.mask(delta, states, nd)
                assert np.isnan(have).sum() == np.isnan(want).sum() and not (np.isnan(have) & ~allowed).any()
                seen["nan"] += int(np.isnan(have).sum())
                seen["pinf"] += int((have == np.inf).sum())
                seen["ninf_allowed"] += int(((have == NINF) & allowed).sum())
    assert all(v > 0 for v in seen.values()), seen


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["edge", "synth3000"])
def test_zero_weights_equal_the_additive_mask(name):
    dec = golden_vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    V, S = len(dec), trie.num_symbols
    rng = np.random.default_rng(13)
    B = 96
    for delta in random_tables(rng, S):
        nodes, states = row_inputs(rng, trie, delta.shape[0], B)
        d, st, nd = cuda(delta, states, nodes)
        bits = oracle.unpack_bits(trie.dfa_token_mask(d, st, nd).cpu().numpy(), V)
        out = trie.dfa_token_logw(d, torch.zeros(delta.shape, device="cuda"), st, nd).cpu().numpy()
        assert np.array_equal(out.view(np.uint32), np.where(bits, np.float32(0), np.float32(NINF)).view(np.uint32))


@pytest.mark.gpu
def test_padded_row_stride_leaves_the_tail_untouched():
    dec = golden_vocab("synth3000")
    trie = ParallelTokenCharacterTrie(dec)
    V, S = len(dec), trie.num_symbols
    rng = np.random.default_rng(14)
    delta = random_tables(rng, S)[2]
    logw = rng.normal(size=delta.shape).astype(np.float32)
    B, ld = 37, V + 13
    nodes, states = row_inputs(rng, trie, delta.shape[0], B)
    d, w, st, nd = cuda(delta, logw, states, nodes)
    buf = torch.full((B, ld), 12345.0, dtype=torch.float32, device="cuda")
    trie._engine.ensure_device(torch.cuda.current_device())  # the raw entry point needs the metadata resident
    _lib.check(_lib.lib.gt_dfa_token_logw(trie._engine._handle, d.data_ptr(), w.data_ptr(), d.shape[0], S, st.data_ptr(),
                                          nd.data_ptr(), B, buf.data_ptr(), ld, torch.cuda.current_stream().cuda_stream),
               "gt_dfa_token_logw")
    have = buf.cpu().numpy()
    assert np.array_equal(have[:, :V], trie.dfa_token_logw(d, w, st, nd).cpu().numpy())
    assert (have[:, V:] == 12345.0).all()


@pytest.mark.gpu
def test_stacked_tables_equal_separate_calls():
    dec = golden_vocab("synth3000")
    trie = ParallelTokenCharacterTrie(dec)
    S = trie.num_symbols
    rng = np.random.default_rng(15)
    _, t8, t256, _ = random_tables(rng, S)
    w8, w256 = (rng.normal(size=t.shape).astype(np.float32) for t in (t8, t256))
    stacked = np.concatenate([t8, np.where(t256 >= 0, t256 + t8.shape[0], -1)]).astype(np.int32)
    B = 48
    nodes, s8 = row_inputs(rng, trie, 8, B)
    s256 = rng.integers(0, 256, B).astype(np.int32)
    which = rng.random(B) < 0.5
    nd = torch.tensor(nodes).cuda()
    sep = torch.where(torch.tensor(which).cuda()[:, None], trie.dfa_token_logw(*cuda(t8, w8, s8), nd),
                      trie.dfa_token_logw(*cuda(t256, w256, s256), nd))
    st = np.where(which, s8, s256 + 8).astype(np.int32)
    st[1] = -1
    st[2] = 8 + 256
    sep[1:3] = float("-inf")
    have = trie.dfa_token_logw(*cuda(stacked, np.concatenate([w8, w256]), st), nd)
    assert torch.equal(have, sep)


@pytest.mark.gpu
def test_bad_weight_tables_raise():
    trie = ParallelTokenCharacterTrie(golden_vocab("sentinel"))
    delta = a_then_b(trie.num_symbols)
    for bad in (np.zeros((3, trie.num_symbols - 1), np.float32), np.zeros((2, trie.num_symbols), np.float32),
                np.zeros(delta.shape, np.int32), delta):
        with pytest.raises(ValueError):
            trie.dfa_token_logw(delta, bad, [0])
    # float64 tables are converted to float32 on the device
    w = a_then_b_weights(trie.num_symbols)
    assert torch.equal(trie.dfa_token_logw(delta, w.astype(np.float64), [0]), trie.dfa_token_logw(delta, w, [0]))


def weighted_step(trie, delta, logw, states, nodes, logp, seed):
    tokw = trie.dfa_token_logw(delta, logw, states, nodes)
    logZ, tok = smc.masked_logsumexp_sample(logp, tokw, seed=seed)
    return tokw, logZ, tok, trie.dfa_advance(delta, states, tok, nodes)


def step_inputs(seed, B, table=2):
    dec = golden_vocab("synth3000")
    trie = ParallelTokenCharacterTrie(dec)
    rng = np.random.default_rng(seed)
    delta = random_tables(rng, trie.num_symbols)[table]
    logw = (rng.normal(size=delta.shape) * 0.5).astype(np.float32)
    nodes, states = row_inputs(rng, trie, delta.shape[0], B)
    logp = torch.tensor(logsoftmax_rows(B, len(dec), seed=seed)).cuda()
    return trie, delta, logw, nodes, states, logp


@pytest.mark.gpu
def test_weighted_step_weight_increment_draws_and_advance():
    trie, delta, logw, nodes, states, logp = step_inputs(16, 64)
    d, w, st, nd = cuda(delta, logw, states, nodes)
    tokw, logZ, tok, adv = weighted_step(trie, d, w, st, nd, logp, seed=3)
    want = torch.logsumexp(logp.double() + tokw.double(), dim=1).cpu().numpy()
    have = logZ.cpu().numpy()
    fin = np.isfinite(want)
    assert fin.sum() > 32 and np.array_equal(np.isfinite(have), fin)
    np.testing.assert_allclose(have[fin], want[fin], rtol=1e-5, atol=1e-6)
    t, a = tok.cpu().numpy(), adv.cpu().numpy()
    assert (t[fin] >= 0).all() and (t[~fin] == -1).all()
    assert np.isfinite(tokw.cpu().numpy()[np.flatnonzero(fin), t[fin]]).all()
    assert (a[fin] >= 0).all() and (a[~fin] == -1).all()
    assert np.array_equal(a, trie_oracle(trie).advance(delta, states, t, nodes))


@pytest.mark.gpu
def test_weighted_draw_follows_the_weighted_distribution():
    from scipy import stats

    dec = golden_vocab("synth3000")
    trie = ParallelTokenCharacterTrie(dec)
    V = len(dec)
    rng = np.random.default_rng(17)
    delta = random_tables(rng, trie.num_symbols)[1]
    logw = rng.normal(size=delta.shape).astype(np.float32)
    q = int(np.flatnonzero(trie_oracle(trie).mask(delta, np.arange(delta.shape[0])).sum(axis=1) > 20)[0])
    rows, calls = 4096, 40
    logp = torch.tensor(logsoftmax_rows(1, V, seed=17)).cuda().expand(rows, -1).contiguous()
    tokw = trie.dfa_token_logw(*cuda(delta, logw, np.full(rows, q, np.int32)))
    p = torch.softmax(logp[0].double() + tokw[0].double(), dim=0).cpu().numpy()
    counts = np.zeros(V, dtype=np.int64)
    for k in range(calls):
        _, tok = smc.masked_logsumexp_sample(logp, tokw, seed=5, offset=k * rows)
        counts += np.bincount(tok.cpu().numpy(), minlength=V)
    n = rows * calls
    assert counts.sum() == n and counts[p == 0].sum() == 0
    big = p * n >= 5
    obs = np.append(counts[big], counts[~big].sum())
    exp = np.append(p[big] * n, p[~big].sum() * n)
    sel = exp > 0
    assert stats.chisquare(obs[sel], exp[sel] * obs[sel].sum() / exp[sel].sum()).pvalue > 1e-4


@pytest.mark.gpu
def test_zero_weights_compose_with_the_masked_next_symbol_draw():
    trie, delta, logw, nodes, states, logp = step_inputs(18, 128)
    d, st = cuda(delta, states)
    tokw = trie.dfa_token_logw(d, torch.zeros(delta.shape, device="cuda"), st)  # one per token, at the root
    bits = trie.dfa_token_mask(d, st)
    internal = np.flatnonzero(np.diff(trie._layout["child_ptr"]) > 0)
    rng = np.random.default_rng(18)
    for n in (np.full(len(states), trie.root), rng.choice(internal, len(states))):
        nt = torch.tensor(n.astype(np.int32)).cuda()
        for k in range(3):
            a = trie.sample_next_symbol(logp + tokw, nt, log_input=True, seed=9, offset=k * 1000)
            b = trie.sample_next_symbol(logp, nt, mask=bits, log_input=True, seed=9, offset=k * 1000)
            for x, y in zip(a, b):
                assert torch.equal(x, y)


@pytest.mark.gpu
def test_weighted_step_in_cuda_graph_matches_eager():
    trie, delta, logw, nodes, states, logp = step_inputs(19, 64, table=1)
    d, w, st, nd = cuda(delta, logw, states, nodes)
    eager = weighted_step(trie, d, w, st, nd, logp, seed=11)
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        weighted_step(trie, d, w, st, nd, logp, seed=11)  # warm-up on the capturing stream
    stream.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        out = weighted_step(trie, d, w, st, nd, logp, seed=11)
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        for have, want in zip(out, eager):
            assert torch.equal(have, want)
