"""Token log-weights under a weighted byte-level pushdown automaton (``gt_pda_token_logw``).

CPU part: the reference of ``pda_logw_oracle`` on hand-checked rows of a bracket automaton, and the argument checks of
the entry point and their order.  GPU part (``-m gpu``): the kernel bit for bit against the reference on the JSON
vocabulary (random weights, a depth penalty), ``synth_vocab`` at 128,256 tokens and the ``vocab_shapes`` families, under
random PDAs of 1 to 4,096 states, rows from depth 0 to capacity and invalid rows, and a padded table; a padded output
row stride; special values; zero weights against the Boolean mask and push-free tables against ``dfa_token_logw``; the
weighted JSON step (log-weights, draw, advance, resampling) in one CUDA graph, with its weight increment and a
chi-square test of its draw; and the exact weighted byte-level route.
"""
import ctypes

import numpy as np
import pytest
import torch

import dfa_oracle
import oracle
import pda_oracle
import vocab_shapes
from genlm_backend_b200 import ParallelTokenCharacterTrie, _lib, dfa, pda, smc
from genlm_backend_b200.synthetic import synth_vocab
from helpers import golden_vocab, tokens
from pda_logw_oracle import WeightedPdaOracle
from test_pda import cuda, json_rows, json_tables, random_rows

NINF = -np.inf
POS = np.inf
BRACKETS = [b"[", b"]", b"[[", b"[]", b"]]", b"[]]"]


def bracket_tables(S, w_push=-1.0, w_pop=-0.25):
    """One state: "[" pushes 0 with log-weight w_push, "]" pops with log-weight w_pop; everything else rejects."""
    delta = np.full((1, S), -1, dtype=np.int32)
    push = np.full((1, S), -1, dtype=np.int32)
    logw = np.zeros((1, S), dtype=np.float32)
    delta[0, ord("[")], push[0, ord("[")], logw[0, ord("[")] = 0, 0, w_push
    delta[0, ord("]")], logw[0, ord("]")] = pda.GT_PDA_POP, w_pop
    return delta, push, logw


def ieee(o, *args):
    with np.errstate(invalid="ignore", over="ignore"):  # inf - inf and sums past the float32 range are the point here
        return o.logw(*args)


def random_weights(rng, shape, scale=1.0):
    return (rng.normal(size=shape) * scale).astype(np.float32)


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_oracle_hand_checked_brackets():
    o = WeightedPdaOracle(BRACKETS)
    delta, push, logw = bracket_tables(256)
    stack = np.zeros((2, 2), dtype=np.int32)
    have = o.logw(delta, push, logw, [0, 0], stack, [0, 1])
    want = np.array([
        # [      ]      [[     []      ]]    []]
        [-1.0, NINF, -2.0, -1.25, NINF, NINF],  # depth 0: no pop from the empty stack
        [-1.0, -0.25, NINF, -1.25, NINF, -1.5],  # depth 1 of 2: "[[" pushes past the capacity, "]]" pops twice
    ], dtype=np.float32)
    assert have.dtype == np.float32 and np.array_equal(have, want)
    have3 = o.logw(delta, push, logw, [0, 0], np.zeros((2, 3), np.int32), [0, 1])
    assert have3[1, 2] == -2.0 and np.array_equal(have3[0], want[0])  # capacity 3: "[[" fits from depth 1
    # zero weights: the additive form of the mask; invalid rows: all -inf
    assert np.array_equal(o.logw(delta, push, np.zeros_like(logw), [0, 0], stack, [0, 1]),
                          np.where(o.mask(delta, push, [0, 0], stack, [0, 1]), np.float32(0), np.float32(NINF)))
    bad = o.logw(delta, push, logw, [1, -1, 0, 0], np.zeros((4, 2), np.int32), [0, 0, 3, -1])
    assert (bad == NINF).all()


def test_oracle_special_values_and_the_empty_item():
    o = WeightedPdaOracle(BRACKETS + [b""])
    delta, push, _ = bracket_tables(256)
    stack = np.zeros((2, 2), dtype=np.int32)
    cases = {  # (w_push, w_pop) -> row at depth 0, row at depth 1
        (NINF, POS): ([NINF, NINF, NINF, np.nan, NINF, NINF, 0], [NINF, POS, NINF, np.nan, NINF, np.nan, 0]),
        (np.nan, -1.0): ([np.nan, NINF, np.nan, np.nan, NINF, NINF, 0], [np.nan, -1.0, NINF, np.nan, NINF, np.nan, 0]),
        (POS, np.nan): ([POS, NINF, POS, np.nan, NINF, NINF, 0], [POS, np.nan, NINF, np.nan, NINF, np.nan, 0]),
    }
    for (wp, wq), want in cases.items():
        _, _, logw = bracket_tables(256, wp, wq)
        have = ieee(o, delta, push, logw, [0, 0], stack, [0, 1])
        assert np.array_equal(have, np.array(want, np.float32), equal_nan=True), (wp, wq)


def test_logw_entry_point_rejects_bad_arguments_in_order_without_a_gpu():
    trie = ParallelTokenCharacterTrie(golden_vocab("sentinel"))
    h = trie._engine._handle
    V, S = trie._engine.V, trie.num_symbols
    lib = _lib.lib
    p = ctypes.c_void_p(1 << 20)  # stands for a device pointer: never dereferenced by the checks

    def call(**kw):
        a = dict(t=h, delta=p, push=p, logw=p, Q=4, ld=S, states=p, stack=p, cap=8, depth=p, n=4, out=p, ld_out=V)
        a.update(kw)
        rc = lib.gt_pda_token_logw(a["t"], a["delta"], a["push"], a["logw"], a["Q"], a["ld"], a["states"], a["stack"],
                                   a["cap"], a["depth"], a["n"], a["out"], a["ld_out"], None)
        return rc, lib.gt_last_error().decode() if rc else ""

    for bad in (dict(t=None), dict(delta=None), dict(push=None), dict(logw=None), dict(states=None), dict(stack=None),
                dict(depth=None), dict(out=None), dict(ld_out=V - 1), dict(ld_out=0), dict(Q=0), dict(Q=-1),
                dict(ld=S - 1), dict(ld=0), dict(n=-1), dict(cap=0), dict(cap=-3)):
        rc, msg = call(**bad)
        assert rc == 1 and "gt_pda_token_logw" in msg, bad
    for bad in (dict(Q=(1 << 31) // S + 1), dict(Q=1 << 40), dict(cap=65), dict(cap=1 << 40)):
        assert call(**bad)[0] == 4, bad
    assert "GT_PDA_MAX_DEPTH" in call(cap=65)[1]
    # the order: null trie, null pointers, ld_out, the table and row counts, the table's size, the capacity, no rows,
    # the grid
    assert "null trie" in call(t=None, logw=None, ld_out=0, Q=0)[1]
    assert "null data pointer" in call(logw=None, ld_out=0, Q=0)[1]
    assert "null data pointer" in call(out=None, ld_out=0, cap=0)[1]
    assert "ld_out" in call(ld_out=V - 1, Q=0, n=-1, cap=65)[1]
    assert "bad n_states" in call(Q=0, n=0, cap=65)[1]
    assert call(Q=(1 << 31) // S + 1, n=0, cap=0)[0] == 4
    assert "stack_ld" in call(cap=0, n=0)[1] and call(cap=65, n=0)[0] == 4
    assert call(n=0)[0] == 0 and call(n=0, cap=64)[0] == 0 and call(n=0, cap=1)[0] == 0
    rc, msg = call(n=65535 * 4 + 1)
    assert rc == 4 and "too many rows" in msg


# ---- GPU ---------------------------------------------------------------------------------------------------------
def check_logw(trie, o, delta, push, logw, states, stack, depth, what=""):
    """The log-weights bit for bit (NaN for NaN) against the reference, their finite-or-not pattern against the Boolean
    mask where the table is finite, and the rows' stacks and depths untouched."""
    V, B = o.V, len(states)
    d, p, st, stk, dep = cuda(delta, push, states, stack, depth)
    out = trie.pda_token_logw(d, p, torch.tensor(logw).cuda(), st, stk, dep)
    assert out.dtype == torch.float32 and out.shape == (B, V) and out.device == d.device
    have = out.cpu().numpy()
    want = ieee(o, delta, push, logw, states, stack, depth)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(have), nan), what  # NaN payloads aside, bit for bit
    assert np.array_equal(have[~nan].view(np.uint32), want[~nan].view(np.uint32)), what
    allowed = oracle.unpack_bits(trie.pda_token_mask(d, p, st, stk, dep).cpu().numpy(), V)
    assert np.array_equal(allowed, o.mask(delta, push, states, stack, depth)), what
    assert (have[~allowed] == NINF).all(), what  # whatever the weights on a rejected walk
    assert torch.equal(stk.cpu(), torch.tensor(stack)) and torch.equal(dep.cpu(), torch.tensor(depth))
    return have, allowed


@pytest.fixture(scope="module")
def json_setup():
    dec = pda_oracle.json_vocab()
    trie = ParallelTokenCharacterTrie(dec)
    assert trie.num_symbols == 257
    return dec, trie, WeightedPdaOracle(dec)


@pytest.mark.gpu
def test_hand_checked_brackets_on_the_device():
    trie = ParallelTokenCharacterTrie(tokens(BRACKETS))
    o = WeightedPdaOracle(BRACKETS)
    S = trie.num_symbols
    delta, push, logw = bracket_tables(S)
    for cap in (2, 3):
        have, _ = check_logw(trie, o, delta, push, logw, [0, 0, 1, 0], np.zeros((4, cap), np.int32), [0, 1, 0, cap + 1])
        want = [[-1.0, NINF, -2.0, -1.25, NINF, NINF], [-1.0, -0.25, NINF if cap == 2 else -2.0, -1.25, NINF, -1.5],
                [NINF] * 6, [NINF] * 6]
        assert np.array_equal(have, np.array(want, np.float32)), cap


@pytest.mark.gpu
@pytest.mark.parametrize("cap", [1, 3, 64])
def test_json_logw_matches_oracle(json_setup, cap):
    """json_pda under random normal weights on every entry, and under a depth penalty: -0.7 on every push, 0
    elsewhere."""
    dec, trie, o = json_setup
    delta, push, start = json_tables()
    rng = np.random.default_rng(200 + cap)
    B = 96
    top = 10 + B // 8
    states, stack, depth = json_rows(rng, B, cap, delta, push, start)
    states[top], depth[top] = start, 0
    normal = random_weights(rng, delta.shape, 2.0)
    penalty = np.where(push >= 0, np.float32(-0.7), np.float32(0)).astype(np.float32)
    for logw in (normal, penalty):
        have, allowed = check_logw(trie, o, delta, push, logw, states, stack, depth, f"json cap {cap}")
        assert allowed[top:].any(axis=1).all()  # every reachable configuration has a next token
    # the depth penalty by hand at the start of a document: outside strings, each "[" or "{" of a token pushes once
    plain = [i for i, t in enumerate(dec) if allowed[top, i] and b'"' not in getattr(t, "byte_string", b'"')]
    assert len(plain) > 100
    for i in plain:
        n_open = sum(dec[i].byte_string.count(c) for c in (b"[", b"{"))
        assert have[top, i] == np.float32(n_open * np.float64(np.float32(-0.7))), dec[i].byte_string


@pytest.mark.gpu
@pytest.mark.parametrize("Q", [1, 2, 8, 61, 256, 4096])
def test_random_pdas_match_oracle(json_setup, Q):
    _, trie, o = json_setup
    rng = np.random.default_rng(300 + Q)
    S = trie.num_symbols
    for cap in (1, 3, 64):
        delta, push = pda_oracle.random_pda(rng, Q, S, p_move=0.75, p_pop=0.15)
        logw = random_weights(rng, delta.shape)
        states, stack, depth = random_rows(rng, Q, 64, cap)
        check_logw(trie, o, delta, push, logw, states, stack, depth, f"Q {Q} cap {cap}")
    # a padded table: ld_delta > S, the padding full of moves, pushes and weights that must never be read
    pad = 9
    dp = np.concatenate([delta, rng.integers(0, Q, (Q, pad)).astype(np.int32)], axis=1)
    pp = np.concatenate([push, rng.integers(0, Q, (Q, pad)).astype(np.int32)], axis=1)
    wp = np.concatenate([logw, np.full((Q, pad), np.nan, np.float32)], axis=1)
    d, p, st, stk, dep = cuda(dp, pp, states, stack, depth)
    have = trie.pda_token_logw(d, p, torch.tensor(wp).cuda(), st, stk, dep).cpu().numpy()
    assert np.array_equal(have, o.logw(delta, push, logw, states, stack, depth)), Q


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["synth128256", "runs", "dups", "no_single_bytes", "wide_alphabet", "chain513"])
def test_vocab_families_match_oracle(name):
    dec = synth_vocab(128256) if name == "synth128256" else vocab_shapes.vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    o = WeightedPdaOracle(dec)
    S = trie.num_symbols
    assert o.S == S
    rng = np.random.default_rng(17)
    B = 24 if name == "synth128256" else 40
    for Q, cap, kw in ((16, 64, dict(p_move=0.85, p_pop=0.1, p_push=0.4)), (300, 7, {})):
        delta, push = pda_oracle.random_pda(rng, Q, S, **kw)
        # a self-loop pushing on every run character, so that long runs reach the capacity
        delta[0, list(vocab_shapes.RUN_CHARS) + [0]] = 0
        push[0, list(vocab_shapes.RUN_CHARS) + [0]] = 1
        logw = random_weights(rng, delta.shape, 0.5)
        states, stack, depth = random_rows(rng, Q, B, cap)
        states[10:14] = 0
        have, allowed = check_logw(trie, o, delta, push, logw, states, stack, depth, f"{name} Q {Q}")
        assert allowed.any()
        if name == "dups":  # the empty items: 0 wherever the row is valid
            empty = np.flatnonzero(o.lens == 0)
            assert empty.size and (have[allowed[:, empty[0]]][:, empty] == 0).all()


@pytest.mark.gpu
def test_padded_output_row_stride_leaves_the_tail_untouched(json_setup):
    _, trie, o = json_setup
    V = o.V
    delta, push, start = json_tables()
    rng = np.random.default_rng(3)
    logw = random_weights(rng, delta.shape)
    B, ld = 37, V + 13
    states, stack, depth = json_rows(rng, B, 16, delta, push, start)
    d, p, st, stk, dep = cuda(delta, push, states, stack, depth)
    w = torch.tensor(logw).cuda()
    buf = torch.full((B, ld), float("nan"), dtype=torch.float32, device="cuda")
    trie._engine.ensure_device(torch.cuda.current_device())  # the raw entry point needs the metadata resident
    _lib.check(_lib.lib.gt_pda_token_logw(trie._engine._handle, d.data_ptr(), p.data_ptr(), w.data_ptr(), d.shape[0],
                                          d.shape[1], st.data_ptr(), stk.data_ptr(), 16, dep.data_ptr(), B,
                                          buf.data_ptr(), ld, torch.cuda.current_stream().cuda_stream),
               "gt_pda_token_logw")
    have = buf.cpu().numpy()
    assert np.array_equal(have[:, :V], o.logw(delta, push, logw, states, stack, depth))
    assert np.isnan(have[:, V:]).all()


@pytest.mark.gpu
def test_special_values_follow_ieee(json_setup):
    """-inf then +inf gives NaN, NaN gives NaN, +inf gives +inf; a rejected item is -inf whatever the weights on its
    walk: on the bracket automaton by hand, and under random PDAs with sprinkled special weights against the
    reference."""
    trie = ParallelTokenCharacterTrie(tokens(BRACKETS))
    o = WeightedPdaOracle(BRACKETS)
    S = trie.num_symbols
    delta, push, _ = bracket_tables(S)
    for wp, wq in ((NINF, POS), (np.nan, -1.0), (POS, np.nan)):
        _, _, logw = bracket_tables(S, wp, wq)
        check_logw(trie, o, delta, push, logw, [0, 0], np.zeros((2, 2), np.int32), [0, 1], (wp, wq))
    _, _, logw = bracket_tables(S, NINF, POS)
    have = trie.pda_token_logw(*cuda(delta, push), torch.tensor(logw).cuda(),
                               *cuda([0, 0], np.zeros((2, 2), np.int32), [0, 1])).cpu().numpy()
    assert np.isnan(have[0, 3]) and np.isnan(have[1, 5]) and have[1, 1] == POS  # "[]": -inf + inf; "]": +inf
    assert have[1, 2] == NINF and have[1, 4] == NINF  # "[[" past capacity, "]]" below the stack: +inf on their walks

    _, trie, o = json_setup
    rng = np.random.default_rng(12)
    seen = {"nan": 0, "pinf": 0, "ninf_allowed": 0}
    for Q in (8, 61):
        delta, push = pda_oracle.random_pda(rng, Q, trie.num_symbols, p_move=0.75, p_pop=0.15)
        states, stack, depth = random_rows(rng, Q, 64, 5)
        for frac in (0.002, 0.02):
            logw = random_weights(rng, delta.shape)
            u = rng.random(delta.shape)
            logw[u < frac] = np.inf
            logw[(u >= frac) & (u < 2 * frac)] = -np.inf
            logw[(u >= 2 * frac) & (u < 3 * frac)] = np.nan
            logw[(delta < 0) & (delta != pda.GT_PDA_POP)] = np.nan  # a rejecting transition's weight never shows
            have, allowed = check_logw(trie, o, delta, push, logw, states, stack, depth, (Q, frac))
            seen["nan"] += int(np.isnan(have).sum())
            seen["pinf"] += int((have == np.inf).sum())
            seen["ninf_allowed"] += int((np.isneginf(have) & allowed).sum())
    assert all(v > 0 for v in seen.values()), seen


@pytest.mark.gpu
@pytest.mark.parametrize("cap", [1, 64])
def test_zero_weights_equal_the_additive_mask(json_setup, cap):
    dec, trie, o = json_setup
    V, S = len(dec), trie.num_symbols
    rng = np.random.default_rng(13)
    delta, push, start = json_tables()
    tables = [(delta, push, json_rows(rng, 96, cap, delta, push, start))]
    for Q in (8, 256):
        d2, p2 = pda_oracle.random_pda(rng, Q, S, p_move=0.75, p_pop=0.15)
        tables.append((d2, p2, random_rows(rng, Q, 96, cap)))
    for delta, push, (states, stack, depth) in tables:
        d, p, st, stk, dep = cuda(delta, push, states, stack, depth)
        bits = oracle.unpack_bits(trie.pda_token_mask(d, p, st, stk, dep).cpu().numpy(), V)
        out = trie.pda_token_logw(d, p, torch.zeros(delta.shape, device="cuda"), st, stk, dep).cpu().numpy()
        want = torch.where(torch.tensor(bits), 0.0, float("-inf")).to(torch.float32).numpy()
        assert np.array_equal(out.view(np.uint32), want.view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["json", "synth3000"])
def test_push_free_tables_equal_dfa_token_logw(json_setup, name):
    dec = json_setup[0] if name == "json" else golden_vocab(name)
    trie = json_setup[1] if name == "json" else ParallelTokenCharacterTrie(dec)
    S = trie.num_symbols
    rng = np.random.default_rng(11)
    for Q in (1, 8, 256):
        delta, acc = dfa_oracle.random_dfa(rng, Q, S, p_live=0.9)
        delta = dfa.trim(delta, acc) if Q > 1 else np.zeros((1, S), np.int32)
        push = np.full_like(delta, -1)
        logw = random_weights(rng, delta.shape)
        B = 48
        states = rng.integers(0, Q, B).astype(np.int32)
        states[1], states[2] = -1, Q
        stack = rng.integers(0, Q, (B, 9)).astype(np.int32)
        d, p, st, stk, dep = cuda(delta, push, states, stack, np.zeros(B))  # empty stacks
        w = torch.tensor(logw).cuda()
        have = trie.pda_token_logw(d, p, w, st, stk, dep)
        want = trie.dfa_token_logw(d, w, st)
        assert torch.equal(have.view(torch.int32), want.view(torch.int32)), (name, Q)
        assert torch.isfinite(have).any()


@pytest.mark.gpu
def test_bad_weight_tables_raise(json_setup):
    _, trie, _ = json_setup
    delta, push, start = json_tables()
    B = 4
    st = torch.full((B,), start, dtype=torch.int32, device="cuda")
    stk = torch.zeros((B, 8), dtype=torch.int32, device="cuda")
    dep = torch.zeros(B, dtype=torch.int32, device="cuda")
    for bad in (np.zeros((delta.shape[0], delta.shape[1] - 1), np.float32), np.zeros((2, delta.shape[1]), np.float32),
                np.zeros(delta.shape, np.int32), delta):
        with pytest.raises(ValueError, match="logw must be a float table of delta's shape"):
            trie.pda_token_logw(delta, push, bad, st, stk, dep)
    with pytest.raises(ValueError):
        trie.pda_token_logw(delta, push, np.zeros(delta.shape, np.float32), st, stk.cpu(), dep)
    # float64 tables are converted to float32 on the device
    w = np.random.default_rng(0).normal(size=delta.shape)
    assert torch.equal(trie.pda_token_logw(delta, push, w, st, stk, dep),
                       trie.pda_token_logw(delta, push, w.astype(np.float32), st, stk, dep))


def weighted_token_step(trie, d, p, w, q, stack, depth, logp, lw, G, seed, offset):
    """The weighted JSON token-level SMC step: log-weights, draw, advance, weight update, resampling and reindexing of
    every per-particle tensor; in place, so that a captured graph can be replayed step after step."""
    B = logp.shape[0]
    tokw = trie.pda_token_logw(d, p, w, q, stack, depth)
    logZ, tok = smc.masked_logsumexp_sample(logp, tokw, seed=seed, offset=offset)
    nq = trie.pda_advance(d, p, q, stack, depth, tok)
    anc, nlw, *_ = smc.resample((lw + logZ).view(G, B // G), "systematic", 0.5, seed=seed, offset=offset)
    idx = anc.view(-1)
    q.copy_(nq.index_select(0, idx))
    stack.copy_(stack.index_select(0, idx))
    depth.copy_(depth.index_select(0, idx))
    lw.copy_(nlw.view(-1))
    return tokw, logZ, tok, idx


def json_weights(rng, delta, push):
    """Normal log-weights on every transition of json_pda (scale 0.5) and -0.5 more on every push: a depth prior."""
    prior = np.where(push >= 0, np.float32(-0.5), np.float32(0))
    return (random_weights(rng, delta.shape, 0.5) + prior).astype(np.float32)


@pytest.mark.gpu
def test_weighted_json_smc_step_in_one_cuda_graph(json_setup):
    dec, trie, o = json_setup
    delta, push, start = json_tables()
    V, B, G, cap = len(dec), 64, 8, 64
    rng = np.random.default_rng(22)
    logw = json_weights(rng, delta, push)
    logits = rng.normal(size=(B, V)).astype(np.float32) * 2
    logits[:, 256] += 8.0  # EOS, wherever it is allowed
    logp = torch.log_softmax(torch.tensor(logits), dim=1).cuda()
    d, p = cuda(delta, push)
    w = torch.tensor(logw).cuda()
    q = torch.full((B,), start, dtype=torch.int32, device="cuda")
    stack = torch.zeros((B, cap), dtype=torch.int32, device="cuda")
    depth = torch.zeros(B, dtype=torch.int32, device="cuda")
    lw = torch.zeros(B, dtype=torch.float32, device="cuda")
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):  # warm-up on the capturing stream, on copies
        weighted_token_step(trie, d, p, w, q.clone(), stack.clone(), depth.clone(), logp, lw.clone(), G, 0, 0)
    stream.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        tokw, logZ, tok, idx = weighted_token_step(trie, d, p, w, q, stack, depth, logp, lw, G, 5, 0)
    texts, finished = [b""] * B, [None] * B
    hp = logp.double().cpu()
    for step in range(60):
        h_q, h_stack, h_depth = q.cpu().numpy(), stack.cpu().numpy(), depth.cpu().numpy()
        g.replay()
        torch.cuda.synchronize()
        want = o.logw(delta, push, logw, h_q, h_stack, h_depth)
        assert np.array_equal(tokw.cpu().numpy(), want), step
        live = [f is None for f in finished]
        assert np.isfinite(want[live]).any(axis=1).all()  # no live particle meets a dead end
        ref = torch.logsumexp(hp + torch.tensor(want, dtype=torch.float64), dim=1).numpy()
        np.testing.assert_allclose(logZ.cpu().numpy(), ref, rtol=1e-5, atol=1e-6)
        t, anc = tok.cpu().numpy(), idx.cpu().numpy()
        assert (t >= 0).all() and np.isfinite(want[np.arange(B), t]).all()
        for b in range(B):
            if finished[b] is None and t[b] == 256:
                finished[b] = texts[b]
            elif finished[b] is None:
                texts[b] += dec[t[b]].byte_string
        texts = [texts[a] for a in anc]
        finished = [finished[a] for a in anc]
        if all(f is not None for f in finished):
            break
    assert any(f is not None for f in finished)
    for f in finished:
        if f is not None:
            assert pda_oracle.json_loads_accepts(f), f
    for b in range(B):  # the live ones stand where the reference walk of their text stands
        if finished[b] is None:
            wq, ws = pda_oracle.walk(delta, push, start, [], list(texts[b]), cap)
            assert wq == int(q[b]) and ws == stack[b, :int(depth[b])].cpu().tolist()


@pytest.mark.gpu
def test_weighted_draw_follows_the_weighted_distribution(json_setup):
    from scipy import stats

    dec, trie, o = json_setup
    delta, push, start = json_tables()
    V = len(dec)
    rng = np.random.default_rng(23)
    logw = json_weights(rng, delta, push)
    # after a number inside an array: a few hundred allowed tokens
    q0, stk0 = pda_oracle.walk(delta, push, start, [], list(b"[1"), 8)
    rows, calls = 4096, 40
    st = torch.full((rows,), q0, dtype=torch.int32, device="cuda")
    stk = torch.zeros((rows, 8), dtype=torch.int32, device="cuda")
    stk[:, :len(stk0)] = torch.tensor(stk0, dtype=torch.int32)
    dep = torch.full((rows,), len(stk0), dtype=torch.int32, device="cuda")
    tokw = trie.pda_token_logw(*cuda(delta, push), torch.tensor(logw).cuda(), st, stk, dep)
    assert 200 <= int(torch.isfinite(tokw[0]).sum()) <= 500
    logp = torch.log_softmax(torch.tensor(rng.normal(size=(1, V)), dtype=torch.float32), dim=1).cuda()
    logp = logp.expand(rows, -1).contiguous()
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
def test_json_exact_weighted_byte_level_route(json_setup):
    """Per token: one tokw at the root in the particle's configuration; byte by byte, sample_next_symbol(logps + tokw,
    log_input=True) draws from p · w / Z.  The root's logZ is masked_logsumexp_sample(logps, tokw)'s; a drawn leaf ends
    the token, which pda_advance consumes; every finished text parses."""
    dec, trie, o = json_setup
    delta, push, start = json_tables()
    V, B, cap = len(dec), 32, 64
    rng = np.random.default_rng(9)
    logw = json_weights(rng, delta, push)
    logits = rng.normal(size=(B, V)).astype(np.float32)
    logits[:, 256] += 10.0  # EOS dominates wherever it is allowed
    logps = torch.log_softmax(torch.tensor(logits), dim=1).cuda()
    d, p = cuda(delta, push)
    w = torch.tensor(logw).cuda()
    q = torch.full((B,), start, dtype=torch.int32, device="cuda")
    stack = torch.zeros((B, cap), dtype=torch.int32, device="cuda")
    depth = torch.zeros(B, dtype=torch.int32, device="cuda")
    root = len(trie) - 1
    texts, finished = [b""] * B, [None] * B
    for step in range(40):
        tokw = trie.pda_token_logw(d, p, w, q, stack, depth)
        assert np.array_equal(tokw.cpu().numpy(), o.logw(delta, push, logw, q.cpu().numpy(), stack.cpu().numpy(),
                                                         depth.cpu().numpy()))
        ws = logps + tokw
        lse, _ = smc.masked_logsumexp_sample(logps, tokw, seed=1, offset=step * B)
        node = torch.full((B,), root, dtype=torch.int32, device="cuda")
        tok = torch.full((B,), -1, dtype=torch.int32, device="cuda")
        for k in range(100):  # the longest item has 80 bytes
            child, label, _, logZ = trie.sample_next_symbol(ws, node, log_input=True, seed=3,
                                                            offset=(step * 100 + k) * B)
            if k == 0:
                np.testing.assert_allclose(logZ.cpu().numpy(), lse.cpu().numpy(), rtol=1e-5, atol=1e-6)
            c, lab = child.cpu().numpy(), label.cpu().numpy()
            pending = tok.cpu().numpy() < 0
            assert (c[pending] >= 0).all()
            leaf = pending & (lab < 0)
            tok[torch.tensor(leaf).cuda()] = torch.tensor(-1 - lab[leaf], dtype=torch.int32).cuda()
            node = torch.where(torch.tensor(pending & ~leaf).cuda(), child, node)
            if (tok >= 0).all():
                break
        assert (tok >= 0).all()
        assert torch.isfinite(tokw.gather(1, tok.long()[:, None])).all()
        q = trie.pda_advance(d, p, q, stack, depth, tok)
        assert (q >= 0).all()
        for b, t in enumerate(tok.cpu().tolist()):
            if finished[b] is None:
                if t == 256:
                    finished[b] = texts[b]
                else:
                    texts[b] += dec[t].byte_string
        if all(f is not None for f in finished):
            break
    assert any(f is not None for f in finished)
    for f in finished:
        if f is not None:
            assert pda_oracle.json_loads_accepts(f), f
