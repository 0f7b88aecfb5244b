"""Token masks under a byte-level pushdown automaton (``gt_pda_token_mask``), the PDA advance over drawn tokens
(``gt_pda_advance``) and the JSON automaton of ``genlm_backend_b200.pda``.

CPU part: ``json_pda`` against Python's JSON parser on seeded documents, their mutations and truncations; every prefix
of a valid document is live and every state can be completed; the reference walk on hand-checked cases; the argument
checks and their order.  GPU part (``-m gpu``): masks and advances bit for bit against ``pda_oracle`` on the JSON
vocabulary, ``synth_vocab`` at 128,256 tokens and the ``vocab_shapes`` families, under random PDAs of 1 to 4,096 states
and rows from depth 0 to capacity; push-free tables against the DFA calls; rejected advances; graph replay; and a
JSON-constrained SMC run, token by token in one CUDA graph and byte by byte through the masked next-symbol draw.
"""
import ctypes
import json

import numpy as np
import pytest
import torch

import oracle
import pda_oracle
import vocab_shapes
from genlm_backend_b200 import ParallelTokenCharacterTrie, _lib, dfa, pda, smc
from genlm_backend_b200.synthetic import synth_vocab
import dfa_oracle
from helpers import golden_vocab

EOS_SYM = 256


def json_tables(S=257, eos=EOS_SYM):
    return pda.json_pda(S, eos=eos)


def mutations(rng, doc, n):
    """n byte mutations of doc: a substitution, a deletion, an insertion or a duplication of a random span."""
    out = []
    special = b'[]{}",:\\0-.eE+ \x00\x80\xbf\xc2\xed\xf4\xff'
    for _ in range(n):
        d = bytearray(doc)
        k = int(rng.integers(0, 4))
        at = int(rng.integers(0, len(d) + 1))
        b = special[int(rng.integers(0, len(special)))] if rng.random() < 0.7 else int(rng.integers(0, 256))
        if k == 0 and d:
            d[min(at, len(d) - 1)] = b
        elif k == 1 and d:
            del d[min(at, len(d) - 1)]
        elif k == 2:
            d.insert(at, b)
        else:
            d[at:at] = d[at:at + int(rng.integers(1, 6))]
        out.append(bytes(d))
    return out


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_json_pda_agrees_with_json_loads():
    delta, push, start = json_tables()
    rng = np.random.default_rng(0)
    docs = [pda_oracle.random_json(rng) for _ in range(300)]
    docs += [b"0", b"-0", b"-0.0e+00", b"1E5", b"01", b"1.", b".5", b"-", b"+1", b"1e", b"1e+", b"[1,]", b"[,1]",
             b'{"a"}', b'{"a":}', b'{,"a":1}', b'{"a":1,}', b"[", b"]", b"", b"   ", b"nul", b"nulls", b"true false",
             b'"\\x"', b'"\\u12"', b'"\\uD800"', b'"\\ud83d\\ude00"', b'"\x1f"', b'"\x7f"', b"\xef\xbb\xbf1",
             b'"\xed\x9f\xbf"', b'"\xed\xa0\x80"', b'"\xc1\xbf"', b'"\xe0\x9f\xbf"', b'"\xf0\x8f\xbf\xbf"',
             b'"\xf4\x8f\xbf\xbf"', b'"\xf4\x90\x80\x80"', b'"\xf5\x80\x80\x80"', b"NaN", b"-Infinity", b"[1 2]",
             b'{"a" "b"}', b"[" * 64 + b"]" * 64, b'"\xf4e', b'"\xf4\x8f\xbf\xbfe"', b'[fals\x8f\x80\x80"]', b"tru\x80", b"{}" * 2, b"[]", b"{}", b' {"":""} ', b"1\n", b"\t[\r]\n"]
    cases = []
    for doc in docs:
        cases.append(doc)
        cases += mutations(rng, doc, 4)
        cases += [doc[:int(rng.integers(0, len(doc) + 1))] for _ in range(2)]
    n_ok = 0
    for doc in cases:
        ok = pda_oracle.json_loads_accepts(doc)
        if ok and max_nesting(doc) > 64:
            continue  # deeper than the stack: a reject by design
        assert pda_oracle.accepts(delta, push, start, doc, EOS_SYM) == ok, doc
        n_ok += ok
    assert 300 < n_ok < len(cases) - 300  # both sides are well represented


def max_nesting(doc):
    """Nesting depth of a document that json.loads accepts (brackets inside strings do not count)."""
    def depth(v):
        if isinstance(v, list):
            return 1 + max(map(depth, v), default=0)
        if isinstance(v, dict):
            return 1 + max(map(depth, v.values()), default=0)
        return 0

    return depth(json.loads(doc.decode("utf-8")))


def test_every_prefix_of_a_valid_document_is_live():
    delta, push, start = json_tables()
    rng = np.random.default_rng(1)
    for _ in range(150):
        doc = pda_oracle.random_json(rng)
        q, stack = start, []
        for k, b in enumerate(doc):
            q, stack = pda_oracle.walk(delta, push, q, stack, [b], 64)
            assert q >= 0, (doc, k)
        assert pda_oracle.walk(delta, push, q, stack, [EOS_SYM], 64) == (q, [])


def test_every_state_can_be_completed():
    """From every state, a push-free path reaches a pop or the EOS self-loop, and every pushed value is such a state:
    so every reachable configuration completes by closing its containers one by one."""
    delta, push, start = json_tables()
    Q = delta.shape[0]
    done = np.zeros(Q, dtype=bool)
    done[(delta == pda.GT_PDA_POP).any(axis=1)] = True
    done[delta[:, EOS_SYM] == np.arange(Q)] = True
    moves = (delta >= 0) & (push < 0)
    while True:
        nxt = done | (moves & done[np.where(moves, delta, 0)]).any(axis=1)
        if (nxt == done).all():
            break
        done = nxt
    assert done.all()
    assert ((push < 0) | done[np.where(push >= 0, push, 0)]).all()
    # only containers push; EOS is a self-loop where it is allowed, and never at the start
    assert set(np.flatnonzero((push >= 0).any(axis=0)).tolist()) == {ord("["), ord("{")}
    assert ((delta[:, EOS_SYM] == -1) | (delta[:, EOS_SYM] == np.arange(Q))).all()
    assert delta[start, EOS_SYM] == -1


def test_json_pda_arguments():
    d, p, start = pda.json_pda(256)
    assert d.dtype == np.int32 and p.dtype == np.int32 and d.shape == p.shape == (d.shape[0], 256)
    assert d.shape[0] < 200
    d2, _, _ = pda.json_pda(300, eos=299)
    assert (d2[:, 256:299] == -1).all() and (d2[:, 299] >= 0).sum() == 5  # top_end and four number ends
    for bad in (dict(num_symbols=255), dict(num_symbols=257, eos=255), dict(num_symbols=257, eos=257)):
        with pytest.raises(ValueError):
            pda.json_pda(**bad)


def test_oracle_hand_checked():
    """A two-state bracket language over "(" and ")" plus a pop-into-the-row-stack case."""
    S = 256
    delta = np.full((2, S), -1, dtype=np.int32)
    push = np.full((2, S), -1, dtype=np.int32)
    delta[0, ord("(")] = 0
    push[0, ord("(")] = 1
    delta[:, ord(")")] = pda.GT_PDA_POP
    delta[1, ord("x")] = 1
    items = [b"(", b")", b"()", b"((", b"(((", b"))", b"x", b"", b")x"]
    o = pda_oracle.PdaOracle([bytes(i) for i in items])
    stack = np.array([[0, 0], [1, 0], [5, 0], [0, 0], [0, 0], [0, 0]], dtype=np.int32)
    have = o.mask(delta, push, [0, 0, 0, 1, 2, 0], stack, [0, 1, 1, 0, 0, 3]).astype(int)
    want = [
        [1, 0, 1, 1, 0, 0, 0, 1, 0],  # empty stack of capacity 2: no pop, at most two pushes
        [1, 1, 1, 0, 0, 0, 0, 1, 1],  # [1]: one push left; ")" returns to 1, where "x" loops
        [1, 0, 1, 0, 0, 0, 0, 1, 0],  # [5]: the popped value is outside [0, Q)
        [0, 0, 0, 0, 0, 0, 1, 1, 0],  # state 1 with an empty stack
        [0] * 9,                      # invalid state
        [0] * 9,                      # invalid depth
    ]
    assert have.tolist() == want
    st, stk, dep = o.advance(delta, push, [0, 0, 0, 0], stack[:4], [1, 1, 0, 1], [2, 1, 3, 4])
    assert st.tolist() == [1, 1, 0, -1]  # "()" pushes and pops its own entry; "(((" passes the capacity
    assert dep.tolist() == [1, 0, 2, 1] and stk[0, 0] == 0 and stk[2].tolist() == [1, 1]
    assert stk[3].tolist() == [0, 0]


def test_pda_entry_points_reject_bad_arguments_without_a_gpu():
    trie = ParallelTokenCharacterTrie(golden_vocab("sentinel"))
    h = trie._engine._handle
    V, S = trie._engine.V, trie.num_symbols
    W = (V + 31) // 32
    lib = _lib.lib
    p = ctypes.c_void_p(1 << 20)  # stands for a device pointer: never dereferenced by the checks

    def mask(**kw):
        a = dict(t=h, delta=p, push=p, Q=4, ld=S, states=p, stack=p, cap=8, depth=p, n=4, bits=p, ld_bits=W)
        a.update(kw)
        return lib.gt_pda_token_mask(a["t"], a["delta"], a["push"], a["Q"], a["ld"], a["states"], a["stack"], a["cap"],
                                     a["depth"], a["n"], a["bits"], a["ld_bits"], None)

    def advance(**kw):
        a = dict(t=h, delta=p, push=p, Q=4, ld=S, states=p, stack=p, cap=8, depth=p, tokens=p, n=4, out=p)
        a.update(kw)
        return lib.gt_pda_advance(a["t"], a["delta"], a["push"], a["Q"], a["ld"], a["states"], a["stack"], a["cap"],
                                  a["depth"], a["tokens"], a["n"], a["out"], None)

    common = (dict(t=None), dict(delta=None), dict(push=None), dict(states=None), dict(stack=None), dict(depth=None),
              dict(Q=0), dict(Q=-1), dict(ld=S - 1), dict(ld=0), dict(n=-1), dict(cap=0), dict(cap=-3))
    for bad in common + (dict(bits=None), dict(ld_bits=W - 1), dict(ld_bits=0)):
        assert mask(**bad) == 1, bad
    for bad in common + (dict(tokens=None), dict(out=None)):
        assert advance(**bad) == 1, bad
    assert b"gt_pda_advance" in lib.gt_last_error()
    for fn in (mask, advance):
        assert fn(Q=(1 << 31) // S + 1) == 4  # a table of 2^31 entries or more
        assert fn(Q=1 << 40, ld=S) == 4
        assert fn(cap=65) == 4 and fn(cap=1 << 40) == 4
        assert b"GT_PDA_MAX_DEPTH" in lib.gt_last_error()
        assert fn(n=0) == 0 and fn(n=0, cap=64) == 0 and fn(n=0, cap=1) == 0
        # the order: null pointers, then the table's scalars, then the capacity, then "no rows"
        assert fn(states=None, Q=0) == 1 and b"null" in lib.gt_last_error()
        assert fn(Q=0, cap=65) == 1 and b"n_states" in lib.gt_last_error()
        assert fn(Q=1 << 40, cap=0) == 4
        assert fn(cap=0, n=0) == 1 and fn(cap=65, n=0) == 4
    assert mask(ld_bits=0, Q=0) == 1 and b"mask_ld" in lib.gt_last_error()
    assert mask(n=65535 * 8 + 1) == 4 and b"too many rows" in lib.gt_last_error()


# ---- GPU ---------------------------------------------------------------------------------------------------------
def cuda(*xs):
    return [torch.as_tensor(np.ascontiguousarray(x)).to(torch.int32).cuda() for x in xs]


def random_rows(rng, Q, B, cap):
    """States (live ones, -1 and Q), depths (0, 1, cap - 1, cap, random, and the invalid -1 and cap + 1) and stacks
    with live entries and a few outside [0, Q)."""
    states = rng.integers(0, Q, B).astype(np.int32)
    states[1], states[2] = -1, Q
    depth = rng.integers(0, cap + 1, B).astype(np.int32)
    depth[3:9] = [0, 1, max(cap - 1, 0), cap, -1, cap + 1]
    depth[9:9 + B // 8] = cap
    stack = rng.integers(0, Q, (B, cap)).astype(np.int32)
    bad = rng.random((B, cap)) < 0.05
    stack[bad] = rng.choice(np.array([-1, -2, Q, Q + 9], dtype=np.int32), int(bad.sum()))
    return states, stack, depth


def check_mask_and_advance(trie, o, delta, push, states, stack, depth, rng, what=""):
    """The mask and the advance (of an allowed token per row where there is one, and of tokens -1, V and a random one)
    bit for bit against the reference; stacks and depths after the advance; rejected rows unchanged."""
    V, B = o.V, len(states)
    d, p, st, stk, dep = cuda(delta, push, states, stack, depth)
    bits = trie.pda_token_mask(d, p, st, stk, dep)
    assert bits.dtype == torch.int32 and bits.shape == (B, (V + 31) // 32)
    hb = bits.cpu().numpy()
    want = o.mask(delta, push, states, stack, depth)
    assert np.array_equal(oracle.unpack_bits(hb, V), want), what
    assert not oracle.unpack_bits(hb, hb.shape[1] * 32)[:, V:].any()
    assert torch.equal(stk.cpu(), torch.tensor(stack)) and torch.equal(dep.cpu(), torch.tensor(depth))
    toks = np.array([rng.choice(np.flatnonzero(m)) if m.any() and rng.random() < 0.8 else rng.integers(0, V)
                     for m in want], np.int32)
    toks[3:6] = [-1, V, -5]
    adv = trie.pda_advance(d, p, st, stk, dep, torch.tensor(toks).cuda()).cpu().numpy()
    w_st, w_stack, w_depth = o.advance(delta, push, states, stack, depth, toks)
    assert np.array_equal(adv, w_st), what
    ok = (toks >= 0) & (toks < V)
    allowed = np.zeros(B, bool)
    allowed[ok] = want[np.flatnonzero(ok), toks[ok]]
    assert np.array_equal(adv >= 0, allowed)
    have_stack, have_depth = stk.cpu().numpy(), dep.cpu().numpy()
    assert np.array_equal(have_depth, w_depth), what
    for b in range(B):
        if adv[b] >= 0:
            assert np.array_equal(have_stack[b, :w_depth[b]], w_stack[b, :w_depth[b]]), (what, b)
        else:  # a rejected row keeps its whole stack
            assert np.array_equal(have_stack[b], stack[b]), (what, b)
    return want, adv


@pytest.fixture(scope="module")
def json_setup():
    dec = pda_oracle.json_vocab()
    trie = ParallelTokenCharacterTrie(dec)
    assert trie.num_symbols == 257
    return dec, trie, pda_oracle.PdaOracle(dec)


def json_rows(rng, B, cap, delta, push, start):
    """Configurations reached by walking prefixes of random documents (depth up to cap), a few from prefixes deep in
    brackets, and the invalid rows of ``random_rows``."""
    states, stack, depth = random_rows(rng, delta.shape[0], B, cap)
    for b in range(10 + B // 8, B):
        doc = pda_oracle.random_json(rng) if rng.random() < 0.8 else b"[" * int(rng.integers(cap - 3, cap + 1)) + b"{"
        q, stk = start, []
        for ch in doc[:int(rng.integers(0, len(doc) + 1))]:
            nq, nstk = pda_oracle.walk(delta, push, q, stk, [ch], cap)
            if nq < 0:
                break
            q, stk = nq, nstk
        states[b], depth[b] = q, len(stk)
        stack[b, :len(stk)] = stk
    return states, stack, depth


@pytest.mark.gpu
@pytest.mark.parametrize("cap", [1, 3, 64])
def test_json_masks_and_advances_match_oracle(json_setup, cap):
    dec, trie, o = json_setup
    delta, push, start = json_tables()
    rng = np.random.default_rng(cap)
    B = 96
    states, stack, depth = json_rows(rng, B, cap, delta, push, start)
    states[10 + B // 8], depth[10 + B // 8] = start, 0
    want, _ = check_mask_and_advance(trie, o, delta, push, states, stack, depth, rng, f"json cap {cap}")
    assert want[10 + B // 8:].any(axis=1).all()  # every reachable configuration has a next token
    if cap == 64:  # the 70-bracket item passes capacity, the 40 + 40 one fits from an empty stack
        i70, i40 = (next(i for i, t in enumerate(dec) if getattr(t, "byte_string", None) == x)
                    for x in (b"[" * 70, b"[" * 40 + b"]" * 40))
        top = (states == start) & (depth == 0)
        assert top.any() and not want[top, i70].any() and want[top, i40].all()


@pytest.mark.gpu
@pytest.mark.parametrize("Q", [1, 2, 8, 61, 256, 4096])
def test_random_pdas_match_oracle(json_setup, Q):
    _, trie, o = json_setup
    rng = np.random.default_rng(100 + Q)
    for cap in (1, 5, 64):
        delta, push = pda_oracle.random_pda(rng, Q, 257, p_move=0.75, p_pop=0.15)
        states, stack, depth = random_rows(rng, Q, 64, cap)
        check_mask_and_advance(trie, o, delta, push, states, stack, depth, rng, f"Q {Q} cap {cap}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["synth128256", "runs", "dups", "no_single_bytes", "wide_alphabet", "chain513"])
def test_vocab_families_match_oracle(name):
    dec = synth_vocab(128256) if name == "synth128256" else vocab_shapes.vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    o = pda_oracle.PdaOracle(dec)
    S = trie.num_symbols
    assert o.S == S
    rng = np.random.default_rng(7)
    B = 24 if name == "synth128256" else 40
    for Q, cap, kw in ((16, 64, dict(p_move=0.85, p_pop=0.1, p_push=0.4)), (300, 7, {})):
        delta, push = pda_oracle.random_pda(rng, Q, S, **kw)
        # a self-loop pushing on every run character, so that long runs reach the capacity
        delta[0, list(vocab_shapes.RUN_CHARS) + [0]] = 0
        push[0, list(vocab_shapes.RUN_CHARS) + [0]] = 1
        states, stack, depth = random_rows(rng, Q, B, cap)
        states[10:14] = 0
        check_mask_and_advance(trie, o, delta, push, states, stack, depth, rng, f"{name} Q {Q}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["json", "synth3000"])
def test_push_free_tables_equal_the_dfa_calls(json_setup, name):
    dec = json_setup[0] if name == "json" else golden_vocab(name)
    trie = json_setup[1] if name == "json" else ParallelTokenCharacterTrie(dec)
    S, V = trie.num_symbols, len(dec)
    rng = np.random.default_rng(11)
    for Q in (1, 8, 256):
        delta, acc = dfa_oracle.random_dfa(rng, Q, S, p_live=0.9)
        delta = dfa.trim(delta, acc) if Q > 1 else np.zeros((1, S), np.int32)
        push = np.full_like(delta, -1)
        B = 48
        states, stack, depth = random_rows(rng, Q, B, 9)
        depth[4], depth[7], depth[8] = 2, 3, 9  # valid depths only: the DFA calls have no stack
        d, p, st, stk, dep = cuda(delta, push, states, stack, depth)
        bits = trie.pda_token_mask(d, p, st, stk, dep)
        assert torch.equal(bits, trie.dfa_token_mask(d, st))
        toks = torch.tensor(np.where(rng.random(B) < 0.9, rng.integers(0, V, B), -1).astype(np.int32)).cuda()
        dfa_bits = oracle.unpack_bits(bits.cpu().numpy(), V)
        toks[: B // 2] = torch.tensor([rng.choice(np.flatnonzero(m)) if m.any() else -1 for m in dfa_bits[: B // 2]])
        adv = trie.pda_advance(d, p, st, stk, dep, toks)
        assert torch.equal(adv, trie.dfa_advance(d, st, toks))
        assert (adv >= 0).any()
        assert torch.equal(stk.cpu(), torch.tensor(stack)) and torch.equal(dep.cpu(), torch.tensor(depth))


@pytest.mark.gpu
def test_python_arguments(json_setup):
    _, trie, _ = json_setup
    delta, push, start = json_tables()
    B = 4
    st = torch.full((B,), start, dtype=torch.int32, device="cuda")
    stk = torch.zeros((B, 8), dtype=torch.int32, device="cuda")
    dep = torch.zeros(B, dtype=torch.int32, device="cuda")
    tok = torch.full((B,), ord("["), dtype=torch.int32, device="cuda")
    for bad_stack, bad_depth in ((stk.cpu(), dep), (stk.long(), dep), (stk, dep.cpu()), (stk, dep.long()),
                                 (torch.zeros((B, 65), dtype=torch.int32, device="cuda"), dep),
                                 (torch.zeros((B, 0), dtype=torch.int32, device="cuda"), dep),
                                 (torch.zeros((B, 16), dtype=torch.int32, device="cuda")[:, ::2], dep),
                                 (stk[:3], dep), (stk, dep[:3]), (stk.view(-1), dep)):
        with pytest.raises(ValueError):
            trie.pda_advance(delta, push, st, bad_stack, bad_depth, tok)
        with pytest.raises(ValueError):
            trie.pda_token_mask(delta, push, st, bad_stack, bad_depth)
    with pytest.raises(ValueError):
        trie.pda_token_mask(delta, push[:, :10], st, stk, dep)
    # host tables, written back into states
    out = trie.pda_advance(delta, push, st, stk, dep, tok)
    assert (out == int(delta[start, ord("[")])).all() and (dep == 1).all() and (stk[:, 0] == int(push[start, ord("[")])).all()
    st2 = st.clone()
    d, p = cuda(delta, push)
    lib_args = (trie._engine._handle, d.data_ptr(), p.data_ptr(), delta.shape[0], delta.shape[1])
    trie._engine.ensure_device(torch.cuda.current_device())
    _lib.check(_lib.lib.gt_pda_advance(*lib_args, st2.data_ptr(), stk.data_ptr(), 8, dep.data_ptr(), tok.data_ptr(), B,
                                       st2.data_ptr(), torch.cuda.current_stream().cuda_stream), "gt_pda_advance")
    assert torch.equal(st2, out) and (dep == 2).all()


@pytest.mark.gpu
def test_padding_words_and_row_stride(json_setup):
    _, trie, o = json_setup
    V, W = o.V, (o.V + 31) // 32
    delta, push, start = json_tables()
    rng = np.random.default_rng(3)
    states, stack, depth = json_rows(rng, 37, 16, delta, push, start)
    d, p, st, stk, dep = cuda(delta, push, states, stack, depth)
    ld = W + 3
    buf = torch.full((37, ld), 0x55555555, dtype=torch.int32, device="cuda")
    trie._engine.ensure_device(torch.cuda.current_device())
    _lib.check(_lib.lib.gt_pda_token_mask(trie._engine._handle, d.data_ptr(), p.data_ptr(), d.shape[0], d.shape[1],
                                          st.data_ptr(), stk.data_ptr(), 16, dep.data_ptr(), 37, buf.data_ptr(), ld,
                                          torch.cuda.current_stream().cuda_stream), "gt_pda_token_mask")
    have = buf.cpu().numpy()
    assert np.array_equal(have[:, :W], trie.pda_token_mask(d, p, st, stk, dep).cpu().numpy())
    assert (have[:, W:] == 0x55555555).all()


def token_step(trie, d, p, q, stack, depth, logp, lw, G, seed, offset):
    """The JSON-constrained token-level SMC step: mask, draw, advance, weight update, resampling and reindexing of every
    per-particle tensor; in place, so that a captured graph can be replayed step after step."""
    B = logp.shape[0]
    bits = trie.pda_token_mask(d, p, q, stack, depth)
    logZ, tok = smc.masked_logsumexp_sample(logp, bits, seed=seed, offset=offset)
    nq = trie.pda_advance(d, p, q, stack, depth, tok)
    anc, nlw, *_ = smc.resample((lw + logZ).view(G, B // G), "systematic", 0.5, seed=seed, offset=offset)
    idx = anc.view(-1)
    q.copy_(nq.index_select(0, idx))
    stack.copy_(stack.index_select(0, idx))
    depth.copy_(depth.index_select(0, idx))
    lw.copy_(nlw.view(-1))
    return bits, tok, idx


@pytest.mark.gpu
def test_json_smc_run_in_one_cuda_graph(json_setup):
    dec, trie, o = json_setup
    delta, push, start = json_tables()
    V, B, G, cap = len(dec), 64, 8, 64
    rng = np.random.default_rng(21)
    logits = rng.normal(size=(B, V)).astype(np.float32) * 2
    logits[:, 256] += 8.0  # EOS, wherever it is allowed: particles finish as soon as their text is a document
    logp = torch.tensor(logits).cuda()
    d, p = cuda(delta, push)
    q = torch.full((B,), start, dtype=torch.int32, device="cuda")
    stack = torch.zeros((B, cap), dtype=torch.int32, device="cuda")
    depth = torch.zeros(B, dtype=torch.int32, device="cuda")
    lw = torch.zeros(B, dtype=torch.float32, device="cuda")
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):  # warm-up on the capturing stream, on copies
        token_step(trie, d, p, q.clone(), stack.clone(), depth.clone(), logp, lw.clone(), G, 0, 0)
    stream.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        bits, tok, idx = token_step(trie, d, p, q, stack, depth, logp, lw, G, 5, 0)
    texts = [b""] * B
    finished = [None] * B
    n_done = 0
    for step in range(60):
        h_q, h_stack, h_depth = q.cpu().numpy(), stack.cpu().numpy(), depth.cpu().numpy()
        g.replay()  # the same seed and offset every step: the logits differ by state through the mask only
        torch.cuda.synchronize()
        hb, t, anc = oracle.unpack_bits(bits.cpu().numpy(), V), tok.cpu().numpy(), idx.cpu().numpy()
        live = [finished[b] is None for b in range(B)]
        want = o.mask(delta, push, h_q, h_stack, h_depth)
        assert np.array_equal(hb, want)
        assert hb[live].any(axis=1).all()  # no live particle meets a dead end
        assert (t >= 0).all()
        for b in range(B):
            if finished[b] is None and t[b] == 256:
                finished[b] = texts[b]
            elif finished[b] is None:
                texts[b] += dec[t[b]].byte_string
        texts = [texts[a] for a in anc]
        finished = [finished[a] for a in anc]
        n_done = sum(f is not None for f in finished)
        if n_done == B:
            break
    assert n_done > 0
    for f in finished:
        if f is not None:
            assert pda_oracle.json_loads_accepts(f), f
    # the live ones are prefixes of documents: their configurations are those the reference walk reaches
    for b in range(B):
        if finished[b] is None:
            wq, ws = pda_oracle.walk(delta, push, start, [], list(texts[b]), cap)
            assert wq == int(q[b]) and ws == stack[b, :int(depth[b])].cpu().tolist()


@pytest.mark.gpu
def test_json_exact_byte_level_route_parses(json_setup):
    """Per token: the root mask in the particle's configuration restricts the byte draw (sample_next_symbol with
    mask=bits); a drawn leaf ends the token, which pda_advance consumes.  Every finished text parses."""
    dec, trie, o = json_setup
    delta, push, start = json_tables()
    V, B, cap = len(dec), 32, 64
    rng = np.random.default_rng(8)
    w = rng.random((B, V)).astype(np.float32) + 0.05
    w[:, 256] = 50.0  # EOS dominates wherever it is allowed
    ws = torch.tensor(w).cuda()
    d, p = cuda(delta, push)
    q = torch.full((B,), start, dtype=torch.int32, device="cuda")
    stack = torch.zeros((B, cap), dtype=torch.int32, device="cuda")
    depth = torch.zeros(B, dtype=torch.int32, device="cuda")
    root = len(trie) - 1
    texts, finished = [b""] * B, [None] * B
    for step in range(40):
        bits = trie.pda_token_mask(d, p, q, stack, depth)
        assert oracle.unpack_bits(bits.cpu().numpy(), V)[[f is None for f in finished]].any(axis=1).all()
        node = torch.full((B,), root, dtype=torch.int32, device="cuda")
        tok = torch.full((B,), -1, dtype=torch.int32, device="cuda")
        for k in range(100):  # the longest item has 80 bytes
            child, label, _, _ = trie.sample_next_symbol(ws, node, mask=bits, seed=3, offset=(step * 100 + k) * B)
            c, lab = child.cpu().numpy(), label.cpu().numpy()
            pending = tok.cpu().numpy() < 0
            assert (c[pending] >= 0).all()
            leaf = pending & (lab < 0)
            tok[torch.tensor(leaf).cuda()] = torch.tensor(-1 - lab[leaf], dtype=torch.int32).cuda()
            node = torch.where(torch.tensor(pending & ~leaf).cuda(), child, node)
            if (tok >= 0).all():
                break
        assert (tok >= 0).all()
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
