"""Byte-level pushdown automata as tables over the trie's symbols, for nested constraints such as JSON.

A regular constraint is a DFA (``genlm_backend_b200.dfa``).  A format that nests -- JSON, bracketed code, arithmetic
expressions, S-expressions -- is not regular: a DFA can only unroll the nesting into states, and every state inside a
container then has to remember the kinds of all enclosing containers (on the order of ``2^d`` copies at depth ``d``
with two container kinds).  A deterministic pushdown automaton keeps those kinds on a stack instead.

Format: a deterministic PDA in return-state form, as a grammar compiles into a recursive transition network: a push
saves the state to return to, a pop goes there.  Two int32 tables of the same shape ``[Q, ld >= S]``
(``S = ParallelTokenCharacterTrie.num_symbols``: bytes 0..255, then the non-byte labels such as EOS):

- ``delta[q, s]`` in ``[0, Q)``: go to that state, first pushing ``push[q, s]`` when it is ``>= 0`` (a push value
  ``>= Q``, or a push onto a full stack, rejects);
- ``delta[q, s] == GT_PDA_POP`` (-2): pop the top of the stack and go to the popped state (an empty stack, or a popped
  value outside ``[0, Q)``, rejects);
- any other value rejects; ``push`` is read only for a move.

A particle's configuration is its state ``states[b]``, its depth ``depth[b]`` and its stack ``stack[b, :depth[b]]``
(bottom first): ``stack`` is an int32 CUDA ``[B, stack_ld]`` tensor, ``stack_ld <= GT_PDA_MAX_DEPTH`` (64) being every
particle's capacity, and ``depth`` an int32 CUDA ``[B]`` tensor.  A particle starts at ``(start, depth 0)``.  A table
with ``push`` all -1 and no ``GT_PDA_POP`` entry is a DFA, and the PDA calls then give what the DFA calls give.

Token-level step (mask, draw, advance; ``stack`` and ``depth`` are advanced in place)::

    bits = trie.pda_token_mask(delta, push, q, stack, depth)
    logZ, tok = smc.masked_logsumexp_sample(logps, bits, seed=seed, offset=step * B)
    q = trie.pda_advance(delta, push, q, stack, depth, tok)       # -1 for "no draw"; stack and depth kept then

Exact byte-level step: the mask, computed once per token at the root, restricts the byte read-outs; drawing byte by
byte from the root under it draws exactly from the masked token distribution::

    bits = trie.pda_token_mask(delta, push, q, stack, depth)      # once per token, at the root
    child, label, logp, logZ = trie.sample_next_symbol(ws, n, mask=bits, seed=s, offset=k)   # per byte
    # a drawn leaf child ends token -1 - label; then q = trie.pda_advance(delta, push, q, stack, depth, tok)

Resampling reindexes every per-particle tensor, the stacks included::

    anc, log_weights, ess, log_mean_w, resampled = smc.resample(log_weights.view(G, P), "systematic", 0.5)
    idx = anc.view(-1)
    q, stack, depth = q.index_select(0, idx), stack.index_select(0, idx), depth.index_select(0, idx)

Weighted automata: a float table ``logw`` of ``delta``'s shape, ``logw[q, s]`` the log-weight of the transition from
``q`` on ``s`` -- a plain move, a move with a push or a pop alike; the EOS column holds the final weights.  This carries a
probabilistic grammar compiled into return-state form (rule probabilities on the transitions that choose a rule), a
prior on the nesting depth (a weight on every push), or a preference per container kind (``json_pda`` copies scalar
states per context, so a weight can depend on where a value sits).  A pop's weight is read at ``(q, s)`` and does not
depend on the popped state: a weight that should depend on the state returned to belongs on the push that saved it.
``pda_token_logw`` gives each token the fp64 sum, rounded once to float32, of the log-weights along its symbols where
``pda_token_mask`` allows it, and ``-inf`` elsewhere; with ``logw`` all zero that is the ``{0, -inf}`` form of the
mask.  It is the sampler's additive mask, whose ``logZ = log sum_i p_i w_i`` is the particle's weight increment.  For a
prefix weight ``phi`` (a weighted grammar), the tables after weight pushing make the row ``log phi(x t) - log phi(x)``,
the exact token-level factor; computing the pushed tables is the caller's job.

Weighted token-level step (``pda_advance`` takes the same ``delta`` and ``push``)::

    tokw = trie.pda_token_logw(delta, push, logw, q, stack, depth)
    logZ, tok = smc.masked_logsumexp_sample(logps, tokw, seed=seed, offset=step * B)   # tok from p * w / Z
    q = trie.pda_advance(delta, push, q, stack, depth, tok)
    log_weights += logZ

Exact weighted byte-level step: one ``tokw`` per token, at the root, and the next-symbol draws from ``logps + tokw``
with ``log_input=True`` (a ``-inf`` is a zero weight, as under ``mask=``)::

    tokw = trie.pda_token_logw(delta, push, logw, q, stack, depth)  # once per token, at the root
    child, label, logp, logZ = trie.sample_next_symbol(logps + tokw, n, log_input=True, seed=s, offset=k)  # per byte
    # the root's logZ is masked_logsumexp_sample(logps, tokw)'s; a drawn leaf ends token -1 - label, then pda_advance

``json_pda`` builds the automaton of RFC 8259 JSON text.
"""
import numpy as np

from ._lib import GT_PDA_MAX_DEPTH, GT_PDA_POP

__all__ = ["GT_PDA_POP", "GT_PDA_MAX_DEPTH", "json_pda"]

_WS = b" \t\n\r"
_DIGITS = b"0123456789"
_HEX = b"0123456789abcdefABCDEF"


def _range(lo, hi):
    return bytes(range(lo, hi + 1))


def json_pda(num_symbols, eos=None):
    """``(delta, push, start)``: host int32 ``[Q, num_symbols]`` tables and the start state of a PDA that accepts RFC
    8259 JSON text over bytes.

    - One value of any kind at the top level, with whitespace ``[ \\t\\n\\r]`` around every token.
    - Numbers by the RFC grammar (``-?(0|[1-9][0-9]*)(.[0-9]+)?([eE][+-]?[0-9]+)?``); ``true``, ``false``, ``null``.
    - Strings with the escapes ``\\" \\\\ \\/ \\b \\f \\n \\r \\t`` and ``\\uXXXX``, no raw byte below 0x20, and
      well-formed UTF-8 only (Unicode Table 3-7: no overlong forms, no encoded surrogates, nothing above U+10FFFF).
    - ``eos`` (a non-byte symbol in ``[256, num_symbols)``, or None) is allowed exactly in the accepting states, where
      ``delta[q, eos] = q``; every other non-byte symbol rejects.

    Only containers push: ``[`` and ``{`` push the state that follows a value in the enclosing context (top level, in an
    array, in an object) and a closing ``]`` or ``}`` pops it.  The states of a scalar are copied per context, so a
    number's last digit already behaves as the state after the value: the ``]`` or ``}`` that ends a number is the
    single pop.  The nesting depth is bounded by the caller's ``stack_ld``; a push past it rejects.  Every
    configuration the automaton reaches can still be completed to a document, so a particle never meets a dead end."""
    S = int(num_symbols)
    if S < 256:
        raise ValueError(f"num_symbols must be at least 256 (the bytes), got {S}")
    if eos is not None and not 256 <= int(eos) < S:
        raise ValueError(f"eos must be a non-byte symbol in [256, {S}), got {eos}")
    ids = {}

    def st(name):
        return ids.setdefault(name, len(ids))

    top, top_end = st("top"), st("top_end")
    arr_first, arr_value, arr_after = st("arr_first"), st("arr_value"), st("arr_after")
    obj_first, obj_key, obj_colon, obj_value, obj_after = (st("obj_first"), st("obj_key"), st("obj_colon"),
                                                           st("obj_value"), st("obj_after"))
    after = {"top": top_end, "arr": arr_after, "obj": obj_after, "key": obj_colon}
    string = ("str", "esc", "u1", "u2", "u3", "u4", "c1", "c2", "c3", "e0", "ed", "f0", "f4")
    number = ("minus", "zero", "int", "dot", "frac", "exp_mark", "exp_sign", "exp")
    literal = {w: tuple(f"{w.decode()}{k}" for k in range(1, len(w))) for w in (b"true", b"false", b"null")}
    for c in after:
        for x in string:
            st(f"{c}:{x}")
    for c in ("top", "arr", "obj"):
        for x in number + sum(literal.values(), ()):
            st(f"{c}:{x}")
    Q = len(ids)
    delta = np.full((Q, S), -1, dtype=np.int32)
    push = np.full((Q, S), -1, dtype=np.int32)

    def move(q, symbols, nq, pu=-1):
        for s in symbols:
            delta[q, s] = nq
            push[q, s] = pu

    def value(q, c):
        """The transitions that start a value in context c from q."""
        move(q, b'"', ids[f"{c}:str"])
        move(q, b"-", ids[f"{c}:minus"])
        move(q, b"0", ids[f"{c}:zero"])
        move(q, _range(0x31, 0x39), ids[f"{c}:int"])
        for word, states in literal.items():
            move(q, word[:1], ids[f"{c}:{states[0]}"])
        move(q, b"[", arr_first, after[c])
        move(q, b"{", obj_first, after[c])

    for q in (top, top_end, arr_first, arr_value, arr_after, obj_first, obj_key, obj_colon, obj_value, obj_after):
        move(q, _WS, q)
    value(top, "top")
    value(arr_first, "arr")
    value(arr_value, "arr")
    value(obj_value, "obj")
    delta[arr_first, ord("]")] = GT_PDA_POP
    move(arr_after, b",", arr_value)
    delta[arr_after, ord("]")] = GT_PDA_POP
    move(obj_first, b'"', ids["key:str"])
    delta[obj_first, ord("}")] = GT_PDA_POP
    move(obj_key, b'"', ids["key:str"])
    move(obj_colon, b":", obj_value)
    move(obj_after, b",", obj_key)
    delta[obj_after, ord("}")] = GT_PDA_POP
    if eos is not None:
        delta[top_end, eos] = top_end

    for c, done in after.items():
        s = {x: ids[f"{c}:{x}"] for x in string}
        move(s["str"], bytes(b for b in range(0x20, 0x80) if b not in b'"\\'), s["str"])
        move(s["str"], b'"', done)
        move(s["str"], b"\\", s["esc"])
        move(s["esc"], b'"\\/bfnrt', s["str"])
        move(s["esc"], b"u", s["u1"])
        move(s["u1"], _HEX, s["u2"])
        move(s["u2"], _HEX, s["u3"])
        move(s["u3"], _HEX, s["u4"])
        move(s["u4"], _HEX, s["str"])
        # UTF-8 (Unicode Table 3-7): a lead byte, then 1-3 continuation bytes, the first one narrowed after E0, ED, F0, F4
        move(s["str"], _range(0xC2, 0xDF), s["c1"])
        move(s["str"], b"\xe0", s["e0"])
        move(s["str"], _range(0xE1, 0xEC) + b"\xee\xef", s["c2"])
        move(s["str"], b"\xed", s["ed"])
        move(s["str"], b"\xf0", s["f0"])
        move(s["str"], _range(0xF1, 0xF3), s["c3"])
        move(s["str"], b"\xf4", s["f4"])
        move(s["c1"], _range(0x80, 0xBF), s["str"])
        move(s["c2"], _range(0x80, 0xBF), s["c1"])
        move(s["c3"], _range(0x80, 0xBF), s["c2"])
        move(s["e0"], _range(0xA0, 0xBF), s["c1"])
        move(s["ed"], _range(0x80, 0x9F), s["c1"])
        move(s["f0"], _range(0x90, 0xBF), s["c2"])
        move(s["f4"], _range(0x80, 0x8F), s["c2"])

    for c in ("top", "arr", "obj"):
        done = after[c]
        n = {x: ids[f"{c}:{x}"] for x in number}
        # a number's end is where a byte cannot continue it: the final states behave as the state after the value
        for x in ("zero", "int", "frac", "exp"):
            delta[n[x]] = delta[done]
            push[n[x]] = push[done]
            if c == "top" and eos is not None:
                delta[n[x], eos] = n[x]
        move(n["minus"], b"0", n["zero"])
        move(n["minus"], _range(0x31, 0x39), n["int"])
        move(n["zero"], b".", n["dot"])
        move(n["int"], _DIGITS, n["int"])
        move(n["int"], b".", n["dot"])
        move(n["dot"], _DIGITS, n["frac"])
        move(n["frac"], _DIGITS, n["frac"])
        for x in ("zero", "int", "frac"):
            move(n[x], b"eE", n["exp_mark"])
        move(n["exp_mark"], b"+-", n["exp_sign"])
        move(n["exp_mark"], _DIGITS, n["exp"])
        move(n["exp_sign"], _DIGITS, n["exp"])
        move(n["exp"], _DIGITS, n["exp"])
        for word, states in literal.items():
            chain = [ids[f"{c}:{x}"] for x in states] + [done]
            for k in range(len(states)):
                move(chain[k], word[k + 1:k + 2], chain[k + 1])
    return delta, push, top
