"""Reference for the token masks under a byte-level pushdown automaton and the PDA advance: a numpy walk with an
explicit stack per item over each item's symbols (``symbol_oracle.item_symbols``), every row at the root.  Unlike the
kernels, which push onto an overlay and read the row's stack below a cursor, the walk copies the row's stack and
pushes and pops on the copy.

Also: ``random_pda``, and a vocabulary shaped after JSON text (``json_vocab``, with ``random_json`` documents).
"""
import json

import numpy as np

import symbol_oracle
from genlm_backend_b200 import Token
from genlm_backend_b200.pda import GT_PDA_POP
from helpers import EOS


def walk(delta, push, q, stack, syms, cap):
    """``(state, stack)`` after ``syms`` from state ``q`` with stack ``stack`` (bottom first), or ``(-1, None)`` on a
    reject; one symbol at a time, for a single byte string."""
    Q = delta.shape[0]
    if not (0 <= q < Q and 0 <= len(stack) <= cap):
        return -1, None
    stack = list(stack)
    for s in syms:
        nq = int(delta[q, s])
        if 0 <= nq < Q:
            pu = int(push[q, s])
            if pu >= 0:
                if pu >= Q or len(stack) >= cap:
                    return -1, None
                stack.append(pu)
            q = nq
        elif nq == GT_PDA_POP and stack and 0 <= stack[-1] < Q:
            q = stack.pop()
        else:
            return -1, None
    return q, stack


def accepts(delta, push, start, doc, eos, cap=64):
    """True iff ``doc`` (bytes) followed by ``eos`` walks from ``(start, [])`` without a reject to an empty stack."""
    q, stack = walk(delta, push, start, [], list(doc) + [eos], cap)
    return q >= 0 and stack == []


class PdaOracle:
    def __init__(self, decode):
        syms, self.S = symbol_oracle.item_symbols(decode)
        self.V = len(syms)
        self.lens = np.array([len(s) for s in syms], dtype=np.int64)
        self.sym = np.zeros((self.V, max(int(self.lens.max(initial=0)), 1)), dtype=np.int64)
        for i, s in enumerate(syms):
            self.sym[i, :len(s)] = s

    def _walk(self, delta, push, q, row_stack, cap, items):
        """Every item of ``items`` walked from ``(q, row_stack)``: ``(states, stacks [n, cap], depths)``, -1 once
        rejected.  The row must be valid."""
        Q = delta.shape[0]
        n = len(items)
        st = np.full(n, q, dtype=np.int64)
        stk = np.zeros((n, cap), dtype=np.int64)
        stk[:, :len(row_stack)] = row_stack
        d = np.full(n, len(row_stack), dtype=np.int64)
        lens, sym = self.lens[items], self.sym[items]
        for k in range(int(lens.max(initial=0))):
            a = np.flatnonzero((st >= 0) & (lens > k))
            if not a.size:
                break
            cur, s, da = st[a], sym[a, k], d[a]
            nq, pu = delta[cur, s], push[cur, s]
            new = np.full(a.size, -1, dtype=np.int64)
            move = (nq >= 0) & (nq < Q)
            plain = move & (pu < 0)
            new[plain] = nq[plain]
            pushes = move & (pu >= 0) & (pu < Q) & (da < cap)
            at = a[pushes]
            stk[at, da[pushes]] = pu[pushes]
            d[at] += 1
            new[pushes] = nq[pushes]
            pops = (nq == GT_PDA_POP) & (da > 0)
            at = a[pops]
            v = stk[at, da[pops] - 1]
            d[at] -= 1
            new[pops] = np.where((v >= 0) & (v < Q), v, -1)
            st[a] = new
        return st, stk, d

    @staticmethod
    def _rows(delta, push, states, stack, depth):
        delta = np.asarray(delta, dtype=np.int64)
        push = np.asarray(push, dtype=np.int64)
        stack = np.asarray(stack, dtype=np.int64)
        return delta, push, np.asarray(states, dtype=np.int64), stack, np.asarray(depth, dtype=np.int64), stack.shape[1]

    def mask(self, delta, push, states, stack, depth):
        """bool [B, V]."""
        delta, push, states, stack, depth, cap = self._rows(delta, push, states, stack, depth)
        out = np.zeros((len(states), self.V), dtype=bool)
        items = np.arange(self.V)
        for b, (q, dep) in enumerate(zip(states.tolist(), depth.tolist())):
            if 0 <= q < delta.shape[0] and 0 <= dep <= cap:
                out[b] = self._walk(delta, push, q, stack[b, :dep], cap, items)[0] >= 0
        return out

    def advance(self, delta, push, states, stack, depth, tokens):
        """``(states_out int64 [B], stack_out, depth_out)``: the state after the token or -1, and the rows' stacks and
        depths after it (unchanged where the state is -1; entries at or above a new depth are those of the input)."""
        delta, push, states, stack, depth, cap = self._rows(delta, push, states, stack, depth)
        out = np.full(len(states), -1, dtype=np.int64)
        stack_out, depth_out = stack.copy(), depth.copy()
        for b, (q, dep, t) in enumerate(zip(states.tolist(), depth.tolist(), np.asarray(tokens).tolist())):
            if 0 <= t < self.V and 0 <= q < delta.shape[0] and 0 <= dep <= cap:
                st, stk, d = self._walk(delta, push, q, stack[b, :dep], cap, np.array([t]))
                if st[0] >= 0:
                    out[b] = st[0]
                    stack_out[b, :d[0]] = stk[0, :d[0]]
                    depth_out[b] = d[0]
        return out, stack_out, depth_out


def random_pda(rng, Q, S, p_move=0.6, p_pop=0.15, p_push=0.25, p_bad=0.03):
    """``(delta, push)`` of Q states over S symbols.  Each delta entry is a pop with probability p_pop, else a uniform
    state with probability p_move, else a reject (-1, another negative value or a value >= Q).  Each push entry is a
    uniform state with probability p_push, a value >= Q with probability p_bad, else -1 or another negative value."""
    u = rng.random((Q, S))
    reject = rng.choice(np.array([-1, -3, Q, Q + 5, 1 << 30], dtype=np.int64), (Q, S))
    delta = np.where(u < p_pop, GT_PDA_POP, np.where(u < p_pop + p_move, rng.integers(0, Q, (Q, S)), reject))
    v = rng.random((Q, S))
    no_push = rng.choice(np.array([-1, -1, -7], dtype=np.int64), (Q, S))
    push = np.where(v < p_push, rng.integers(0, Q, (Q, S)), np.where(v < p_push + p_bad, Q + rng.integers(0, 3, (Q, S)), no_push))
    return delta.astype(np.int32), push.astype(np.int32)


# ---- JSON text -------------------------------------------------------------------------------------------------------
_CHARS = list("abcxyz ABC019_-/\\\"\t\n\x01\x1f\x7f") + ["é", "€", "\U0001f600", "中", "퟿", "",
                                                       "￿", "\U00010000", "\U0010ffff"]


def _random_value(rng, depth):
    k = int(rng.integers(0, 9 if depth < 6 else 6))
    if k == 0:
        return None
    if k == 1:
        return bool(rng.integers(0, 2))
    if k == 2:
        return int(rng.integers(-10**12, 10**12)) // int(10 ** rng.integers(0, 12))
    if k == 3:
        return float(rng.normal() * 10.0 ** int(rng.integers(-30, 30)))
    if k in (4, 5):
        return "".join(_CHARS[int(i)] for i in rng.integers(0, len(_CHARS), int(rng.integers(0, 8))))
    if k in (6, 7):
        return [_random_value(rng, depth + 1) for _ in range(int(rng.integers(0, 4)))]
    return {_random_value(rng, 9) if rng.random() < 0.9 else "": _random_value(rng, depth + 1)
            for _ in range(int(rng.integers(0, 4)))}


def random_json(rng):
    """One seeded JSON document as UTF-8 bytes: any top-level value, random separators and indentation, escaped or
    raw non-ASCII, and numbers with fractions and exponents."""
    v = _random_value(rng, 0)
    seps = [(",", ":"), (", ", ": "), (" ,\t", " :\r\n")][int(rng.integers(0, 3))]
    indent = [None, 0, 2, "\t"][int(rng.integers(0, 4))]
    text = json.dumps(v, ensure_ascii=bool(rng.integers(0, 2)), separators=seps, indent=indent)
    pad = [" ", "\n", "\r\n", "\t", ""]
    return (pad[int(rng.integers(0, 5))] + text + pad[int(rng.integers(0, 5))]).encode("utf-8")


def json_loads_accepts(doc):
    """Whether Python's JSON parser (the C scanner, NaN and Infinity refused) accepts ``doc`` decoded as strict UTF-8."""
    def refuse(name):
        raise ValueError(name)

    try:
        json.loads(doc.decode("utf-8"), parse_constant=refuse)
    except (UnicodeDecodeError, ValueError, RecursionError):
        return False
    return True


ADVERSARIAL = [b"[" * 70, b"[" * 40 + b"]" * 40, b"}}}}", b"12}", b'"]}', b"\\u00", b'"\\u00', b'{"a":[1,{"b":null}]}',
               b"[]", b"{}", b"]]", b"[[", b"1]", b"0.5e-3]", b"]," + b" " * 6, b"true}", b'","', b'":"',
               "é".encode()[:1], "é".encode()[1:], "€".encode()[:2], "€".encode()[1:],
               "\U0001f600".encode()[:3], "\U0001f600".encode()[1:], "\U0001f600".encode()[2:], b"\xed\xa0\x80",
               b"\xc0\xaf", b"\xf4\x90\x80\x80", b"\xe0\x80\x80"]


def json_vocab(n_docs=200, seed=0):
    """All 256 single bytes, an EOS sentinel (symbol 256), seeded chunks of 2-8 bytes cut from random JSON documents,
    and ``ADVERSARIAL`` items: ``Token`` items, EOS at index 256."""
    rng = np.random.default_rng(seed)
    items = [bytes([b]) for b in range(256)]
    chunks = []
    for _ in range(n_docs):
        doc = random_json(rng)
        at = 0
        while at < len(doc):
            n = int(rng.integers(2, 9))
            chunks.append(doc[at:at + n])
            at += n
    rest = list(dict.fromkeys(c for c in chunks + ADVERSARIAL if len(c) > 1))
    return [Token(i, b) for i, b in enumerate(items)] + [EOS()] + [Token(257 + i, b) for i, b in enumerate(rest)]
