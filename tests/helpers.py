"""Shared helpers for the test-suite."""
import os

import numpy as np

import oracle
from genlm_backend_b200 import Token
from genlm_backend_b200.synthetic import synth_vocab

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def unflat(blob, lens):
    """Inverse of make_golden.flat: list of byte strings."""
    out, at = [], 0
    data = blob.tobytes()
    for n in lens.tolist():
        out.append(data[at:at + n])
        at += n
    return out


def tokens(byte_strings):
    return [Token(i, b) for i, b in enumerate(byte_strings)]


def golden_vocab(name):
    """The vocabulary of golden file ``name``, or ``sentinel`` (a repeated item, the empty item, an EOS sentinel and
    plain bytes), or ``synth128256`` (the synthetic vocabulary of 128,256 tokens)."""
    if name == "sentinel":
        return [Token(0, b"ab"), Token(1, b""), Token(2, b"ab"), Token(3, b"a"), EOS(), b"plain"]
    if name == "synth128256":
        return synth_vocab(128256)
    g = load_golden(name)
    return tokens(unflat(g["blob"], g["lens"]))


def golden_layout(name):
    """The reference's layout of golden file ``name``, and the file."""
    g = load_golden(name)
    return oracle.OracleLayout(g["idx_to_leaf"], g["jump_ptr"], g["jump_idx"]), g


def trie_layout(trie):
    """``trie``'s own layout in the oracle's terms."""
    return oracle.OracleLayout(trie.idx_to_leaf, trie._layout["child_ptr"], trie._layout["child_idx"])


def depth1_node(trie):
    """The child of the root with the most children."""
    kids = trie.jump[trie.root]
    internal = [int(c) for c in kids if len(trie.jump[c])]
    return max(internal, key=lambda c: len(trie.jump[c]))


def assert_within_ulp(have, want):
    """fp32 results within one fp32 ulp of fp64 values; exact zeros and infinities kept."""
    have = np.asarray(have, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    fin = np.isfinite(want)
    assert np.array_equal(have[~fin], want[~fin], equal_nan=True)
    assert (have[want == 0] == 0).all()
    ulp = np.spacing(np.abs(want[fin]).astype(np.float32)).astype(np.float64)
    err = np.abs(have[fin] - want[fin])
    assert (err <= ulp).all(), float((err / np.maximum(ulp, 1e-300)).max())


def rel_err(have, want):
    """Max relative error where want != 0, and max |have| where want == 0 (must be exactly 0 for masses)."""
    have = np.asarray(have, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    nz = want != 0
    r = np.abs(have[nz] - want[nz]) / np.abs(want[nz]) if nz.any() else np.zeros(1)
    z = np.abs(have[~nz]) if (~nz).any() else np.zeros(1)
    return float(r.max()), float(z.max())


class EOS:
    """A non-byte vocabulary item: iterating it yields itself (the reference's EndOfSequence pattern)."""

    def __iter__(self):
        return iter([self])

    def __repr__(self):
        return "EOS"
