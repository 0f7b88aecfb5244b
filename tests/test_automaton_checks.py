"""Host argument checks of the seven automaton entry points that the per-call tests leave open: the full check order
of ``gt_dfa_token_mask``, and the exact row limit of every call (``65535 x GT_DFA_ROWS`` or ``65535 x GT_PDA_ROWS`` for
the masks and log-weights, ``INT32_MAX`` for the advances), on both sides.

The trie is this module's own and is never uploaded, so a call that gets past every argument check stops at the
resident-plan lookup (``GT_ERR_CUDA`` without a device, ``GT_ERR_STATE`` with one) and launches nothing: the data
pointers here are placeholders that are never dereferenced.
"""
import ctypes

import pytest

from genlm_backend_b200 import ParallelTokenCharacterTrie, _lib
from helpers import golden_vocab

GT_OK, GT_ERR_ARG, GT_ERR_CUDA, GT_ERR_STATE, GT_ERR_LIMIT = 0, 1, 2, 3, 4
DFA_ROWS, PDA_ROWS = 8, 4  # GT_DFA_ROWS, GT_PDA_ROWS: rows per CTA of the mask kernels, 65535 CTAs high at most
P = ctypes.c_void_p(1 << 20)  # stands for a device pointer

# entry point -> its parameters in C order (the stream follows), and the row limit
CALLS = {
    "gt_dfa_token_mask": ("t delta Q ld states nodes n bits ld_bits", 65535 * DFA_ROWS),
    "gt_dfa_token_logw": ("t delta logw Q ld states nodes n out ld_out", 65535 * DFA_ROWS),
    "gt_dfa_advance": ("t delta Q ld states nodes tokens n out", (1 << 31) - 1),
    "gt_pda_token_mask": ("t delta push Q ld states stack cap depth n bits ld_bits", 65535 * PDA_ROWS),
    "gt_pda_token_logw": ("t delta push logw Q ld states stack cap depth n out ld_out", 65535 * PDA_ROWS),
    "gt_pda_advance": ("t delta push Q ld states stack cap depth tokens n out", (1 << 31) - 1),
}


@pytest.fixture(scope="module")
def trie():
    return ParallelTokenCharacterTrie(golden_vocab("sentinel"))


def call(trie, fn, **kw):
    """``(return code, last error)`` of ``fn`` with valid arguments but for ``kw``."""
    eng = trie._engine
    assert not eng._uploaded  # a resident trie would take a call past every check to a launch
    a = dict(t=eng._handle, delta=P, logw=P, push=P, Q=4, ld=trie.num_symbols, states=P, nodes=P, stack=P, cap=8, depth=P,
             tokens=P, n=4, bits=P, ld_bits=(eng.V + 31) // 32, out=P, ld_out=eng.V)
    a.update(kw)
    rc = getattr(_lib.lib, fn)(*(a[k] for k in CALLS[fn][0].split()), None)
    return rc, lib_error() if rc else ""


def lib_error():
    return _lib.lib.gt_last_error().decode()


def test_dfa_mask_checks_run_in_order(trie):
    """Each case breaks one check and every later one; the earliest broken check decides the result."""
    W, S = (trie._engine.V + 31) // 32, trie.num_symbols
    over = 65535 * DFA_ROWS + 1
    cases = [  # (arguments, return code, message)
        (dict(t=None, delta=None, ld_bits=W - 1, Q=0, n=over), GT_ERR_ARG, "null trie"),
        (dict(delta=None, ld_bits=W - 1, Q=0, n=over), GT_ERR_ARG, "null data pointer"),
        (dict(bits=None, ld_bits=0, Q=0, n=over), GT_ERR_ARG, "null data pointer"),
        (dict(ld_bits=W - 1, Q=0, n=-1), GT_ERR_ARG, "mask_ld"),
        (dict(Q=0, n=over), GT_ERR_ARG, "bad n_states"),
        (dict(ld=S - 1, n=over), GT_ERR_ARG, "bad n_states"),
        (dict(Q=(1 << 31) // S + 1, n=over), GT_ERR_LIMIT, "reaches 2^31"),
        (dict(Q=(1 << 31) // S + 1, n=0), GT_ERR_LIMIT, "reaches 2^31"),
        (dict(n=0), GT_OK, ""),
        (dict(n=0, nodes=None), GT_OK, ""),
        (dict(n=over), GT_ERR_LIMIT, "too many rows"),
    ]
    for kw, rc, msg in cases:
        have_rc, have_msg = call(trie, "gt_dfa_token_mask", **kw)
        assert have_rc == rc and msg in have_msg, (kw, have_rc, have_msg)
        assert rc == GT_OK or have_msg.startswith("gt_dfa_token_mask: "), have_msg
    # past every argument check: the resident-plan lookup is next
    assert call(trie, "gt_dfa_token_mask", n=over - 1)[0] in (GT_ERR_CUDA, GT_ERR_STATE)


@pytest.mark.parametrize("fn", list(CALLS))
def test_row_limit_is_exact(trie, fn):
    limit = CALLS[fn][1]
    rc, msg = call(trie, fn, n=limit + 1)
    assert rc == GT_ERR_LIMIT and msg == f"{fn}: too many rows", (rc, msg)
    for nodes in ((P, None) if "nodes" in CALLS[fn][0] else (P,)):
        rc, msg = call(trie, fn, n=limit, nodes=nodes)
        assert rc in (GT_ERR_CUDA, GT_ERR_STATE), (rc, msg)  # not GT_ERR_LIMIT, and no launch
