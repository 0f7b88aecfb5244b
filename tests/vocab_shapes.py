"""Vocabularies shaped like real tokenizers' rather than like ``synth_vocab``, and the tile kernel's shared-memory need.

``synth_vocab`` has every single byte, items of at most 32 bytes, no repeated byte strings and first bytes spread
evenly.  Tokenizer vocabularies put a large share of their items under one prefix (GPT-2 has ~40 % under ``b" "``),
have whitespace and punctuation runs hundreds of bytes long, repeat byte strings under different ids, and (for
``str`` vocabularies) have thousands of symbols.  Each generator here is deterministic, returns ``Token`` items (or
``str`` items for ``wide_alphabet``) and stays under ~60k items so that the fp64 oracles stay fast.

``tile_smem_bytes`` is the Python twin of ``MassSmem`` (csrc/mass_kernels.cu), computed from the exported plan the
way ``plan_emulator.swizzle_slot`` restates ``swizzle_slot``.
"""
import numpy as np

from genlm_backend_b200 import Token
from genlm_backend_b200.synthetic import synth_vocab_bytes

SMEM_LIMIT = 227 * 1024  # dynamic shared memory one CTA of sm_100a may use
TILE_SIZES = (1024, 2048)  # what the planner accepts


def _tokens(byte_strings):
    return [Token(i, b) for i, b in enumerate(byte_strings)]


def _unique(byte_strings):
    return list(dict.fromkeys(byte_strings))


def space_heavy():
    """GPT-2-like: synthetic items, then as many again under ``b" "``, with three nested prefixes ``b" "``, ``b" t"``,
    ``b" th"`` each holding more than 8 tiles of 1,024 leaves (heavy spanning nodes of ``span_kernel``, several of them in
    one warp)."""
    base = synth_vocab_bytes(30000, seed=1)
    under = [b" th" + t for t in synth_vocab_bytes(9000, seed=2)]
    under += [b" t" + t for t in synth_vocab_bytes(3000, seed=3)[256:]]
    under += [b" " + t for t in synth_vocab_bytes(12000, seed=4)]
    return _tokens(_unique(base + under))


RUN_CHARS = b" -=\n\t#*"


def runs():
    """Synthetic items plus runs ``c * k``, k = 2 .. 256, of whitespace and punctuation: depth 256, and node tables near
    the shared-memory bound at T = 2048."""
    v = synth_vocab_bytes(20000, seed=3)
    for c in RUN_CHARS:
        v += [bytes([c]) * k for k in range(2, 257)]
    return _tokens(_unique(v))


def long_mixed():
    """``synth_vocab(50257)`` plus 2,000 items of 64-200 random printable bytes after a common prefix: its node table
    fits at T = 1024 and not at T = 2048."""
    rng = np.random.default_rng(4)
    v = synth_vocab_bytes(50257, seed=4)
    extra = [v[rng.integers(0, 5000)] + bytes(rng.integers(32, 127, size=int(n), dtype=np.uint8))
             for n in rng.integers(64, 200, size=2000)]
    return _tokens(_unique(v + extra))


def dups():
    """300 more ``b"a"``, 40 more ``b"ab"`` and 3 empty items on top of synthetic items: a node with more than 256
    children, most of them leaves, and several leaf children of the root."""
    return _tokens([b"a"] * 300 + [b"ab"] * 40 + synth_vocab_bytes(5000, seed=5) + [b""] * 3)


def no_single_bytes():
    """Synthetic items without the 256 single bytes: no leaf child of the root, and the first leaf in DFS order deep."""
    return _tokens(synth_vocab_bytes(20000, seed=6)[256:])


CJK = [chr(0x4E00 + i) for i in range(3000)]


def wide_alphabet():
    """``str`` items of 1-4 characters over 3,000 CJK code points: S = 3,256 symbols and a root with 2,999 children."""
    rng = np.random.default_rng(0)
    lens = rng.integers(1, 5, size=20000)
    chars = rng.integers(0, len(CJK), size=int(lens.sum())).tolist()
    ends = np.cumsum(lens).tolist()
    return list(dict.fromkeys("".join(CJK[c] for c in chars[e - n:e]) for n, e in zip(lens.tolist(), ends)))


def nested_chain(V):
    """``b"\\0" * k`` for k = 1 .. V: one chain, each node with one leaf child and one internal child."""
    return _tokens([b"\0" * k for k in range(1, V + 1)])


CHAIN_LENGTHS = (1, 2, 31, 32, 33, 511, 513)  # around a 32-bit mask word and a 512-rank block


def over_limit():
    """3,000 random items of 100-300 bytes: ~600k nodes in three tiles, a node table no tile size fits."""
    rng = np.random.default_rng(7)
    return _tokens(_unique(bytes(rng.integers(0, 256, size=int(n), dtype=np.uint8))
                           for n in rng.integers(100, 300, size=3000)))


FAMILIES = {
    "space_heavy": space_heavy, "runs": runs, "long_mixed": long_mixed, "dups": dups,
    "no_single_bytes": no_single_bytes, "wide_alphabet": wide_alphabet, "over_limit": over_limit,
}


def vocab(name):
    """The vocabulary of family ``name``; ``chain<V>`` is ``nested_chain(V)``."""
    if name.startswith("chain"):
        return nested_chain(int(name[5:]))
    return FAMILIES[name]()


def tile_smem_bytes(engine):
    """Dynamic shared memory one CTA of the tile kernel needs for ``engine``'s plan (``MassSmem(P, 16).total``: both
    pipelines use 16-byte value slots): two leaf blocks, two rest buffers and two metadata blocks, each section rounded
    up to 128 bytes, plus the barriers."""
    def up(x):
        return (int(x) + 127) & ~127

    info = engine.plan_info()
    T, SV = info["tile_leaves"], info["max_tile_values"]
    lo = engine.plan_array("tile_node_lo").astype(np.int64)
    # the emit stage is copied from the 16-byte aligned start at or below each tile's node interval
    nodes = int((((lo[1:] - (lo[:-1] & ~7)) + 7) & ~7).max(initial=0))
    rows = int(np.diff(engine.plan_array("ell_row_ptr")).max(initial=0))
    chunks = int(np.diff(engine.plan_array("ell_chunk_ptr")).max(initial=0))
    meta = up(rows * 64) + up((chunks + 2) * 8) + up(nodes * 2 + 16) + 128
    return 2 * up(T * 16) + 2 * up((SV - T) * 16) + 2 * meta + 128
