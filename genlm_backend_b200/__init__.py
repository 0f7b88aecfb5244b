"""genlm_backend_b200: the trie-mass / SMC-sampling hot path of genlm-backend, rebuilt for B200 (sm_100a).

Public names mirror the reference package for this path: ``Token``, ``TokenCharacterTrie``,
``ParallelTokenCharacterTrie``, ``AsyncTokenCharacterTrie``; ``smc`` holds the fused masked
logsumexp + categorical draw of the particle step; ``dfa`` the host helpers for byte-level DFA constraints;
``pda`` the pushdown-automaton format for nested constraints and a JSON automaton.
"""
from .tokenization import Token
from .trie import TokenCharacterTrie, ParallelTokenCharacterTrie, AsyncTokenCharacterTrie
from . import dfa, pda, smc

__all__ = ["Token", "TokenCharacterTrie", "ParallelTokenCharacterTrie", "AsyncTokenCharacterTrie", "dfa", "pda", "smc"]
