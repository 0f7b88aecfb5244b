"""Byte-level DFAs as tables over the trie's symbols, for constrained sampling.

A DFA is an int32 table ``delta[Q, S]`` (``S = ParallelTokenCharacterTrie.num_symbols``: bytes 0..255, then the non-byte
labels such as EOS): ``delta[q, s]`` is the state after symbol ``s`` from state ``q``, or -1 to reject.  One table drives
both proposals of a constrained sampler:

- token level: ``trie.dfa_token_mask(delta, states)`` -> ``smc.masked_logsumexp_sample`` -> ``trie.dfa_advance``;
- byte level: ``symbol_logw(delta, states)`` -> ``trie.sample_next_symbol_weighted``; after a byte draw the next state is
  ``delta[states, symbol]``, a plain gather (a drawn end of token, symbol ``S``, keeps the state).  This looks one symbol
  ahead only: a byte can get weight 1 although most tokens below it are rejected later.
- exact byte level: the token mask, computed once per token at the root, restricts the byte read-outs; drawing byte by
  byte from the root under it draws exactly from the masked token distribution of ``smc.masked_logsumexp_sample``::

      bits = trie.dfa_token_mask(delta, q)                    # once per token, at the root
      child, label, logp, logZ = trie.sample_next_symbol(ws, n, mask=bits, seed=s, offset=k)   # per byte; logZ at the root = the token's weight increment
      # a drawn leaf child ends token -1 - label; then q = trie.dfa_advance(delta, q, tok)

  The mask stays valid for every byte of the token: the walk from the root equals the walk from ``n`` in the state
  reached at ``n``.

Soft constraints: a deterministic weighted byte automaton adds a float32 table ``logw[Q, S]`` of the same shape,
``logw[q, s]`` the log-weight of the transition from ``q`` on ``s`` (the EOS column holds the final weights).  A weighted
regex, a byte n-gram prior or a length or format penalty are all such tables.  A token's log-weight is the sum of the
transition log-weights along its remaining bytes, ``-inf`` where the Boolean mask rejects it:

- token level: ``tokw = trie.dfa_token_logw(delta, logw, q)`` -> ``logZ, tok = smc.masked_logsumexp_sample(logps, tokw)``
  -> ``q = trie.dfa_advance(delta, q, tok)``; ``logZ = log sum_i p_i w_i`` is the particle's weight increment and
  ``tok`` is drawn from ``p w / Z``;
- exact byte level: ``trie.sample_next_symbol(logps + tokw, n, log_input=True, seed=s, offset=k)`` per byte, with one
  ``tokw`` per token, computed at the root; the root's ``logZ`` is the token-level weight increment;
- one symbol ahead: ``symbol_logw(delta, q, logw=logw)`` -> ``trie.sample_next_symbol_weighted``.

Prefix weights: when the potential is a prefix weight ``phi`` given by a deterministic weighted automaton, the table
after standard weight pushing makes the log-weights along token ``t`` sum to ``log phi(x t) - log phi(x)``, the exact
token-level factor.  Computing the pushed table (a linear solve for cyclic automata) is left to the caller.

Several constraints in one call: stack their tables into one ``delta`` with disjoint state ranges (add each table's
offset to its non-negative entries; their ``logw`` tables stack the same way, unchanged) and give each row its own start
state.
"""
import numpy as np
import torch


def trim(delta, accepting):
    """Trimmed copy of ``delta`` (host numpy, int32): every transition into a state that cannot reach an accepting
    state becomes -1, as does every entry outside ``[0, Q)``.  State numbering is kept, so callers' state ids stay
    valid.  ``accepting``: state ids, or a bool mask of length ``Q``."""
    delta = np.array(delta, dtype=np.int64)
    if delta.ndim != 2:
        raise ValueError(f"delta must be a 2-D [states, symbols] table, got shape {delta.shape}")
    Q = delta.shape[0]
    acc = np.asarray(accepting)
    good = acc.astype(bool).copy() if acc.dtype == bool else np.zeros(Q, dtype=bool)
    if acc.dtype != bool:
        good[acc.astype(np.int64)] = True
    if good.shape != (Q,):
        raise ValueError(f"accepting must name states of a {Q}-state table")
    valid = (delta >= 0) & (delta < Q)
    src, _ = np.nonzero(valid)
    dst = delta[valid]
    order = np.argsort(dst, kind="stable")
    src, dst = src[order], dst[order]
    first = np.searchsorted(dst, np.arange(Q + 1))  # the sources of transitions into q: src[first[q]:first[q+1]]
    frontier = np.flatnonzero(good)
    while frontier.size:  # reverse BFS from the accepting states
        preds = np.concatenate([src[first[q]:first[q + 1]] for q in frontier.tolist()])
        preds = np.unique(preds[~good[preds]])
        good[preds] = True
        frontier = preds
    keep = valid & good[np.where(valid, delta, 0)]
    return np.where(keep, delta, -1).astype(np.int32)


def symbol_logw(delta, states, num_symbols=None, logw=None):
    """``float32[B, S+1]`` log-weights for ``sample_next_symbol_weighted``: column ``s < S`` is 0 (``logw[q, s]`` when
    a weighted table ``logw`` of ``delta``'s shape is given) where ``delta[q, s]`` is a live state and ``-inf``
    elsewhere; column ``S`` ("the token ends here") is 0 iff ``q`` itself is live.  A state outside ``[0, Q)`` gives an
    all ``-inf`` row.  ``S`` is ``num_symbols`` (default: the table's width).  The result is on the device of ``delta``
    when it is a tensor."""
    delta = torch.as_tensor(delta)
    states = torch.as_tensor(states, device=delta.device).reshape(-1).long()
    Q = delta.shape[0]
    S = delta.shape[1] if num_symbols is None else int(num_symbols)
    live = (states >= 0) & (states < Q)
    rows = states.clamp(0, Q - 1)
    nxt = delta[rows, :S]
    ok = live[:, None] & (nxt >= 0) & (nxt < Q)
    zero = torch.zeros((), dtype=torch.float32, device=delta.device)
    ninf = torch.full((), float("-inf"), dtype=torch.float32, device=delta.device)
    w = zero
    if logw is not None:
        logw = torch.as_tensor(logw)
        if not logw.is_floating_point() or logw.shape != delta.shape:
            raise ValueError(f"logw must be a float table of delta's shape {tuple(delta.shape)}, got {logw.dtype} "
                             f"{tuple(logw.shape)}")
        w = logw.to(device=delta.device, dtype=torch.float32)[rows, :S]
    return torch.cat([torch.where(ok, w, ninf), torch.where(live, zero, ninf)[:, None]], dim=1)
