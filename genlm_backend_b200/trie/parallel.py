"""``ParallelTokenCharacterTrie``: batched ``weight_sum`` / ``weight_max`` on the GPU.

Drop-in for the reference's ``genlm/backend/trie/parallel.py``.  The reference computes
``ws[:, positions] @ M`` with a sparse leaf x node reachability matrix (``parallel.py:92-103``) and a
``scatter_reduce_(amax)`` over every (leaf, ancestor) pair (``parallel.py:120-145``).  Here both are one
pass of the sm_100a kernels behind ``gt_weight_reduce``: rows are permuted into DFS leaf order through
shared memory, and every node is a short subtraction-free reduction over aligned leaf blocks.

Same signatures, same float32 numpy results in the reference's node order.  Additions (never changes
of defaults): ``*_tensor`` methods that keep results on the device, ``log_input=True`` to fuse the
``exp`` of log-probabilities, and ``devices=[...]`` to shard batch rows over several GPUs.
"""
import os
import threading

import numpy as np
import torch

from .base import TokenCharacterTrie
from ._engine import require_cuda
from ..sharding import row_blocks

# rows per pipelined slice of the host->device->host path
_PIPE_ROWS = 32
_PIPE_FIRST = 8
_PIPE_SLOTS = 3
# batches of at most this many rows take the single-stream latency path
_SMALL_BATCH = 8


# CPU rows are gathered into the pinned staging buffer by a few threads: one thread copies ~10 GB/s, which would make the
# host copy (0.5 MB per row at 128k tokens) the bottleneck of a 1,024-request batch (torch's copy releases the GIL)
_COPY_THREADS = int(os.environ.get("GT_COPY_THREADS", "4"))
_copy_pool = None


def _copy_block(stage, rows, a, b):
    for i in range(a, b):
        stage[i].copy_(rows[i])


def _gather_rows(rows, stage):
    """``stage[i] = rows[i]`` for a list of 1-D CPU tensors."""
    global _copy_pool
    n = len(rows)
    if n < 2 * _COPY_THREADS:
        _copy_block(stage, rows, 0, n)
        return
    if _copy_pool is None:
        from concurrent.futures import ThreadPoolExecutor

        _copy_pool = ThreadPoolExecutor(max_workers=_COPY_THREADS, thread_name_prefix="trie-stage")
    step = -(-n // _COPY_THREADS)
    futs = [_copy_pool.submit(_copy_block, stage, rows, a, min(n, a + step)) for a in range(0, n, step)]
    for f in futs:
        f.result()


def _pipe_slices(lo, hi):
    """Row slices of the host->device->host pipeline.  The first slice is short: nothing overlaps its H2D copy, and
    the D2H stream -- the PCIe-bound part, 2.7 MB per row and reduction at 128k tokens -- starts as soon as it is
    reduced; the following slices are ``_PIPE_ROWS`` rows."""
    out, r0 = [], lo
    while r0 < hi:
        r1 = min(hi, r0 + (_PIPE_FIRST if r0 == lo else _PIPE_ROWS))
        out.append((r0, r1))
        r0 = r1
    return out


class ParallelTokenCharacterTrie(TokenCharacterTrie):
    """A GPU version of ``TokenCharacterTrie`` that performs weight sum and max operations in parallel."""

    def __init__(self, decode, device=None, devices=None, **kwargs):
        """
        Args:
            decode (list): the token vocabulary.
            device (str|None): ``"cuda"``, ``"cpu"`` or ``None`` as in the reference (``parallel.py:8-13``).  It
                names where ``_preprocess_ws`` stages the rows; the reduction itself always runs on a GPU.
            devices (list[int]|None): CUDA device indices to shard batch rows over (default: the current one).
        """
        super().__init__(decode, **kwargs)
        self.device = device or ("cuda" if torch.cuda.is_available() else "cpu")
        if self.device not in ["cpu", "cuda"]:
            raise ValueError(f"Invalid device: {device}. Must be 'cpu', 'cuda' or None")
        self._devices = None if devices is None else [int(d) for d in devices]
        self._reach = None
        self._streams = {}
        self._stage = {}  # (device, pipeline slot) -> (pinned [rows, V] staging buffer, event of its last H2D copy)
        # the pipeline streams and staging buffers are per trie: one host-returning batch at a time (the async wrapper's
        # worker thread and a direct caller may both be at it)
        self._host_lock = threading.Lock()
        # position of each leaf's weight in the input rows (the identity: idx_to_leaf[:, 0])
        self.positions = torch.tensor(self.idx_to_leaf[:, 0], dtype=torch.long, device=self.device)

    # ---- reference attributes kept for compatibility (not used by the kernels) ----------------------------
    def _reachability(self):
        if self._reach is None:
            rows, cols = self._engine.reachability()
            self._reach = (torch.from_numpy(rows).to(self.device), torch.from_numpy(cols).to(self.device))
        return self._reach

    @property
    def src_indices(self):
        return self._reachability()[0]

    @property
    def dst_indices(self):
        return self._reachability()[1]

    @property
    def M(self):
        """Sparse CSR leaf x node reachability matrix of the reference (``parallel.py:33-64``)."""
        rows, cols = self._reachability()
        values = torch.ones(len(rows), device=self.device)
        return torch.sparse_coo_tensor(
            torch.stack([rows, cols]), values, (len(self.decode), len(self))
        ).to_sparse_csr()

    def _build_parent_map(self):
        parent = self._layout["parent"]
        return {child: int(p) for child, p in enumerate(parent.tolist()) if p >= 0}

    # ---- input handling ------------------------------------------------------------------------------------
    def _preprocess_ws(self, batch_ws):
        """Rows -> stacked float32 tensor on ``self.device`` (``parallel.py:66-75``)."""
        processed = []
        for ws in batch_ws:
            if not isinstance(ws, torch.Tensor):
                ws = torch.tensor(ws, device=self.device, dtype=torch.float32)
            elif ws.device.type != self.device or ws.dtype != torch.float32:
                ws = ws.to(device=self.device, dtype=torch.float32)
            assert ws.shape[0] == len(self.decode), [ws.shape[0], len(self.decode)]
            processed.append(ws)
        return torch.stack(processed)

    def _as_batch(self, ws):
        """Anything the reference accepts -> one ``[B, V]`` tensor, without touching dtype or device when the
        input already is a 2-D float tensor (so fp16 / bf16 rows are converted inside the kernel)."""
        if isinstance(ws, torch.Tensor) and ws.dim() == 2 and ws.dtype in (torch.float16, torch.bfloat16, torch.float32):
            assert ws.shape[1] == len(self.decode), [ws.shape[1], len(self.decode)]
            return ws
        return self._preprocess_ws(ws)

    def _device_list(self):
        require_cuda()
        return self._devices if self._devices else [torch.cuda.current_device()]

    # ---- device-resident API (additions) ---------------------------------------------------------------------
    def batch_weight_tensor(self, ws, ops=("sum",), log_input=False, out_sum=None, out_max=None, dfs_order=False):
        """Node masses for a ``[B, V]`` batch, kept on the GPU.  Returns ``(sum, max)`` float32 ``[B, N]`` tensors
        (``None`` for an op not requested).  Launches on the current stream of the input's device; no sync.

        ``dfs_order=True``: column ``r`` of ``ws`` holds the weight of token ``self.dfs_token_order[r]`` -- rows produced
        by an LM head whose output rows were permuted once with ``dfs_token_order`` -- which spares the kernels the
        scatter of every row into DFS leaf order (``GT_FLAG_DFS_ORDER``); the results are the same."""
        ws = self._as_batch(ws)
        if not ws.is_cuda:
            ws = ws.to(torch.device("cuda", self._device_list()[0]), non_blocking=True)
        return self._engine.reduce(ws, ops, out_dtype=torch.float32, log_input=log_input, out_sum=out_sum, out_max=out_max,
                                   dfs_order=dfs_order)

    @property
    def dfs_token_order(self):
        """``int64[V]``: position in ``decode`` of the token whose leaf has DFS rank ``r``.  ``ws[:, dfs_token_order]`` is
        the DFS-ordered form of a batch; applied once to the rows of an LM head's output projection it makes the model
        emit DFS-ordered rows for ``batch_weight_tensor(..., dfs_order=True)``."""
        return torch.from_numpy(self._layout["perm"].astype(np.int64))

    def batch_weight_sum_tensor(self, ws, log_input=False, out=None):
        return self.batch_weight_tensor(ws, ("sum",), log_input=log_input, out_sum=out)[0]

    def batch_weight_max_tensor(self, ws, log_input=False, out=None):
        return self.batch_weight_tensor(ws, ("max",), log_input=log_input, out_max=out)[1]

    def gather_nodes(self, mass, node_ids, normalizer=None, log=False):
        """Read a few nodes per row out of a device-resident ``[B, N]`` mass slab (a ``*_tensor`` result):
        ``out[b, k] = mass[b, node_ids[b, k]]``; with ``normalizer`` (a node id per row) the value is divided by
        that node's mass, with ``log=True`` logs are returned.  The result is a ``[B, K]`` device tensor, so only
        ``B * K`` values ever cross PCIe instead of the whole slab (``parallel.py:103,145``)."""
        return self._engine.gather_nodes(mass, node_ids, normalizer=normalizer, log=log)

    def batch_weight_sum_at(self, ws, node_ids, normalizer=None, log=False, log_input=False):
        """``batch_weight_sum(ws)[b, node_ids[b, k]]`` as a ``[B, K]`` float32 numpy array, without moving the
        ``[B, N]`` slab to the host."""
        sums = self.batch_weight_sum_tensor(ws, log_input=log_input)
        return self.gather_nodes(sums, node_ids, normalizer=normalizer, log=log).cpu().numpy()

    def batch_weight_sum_max_at(self, ws, node_ids, normalizer=None, log=False, log_input=False):
        """Both reductions from one staging pass, read out at ``node_ids``: ``(sums, maxes)`` as ``[B, K]`` float32
        numpy arrays (``normalizer`` applies to the sums only)."""
        ws = self._as_batch(ws)
        if not ws.is_cuda:
            ws = ws.to(torch.device("cuda", self._device_list()[0]), non_blocking=True)
        sums, maxes = self._engine.reduce(ws, ("sum", "max"), log_input=log_input)
        out_s = self.gather_nodes(sums, node_ids, normalizer=normalizer, log=log)
        out_m = self.gather_nodes(maxes, node_ids, log=log)
        return out_s.cpu().numpy(), out_m.cpu().numpy()

    def batch_weight_max_at(self, ws, node_ids, log=False, log_input=False):
        """``batch_weight_max(ws)[b, node_ids[b, k]]`` as a ``[B, K]`` float32 numpy array."""
        maxes = self.batch_weight_max_tensor(ws, log_input=log_input)
        return self.gather_nodes(maxes, node_ids, log=log).cpu().numpy()

    def subtree_token_mask(self, nodes, device=None):
        """Keep-bitmask of the tokens in the subtree of each node in ``nodes`` -- the tokens whose spelling extends
        that node's prefix, i.e. column ``nodes[b]`` of the reachability matrix ``M`` (``parallel.py:33-64``) -- as
        an ``int32[B, ceil(V/32)]`` device tensor in the bit-mask layout of ``smc.masked_logsumexp_sample``."""
        return self._engine.subtree_token_mask(nodes, device=device)

    # ---- token masks under a byte-level DFA (a constrained token-level SMC step) ------------------------------------
    def dfa_token_mask(self, delta, states, nodes=None):
        """Keep-bitmask ``int32[B, ceil(V/32)]`` of the tokens each particle may emit next without leaving its
        constraint's language, in the bit-mask layout of ``smc.masked_logsumexp_sample``.

        ``delta`` is a DFA over the trie's symbols (``num_symbols``): an int32 ``[Q, ld >= S]`` table, ``delta[q, s]``
        the next state or -1 to reject (see ``genlm_backend_b200.dfa``: ``trim`` it first).  ``states[b]`` is row
        ``b``'s state after the symbols of the path to ``nodes[b]`` (every row at the root when ``nodes`` is None); a
        token is allowed iff it lies under that node and the walk over its remaining symbols never rejects.  An invalid
        node or state gives an all-zero row.  Runs on the current stream of the inputs' device; no sync."""
        return self._engine.dfa_token_mask(delta, states, nodes)

    def dfa_token_logw(self, delta, logw, states, nodes=None):
        """``float32[B, V]``: the log-weight of each token under a weighted byte automaton, the additive mask of
        ``smc.masked_logsumexp_sample``.

        ``delta`` as in ``dfa_token_mask``; ``logw`` is a float table of ``delta``'s shape, ``logw[q, s]`` the
        log-weight of the transition from ``q`` on symbol ``s`` (converted to float32 on the device).  A token that
        ``dfa_token_mask`` allows gets the fp64 sum, rounded once to float32, of the log-weights along its remaining
        symbols (0 when none remain); every other token gets ``-inf``.  IEEE arithmetic decides special values (a
        ``-inf`` weight on the walk gives ``-inf``, a NaN gives NaN).  With ``logw`` all zero the result is the
        ``{0, -inf}`` form of ``dfa_token_mask``.  Runs on the current stream of the inputs' device; no sync."""
        return self._engine.dfa_token_logw(delta, logw, states, nodes)

    def dfa_advance(self, delta, states, tokens, nodes=None):
        """``int32[B]``: row ``b``'s DFA state after the remaining symbols of token ``tokens[b]`` (those past
        ``nodes[b]``'s depth), or -1 for a token that ``dfa_token_mask`` does not allow -- also the sampler's "no draw"
        (-1).  Keeps ``mask -> masked_logsumexp_sample -> advance`` on the device."""
        return self._engine.dfa_advance(delta, states, tokens, nodes)

    # ---- token masks under a byte-level pushdown automaton (nested constraints such as JSON) ------------------------
    def pda_token_mask(self, delta, push, states, stack, depth):
        """Keep-bitmask ``int32[B, ceil(V/32)]`` of the tokens each particle may emit next under a deterministic
        byte-level pushdown automaton, in the bit-mask layout of ``smc.masked_logsumexp_sample``.

        ``delta`` and ``push`` are int32 ``[Q, ld >= S]`` tables in the format of ``genlm_backend_b200.pda`` (a move,
        optionally pushing a return state; ``GT_PDA_POP`` = -2 to return to the popped state; anything else rejects).
        Row ``b`` stands at the root in state ``states[b]`` with the stack ``stack[b, :depth[b]]`` (bottom first);
        ``stack`` is an int32 CUDA ``[B, stack_ld]`` tensor with contiguous rows (``stack_ld <= 64`` is every row's
        capacity) and ``depth`` an int32 CUDA ``[B]`` tensor.  A token is allowed iff the walk over its symbols never
        rejects; an invalid state or depth gives an all-zero row.  Runs on the current stream of the inputs' device; no
        sync."""
        return self._engine.pda_token_mask(delta, push, states, stack, depth)

    def pda_token_logw(self, delta, push, logw, states, stack, depth):
        """``float32[B, V]``: the log-weight of each token under a weighted byte-level pushdown automaton, the additive
        mask of ``smc.masked_logsumexp_sample``.

        ``delta``, ``push``, ``states``, ``stack`` and ``depth`` as in ``pda_token_mask``; ``logw`` is a float table of
        ``delta``'s shape, ``logw[q, s]`` the log-weight of the transition from ``q`` on symbol ``s`` -- a move, a move
        with a push or a pop alike (converted to float32 on the device).  A pop's weight does not depend on the popped
        state: a weight that should belongs on the push that saved it.  A token that ``pda_token_mask`` allows gets the
        fp64 sum, rounded once to float32, of the log-weights along its symbols (0 for an empty token); every other
        token gets ``-inf``.  IEEE arithmetic decides special values (a ``-inf`` weight on the walk gives ``-inf``, a
        NaN gives NaN).  With ``logw`` all zero the result is the ``{0, -inf}`` form of ``pda_token_mask``.  Runs on the
        current stream of the inputs' device; no sync."""
        return self._engine.pda_token_logw(delta, push, logw, states, stack, depth)

    def pda_advance(self, delta, push, states, stack, depth, tokens):
        """``int32[B]``: row ``b``'s state after token ``tokens[b]``, or -1 for a token that ``pda_token_mask`` does not
        allow -- also the sampler's "no draw" (-1).  Where the result is not -1, ``stack`` and ``depth`` are advanced in
        place (entries at or above the new depth are unspecified); elsewhere the row's stack and depth are unchanged.
        ``stack`` and ``depth`` must be int32 CUDA tensors as in ``pda_token_mask``: anything else raises ``ValueError``,
        since a converted copy would lose the update.  The result may be written back into ``states``."""
        return self._engine.pda_advance(delta, push, states, stack, depth, tokens)

    # ---- child masses of one node per row (the next-symbol distribution of a character-level sampler) ------------
    @property
    def max_children(self):
        """``D``: the largest child count of any node, the width of the child read-outs."""
        return self._engine.max_children

    @property
    def edge_labels(self):
        """``int32[N]``: label of the edge into each node: a symbol ``>= 0``; ``-1 - i`` for the leaf of item ``i``
        ("token ``i`` ends here"); ``INT32_MIN`` for the root."""
        return self._layout["edge_label"]

    def _child_rows(self, ws):
        if isinstance(ws, torch.Tensor) and ws.dim() == 2 and ws.dtype in (torch.float16, torch.bfloat16, torch.float32, torch.float64):
            assert ws.shape[1] == len(self.decode), [ws.shape[1], len(self.decode)]
        else:
            ws = self._as_batch(ws)
        if not ws.is_cuda:
            ws = ws.to(torch.device("cuda", self._device_list()[0]), non_blocking=True)
        return ws

    def batch_child_masses_tensor(self, ws, nodes, ops=("sum",), log_input=False, dfs_order=False, normalize=False, log=False,
                                  mask=None):
        """Masses of the children of one node per row, computed from the rows alone (the ``[B, N]`` slab is never
        formed; only the leaves under ``nodes[b]`` are read).

        Returns ``(child_ids int32[B, D], sums float32[B, D] | None, maxes float32[B, D] | None)`` on the input's device,
        on its current stream, without a sync.  Column ``j`` is child ``jump[nodes[b]][j]``; columns past the node's
        degree are padding (id ``-1``, mass 0 -- ``-inf`` with ``log``); an invalid id or a leaf gives a padding row.
        Sums are accumulated in fp64 and rounded once; ``normalize`` divides them by the node's mass (the conditional
        next-symbol distribution); ``log`` returns logs of both.  Maxes equal ``batch_weight_max_tensor(ws)`` at the ids.
        ``dfs_order`` as for ``batch_weight_tensor``.

        ``mask``: restrict the rows to the tokens a keep-mask allows -- an int32 keep-bitmask ``[ceil(V/32)]`` (shared) or
        ``[B, ceil(V/32)]`` (what ``dfa_token_mask`` and ``subtree_token_mask`` return; any row stride of at least
        ``ceil(V/32)``), or a bool keep-mask ``[V]`` / ``[B, V]``, always in token order.  The results are bit for bit those
        for rows whose masked-out weights are 0 (``-inf`` with ``log_input``), computed without that ``[B, V]`` pass: a
        masked-out weight (NaN and inf included) never contributes, and a child without an allowed token has mass 0."""
        return self._engine.child_masses(self._child_rows(ws), nodes, ops=ops, log_input=log_input, dfs_order=dfs_order,
                                         normalize=normalize, log=log, mask=mask)

    def batch_child_masses(self, ws, nodes, ops=("sum",), log_input=False, dfs_order=False, normalize=False, log=False,
                           mask=None):
        """``batch_child_masses_tensor`` as numpy arrays."""
        out = self.batch_child_masses_tensor(ws, nodes, ops=ops, log_input=log_input, dfs_order=dfs_order,
                                             normalize=normalize, log=log, mask=mask)
        return tuple(None if t is None else t.cpu().numpy() for t in out)

    def _edge_labels_on(self, device):
        cache = self.__dict__.setdefault("_edge_label_dev", {})
        lab = cache.get(device.index)
        if lab is None:
            lab = cache[device.index] = torch.from_numpy(self.edge_labels).to(device)
        return lab

    def sample_next_symbol(self, ws, nodes, seed=0, offset=0, log_input=False, dfs_order=False, check_valid=False, mask=None):
        """One draw of the next symbol per row from the children of ``nodes[b]``, in proportion to their masses.

        Returns ``(child, label, logp, logZ)`` device tensors: the chosen child (int32), its ``edge_labels`` entry (a
        symbol, or ``-1 - i`` when the draw ends token ``i``), ``log mass(child) - log mass(node)`` and ``log mass(node)``.
        Row ``b`` uses the Philox counter ``offset + b`` under key ``seed`` (as ``smc.masked_logsumexp_sample``).  A row
        without mass (also a leaf or an invalid id) gives ``child = -1``, ``label = INT32_MIN`` and ``logZ = -inf``; a NaN
        weight under the node gives ``logZ = NaN``.  ``check_valid``: synchronise and raise ``RuntimeError`` like
        ``torch.multinomial`` when a row has no mass or a NaN.

        ``mask`` (as for ``batch_child_masses_tensor``): draw among the allowed tokens only.  With one token mask per
        particle, drawing symbol by symbol from the root until a leaf child draws exactly from the masked token
        distribution of ``smc.masked_logsumexp_sample``, and ``logZ`` at the root is that call's ``logZ``."""
        ws = self._child_rows(ws)
        child, logp, logZ = self._engine.child_sample(ws, nodes, seed=seed, offset=offset, log_input=log_input,
                                                      dfs_order=dfs_order, mask=mask)
        lab = self._edge_labels_on(child.device)
        label = torch.where(child >= 0, lab[child.clamp(min=0).long()], torch.full_like(child, np.iinfo(np.int32).min))
        if check_valid and child.numel():
            bad = child < 0
            if bool(bad.any()):
                if bool(torch.isnan(logZ[bad]).any()):
                    raise RuntimeError("probability tensor contains either `inf`, `nan` or element < 0")
                raise RuntimeError("invalid multinomial distribution (sum of probabilities <= 0)")
        return child, label, logp, logZ

    # ---- the same indexed by symbol, and a draw under per-row symbol weights (a byte-level potential) -------------
    @property
    def num_symbols(self):
        """``S``: symbols ``0 .. S-1`` are the edge labels (bytes first, then other labels); the symbol read-outs have
        ``S + 1`` columns, the last one (``end_symbol``) being "the token ends here"."""
        return self._engine.num_symbols

    @property
    def end_symbol(self):
        """Column of "the token ends here" (the node's leaf children) in the symbol read-outs: ``S``."""
        return self._engine.num_symbols

    @property
    def symbol_labels(self):
        """The ``S`` edge-label objects by symbol: byte ``s`` for ``s < 256``, then the other labels of the vocabulary
        in order of first appearance."""
        return list(self._edge_labels)

    def batch_symbol_masses_tensor(self, ws, nodes, ops=("sum",), log_input=False, dfs_order=False, normalize=False, log=False,
                                   mask=None):
        """``batch_child_masses_tensor`` laid out by symbol: ``(sums float32[B, S+1] | None, maxes float32[B, S+1] |
        None)`` on the input's device, on its current stream, without a sync.

        Column ``s < S`` is the child of ``nodes[b]`` whose edge symbol is ``s`` (0 -- ``-inf`` with ``log`` -- when
        there is none); column ``S`` adds up (sum) or maxes over all leaf children of the node, i.e. the items whose
        spelling ends there.  The values of the non-end columns are bit-equal to those of ``batch_child_masses_tensor``
        under the same flags; an invalid id or a leaf gives a padding row.  ``mask`` as for ``batch_child_masses_tensor``."""
        return self._engine.symbol_masses(self._child_rows(ws), nodes, ops=ops, log_input=log_input, dfs_order=dfs_order,
                                          normalize=normalize, log=log, mask=mask)

    def batch_symbol_masses(self, ws, nodes, ops=("sum",), log_input=False, dfs_order=False, normalize=False, log=False,
                            mask=None):
        """``batch_symbol_masses_tensor`` as numpy arrays."""
        out = self.batch_symbol_masses_tensor(ws, nodes, ops=ops, log_input=log_input, dfs_order=dfs_order,
                                              normalize=normalize, log=log, mask=mask)
        return tuple(None if t is None else t.cpu().numpy() for t in out)

    def sample_next_symbol_weighted(self, ws, nodes, symbol_logw, seed=0, offset=0, log_input=False, dfs_order=False,
                                    check_valid=False, mask=None):
        """One draw of the next symbol per row in proportion to ``mass(child) * exp(symbol_logw[b, symbol(child)])``.

        ``symbol_logw`` holds log-weights by symbol, ``[S+1]`` (shared by every row) or ``[B, S+1]``; its last column
        weighs "the token ends here".  Returns ``(child, symbol, logp, logZ, log_mass)`` device tensors: the chosen
        child (int32; among several items ending at the node, the one drawn), its symbol (``S`` for a leaf child),
        ``log q(child) - logZ``, ``logZ = log sum_j q_j`` (the particle's weight increment) and the node's
        log-mass.  Counters and key as in ``sample_next_symbol``; with all log-weights 0 the child, ``logp`` and
        ``logZ`` are those of ``sample_next_symbol``.  A row without a draw gives child and symbol ``-1`` and
        ``logZ = -inf`` (no weighted mass), NaN (a NaN weight or log-weight) or ``+inf``.  ``check_valid``:
        synchronise and raise ``RuntimeError`` like ``torch.multinomial`` for such rows.  ``mask`` as for
        ``sample_next_symbol``: the masses, and so ``log_mass``, count the allowed tokens only."""
        ws = self._child_rows(ws)
        child, symbol, logp, logZ, logM = self._engine.symbol_sample(ws, nodes, symbol_logw, seed=seed, offset=offset,
                                                                     log_input=log_input, dfs_order=dfs_order, mask=mask)
        if check_valid and child.numel():
            bad = child < 0
            if bool(bad.any()):
                z = logZ[bad]
                if bool((torch.isnan(z) | (z == float("inf"))).any()):
                    raise RuntimeError("probability tensor contains either `inf`, `nan` or element < 0")
                raise RuntimeError("invalid multinomial distribution (sum of probabilities <= 0)")
        return child, symbol, logp, logZ, logM

    # ---- reference API: numpy results on the host --------------------------------------------------------------
    def _pipe_streams(self, index):
        if index not in self._streams:
            with torch.cuda.device(index):
                self._streams[index] = [torch.cuda.Stream(device=index) for _ in range(_PIPE_SLOTS)]
        return self._streams[index]

    def _host_rows(self, ws):
        """A list / tuple of 1-D CPU float32 rows of the right length (what the async wrapper hands over for requests
        that arrive as host tensors), or ``None``.  Such a batch is staged slice by slice through pinned buffers
        instead of being stacked first: the host copy of a slice overlaps the device work of the slices before it."""
        if not isinstance(ws, (list, tuple)) or len(ws) < 2:
            return None
        V = len(self.decode)
        for r in ws:
            if not (isinstance(r, torch.Tensor) and r.device.type == "cpu" and r.dtype == torch.float32 and r.dim() == 1):
                return None
            assert r.shape[0] == V, [r.shape[0], V]
        return ws

    def _stage_buffer(self, index, slot, rows):
        key = (index, slot)
        buf, ev = self._stage.get(key, (None, None))
        if buf is None or buf.shape[0] < rows:
            buf = torch.empty((rows, len(self.decode)), dtype=torch.float32, pin_memory=True)
            ev = torch.cuda.Event()
            self._stage[key] = (buf, ev)
        else:
            ev.synchronize()  # the H2D copy that last read this buffer has finished
        return buf, ev

    def _small_to_host(self, ws, host_rows, ops, log_input, as_rows):
        """Latency path for a handful of rows: the caller's current stream only (no pipeline streams, no events), cached
        device scratch, one H2D copy, the three kernels, one pitched D2H copy per reduction, one stream synchronisation;
        the engine is called through its check-free entry points (everything was validated on the way here)."""
        index = self._device_list()[0]
        N = len(self)
        switch = torch.cuda.current_device() != index
        if switch:
            prev = torch.cuda.current_device()
            torch.cuda.set_device(index)
        try:
            st = torch.cuda.current_stream(index)
            if host_rows is not None:
                ws = torch.stack(host_rows)
            if not ws.is_cuda or ws.device.index != index:
                ws = ws.to(torch.device("cuda", index), non_blocking=True)
            if ws.stride(-1) != 1 or (ws.shape[0] > 1 and ws.stride(0) != ws.shape[1]):
                ws = ws.contiguous()
            B = ws.shape[0]
            opmask = (1 if "sum" in ops else 0) | (2 if "max" in ops else 0)
            sp = st.cuda_stream
            slabs = self._engine.reduce_raw(ws, opmask, log_input, index, sp)
            outs = {}
            for op, o in zip(("sum", "max"), slabs):
                if o is not None:
                    h = outs[op] = torch.empty((B, N), dtype=torch.float32, pin_memory=True)
                    self._engine.download_raw(o, h, sp)
            st.synchronize()
        finally:
            if switch:
                torch.cuda.set_device(prev)
        if as_rows:
            return {op: list(o.numpy()) for op, o in outs.items()}
        return {op: o.numpy() for op, o in outs.items()}

    def _batch_to_host(self, ws, ops, log_input=False, as_rows=False):
        """Run ``ops`` over the batch and return host arrays: C-contiguous float32 ``[B, N]`` like the reference's
        ``.cpu().numpy()`` (``parallel.py:103,145``), or with ``as_rows`` a list of ``B`` row arrays (what the async
        wrapper hands to its futures).  Rows are split contiguously over the configured GPUs; on each GPU slices of
        ``_PIPE_ROWS`` rows flow H2D -> kernels -> D2H on rotating streams so the copies overlap the kernels and each
        other.  Results land in page-locked host memory owned by the returned arrays (torch's caching host allocator
        recycles it when they are dropped): one ``[B, N]`` block, or with ``as_rows`` one block per slice, so that a row
        kept by a caller holds on to at most ``_PIPE_ROWS`` rows."""
        host_rows = self._host_rows(ws)
        if host_rows is None:
            ws = self._as_batch(ws)
        B, N = (len(host_rows) if host_rows is not None else ws.shape[0]), len(self)
        devices = self._device_list()
        if B == 0:
            return {op: ([] if as_rows else np.empty((0, N), dtype=np.float32)) for op in ops}
        if B <= _SMALL_BATCH:
            return self._small_to_host(ws, host_rows, ops, log_input, as_rows)
        with self._host_lock:
            return self._pipelined_to_host(ws, host_rows, ops, log_input, as_rows, B, N, devices)

    def _pipelined_to_host(self, ws, host_rows, ops, log_input, as_rows, B, N, devices):
        whole = None if as_rows else {op: torch.empty((B, N), dtype=torch.float32, pin_memory=True) for op in ops}
        row_lists = {op: [None] * B for op in ops} if as_rows else None
        used = []
        keep = []
        for index, (lo, hi) in zip(devices, row_blocks(B, len(devices))):
            if lo >= hi:
                continue
            dev = torch.device("cuda", index)
            streams = self._pipe_streams(index)
            start = torch.cuda.Event()
            start.record(torch.cuda.current_stream(ws.device.index if host_rows is None and ws.is_cuda else index))
            for k, (r0, r1) in enumerate(_pipe_slices(lo, hi)):
                st = streams[k % _PIPE_SLOTS]
                st.wait_event(start)  # inputs produced on the caller's stream are ready
                with torch.cuda.device(index), torch.cuda.stream(st):
                    if host_rows is not None:
                        stage, staged = self._stage_buffer(index, k % _PIPE_SLOTS, _PIPE_ROWS)
                        _gather_rows(host_rows[r0:r1], stage)
                        chunk = stage[: r1 - r0].to(dev, non_blocking=True)
                        staged.record(st)
                    else:
                        chunk = ws[r0:r1]
                        if chunk.device != dev:
                            chunk = chunk.to(dev, non_blocking=True)
                    o_sum, o_max = self._engine.reduce(chunk, ops, log_input=log_input)
                    for op, o in (("sum", o_sum), ("max", o_max)):
                        if o is None:
                            continue
                        if as_rows:
                            slab = torch.empty((r1 - r0, N), dtype=torch.float32, pin_memory=True)
                            row_lists[op][r0:r1] = list(slab.numpy())
                        else:
                            slab = whole[op][r0:r1]
                        self._engine.download(o, slab, st)
                        keep.append(slab)
                    keep.append((chunk, o_sum, o_max))
            used.extend(streams)
        for st in used:
            st.synchronize()
        del keep
        if as_rows:
            return row_lists
        return {op: o.numpy() for op, o in whole.items()}

    def _single(self, ws, op):
        """One weight vector (anything ``_preprocess_ws`` takes) through the small-batch latency path: a ``[1, V]`` view
        instead of a stacked copy, no staging on ``self.device`` first."""
        if not isinstance(ws, torch.Tensor):
            ws = torch.tensor(ws, dtype=torch.float32)
        assert ws.dim() == 1 and ws.shape[0] == len(self.decode), [ws.shape[0], len(self.decode)]
        if ws.dtype not in (torch.float32, torch.float16, torch.bfloat16):
            ws = ws.to(torch.float32)
        return self._batch_to_host(ws.reshape(1, -1), (op,))[op][0]

    def weight_sum(self, ws):
        """Node sums for one weight vector -> ``float32[num_nodes]`` (``parallel.py:77-90``)."""
        return self._single(ws, "sum")

    def batch_weight_sum(self, ws):
        """Node sums for a batch -> ``float32[batch, num_nodes]`` numpy array (``parallel.py:92-103``)."""
        return self._batch_to_host(ws, ("sum",))["sum"]

    def weight_max(self, ws):
        """Node maxima for one weight vector -> ``float32[num_nodes]`` (``parallel.py:105-118``)."""
        return self._single(ws, "max")

    def batch_weight_max(self, ws):
        """Node maxima for a batch -> ``float32[batch, num_nodes]`` numpy array (``parallel.py:120-145``)."""
        return self._batch_to_host(ws, ("max",))["max"]

    def batch_weight_rows(self, ws, op):
        """``batch_weight_sum`` / ``batch_weight_max`` (``op`` = ``"sum"`` / ``"max"``) as a list of per-row float32
        arrays: the form ``AsyncTokenCharacterTrie`` hands to its futures.  The rows live in page-locked blocks of at most
        ``_PIPE_ROWS`` rows, so a caller that keeps one row does not keep the whole batch's results alive."""
        return self._batch_to_host(ws, (op,), as_rows=True)[op]

    def batch_weight_sum_max(self, ws, log_input=False):
        """Both reductions from one staging pass -> ``(sums, maxes)`` numpy arrays."""
        out = self._batch_to_host(ws, ("sum", "max"), log_input=log_input)
        return out["sum"], out["max"]
