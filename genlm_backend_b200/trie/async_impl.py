"""``AsyncTokenCharacterTrie``: asyncio front end that batches concurrent mass queries.

Same contract as the reference's ``genlm/backend/trie/async_impl.py``: requests are queued as ``(weights, future, op)``;
a background task drains whatever is queued, groups by operation, issues ONE batched call per group and resolves the
futures; an exception fails every pending future of that drain and ends the task (the next request restarts it).

What differs from the reference (``async_impl.py:96-137`` runs the batched call on the event-loop thread, which blocks
every coroutine for the whole batch): the batched call runs on a worker thread, so the event loop keeps accepting
requests while a batch's kernels and copies are in flight -- the next drain picks up everything that arrived meanwhile.
One batch is in flight at a time (the GPU pipeline inside a batch already overlaps H2D, kernels and D2H).  Every future of
a ``weight_sum`` / ``weight_max`` request resolves to its own float32 numpy row backed by a page-locked block of at most
32 rows.  ``weight_sum_at`` / ``weight_max_at`` are the sparse read-out for SMC callers that need a few nodes per request:
the ``[B, N]`` slab never leaves the GPU.  ``child_masses`` is the read-out of a character-level sampler: the masses of
one node's children per request, computed from the leaves under that node only; ``symbol_masses`` gives the same
masses laid out by symbol, aligned with the per-symbol weights of a byte-level potential.
"""
import asyncio
import logging
from collections import defaultdict
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from .base import TokenCharacterTrie
from .parallel import ParallelTokenCharacterTrie

logger = logging.getLogger(__name__)


class AsyncTokenCharacterTrie:
    """An asynchronous wrapper for trie implementations that provides automatic request batching."""

    def __init__(self, trie):
        self.trie = trie
        self._queue = None
        self._task = None
        self._executor = None

    @classmethod
    def from_vocab(cls, vocab, backend="parallel", **kwargs):
        """Build the trie for ``vocab`` with the ``"sequential"`` or ``"parallel"`` implementation."""
        if backend == "sequential":
            trie = TokenCharacterTrie(decode=vocab, **kwargs)
        elif backend == "parallel":
            trie = ParallelTokenCharacterTrie(decode=vocab, **kwargs)
        else:
            raise ValueError(f"Unknown backend: {backend}. Must be one of ['sequential', 'parallel']")
        return cls(trie)

    async def _queue_request(self, request, op):
        if not self._task or self._task.done():
            self.start()
        future = asyncio.get_running_loop().create_future()
        await self._queue.put((request, future, op))
        return future

    async def weight_sum(self, ws):
        """Queue a ``weight_sum`` request; concurrent calls are batched together."""
        future = await self._queue_request(ws, "sum")
        return await future

    async def weight_max(self, ws):
        """Queue a ``weight_max`` request; concurrent calls are batched together."""
        future = await self._queue_request(ws, "max")
        return await future

    async def weight_sum_at(self, ws, node_ids, normalizer=None, log=False):
        """``weight_sum(ws)[node_ids]`` (optionally divided by the mass of node ``normalizer``, optionally as logs) as a
        float32 array of ``len(node_ids)`` values.  Batched like ``weight_sum``; only the requested nodes cross PCIe
        (``gt_gather_nodes``).  Requests that share ``len(node_ids)``, ``log`` and the use of a normaliser share a batch."""
        ids = np.asarray(node_ids, dtype=np.int32).reshape(-1)
        op = ("sum_at", len(ids), bool(log), normalizer is not None)
        future = await self._queue_request((ws, ids, normalizer), op)
        return await future

    async def weight_max_at(self, ws, node_ids, log=False):
        """``weight_max(ws)[node_ids]`` as a float32 array; see ``weight_sum_at``."""
        ids = np.asarray(node_ids, dtype=np.int32).reshape(-1)
        op = ("max_at", len(ids), bool(log), False)
        future = await self._queue_request((ws, ids, None), op)
        return await future

    async def child_masses(self, ws, node, normalize=False, log=False):
        """Masses of the children of ``node`` under the weights ``ws`` -> ``(child_ids int32[deg], masses float32[deg])``,
        in ``jump[node]`` order (``ParallelTokenCharacterTrie.batch_child_masses``: only the leaves under the node are
        read).  Concurrent requests with the same ``normalize`` / ``log`` share one batched call."""
        future = await self._queue_request((ws, int(node)), ("child", bool(normalize), bool(log)))
        return await future

    async def symbol_masses(self, ws, node, normalize=False, log=False, log_input=False):
        """Masses of the children of ``node`` by symbol -> float32 ``[S+1]`` (``ParallelTokenCharacterTrie.
        batch_symbol_masses``: column ``S`` is "the token ends here").  Concurrent requests with the same flags share
        one batched call."""
        future = await self._queue_request((ws, int(node)), ("symbol", bool(normalize), bool(log), bool(log_input)))
        return await future

    def start(self):
        """Start the background task (binds a fresh queue to the running loop)."""
        if not self._task or self._task.done():
            self._queue = asyncio.Queue()
            if self._executor is None:
                self._executor = ThreadPoolExecutor(max_workers=1, thread_name_prefix="trie-batch")
            self._task = asyncio.create_task(self._background_loop())

    def _do_weight_sums(self, batch_weights):
        if hasattr(self.trie, "batch_weight_rows"):
            return self.trie.batch_weight_rows(batch_weights, "sum")
        return self.trie.batch_weight_sum(batch_weights)

    def _do_weight_maxs(self, batch_weights):
        if hasattr(self.trie, "batch_weight_rows"):
            return self.trie.batch_weight_rows(batch_weights, "max")
        return self.trie.batch_weight_max(batch_weights)

    def _do_at(self, op, requests):
        kind, _, log, has_norm = op
        rows = self.trie._preprocess_ws([r[0] for r in requests])
        ids = np.stack([r[1] for r in requests])
        if kind == "sum_at":
            norm = np.asarray([int(r[2]) for r in requests], dtype=np.int32) if has_norm else None
            return self.trie.batch_weight_sum_at(rows, ids, normalizer=norm, log=log)
        return self.trie.batch_weight_max_at(rows, ids, log=log)

    def _do_child(self, op, requests):
        _, normalize, log = op
        rows = self.trie._preprocess_ws([r[0] for r in requests])
        nodes = np.asarray([r[1] for r in requests], dtype=np.int32)
        ids, masses, _ = self.trie.batch_child_masses(rows, nodes, normalize=normalize, log=log)
        degs = (ids >= 0).sum(axis=1)  # padding columns come last
        return [(ids[b, :d], masses[b, :d]) for b, d in enumerate(degs.tolist())]

    def _do_symbol(self, op, requests):
        _, normalize, log, log_input = op
        rows = self.trie._preprocess_ws([r[0] for r in requests])
        nodes = np.asarray([r[1] for r in requests], dtype=np.int32)
        sums, _ = self.trie.batch_symbol_masses(rows, nodes, normalize=normalize, log=log, log_input=log_input)
        return list(sums)

    def _run_group(self, op, requests):
        """One batched call (worker thread)."""
        if op == "sum":
            logger.debug(f"processing {len(requests)} sum requests")
            return self._do_weight_sums(requests)
        if op == "max":
            logger.debug(f"processing {len(requests)} max requests")
            return self._do_weight_maxs(requests)
        if isinstance(op, tuple) and op[0] in ("sum_at", "max_at") and hasattr(self.trie, "batch_weight_sum_at"):
            logger.debug(f"processing {len(requests)} {op[0]} requests")
            return self._do_at(op, requests)
        if isinstance(op, tuple) and op[0] == "child" and hasattr(self.trie, "batch_child_masses"):
            logger.debug(f"processing {len(requests)} child-mass requests")
            return self._do_child(op, requests)
        if isinstance(op, tuple) and op[0] == "symbol" and hasattr(self.trie, "batch_symbol_masses"):
            logger.debug(f"processing {len(requests)} symbol-mass requests")
            return self._do_symbol(op, requests)
        raise ValueError(f"Unknown operation: {op}")

    async def _background_loop(self):
        loop = asyncio.get_running_loop()
        while True:
            groups = defaultdict(list)
            try:
                request, future, op = await self._queue.get()
                groups[op].append((request, future))
                while not self._queue.empty():
                    request, future, op = self._queue.get_nowait()
                    groups[op].append((request, future))

                for op, group in groups.items():
                    requests, futures = zip(*group)
                    # off the event-loop thread: requests that arrive while this batch runs queue up for the next drain
                    results = await loop.run_in_executor(self._executor, self._run_group, op, requests)
                    for future, result in zip(futures, results):
                        if not future.done():
                            future.set_result(result)
            except asyncio.CancelledError:
                for group in groups.values():
                    for _, future in group:
                        if not future.done():
                            future.cancel()
                raise
            except Exception as e:
                for group in groups.values():
                    for _, future in group:
                        if not future.done():
                            future.set_exception(e)
                raise

    async def cleanup(self):
        """Cancel the background task and wait for it to finish."""
        if self._task and not self._task.done():
            self._task.cancel()
            try:
                await self._task
            except asyncio.CancelledError:
                pass
            self._task = None
        self._stop_executor()

    def _stop_executor(self):
        if self._executor is not None:
            self._executor.shutdown(wait=False)
            self._executor = None

    def shutdown(self):
        """Cancel the background task without awaiting it (safe when the loop is already closed)."""
        if self._task is not None:
            try:
                self._task.cancel()
            except RuntimeError:
                pass
            self._task = None
        self._stop_executor()

    def __del__(self):
        self.shutdown()
