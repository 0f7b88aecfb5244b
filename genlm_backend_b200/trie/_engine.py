"""Device-side driver shared by the trie classes: owns the C handle, keeps the plan metadata resident
per GPU, caches scratch buffers, and launches ``gt_weight_reduce`` on torch's current stream.

PyTorch is used for device memory, streams and host<->device copies only; every reduction runs in the
hand-written kernels behind the C ABI (``csrc/mass_kernels.cu``).  There is no CPU path.
"""
import ctypes
import os

import numpy as np
import torch

from .. import _lib
from .._lib import lib, check

_IN_TYPES = {
    torch.float32: _lib.GT_F32,
    torch.float64: _lib.GT_F64,
    torch.float16: _lib.GT_F16,
    torch.bfloat16: _lib.GT_BF16,
}
_OUT_TYPES = {torch.float32: _lib.GT_F32, torch.float64: _lib.GT_F64}
OPS = {"sum": _lib.GT_OP_SUM, "max": _lib.GT_OP_MAX}

# rows the per-stream scratch is sized for: gt_workspace_bytes caps the staging part at one 64-row chunk (34 MB at 128k
# tokens: it stays in L2 between the permute and the tile kernel) and keeps spanning-node pieces for up to 1,024 rows, so
# that one span kernel serves a whole large batch
_WORKSPACE_ROWS = int(os.environ.get("GT_WORKSPACE_ROWS", "1024"))
_MAX_WORKSPACES = 16  # per engine: (device, stream) pairs we keep scratch for


def _opmask(ops):
    mask = 0
    for op in ops:
        mask |= OPS[op]
    return mask


def _flags(log_input=False, dfs_order=False, normalize=False, log=False):
    return ((_lib.GT_FLAG_LOG_INPUT if log_input else 0) | (_lib.GT_FLAG_DFS_ORDER if dfs_order else 0)
            | (_lib.GT_CHILD_NORMALIZE if normalize else 0) | (_lib.GT_CHILD_LOG if log else 0))


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError(
            "genlm_backend_b200 computes trie masses with CUDA kernels only (sm_100a); "
            "no CUDA device is available and there is no CPU fallback"
        )


class TrieEngine:
    """Owns a ``gt_trie*`` and everything resident on the GPUs for it."""

    def __init__(self, symbols, offsets, n_tokens):
        symbols = np.ascontiguousarray(symbols, dtype=np.int32)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        handle = ctypes.c_void_p()
        check(lib.gt_build(symbols.ctypes.data, offsets.ctypes.data, int(n_tokens), ctypes.byref(handle)), "gt_build")
        self._handle = handle
        self.V = int(lib.gt_num_tokens(handle))
        self.N = int(lib.gt_num_nodes(handle))
        self.nnz = int(lib.gt_num_reach(handle))
        self._uploaded = set()
        self._workspaces = {}
        self._child_workspaces = {}
        self._ld32 = None
        self.max_children = int(lib.gt_max_children(handle))  # D: columns of the child read-outs
        self.num_symbols = int(lib.gt_num_symbols(handle))  # S: the symbol read-outs have S + 1 columns

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h:
            try:
                lib.gt_free(h)
            except Exception:
                pass
            self._handle = None

    # ---- host layout ---------------------------------------------------------------------------------
    def layout(self):
        V, N = self.V, self.N
        out = {
            "leaf_node": np.empty(V, np.int32), "parent": np.empty(N, np.int32), "edge_label": np.empty(N, np.int32),
            "child_ptr": np.empty(N + 1, np.int32), "child_idx": np.empty(max(N - 1, 0), np.int32),
            "perm": np.empty(V, np.int32), "lo": np.empty(N, np.int32), "hi": np.empty(N, np.int32),
        }
        check(lib.gt_export_layout(self._handle, *[a.ctypes.data for a in out.values()]), "gt_export_layout")
        return out

    def reachability(self):
        rows = np.empty(self.nnz, np.int64)
        cols = np.empty(self.nnz, np.int64)
        check(lib.gt_export_reachability(self._handle, rows.ctypes.data, cols.ctypes.data), "gt_export_reachability")
        return rows, cols

    def plan(self, tile_leaves=0):
        check(lib.gt_plan(self._handle, tile_leaves), "gt_plan")

    def plan_info(self):
        self.plan()
        info = _lib.PlanInfo()
        check(lib.gt_get_plan_info(self._handle, ctypes.byref(info)), "gt_get_plan_info")
        return {name: getattr(info, name) for name, _ in info._fields_}

    def plan_array(self, name):
        self.plan()
        es = ctypes.c_int32()
        n = lib.gt_export_plan_array(self._handle, name.encode(), None, 0, ctypes.byref(es))
        if n < 0:
            check(1, "gt_export_plan_array")
        arr = np.empty(n, np.uint16 if es.value == 2 else np.int32)
        lib.gt_export_plan_array(self._handle, name.encode(), arr.ctypes.data, n, ctypes.byref(es))
        return arr

    # ---- device ----------------------------------------------------------------------------------------
    def ensure_device(self, index):
        if index not in self._uploaded:
            check(lib.gt_upload(self._handle, int(index)), "gt_upload")
            self._uploaded.add(index)

    def _workspace(self, index, stream, rows):
        """Scratch for launches on ``stream`` (a raw ``cudaStream_t``) of device ``index``.  One buffer per
        (device, stream): calls on one stream are ordered, so they may share it; calls on different streams (or
        threads using different streams) never do."""
        need = int(lib.gt_workspace_bytes(self._handle, min(max(rows, 1), _WORKSPACE_ROWS)))
        return self._scratch(self._workspaces, need, index, stream)

    def _child_workspace(self, index, stream, rows):
        """Scratch of ``gt_child_masses`` / ``gt_child_sample``, cached per (device, stream) like ``_workspace``."""
        need = int(lib.gt_child_workspace_bytes(self._handle, min(max(rows, 1), _WORKSPACE_ROWS)))
        return self._scratch(self._child_workspaces, need, index, stream)

    def _launch(self, fn, index, *args, workspace=None, rows=0):
        """``lib.<fn>(*args, [scratch, scratch bytes,] stream)`` on the current stream of device ``index``, checked.
        ``workspace`` (``_workspace`` or ``_child_workspace``) gives the call its scratch for ``rows`` rows."""
        with torch.cuda.device(index):
            stream = torch.cuda.current_stream(index).cuda_stream
            if workspace is not None:
                work = workspace(index, stream, rows)
                args += (work.data_ptr(), work.numel())
            check(getattr(lib, fn)(*args, stream), fn)

    @staticmethod
    def _scratch(cache, need, index, stream):
        key = (index, int(stream or 0))
        buf = cache.get(key)
        if buf is None or buf.numel() < need:
            if buf is None and len(cache) >= _MAX_WORKSPACES:
                cache.pop(next(iter(cache)))  # the caching allocator keeps the block stream-ordered
            # allocated on `stream` (the caller made it current), so a later reuse of the block is ordered after our kernels
            buf = torch.empty(max(need, 4096), dtype=torch.uint8, device=torch.device("cuda", index))
            cache[key] = buf
        return buf

    def row_stride(self, dtype=torch.float32):
        """Row stride (elements) of the output slabs the engine allocates: N rounded up to a whole number of
        128-byte lines, so every row starts line-aligned and the emit stores of all rows of a row group are
        line-aligned together."""
        per_line = 128 // torch.empty((), dtype=dtype).element_size()
        return (self.N + per_line - 1) // per_line * per_line

    def alloc_out(self, B, dtype, device):
        """``[B, N]`` view of a ``[B, row_stride]`` device slab (rows are padded to 128-byte lines)."""
        ld = self.row_stride(dtype)
        return torch.empty((max(B, 1), ld), dtype=dtype, device=device)[:B, : self.N]

    def reduce(self, ws, ops, out_dtype=torch.float32, log_input=False, out_sum=None, out_max=None, phases=0, dfs_order=False):
        """Launch the mass kernels for a ``[B, V]`` CUDA tensor on its device's current stream.

        Returns ``(out_sum, out_max)`` device tensors of shape ``[B, N]`` (``None`` for an op not asked for).
        Nothing is synchronised here.  ``dfs_order``: column ``r`` of ``ws`` is the weight of item ``perm[r]`` (the rows
        are already in DFS leaf order, ``GT_FLAG_DFS_ORDER``).
        """
        require_cuda()
        if not (isinstance(ws, torch.Tensor) and ws.is_cuda and ws.dim() == 2):
            raise ValueError("reduce expects a 2-D CUDA tensor")
        if ws.shape[1] != self.V:
            raise AssertionError([ws.shape[1], self.V])
        if ws.dtype not in _IN_TYPES:
            ws = ws.to(torch.float32)
        if ws.shape[1] > 1 and ws.stride(1) != 1:
            ws = ws.contiguous()
        B = ws.shape[0]
        index = ws.device.index
        self.ensure_device(index)
        opmask = _opmask(ops)

        def _out(t):
            if t is None:
                return self.alloc_out(B, out_dtype, ws.device)
            if not (t.is_cuda and t.device == ws.device and t.dtype == out_dtype and t.shape == (B, self.N) and (t.stride(1) == 1 or self.N <= 1)):
                raise ValueError("out tensor must be a [B, N] tensor of the output dtype on the input's device")
            return t

        out_sum = _out(out_sum) if opmask & _lib.GT_OP_SUM else None
        out_max = _out(out_max) if opmask & _lib.GT_OP_MAX else None
        if B == 0:
            return out_sum, out_max
        ld_out = (out_sum if out_sum is not None else out_max).stride(0) if B > 1 else self.N
        if out_sum is not None and out_max is not None and B > 1 and out_sum.stride(0) != out_max.stride(0):
            raise ValueError("out_sum and out_max must share a row stride")
        ld_ws = ws.stride(0) if B > 1 else max(self.V, 1)
        self._launch(
            "gt_weight_reduce", index, self._handle, ws.data_ptr(), _IN_TYPES[ws.dtype], B, ld_ws,
            out_sum.data_ptr() if out_sum is not None else None, out_max.data_ptr() if out_max is not None else None,
            _OUT_TYPES[out_dtype], ld_out, opmask, _flags(log_input, dfs_order) | int(phases),
            workspace=self._workspace, rows=B,
        )
        return out_sum, out_max

    def reduce_raw(self, ws, opmask, log_input, index, stream_ptr):
        """``reduce`` without the checks, for the few-row latency path: ``ws`` is a contiguous float32 / fp16 / bf16
        ``[B, V]`` tensor on device ``index``, which is the current device; launches on the raw stream ``stream_ptr``.
        Returns the padded ``[B, row_stride]`` float32 slabs ``(sum, max)`` (``None`` for an op not in ``opmask``)."""
        B = ws.shape[0]
        if index not in self._uploaded:
            self.ensure_device(index)
        ld = self._ld32
        if ld is None:
            ld = self._ld32 = self.row_stride(torch.float32)
        out_sum = torch.empty((B, ld), dtype=torch.float32, device=ws.device) if opmask & 1 else None
        out_max = torch.empty((B, ld), dtype=torch.float32, device=ws.device) if opmask & 2 else None
        work = self._workspace(index, stream_ptr, B)
        rc = lib.gt_weight_reduce(
            self._handle, ws.data_ptr(), _IN_TYPES[ws.dtype], B, self.V,
            out_sum.data_ptr() if out_sum is not None else None, out_max.data_ptr() if out_max is not None else None,
            _lib.GT_F32, ld, opmask, _lib.GT_FLAG_LOG_INPUT if log_input else 0, work.data_ptr(), work.numel(), stream_ptr)
        if rc:
            check(rc, "gt_weight_reduce")
        return out_sum, out_max

    def download_raw(self, slab, host_out, stream_ptr):
        """Pitched D2H copy of a padded float32 slab from ``reduce_raw`` into a C-contiguous ``[B, N]`` pinned tensor."""
        rc = lib.gt_download_rows(host_out.data_ptr(), self.N * 4, slab.data_ptr(), slab.stride(0) * 4, self.N * 4, slab.shape[0], stream_ptr)
        if rc:
            check(rc, "gt_download_rows")

    def download(self, dev_out, host_out, stream):
        """Pitched D2H copy (``gt_download_rows``) of a ``[rows, N]`` device result (row stride = the slab's padded
        stride) into a C-contiguous ``[rows, N]`` page-locked host tensor, on ``stream``.  The caller keeps both alive
        until it has synchronised the stream."""
        rows = dev_out.shape[0]
        if rows == 0 or self.N == 0:
            return
        es = dev_out.element_size()
        check(
            lib.gt_download_rows(host_out.data_ptr(), host_out.stride(0) * es if rows > 1 else self.N * es, dev_out.data_ptr(),
                                 dev_out.stride(0) * es if rows > 1 else self.N * es, self.N * es, rows, stream.cuda_stream),
            "gt_download_rows",
        )

    # ---- read-outs that keep the [B, N] slab on the GPU --------------------------------------------------------
    def gather_nodes(self, mass, node_ids, normalizer=None, log=False):
        """``out[b, k] = mass[b, node_ids[b, k]]`` (``node_ids`` 1-D: shared by all rows), optionally divided by
        ``mass[b, normalizer[b]]`` and / or returned as logs.  Everything stays on ``mass``'s device."""
        require_cuda()
        if not (isinstance(mass, torch.Tensor) and mass.is_cuda and mass.dim() == 2 and mass.dtype in _OUT_TYPES):
            raise ValueError("mass must be a 2-D float32 / float64 CUDA tensor")
        if mass.shape[1] != self.N:
            raise AssertionError([mass.shape[1], self.N])
        if mass.shape[1] > 1 and mass.stride(1) != 1:
            mass = mass.contiguous()
        B, dev = mass.shape[0], mass.device
        ids = torch.as_tensor(node_ids).to(device=dev, dtype=torch.int32)
        if ids.dim() == 1:
            ids, ids_ld = ids.contiguous(), 0
        elif ids.dim() == 2 and ids.shape[0] == B:
            ids = ids.contiguous()
            ids_ld = ids.shape[1]
        else:
            raise ValueError("node_ids must be [K] or [B, K]")
        K = ids.shape[-1]
        norm = None
        if normalizer is not None:
            norm = torch.as_tensor(normalizer).to(device=dev, dtype=torch.int32)
            norm = norm.expand(B).contiguous() if norm.dim() == 0 else norm.contiguous()
            if norm.shape != (B,):
                raise ValueError("normalizer must be a node id or one node id per row")
        out = torch.empty((B, K), dtype=mass.dtype, device=dev)
        if B and K:
            self._launch(
                "gt_gather_nodes", dev.index, mass.data_ptr(), _OUT_TYPES[mass.dtype], B, self.N,
                mass.stride(0) if B > 1 else self.N, ids.data_ptr(), K, ids_ld, norm.data_ptr() if norm is not None else None,
                _lib.GT_GATHER_LOG if log else 0, out.data_ptr(), K,
            )
        return out

    def subtree_token_mask(self, nodes, device=None):
        """Keep-bitmask ``int32[B, ceil(V/32)]`` of the tokens under each node (bit ``i % 32`` of word ``i // 32``):
        the layout ``smc.masked_logsumexp_sample`` takes as a bit mask."""
        require_cuda()
        nodes = torch.as_tensor(nodes)
        if device is None:
            device = nodes.device if nodes.is_cuda else torch.device("cuda", torch.cuda.current_device())
        device = torch.device(device)
        nodes = nodes.to(device=device, dtype=torch.int32).reshape(-1).contiguous()
        B, W = nodes.shape[0], (self.V + 31) // 32
        self.ensure_device(device.index)
        bits = torch.empty((B, W), dtype=torch.int32, device=device)
        if B and W:
            self._launch("gt_subtree_token_mask", device.index, self._handle, nodes.data_ptr(), B, bits.data_ptr(), W)
        return bits

    # ---- token masks under a byte DFA or pushdown automaton, and the advance ------------------------------------
    def _automaton_args(self, delta, states, nodes=None, tokens=None, logw=None, pda=None):
        """The leading arguments of an automaton entry point, the trie handle to ``n_rows``, as ``(args, B, device,
        keep)``; ``keep`` holds the converted tensors until the launch.  The device is that of ``states`` when it is a
        CUDA tensor, else that of ``delta``, else the current device.  ``delta`` and ``states``, and ``nodes`` and
        ``tokens`` where given (one entry per row), become contiguous int32 tensors on it.  ``pda = (push, stack,
        depth)`` makes it a PDA call: ``push`` is an integer table of ``delta``'s shape, converted the same way, and the
        rows' stacks must already be int32 tensors on the device, ``stack`` ``[B, stack_ld]`` with contiguous rows and
        ``depth`` ``[B]``, since the advance updates them in place and a converted copy would lose the update.
        ``logw``, the transition log-weights of the weighted calls, is a float table of ``delta``'s shape, converted to
        contiguous float32."""
        require_cuda()
        delta, states = torch.as_tensor(delta), torch.as_tensor(states)
        device = states.device if states.is_cuda else delta.device if delta.is_cuda else torch.device("cuda", torch.cuda.current_device())
        if delta.dim() != 2:
            raise ValueError(f"delta must be a 2-D [states, symbols] table, got shape {tuple(delta.shape)}")
        delta = delta.to(device=device, dtype=torch.int32).contiguous()
        states = states.to(device=device, dtype=torch.int32).reshape(-1).contiguous()
        B = states.shape[0]

        def per_row(x, what):
            x = torch.as_tensor(x).to(device=device, dtype=torch.int32).reshape(-1).contiguous()
            if x.shape[0] != B:
                raise ValueError(f"{what} must hold one entry per row ({B}), got {x.shape[0]}")
            return x

        nodes = None if nodes is None else per_row(nodes, "nodes")
        tokens = None if tokens is None else per_row(tokens, "tokens")
        self.ensure_device(device.index)
        keep = [delta, states, nodes, tokens]
        args = [self._handle, delta.data_ptr()]
        if pda is not None:
            push, stack, depth = pda
            push = torch.as_tensor(push)
            if push.shape != delta.shape or push.is_floating_point() or push.is_complex():
                raise ValueError(f"push must be an integer table of delta's shape {tuple(delta.shape)}, got {push.dtype} "
                                 f"{tuple(push.shape)}")
            push = push.to(device=device, dtype=torch.int32).contiguous()
            for x, what, dim in ((stack, "stack", 2), (depth, "depth", 1)):
                if not (isinstance(x, torch.Tensor) and x.dtype == torch.int32 and x.device == device and x.dim() == dim
                        and x.shape[0] == B):
                    raise ValueError(f"{what} must be an int32 tensor on {device} of {dim} dimensions with one row per "
                                     f"state ({B})")
            if not (1 <= stack.shape[1] <= _lib.GT_PDA_MAX_DEPTH):
                raise ValueError(f"stack must be [B, stack_ld] with 1 <= stack_ld <= {_lib.GT_PDA_MAX_DEPTH}, got "
                                 f"{tuple(stack.shape)}")
            if not stack.is_contiguous() or not depth.is_contiguous():
                raise ValueError("stack and depth must be contiguous: [B, stack_ld] rows of stack_ld entries and [B]")
            keep.append(push)
            args.append(push.data_ptr())
        if logw is not None:
            logw = torch.as_tensor(logw)
            if not logw.is_floating_point() or logw.shape != delta.shape:
                raise ValueError(f"logw must be a float table of delta's shape {tuple(delta.shape)}, got {logw.dtype} "
                                 f"{tuple(logw.shape)}")
            logw = logw.to(device=device, dtype=torch.float32).contiguous()
            keep.append(logw)
            args.append(logw.data_ptr())
        args += [delta.shape[0], delta.shape[1], states.data_ptr()]
        if pda is None:
            args.append(nodes.data_ptr() if nodes is not None else None)
        else:
            args += [stack.data_ptr(), stack.shape[1], depth.data_ptr()]
        if tokens is not None:
            args.append(tokens.data_ptr())
        return args + [B], B, device, keep

    def dfa_token_mask(self, delta, states, nodes=None):
        """``gt_dfa_token_mask`` on the current stream of the inputs' device: keep-bitmask ``int32[B, ceil(V/32)]`` of the
        items allowed under the DFA ``delta`` (``[Q, ld >= S]``) from ``states[b]`` at ``nodes[b]`` (the root when None)."""
        args, B, device, _keep = self._automaton_args(delta, states, nodes=nodes)
        bits = torch.empty((B, (self.V + 31) // 32), dtype=torch.int32, device=device)
        if bits.numel():
            self._launch("gt_dfa_token_mask", device.index, *args, bits.data_ptr(), bits.shape[1])
        return bits

    def dfa_token_logw(self, delta, logw, states, nodes=None):
        """``gt_dfa_token_logw`` on the current stream of the inputs' device: ``float32[B, V]``, each allowed item's
        summed transition log-weights under ``logw`` (a float table of ``delta``'s shape), ``-inf`` elsewhere."""
        args, B, device, _keep = self._automaton_args(delta, states, nodes=nodes, logw=logw)
        out = torch.empty((B, self.V), dtype=torch.float32, device=device)
        if out.numel():
            self._launch("gt_dfa_token_logw", device.index, *args, out.data_ptr(), self.V)
        return out

    def dfa_advance(self, delta, states, tokens, nodes=None):
        """``gt_dfa_advance`` on the current stream of the inputs' device: ``int32[B]``, the state after the remaining
        symbols of item ``tokens[b]``, or -1."""
        args, B, device, _keep = self._automaton_args(delta, states, nodes=nodes, tokens=tokens)
        out = torch.empty(B, dtype=torch.int32, device=device)
        if B:
            self._launch("gt_dfa_advance", device.index, *args, out.data_ptr())
        return out

    def pda_token_mask(self, delta, push, states, stack, depth):
        """``gt_pda_token_mask`` on the current stream of the inputs' device: keep-bitmask ``int32[B, ceil(V/32)]`` of the
        items the PDA (``delta``, ``push``) accepts from each row's configuration at the root."""
        args, B, device, _keep = self._automaton_args(delta, states, pda=(push, stack, depth))
        bits = torch.empty((B, (self.V + 31) // 32), dtype=torch.int32, device=device)
        if bits.numel():
            self._launch("gt_pda_token_mask", device.index, *args, bits.data_ptr(), bits.shape[1])
        return bits

    def pda_token_logw(self, delta, push, logw, states, stack, depth):
        """``gt_pda_token_logw`` on the current stream of the inputs' device: ``float32[B, V]``, each allowed item's
        summed transition log-weights under ``logw`` (a float table of ``delta``'s shape), ``-inf`` elsewhere."""
        args, B, device, _keep = self._automaton_args(delta, states, logw=logw, pda=(push, stack, depth))
        out = torch.empty((B, self.V), dtype=torch.float32, device=device)
        if out.numel():
            self._launch("gt_pda_token_logw", device.index, *args, out.data_ptr(), self.V)
        return out

    def pda_advance(self, delta, push, states, stack, depth, tokens):
        """``gt_pda_advance`` on the current stream of the inputs' device: ``int32[B]``, the state after item
        ``tokens[b]``, or -1; ``stack`` and ``depth`` are updated in place where the result is not -1."""
        args, B, device, _keep = self._automaton_args(delta, states, tokens=tokens, pda=(push, stack, depth))
        out = torch.empty(B, dtype=torch.int32, device=device)
        if B:
            self._launch("gt_pda_advance", device.index, *args, out.data_ptr())
        return out

    # ---- child masses of one node per row, straight from the rows -----------------------------------------------
    def _child_inputs(self, ws, nodes):
        """Checks shared by the child read-outs (those of ``reduce``, plus one node id per row)."""
        require_cuda()
        if not (isinstance(ws, torch.Tensor) and ws.is_cuda and ws.dim() == 2):
            raise ValueError("expected a 2-D CUDA tensor of rows")
        if ws.shape[1] != self.V:
            raise AssertionError([ws.shape[1], self.V])
        if ws.dtype not in _IN_TYPES:
            ws = ws.to(torch.float32)
        B = ws.shape[0]
        if (ws.shape[1] > 1 and ws.stride(1) != 1) or (B > 1 and ws.stride(0) < self.V):
            ws = ws.contiguous()
        nodes = torch.as_tensor(nodes)
        if nodes.dim() != 1 or nodes.shape[0] != B:
            raise ValueError(f"nodes must be 1-D with one node id per row ({B}), got shape {tuple(nodes.shape)}")
        nodes = nodes.to(device=ws.device, dtype=torch.int32).contiguous()
        self.ensure_device(ws.device.index)
        return ws, nodes, B, (ws.stride(0) if B > 1 else max(self.V, 1))

    def keep_bits(self, mask, B, device):
        """A keep-mask for ``B`` rows as ``(bits, mask_ld)`` in ``GT_MASK_BITS_U32`` layout on ``device``: an int32
        bitmask ``[ceil(V/32)]`` (shared, ``mask_ld = 0``) or ``[B, ceil(V/32)]`` (per row, any row stride of at least
        ``ceil(V/32)``), or a bool keep-mask ``[V]`` / ``[B, V]``, packed.  Anything else raises ``ValueError``."""
        from ..smc import _pack_keep_bits

        V, W = self.V, (self.V + 31) // 32
        mask = torch.as_tensor(mask)
        if mask.dtype == torch.bool and mask.dim() in (1, 2) and mask.shape[-1] == V and (mask.dim() == 1 or mask.shape[0] == B):
            keep = torch.nn.functional.pad(mask.to(device), (0, W * 32 - V))  # each row a whole number of words
            mask = _pack_keep_bits(keep.reshape(-1)).view(keep.shape[:-1] + (W,))
        elif mask.dtype != torch.int32 or mask.dim() not in (1, 2) or mask.shape[-1] != W or (mask.dim() == 2 and mask.shape[0] != B):
            raise ValueError(f"mask must be an int32 keep-bitmask [{W}] or [{B}, {W}] (ceil(V/32) words per row), or a bool "
                             f"keep-mask [{V}] or [{B}, {V}]; got {mask.dtype} of shape {tuple(mask.shape)}")
        mask = mask.to(device)
        if mask.dim() == 1:
            return mask.contiguous(), 0
        if mask.stride(1) != 1 or (B > 1 and mask.stride(0) < W):
            mask = mask.contiguous()
        return mask, (mask.stride(0) if B > 1 else W)

    def _read_out(self, fn, mask, B, device):
        """The entry point of a next-symbol read-out and the arguments that follow ``nodes``: ``fn`` without a mask,
        ``fn + "_masked"`` with the mask's bits and row stride otherwise (``keep`` holds the bits until the launch)."""
        if mask is None:
            return fn, (), None
        bits, ld = self.keep_bits(mask, B, device)
        return fn + "_masked", (bits.data_ptr(), ld), bits

    def child_masses(self, ws, nodes, ops=("sum",), log_input=False, dfs_order=False, normalize=False, log=False, mask=None):
        """``gt_child_masses`` (``gt_child_masses_masked`` with a ``mask``, see ``keep_bits``) on the current stream of
        the input's device.  Returns ``(child_ids int32[B, D], sums float32[B, D] | None, maxes float32[B, D] | None)``;
        nothing is synchronised."""
        ws, nodes, B, ld_ws = self._child_inputs(ws, nodes)
        opmask = _opmask(ops)
        D, dev = self.max_children, ws.device
        fn, margs, _keep = self._read_out("gt_child_masses", mask, B, dev)
        ids = torch.empty((B, D), dtype=torch.int32, device=dev)
        sums = torch.empty((B, D), dtype=torch.float32, device=dev) if opmask & _lib.GT_OP_SUM else None
        maxes = torch.empty((B, D), dtype=torch.float32, device=dev) if opmask & _lib.GT_OP_MAX else None
        if B and D:
            self._launch(
                fn, dev.index, self._handle, ws.data_ptr(), _IN_TYPES[ws.dtype], B, ld_ws, nodes.data_ptr(), *margs,
                ids.data_ptr(), sums.data_ptr() if sums is not None else None,
                maxes.data_ptr() if maxes is not None else None, D, opmask, _flags(log_input, dfs_order, normalize, log),
                workspace=self._child_workspace, rows=B,
            )
        return ids, sums, maxes

    def child_sample(self, ws, nodes, seed=0, offset=0, log_input=False, dfs_order=False, mask=None):
        """``gt_child_sample`` (``gt_child_sample_masked`` with a ``mask``) on the current stream of the input's device:
        ``(child int32[B], logp float32[B], logZ float32[B])``; nothing is synchronised."""
        ws, nodes, B, ld_ws = self._child_inputs(ws, nodes)
        dev = ws.device
        fn, margs, _keep = self._read_out("gt_child_sample", mask, B, dev)
        child = torch.empty(B, dtype=torch.int32, device=dev)
        logp = torch.empty(B, dtype=torch.float32, device=dev)
        logZ = torch.empty(B, dtype=torch.float32, device=dev)
        if B:
            self._launch(
                fn, dev.index, self._handle, ws.data_ptr(), _IN_TYPES[ws.dtype], B, ld_ws, nodes.data_ptr(), *margs,
                _flags(log_input, dfs_order), int(seed) & (2**64 - 1), int(offset) & (2**64 - 1), child.data_ptr(),
                logp.data_ptr(), logZ.data_ptr(), workspace=self._child_workspace, rows=B,
            )
        return child, logp, logZ

    # ---- the same, indexed by symbol ---------------------------------------------------------------------------
    def symbol_masses(self, ws, nodes, ops=("sum",), log_input=False, dfs_order=False, normalize=False, log=False, mask=None):
        """``gt_symbol_masses`` (``gt_symbol_masses_masked`` with a ``mask``) on the current stream of the input's device.
        Returns ``(sums float32[B, S+1] | None, maxes float32[B, S+1] | None)``; nothing is synchronised."""
        ws, nodes, B, ld_ws = self._child_inputs(ws, nodes)
        opmask = _opmask(ops)
        W, dev = self.num_symbols + 1, ws.device
        fn, margs, _keep = self._read_out("gt_symbol_masses", mask, B, dev)
        sums = torch.empty((B, W), dtype=torch.float32, device=dev) if opmask & _lib.GT_OP_SUM else None
        maxes = torch.empty((B, W), dtype=torch.float32, device=dev) if opmask & _lib.GT_OP_MAX else None
        if B:
            self._launch(
                fn, dev.index, self._handle, ws.data_ptr(), _IN_TYPES[ws.dtype], B, ld_ws, nodes.data_ptr(), *margs,
                sums.data_ptr() if sums is not None else None, maxes.data_ptr() if maxes is not None else None, W, opmask,
                _flags(log_input, dfs_order, normalize, log), workspace=self._child_workspace, rows=B,
            )
        return sums, maxes

    def symbol_sample(self, ws, nodes, symbol_logw, seed=0, offset=0, log_input=False, dfs_order=False, mask=None):
        """``gt_symbol_sample`` (``gt_symbol_sample_masked`` with a ``mask``) on the current stream of the input's device:
        ``(child int32[B], symbol int32[B], logp float32[B], logZ float32[B], logM float32[B])``; nothing is
        synchronised.  ``symbol_logw``: ``[S+1]`` (shared by all rows) or ``[B, S+1]``, converted to contiguous float32
        on the input's device."""
        ws, nodes, B, ld_ws = self._child_inputs(ws, nodes)
        W, dev = self.num_symbols + 1, ws.device
        logw = torch.as_tensor(symbol_logw)
        if not (logw.dim() == 1 and logw.shape[0] == W) and not (logw.dim() == 2 and tuple(logw.shape) == (B, W)):
            raise ValueError(f"symbol_logw must be [{W}] or [{B}, {W}] (S + 1 = {W} columns), got shape {tuple(logw.shape)}")
        if not logw.is_floating_point():
            raise ValueError(f"symbol_logw must hold floating-point log-weights, got {logw.dtype}")
        logw = logw.to(device=dev, dtype=torch.float32).contiguous()
        ld_w = 0 if logw.dim() == 1 else W
        fn, margs, _keep = self._read_out("gt_symbol_sample", mask, B, dev)
        child = torch.empty(B, dtype=torch.int32, device=dev)
        symbol = torch.empty(B, dtype=torch.int32, device=dev)
        logp = torch.empty(B, dtype=torch.float32, device=dev)
        logZ = torch.empty(B, dtype=torch.float32, device=dev)
        logM = torch.empty(B, dtype=torch.float32, device=dev)
        if B:
            self._launch(
                fn, dev.index, self._handle, ws.data_ptr(), _IN_TYPES[ws.dtype], B, ld_ws, nodes.data_ptr(), *margs,
                logw.data_ptr(), ld_w, _flags(log_input, dfs_order), int(seed) & (2**64 - 1), int(offset) & (2**64 - 1),
                child.data_ptr(), symbol.data_ptr(), logp.data_ptr(), logZ.data_ptr(), logM.data_ptr(),
                workspace=self._child_workspace, rows=B,
            )
        return child, symbol, logp, logZ, logM
