"""Fused SMC particle step: masked logsumexp + one categorical draw per row, in one kernel launch.

Replaces the per-particle torch sequence of the reference idiom (``README.md:82-91``; temperature variant
``genlm/backend/llm/base.py:131-146``)::

    masked = logps + mask            # mask in {0, -inf}
    logZ   = masked.logsumexp(-1)    # particle weight increment
    tok    = torch.multinomial((masked - logZ).exp(), 1).item()

``masked_logsumexp_sample`` does this for a whole ``[B, V]`` batch of particles without a host sync per row.
Draws use one Philox uniform per row through an exact inverse CDF: distribution-equal to
``torch.multinomial``, not stream-equal.  ``resample`` takes the step an SMC driver takes next: each particle group's
effective sample size and, below a threshold, its ancestors, again without a host sync.
"""
import weakref

import torch

from . import _lib
from ._lib import lib, check
from .trie._engine import require_cuda

_IN_TYPES = {torch.float32: _lib.GT_F32, torch.float64: _lib.GT_F64, torch.float16: _lib.GT_F16, torch.bfloat16: _lib.GT_BF16}


# Shared additive {0, -inf} masks (the reference idiom: `valid_ids = torch.tensor([...], dtype=torch.float).log()`, built once
# and added to every particle's row, README.md:59-70) are packed into keep-bitmasks once and cached: the kernel then reads
# V/8 mask bytes per row instead of 4V (shared fp32 mask: 0.79 of the HBM peak at 512 rows, bit mask: 0.87).  An entry
# belongs to one live tensor object (weak reference: a new tensor that reuses the address or id of a dead one never
# matches) at one version (torch bumps it on every in-place write), so a mask that is written to is packed again.
_BITMASK_CACHE = {}  # id(mask) -> (weakref to the mask, its _version, bits or None)
_BITMASK_CACHE_MAX = 16


def _pack_keep_bits(keep):
    """bool ``[V]`` -> int32 ``[ceil(V/32)]`` (bit ``i % 32`` of word ``i // 32``)."""
    V = keep.shape[0]
    pad = (-V) % 32
    k = torch.nn.functional.pad(keep, (0, pad)).view(-1, 32).to(torch.int64)
    w = (k << torch.arange(32, device=keep.device, dtype=torch.int64)).sum(-1)
    return torch.where(w >= 2**31, w - 2**32, w).to(torch.int32)


def _cached_bits(mask):
    """Cache entry of this very tensor at its current version, or ``None``."""
    hit = _BITMASK_CACHE.get(id(mask))
    if hit is not None and hit[0]() is mask and hit[1] == mask._version:
        return hit
    return None


def _shared_additive_as_bits(mask):
    """int32 keep-bitmask of a 1-D additive float mask whose values are all 0 or -inf, else ``None``."""
    hit = _cached_bits(mask)
    if hit is None:
        keep = mask == 0
        exact = bool((keep | (mask == float("-inf"))).all())  # one sync per distinct mask
        for k in [k for k, h in _BITMASK_CACHE.items() if h[0]() is None]:  # entries of dead tensors
            del _BITMASK_CACHE[k]
        if len(_BITMASK_CACHE) >= _BITMASK_CACHE_MAX:
            _BITMASK_CACHE.pop(next(iter(_BITMASK_CACHE)))
        hit = (weakref.ref(mask), mask._version, _pack_keep_bits(keep) if exact else None)
        _BITMASK_CACHE[id(mask)] = hit
    return hit[2]


def _mask_args(mask, B, V, device):
    if mask is None:
        return None, _lib.GT_MASK_NONE, 0, None
    if not isinstance(mask, torch.Tensor):
        mask = torch.as_tensor(mask)
    mask = mask.to(device)
    if mask.dtype == torch.bool:
        kind, m = _lib.GT_MASK_BOOL_U8, mask.view(torch.uint8)  # same bytes: no conversion pass
    elif mask.dtype == torch.uint8:
        kind, m = _lib.GT_MASK_BOOL_U8, mask
    elif mask.dtype == torch.int32 and mask.shape[-1] == (V + 31) // 32:
        kind, m = _lib.GT_MASK_BITS_U32, mask
    elif mask.is_floating_point():
        bits = None
        if mask.dim() == 1 and mask.shape[0] == V and not torch.cuda.is_current_stream_capturing():
            bits = _shared_additive_as_bits(mask)
        elif mask.dim() == 1 and mask.shape[0] == V:
            hit = _cached_bits(mask)
            bits = hit[2] if hit else None  # during graph capture: only what was packed before
        if bits is not None:
            kind, m = _lib.GT_MASK_BITS_U32, bits
        else:
            kind, m = _lib.GT_MASK_ADD_F32, mask.to(torch.float32)
    else:
        raise ValueError(f"unsupported mask dtype {mask.dtype}")
    width = (V + 31) // 32 if kind == _lib.GT_MASK_BITS_U32 else V
    if m.dim() == 1:
        if m.shape[0] != width:
            raise ValueError(f"mask length {m.shape[0]} does not match {width}")
        m = m.contiguous()
        ld = 0
    elif m.dim() == 2:
        if m.shape != (B, width):
            raise ValueError(f"mask shape {tuple(m.shape)} does not match {(B, width)}")
        if m.stride(1) != 1:
            m = m.contiguous()
        ld = m.stride(0) if B > 1 else width
    else:
        raise ValueError("mask must be 1-D (shared) or 2-D (per row)")
    return m, kind, ld, m


def masked_logsumexp_sample(logps, mask=None, temperature=1.0, seed=0, offset=0, check_valid=False):
    """Masked logsumexp and one categorical draw per row.

    Args:
        logps (torch.Tensor): ``[B, V]`` (or ``[V]``) log-probabilities / logits on a CUDA device; fp32, fp16,
            bf16 or fp64.
        mask: ``None``; an additive float mask (``{0, -inf}``, the reference idiom); a bool / uint8 keep-mask;
            or an int32 bitmask of ``ceil(V/32)`` words.  1-D masks are shared by all rows.
        temperature (float): logits are divided by it before masking (``llm/base.py:136``).
        seed, offset (int): Philox key and counter base; row ``b`` uses counter ``offset + b``.
        check_valid (bool): synchronise and raise ``RuntimeError`` like ``torch.multinomial`` when a row has no
            mass or a NaN.

    Returns:
        ``(logZ float32[B], tokens int32[B])`` on the device; rows without mass give ``(-inf, -1)``.  As
        ``torch.logsumexp``, a row with an allowed NaN gives ``(NaN, -1)``, else one with an allowed ``+inf``
        ``(+inf, -1)``.  A bool or bit mask drops a masked-out value whatever it is; an additive mask adds ``-inf`` to
        it, so a masked-out ``+inf`` gives NaN, as in torch.  A shared ``{0, -inf}`` float mask is packed into bits and
        so drops it too.
    """
    require_cuda()
    if not isinstance(logps, torch.Tensor) or not logps.is_cuda:
        raise ValueError("logps must be a CUDA tensor")
    squeeze = logps.dim() == 1
    if squeeze:
        logps = logps.unsqueeze(0)
    if logps.dim() != 2:
        raise ValueError("logps must be 1-D or 2-D")
    if logps.dtype not in _IN_TYPES:
        logps = logps.to(torch.float32)
    if logps.shape[1] > 1 and logps.stride(1) != 1:
        logps = logps.contiguous()
    B, V = logps.shape
    dev = logps.device
    m, kind, mask_ld, _keep = _mask_args(mask, B, V, dev)
    logZ = torch.empty(B, dtype=torch.float32, device=dev)
    tok = torch.empty(B, dtype=torch.int32, device=dev)
    if B:
        with torch.cuda.device(dev.index):
            check(
                lib.gt_lse_sample(
                    logps.data_ptr(), _IN_TYPES[logps.dtype], B, V, logps.stride(0) if B > 1 else V,
                    m.data_ptr() if m is not None else None, kind, mask_ld, float(temperature),
                    int(seed) & (2**64 - 1), int(offset) & (2**64 - 1), logZ.data_ptr(), tok.data_ptr(),
                    torch.cuda.current_stream(dev.index).cuda_stream,
                ),
                "gt_lse_sample",
            )
    if check_valid and B:
        bad = tok < 0
        if bool(bad.any()):
            if bool(torch.isnan(logZ[bad]).any()):
                raise RuntimeError("probability tensor contains either `inf`, `nan` or element < 0")
            raise RuntimeError("invalid multinomial distribution (sum of probabilities <= 0)")
    if squeeze:
        return logZ[0], tok[0]
    return logZ, tok


_RESAMPLE_METHODS = {"multinomial": _lib.GT_RESAMPLE_MULTINOMIAL, "stratified": _lib.GT_RESAMPLE_STRATIFIED,
                     "systematic": _lib.GT_RESAMPLE_SYSTEMATIC}


def resample(log_weights, method="systematic", ess_threshold=0.5, seed=0, offset=0):
    """Per-group effective sample size and, where it falls below ``ess_threshold * P``, ancestors drawn on the device.

    The constrained SMC step, weight bookkeeping and reindexing included, runs as one CUDA graph::

        tokw = trie.dfa_token_logw(delta, logw, q)                  # [B, V] token log-weights at the root
        logZ, tok = smc.masked_logsumexp_sample(logps, tokw, seed=seed, offset=step * B)
        q = trie.dfa_advance(delta, q, tok)
        log_weights += logZ
        anc, log_weights, ess, log_mean_w, resampled = smc.resample(
            log_weights.view(G, P), "systematic", 0.5, seed=seed, offset=step * B)
        log_weights = log_weights.view(-1)
        q = q.index_select(0, anc.view(-1))                        # and every per-particle state of the caller
        tokens = tokens.index_select(0, anc.view(-1))

    Args:
        log_weights (torch.Tensor): CUDA log-weights, ``[P]`` for one group or ``[G, P]`` for ``G`` groups of ``P``
            particles (``P <= 16384``); other float dtypes are converted to float32.
        method (str): ``"multinomial"``, ``"stratified"`` or ``"systematic"``.
        ess_threshold (float): a group resamples iff its ESS ``S^2 / Q`` is below ``ess_threshold * P`` (0: never,
            ``inf``: every group with a positive, finite total).
        seed, offset (int): Philox key and counter base; particle ``b = g * P + j`` uses counter ``offset + b`` (with
            the third counter word 1, so the sampler's ``seed`` and ``offset`` give independent uniforms).

    Returns:
        ``(ancestors, new_log_weights, ess, log_mean_w, resampled)``: ancestors int32 and new log-weights (the group's
        log mean weight where it resampled, else unchanged) shaped like the input, ancestors as flat indices into the
        ``G * P`` particles; ``ess`` and ``log_mean_w`` float32 ``[G]``; ``resampled`` bool ``[G]``.  A group with a NaN
        weight gives ess and log mean weight NaN; one with a ``+inf`` weight ess NaN and ``+inf``; an all ``-inf`` group
        ess 0 and ``-inf``; none of them resamples.  The full semantics are those of ``gt_resample``
        (``include/genlm_trie_b200.h``).
    """
    if method not in _RESAMPLE_METHODS:
        raise ValueError(f"unknown resampling method {method!r}: one of {sorted(_RESAMPLE_METHODS)}")
    if not isinstance(log_weights, torch.Tensor):
        raise ValueError("log_weights must be a tensor")
    if log_weights.dim() not in (1, 2):
        raise ValueError("log_weights must be [P] or [G, P]")
    if not 1 <= log_weights.shape[-1] <= _lib.GT_RESAMPLE_MAX_GROUP:
        raise ValueError(f"group size {log_weights.shape[-1]} is not in [1, {_lib.GT_RESAMPLE_MAX_GROUP}]")
    if not log_weights.is_floating_point():
        raise ValueError(f"log_weights must be a float tensor, not {log_weights.dtype}")
    if not log_weights.is_cuda:
        raise ValueError("log_weights must be a CUDA tensor")
    shape = log_weights.shape
    lw = log_weights.to(torch.float32).reshape(-1, shape[-1]).contiguous()
    G, P = lw.shape
    dev = lw.device
    anc = torch.empty((G, P), dtype=torch.int32, device=dev)
    out = torch.empty((G, P), dtype=torch.float32, device=dev)
    ess = torch.empty(G, dtype=torch.float32, device=dev)
    lmw = torch.empty(G, dtype=torch.float32, device=dev)
    res = torch.empty(G, dtype=torch.bool, device=dev)
    if G:
        with torch.cuda.device(dev.index):
            check(
                lib.gt_resample(
                    lw.data_ptr(), G, P, _RESAMPLE_METHODS[method], float(ess_threshold), int(seed) & (2**64 - 1),
                    int(offset) & (2**64 - 1), anc.data_ptr(), out.data_ptr(), ess.data_ptr(), lmw.data_ptr(),
                    res.data_ptr(), torch.cuda.current_stream(dev.index).cuda_stream,
                ),
                "gt_resample",
            )
    return anc.view(shape), out.view(shape), ess, lmw, res
