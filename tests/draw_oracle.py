"""fp64 replay of the draws of ``gt_lse_sample`` and of the next-symbol draws (``gt_child_sample``,
``gt_symbol_sample`` and their masked forms), from the Philox uniforms of ``resample_oracle.uniforms(..., stream=0)``.

Both draws are inverse CDFs over a fixed order.  The next-symbol draws walk a node's children in child order, with
every term in fp64.  ``gt_lse_sample`` walks the vocabulary in the order of its work split (``lse_draw_order``), with
pass-1 sums in fp32, so a token is checked by the interval rule of ``in_interval`` rather than by equality.
"""
import math

import numpy as np

import oracle
from resample_oracle import uniforms

LOG2E = 1.0 / math.log(2.0)


def sampler_threads(dtype, mask_kind):
    """Threads per row of ``gt_lse_sample`` (``launch_sampler_mk``): 512 for 2-byte rows under an additive mask, else
    256.  ``dtype`` is a numpy or torch dtype; ``mask_kind`` one of ``"none"``, ``"add"``, ``"bool"``, ``"bits"``."""
    return 512 if _itemsize(dtype) == 2 and mask_kind == "add" else 256


def _itemsize(dtype):
    size = getattr(dtype, "itemsize", None)  # a torch dtype; numpy scalar types have a descriptor there
    return size if isinstance(size, int) else np.dtype(dtype).itemsize


def lse_draw_order(V, phase, EPV, NT):
    """int64 ``[V]``: the vocabulary in the order ``gt_lse_sample``'s inverse CDF walks it, a permutation of
    ``[0, V)``.

    The row is cut into ``ng = ceil((phase + V) / EPV)`` 16-byte groups; group ``g`` holds elements
    ``g*EPV - phase + k``, ``k < EPV``, those in ``[0, V)``.  Pass 1 gives thread ``t`` the groups ``t + c*NT``, and the
    first pick is over threads in order.  Pass 2 hands candidate ``c`` of the picked thread to sub-thread ``c % NT``,
    picks a sub-thread in order, and that sub-thread walks its candidates ``c``, ``c + NT``, ... element by element.
    So the order is: thread ``t``, then sub-thread ``c % NT``, then ``c // NT``, then ``k``.  With at most ``NT``
    candidates per thread (rows of at most ``NT**2`` groups) a thread's groups come in increasing order."""
    ng = (phase + V + EPV - 1) // EPV
    C = max(1, -(-ng // (NT * NT)))
    # group g = t + NT * (t2 + NT * cc): indexed [cc, t2, t], walked t, then t2, then cc
    g = np.arange(C * NT * NT, dtype=np.int64).reshape(C, NT, NT).transpose(2, 1, 0).ravel()
    g = g[g < ng]
    e = (g[:, None] * EPV - phase + np.arange(EPV, dtype=np.int64)).ravel()
    return e[(e >= 0) & (e < V)]


def _working_rows(logp, mask, mask_kind, temperature):
    """fp64 ``logp / T + mask`` of the rows as the kernel reads them (fp16 / bf16 exactly, fp64 rounded to fp32);
    a keep-mask (``"bool"``, ``"bits"``) replaces masked-out elements by ``-inf`` whatever their value."""
    x = np.asarray(logp, dtype=np.float32).astype(np.float64) / float(temperature)
    if mask_kind == "add":
        with np.errstate(invalid="ignore"):
            x = x + np.asarray(mask, dtype=np.float32).astype(np.float64)
    elif mask_kind in ("bool", "bits"):
        x = np.where(np.asarray(mask, dtype=bool), x, -np.inf)
    else:
        assert mask_kind == "none" and mask is None, mask_kind
    return x


class LseReplay:
    """Per-row results of ``lse_replay``: ``logZ`` float64 ``[B]``; ``u`` the row's uniform; ``M`` the largest
    working value (``-inf`` for no mass); and per row ``order[b]`` (``lse_draw_order``), ``cdf[b]`` (the running
    sum of ``exp(x - M)`` in that order, so ``Z[b] = cdf[b][-1]``), ``tok[b]`` (the oracle's token, -1 for a row
    without a draw) and ``delta[b]`` (the tolerance of ``in_interval``)."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


def lse_delta(n_t, M_SC):
    """Tolerance of the draw check, as a fraction of ``Z``.  The kernel's CDF differs from the fp64 one by:

    - the fp32 running sum of a thread's pass-1 mass over its ``n_t`` elements (``n_t * 2**-24`` relative);
    - the rounding of the exponent offset ``-m * SC`` to fp32, ``|M * SC| * 2**-24`` in the exponent, and the same
      order for the fp32 working value ``logp * inv_temp + mask`` of an additive mask; both grow at low temperature;
    - ``ex2.approx`` (2 ulp) and the fp32 rounding of ``SC = inv_temp * log2(e)`` and of each exponent, which are a
      few ulp weighted by the row's entropy in bits.
    The draw is a two-level inverse CDF (a thread by its pass-1 mass, then an element by pass-2 masses): these
    relative errors displace ``u * Z`` against the fp64 CDF by at most a few times their sum, hence the factor 4."""
    return 4.0 * 2.0 ** -24 * (n_t + abs(M_SC) + 8)


def lse_replay(logp, mask=None, mask_kind="none", temperature=1.0, seed=0, offset=0, phases=None, dtype=np.float32):
    """fp64 replay of ``gt_lse_sample`` on ``logp`` ``[B, V]`` (float32 values as the kernel reads them).

    ``mask``: ``None``; additive float ``[B, V]`` or ``[V]`` (``"add"``); a keep-mask bool ``[B, V]`` or ``[V]``
    (``"bool"`` and ``"bits"``: pass the unpacked bits).  ``phases[b]``: the element offset of row ``b`` inside its
    16-byte line, ``(data_ptr + b * stride * itemsize) % 16 // itemsize``.  ``dtype`` is the row type on the device
    (it sets ``EPV = 16 / itemsize`` and, with ``mask_kind``, the thread count).

    ``logZ`` follows ``torch.logsumexp`` in fp64: NaN when an allowed value is NaN (also ``+inf - inf`` under an
    additive mask), else ``+inf`` when one is ``+inf``, else ``-inf`` for no mass.  Such rows have no draw.  Otherwise
    the token is the first in draw order whose CDF value exceeds ``u * Z``, else the last one with positive mass (the
    kernel's fall-back when rounding pushes ``u * Z`` past its total)."""
    x = _working_rows(logp, mask, mask_kind, temperature)
    B, V = x.shape
    if mask_kind == "add":
        logZ = oracle.masked_logsumexp(np.asarray(logp, dtype=np.float32), np.asarray(mask, dtype=np.float32),
                                       temperature)
    else:
        logZ = oracle.masked_logsumexp(x)  # the temperature and a keep-mask are in x already
    EPV = 16 // _itemsize(dtype)
    NT = sampler_threads(dtype, mask_kind)
    phases = np.zeros(B, dtype=np.int64) if phases is None else np.asarray(phases, dtype=np.int64)
    u = uniforms(seed, np.uint64(offset) + np.arange(B, dtype=np.uint64), stream=0)
    out = dict(u=u, logZ=np.broadcast_to(logZ, (B,)).copy(), M=np.empty(B), order=[], cdf=[],
               tok=np.full(B, -1, dtype=np.int64), delta=np.zeros(B))
    orders = {}
    for b in range(B):
        ph = int(phases[b])
        if ph not in orders:
            orders[ph] = lse_draw_order(V, ph, EPV, NT)
        order = orders[ph]
        xb = x[b]
        M = np.nan if np.isnan(xb).any() else xb.max()
        out["M"][b] = M
        out["order"].append(order)
        if not np.isfinite(M):
            out["cdf"].append(np.zeros(V))
            continue
        w = np.exp(xb[order] - M)
        cdf = np.cumsum(w)
        Z = cdf[-1]
        out["cdf"].append(cdf)
        i = int(np.searchsorted(cdf, u[b] * Z, side="right"))  # the first position with cdf > u * Z
        if i == V:
            i = int(np.flatnonzero(w > 0)[-1])
        out["tok"][b] = order[i]
        ng = (ph + V + EPV - 1) // EPV
        out["delta"][b] = lse_delta(-(-ng // NT) * EPV, M * LOG2E)
    return LseReplay(**out)


def draw_displacement(tok, u, cdf, order):
    """How far ``u * Z`` lies outside the CDF interval of token ``tok`` (``[cdf before it, cdf at it]``), as a
    fraction of ``Z = cdf[-1]``; 0 inside.  ``inf`` for a token outside the row."""
    pos = np.flatnonzero(order == tok)
    if len(pos) != 1:
        return math.inf
    p = int(pos[0])
    Z = cdf[-1]
    lo = cdf[p - 1] if p else 0.0
    t = u * Z
    return max(lo - t, t - cdf[p], 0.0) / Z


def in_interval(tok, u, cdf, order, delta):
    """The draw check of ``gt_lse_sample``: ``u * Z`` lies inside the drawn token's CDF interval widened by
    ``delta * Z`` on both sides (see ``lse_delta``)."""
    return draw_displacement(tok, u, cdf, order) <= delta


def child_replay(q, u, near_tol=1e-12):
    """The next-symbol draw over one node's children: ``q`` float64 ``[D]``, the terms in child order (0 for padding
    and for children without mass).  Returns ``(j, near)``: the first ``j`` with ``cumsum(q)[j] > u * Z``, else the
    last ``q_j > 0`` (-1 when ``Z`` is not positive and finite); ``near`` marks ``u * Z`` within ``near_tol * Z`` of
    a CDF value, where the kernel's fp64 summation order can decide the child."""
    q = np.asarray(q, dtype=np.float64)
    c = np.cumsum(q)
    Z = c[-1] if len(c) else 0.0
    if not (0.0 < Z < math.inf):
        return -1, False
    t = u * Z
    j = int(np.searchsorted(c, t, side="right"))
    if j == len(q):
        j = int(np.flatnonzero(q > 0)[-1])
    near = bool((np.abs(c - t) <= near_tol * Z).any())
    return j, near

