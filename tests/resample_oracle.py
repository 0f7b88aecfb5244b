"""numpy restatement of ``gt_resample``: Philox4x32-10 uniforms with the resampler's counter layout, and the fp64
definition of the effective sample size and the ancestors with a sequential CDF (``include/genlm_trie_b200.h``)."""
import numpy as np

MULTINOMIAL, STRATIFIED, SYSTEMATIC = "multinomial", "stratified", "systematic"
_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 of uint32 counter words (arrays broadcast) under the key (k0, k1)."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & _M32 for c in (c0, c1, c2, c3))
    k0, k1 = np.uint64(k0) & _M32, np.uint64(k1) & _M32
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _M32
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & _M32, (k1 + np.uint64(0xBB67AE85)) & _M32
    return c0, c1, c2, c3


def uniforms(seed, counters, stream=1):
    """53-bit uniforms in [0, 1) for the counters (first two words), ``stream`` in the third word, key ``seed``.
    ``stream=0`` is the samplers' stream, ``stream=1`` the resampler's."""
    ctr = np.asarray(counters, dtype=np.uint64)
    seed = np.uint64(seed)
    r0, r1, _, _ = philox4x32_10(ctr & _M32, ctr >> np.uint64(32), np.full(ctr.shape, stream, np.uint64), 0,
                                 seed & _M32, seed >> np.uint64(32))
    bits = ((r0 >> np.uint64(5)) << np.uint64(26)) | (r1 >> np.uint64(6))
    return bits.astype(np.float64) * (1.0 / 9007199254740992.0)


def resample(logw, method, ess_threshold, seed=0, offset=0, stream=1):
    """``logw`` float32 ``[G, P]``.  Returns ``(ancestors, logw_out, ess, log_mean_w, resampled, near)``; ``near[g, j]``
    marks a point within ``1e-12 * S`` of a CDF value, where the summation order can decide the ancestor."""
    logw = np.asarray(logw, dtype=np.float32)
    G, P = logw.shape
    anc = np.tile(np.arange(P, dtype=np.int64), (G, 1)) + np.arange(G, dtype=np.int64)[:, None] * P
    out = logw.copy()
    ess = np.zeros(G, dtype=np.float32)
    lmw = np.zeros(G, dtype=np.float32)
    res = np.zeros(G, dtype=bool)
    near = np.zeros((G, P), dtype=bool)
    thr = np.float64(np.float32(ess_threshold)) * P
    j = np.arange(P, dtype=np.float64)
    for g in range(G):
        lw = logw[g]
        if np.isnan(lw).any():
            ess[g], lmw[g] = np.nan, np.nan
            continue
        if (lw == np.inf).any():
            ess[g], lmw[g] = np.nan, np.inf
            continue
        if (lw == -np.inf).all():
            ess[g], lmw[g] = 0.0, -np.inf
            continue
        m = np.float64(lw.max())
        w = np.exp(lw.astype(np.float64) - m)
        c = np.cumsum(w)  # sequential
        S, Q = c[-1], np.sum(w * w)
        e = S * S / Q
        ess[g] = np.float32(e)
        lmw[g] = np.float32(m + np.log(S) - np.log(np.float64(P)))
        if not e < thr:
            continue
        res[g] = True
        ctr = np.uint64(offset) + np.uint64(g * P) + np.arange(P, dtype=np.uint64)
        if method == MULTINOMIAL:
            t = uniforms(seed, ctr, stream) * S
        elif method == STRATIFIED:
            t = (j + uniforms(seed, ctr, stream)) / P * S
        elif method == SYSTEMATIC:
            t = (j + uniforms(seed, ctr[:1], stream)[0]) / P * S
        else:
            raise ValueError(method)
        i = np.searchsorted(c, t, side="right")  # the first index with c_i > t
        i[i == P] = np.flatnonzero(w > 0)[-1]
        anc[g] = g * P + i
        out[g] = lmw[g]
        k = np.clip(np.searchsorted(c, t), 0, P - 1)
        near[g] = (np.abs(c[k] - t) <= 1e-12 * S) | (np.abs(c[np.maximum(k - 1, 0)] - t) <= 1e-12 * S)
    return anc, out, ess, lmw, res, near
