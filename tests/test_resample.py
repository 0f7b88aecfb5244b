"""Particle resampling (``gt_resample`` / ``smc.resample``).

CPU part: the argument checks of the entry point and their order, and the ``ValueError``s of ``smc.resample`` that need
no device.  GPU part (``-m gpu``): ancestors, effective sample sizes and log mean weights against the fp64 oracle of
``resample_oracle`` over group sizes 1-16384 and 1-512 groups, the properties that hold without the oracle (no dead
ancestor, sorted stratified and systematic ancestors, systematic offspring counts, unbiased offspring), the threshold,
special values beside normal groups, determinism (a group alone, in place, repeated calls, graph replay), the whole
weighted-DFA SMC step with resampling in one CUDA graph, and the Philox stream shared with the sampler.
"""
import ctypes
import math

import numpy as np
import pytest
import torch

import resample_oracle as ro
from genlm_backend_b200 import _lib, smc

METHODS = (ro.MULTINOMIAL, ro.STRATIFIED, ro.SYSTEMATIC)
MAXG = _lib.GT_RESAMPLE_MAX_GROUP


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_entry_point_rejects_bad_arguments_in_order_without_a_gpu():
    lib = _lib.lib
    p = ctypes.c_void_p(1 << 20)  # stands for a device pointer: never dereferenced by the checks

    def call(**kw):
        a = dict(logw=p, G=4, P=8, method=2, thr=0.5, anc=p, out=p, ess=p, lmw=p, res=p)
        a.update(kw)
        rc = lib.gt_resample(a["logw"], a["G"], a["P"], a["method"], a["thr"], 1, 0, a["anc"], a["out"], a["ess"],
                             a["lmw"], a["res"], None)
        return rc, lib.gt_last_error().decode() if rc else ""

    for bad in (dict(G=-1), dict(P=0), dict(P=-3), dict(method=-1), dict(method=3), dict(thr=math.nan), dict(logw=None),
                dict(anc=None), dict(out=None), dict(ess=None), dict(lmw=None), dict(res=None)):
        rc, msg = call(**bad)
        assert rc == 1 and "gt_resample" in msg, bad
    for bad in (dict(P=MAXG + 1), dict(G=(2**31 - 1) // 8 + 1), dict(G=2**40)):
        rc, msg = call(**bad)
        assert rc == 4 and "gt_resample" in msg, bad
    for thr in (0.0, math.inf, -1.0):
        assert call(G=0, thr=thr)[0] == 0
    assert "null pointer" in call(P=MAXG, G=(2**31 - 1) // MAXG, logw=None)[1]  # the largest batch passes the limits
    # the order: scalars (sizes, method, threshold, limits), then no groups, then pointers
    assert "n_groups" in call(G=-1, method=7, thr=math.nan, P=MAXG + 1, logw=None)[1]
    assert "method" in call(method=7, thr=math.nan, P=MAXG + 1, logw=None)[1]
    assert "NaN" in call(thr=math.nan, P=MAXG + 1, logw=None)[1]
    assert call(P=MAXG + 1, G=0, logw=None)[0] == 4
    assert call(G=2**40, logw=None)[0] == 4
    assert call(G=0, logw=None, anc=None, out=None, ess=None, lmw=None, res=None) == (0, "")
    assert "null pointer" in call(res=None)[1]


def test_oracle_philox_matches_the_random123_known_answers():
    for ctr, key, want in (((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
                           ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
                           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
                            (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))):
        assert tuple(int(x) for x in ro.philox4x32_10(*ctr, *key)) == want


def test_python_rejects_bad_inputs_without_a_gpu():
    ok = torch.zeros(4, 8)
    with pytest.raises(ValueError, match="method"):
        smc.resample(ok, method="residual")
    for bad in (torch.tensor(0.0), torch.zeros(2, 3, 4), torch.zeros(2, MAXG + 1), torch.zeros(3, 0),
                torch.zeros(4, 8, dtype=torch.int32), np.zeros((4, 8), np.float32), ok):  # ok: not on a CUDA device
        with pytest.raises(ValueError):
            smc.resample(bad)


# ---- GPU ---------------------------------------------------------------------------------------------------------
def skewed(G, P, seed, dead=0.1):
    """Normal log-weights (scale 2) with a share of dead (-inf) particles; every group keeps a live one."""
    rng = np.random.default_rng(seed)
    lw = (rng.normal(size=(G, P)) * 2).astype(np.float32)
    lw[rng.random((G, P)) < dead] = -np.inf
    lw[np.arange(G), rng.integers(0, P, G)] = rng.normal(size=G).astype(np.float32)
    return lw


def run(lw, method, thr, seed=0, offset=0):
    out = smc.resample(torch.tensor(lw).cuda(), method, thr, seed=seed, offset=offset)
    return [x.cpu().numpy() for x in out]


def within_one_ulp(have, want):
    have, want = np.asarray(have, np.float32), np.asarray(want, np.float32)
    same = (have == want) | (np.isnan(have) & np.isnan(want))
    fin = np.isfinite(want) & np.isfinite(have)
    close = np.zeros_like(same)
    close[fin] = np.abs(have[fin].astype(np.float64) - want[fin]) <= np.spacing(np.abs(want[fin]))
    return bool((same | close).all())


def check_ancestors(anc, want, near):
    """Equal to the oracle except at points within 1e-12 * S of a CDF value, which must be rare."""
    diff = anc != want
    assert not (diff & ~near).any(), np.argwhere(diff & ~near)[:5]
    assert near.sum() <= max(2, near.size // 10000), near.sum()


@pytest.mark.gpu
@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("G", [1, 3, 512])
@pytest.mark.parametrize("P", [1, 2, 7, 32, 33, 1000, 4096, 16384])
def test_matches_oracle_and_properties(P, G, method):
    lw = skewed(G, P, seed=P * 7 + G)
    seed, offset = 1234 + G, 99 * P
    anc, out, ess, lmw, res = run(lw, method, math.inf, seed, offset)
    w_anc, w_out, w_ess, w_lmw, w_res, near = ro.resample(lw, method, math.inf, seed, offset)
    assert anc.shape == (G, P) and anc.dtype == np.int32 and out.dtype == np.float32
    assert ess.shape == lmw.shape == res.shape == (G,) and res.dtype == bool
    assert within_one_ulp(ess, w_ess) and within_one_ulp(lmw, w_lmw)
    assert np.array_equal(res, w_res) and res.all()  # threshold inf: every live group resamples
    check_ancestors(anc, w_anc, near)
    assert np.array_equal(out, np.broadcast_to(lmw[:, None], (G, P)))
    # without the oracle: a dead particle is never an ancestor, ancestors stay in their group
    flat = lw.reshape(-1)
    assert np.isfinite(flat[anc.reshape(-1)]).all()
    assert ((anc // P) == np.arange(G)[:, None]).all()
    if method != ro.MULTINOMIAL:
        assert (np.diff(anc, axis=1) >= 0).all()
    if method == ro.SYSTEMATIC:
        w = np.exp(lw.astype(np.float64) - lw.max(axis=1, keepdims=True))
        expect = P * w / w.sum(axis=1, keepdims=True)
        counts = np.stack([np.bincount(a - g * P, minlength=P) for g, a in enumerate(anc)])
        slack = near.any(axis=1, keepdims=True) * 1  # the near-boundary exception moves at most one offspring
        assert ((counts >= np.floor(expect - 1e-7) - slack) & (counts <= np.ceil(expect + 1e-7) + slack)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("method", METHODS)
def test_mean_offspring_counts_are_unbiased(method):
    """z-test per particle over G groups x K offsets of the same weights: the mean offspring count of particle i is
    P * w_i / S.  The variance per draw is bounded by P w (1 - w) (multinomial; stratified has no more) and by
    f (1 - f), f = frac(P w), for systematic; |z| < 5 for all P particles (a false alarm below 1e-4 in all)."""
    G, P, K = 256, 64, 40
    row = skewed(1, P, seed=5, dead=0.2)[0]
    lw = np.tile(row, (G, 1))
    w = np.exp(row.astype(np.float64) - row.max())
    wb = w / w.sum()
    counts = np.zeros(P)
    for k in range(K):
        anc, *_ = run(lw, method, math.inf, seed=17, offset=k * G * P)
        counts += np.bincount((anc - np.arange(G)[:, None] * P).reshape(-1), minlength=P)
    n = G * K
    mean = P * wb
    if method == ro.SYSTEMATIC:
        f = mean - np.floor(mean)
        var = f * (1 - f)
    else:
        var = P * wb * (1 - wb)
    assert counts[wb == 0].sum() == 0
    live = var > 0
    z = (counts[live] / n - mean[live]) / np.sqrt(var[live] / n)
    assert np.abs(z).max() < 5, z
    assert np.array_equal(counts[~live & (wb > 0)], n * mean[~live & (wb > 0)])  # an integral P w: exactly that many


@pytest.mark.gpu
def test_threshold():
    G, P = 64, 256
    rng = np.random.default_rng(3)
    lw = (rng.normal(size=(G, P)) * rng.uniform(0, 3, (G, 1))).astype(np.float32)  # ESS from ~P down to a few
    for method in METHODS:
        anc, out, ess, lmw, res = run(lw, method, 0.5, seed=2)
        w_anc, w_out, w_ess, w_lmw, w_res, near = ro.resample(lw, method, 0.5, seed=2)
        away = np.abs(w_ess.astype(np.float64) - 0.5 * P) > 1e-5 * P
        assert 8 < res.sum() < G - 8
        assert np.array_equal(res[away], w_res[away])
        keep = ~res
        assert np.array_equal(anc[keep], (np.arange(G)[:, None] * P + np.arange(P))[keep])
        assert np.array_equal(out[keep].view(np.uint32), lw[keep].view(np.uint32))
        sel = res & w_res
        check_ancestors(anc[sel], w_anc[sel], near[sel])
        assert run(lw, method, math.inf)[4].all()
        never = run(lw, method, 0.0)
        assert not never[4].any() and np.array_equal(never[1].view(np.uint32), lw.view(np.uint32))
    uni = np.full((3, 100), -1.5, dtype=np.float32)
    anc, out, ess, lmw, res = run(uni, ro.SYSTEMATIC, 1.0)
    assert (ess == 100).all() and not res.any() and np.array_equal(out, uni)
    assert np.allclose(lmw, -1.5, rtol=0, atol=1e-6)


@pytest.mark.gpu
def test_special_values_beside_normal_groups():
    P = 33
    lw = skewed(6, P, seed=8)
    lw[1, 5] = np.nan
    lw[2, 7] = np.inf
    lw[3] = -np.inf
    lw[4, 3], lw[4, 9] = np.nan, np.inf  # NaN wins over +inf
    for method in METHODS:
        anc, out, ess, lmw, res = run(lw, method, math.inf, seed=4)
        assert np.isnan(ess[1]) and np.isnan(lmw[1])
        assert np.isnan(ess[2]) and lmw[2] == np.inf
        assert ess[3] == 0 and lmw[3] == -np.inf
        assert np.isnan(ess[4]) and np.isnan(lmw[4])
        assert not res[1:5].any() and res[0] and res[5]
        ident = np.arange(P)[None, :] + np.arange(1, 5)[:, None] * P
        assert np.array_equal(anc[1:5], ident)
        assert np.array_equal(out[1:5].view(np.uint32), lw[1:5].view(np.uint32))
        alone = [run(lw[g:g + 1], method, math.inf, seed=4, offset=g * P) for g in (0, 5)]
        for g, a in zip((0, 5), alone):
            assert np.array_equal(anc[g], a[0][0] + g * P) and np.array_equal(out[g], a[1][0])
            assert np.array_equal(ess[g:g + 1], a[2]) and np.array_equal(lmw[g:g + 1], a[3])


@pytest.mark.gpu
@pytest.mark.parametrize("P", [7, 1000, 16384])
def test_determinism(P):
    G = 5
    lw = skewed(G, P, seed=P)
    x = torch.tensor(lw).cuda()
    for method in METHODS:
        ref = smc.resample(x, method, 0.9, seed=3, offset=11)
        for g in range(G):  # a group alone at offset + g * P, whatever the other groups hold
            anc, out, ess, lmw, res = smc.resample(x[g], method, 0.9, seed=3, offset=11 + g * P)
            assert torch.equal(anc + g * P, ref[0][g]) and torch.equal(out, ref[1][g])  # ancestors: flat indices
            for have, want in zip((ess, lmw, res), ref[2:]):
                assert torch.equal(have, want[g:g + 1])
        y = x.clone()
        y[1:] = torch.tensor(skewed(G - 1, P, seed=P + 1)).cuda()
        mixed = smc.resample(y, method, 0.9, seed=3, offset=11)
        for have, want in zip(mixed, ref):
            assert torch.equal(have[0], want[0])
        for _ in range(3):
            for have, want in zip(smc.resample(x, method, 0.9, seed=3, offset=11), ref):
                assert torch.equal(have, want)
        # in place: logw_out == logw
        z = x.clone()
        anc, ess, lmw, res = (torch.empty_like(ref[0]), torch.empty_like(ref[2]), torch.empty_like(ref[3]),
                              torch.empty(G, dtype=torch.bool, device="cuda"))
        rc = _lib.lib.gt_resample(z.data_ptr(), G, P, smc._RESAMPLE_METHODS[method], 0.9, 3, 11, anc.data_ptr(),
                                  z.data_ptr(), ess.data_ptr(), lmw.data_ptr(), res.data_ptr(),
                                  torch.cuda.current_stream().cuda_stream)
        assert rc == 0
        for have, want in zip((anc, z, ess, lmw, res), ref):
            assert torch.equal(have, want)
    # graph replay
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        smc.resample(x, "stratified", 0.9, seed=3, offset=11)  # warm-up: the shared-memory opt-in is not captured
    stream.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        cap = smc.resample(x, "stratified", 0.9, seed=3, offset=11)
    want = smc.resample(x, "stratified", 0.9, seed=3, offset=11)
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        for have, w in zip(cap, want):
            assert torch.equal(have, w)


def smc_step(trie, delta, logw, states, nodes, logp, log_weights, G, seed, offset):
    """The weighted-DFA step of DESIGN section 5.12 followed by resampling and reindexing."""
    B = logp.shape[0]
    tokw = trie.dfa_token_logw(delta, logw, states, nodes)
    logZ, tok = smc.masked_logsumexp_sample(logp, tokw, seed=seed, offset=offset)
    q = trie.dfa_advance(delta, states, tok, nodes)
    lw = log_weights + logZ
    anc, lw, ess, lmw, res = smc.resample(lw.view(G, B // G), "systematic", 0.5, seed=seed, offset=offset)
    idx = anc.view(-1)
    return q.index_select(0, idx), nodes.index_select(0, idx), tok.index_select(0, idx), lw.view(-1), ess, lmw, res


@pytest.mark.gpu
def test_weighted_dfa_step_with_resampling_in_one_cuda_graph():
    from test_dfa_logw import cuda, step_inputs

    trie, delta, logw, nodes, states, logp = step_inputs(21, 256, table=1)
    d, w, st, nd = cuda(delta, logw, states, nodes)
    G = 8
    lw0 = torch.tensor((np.random.default_rng(2).normal(size=256) * 2).astype(np.float32)).cuda()
    eager = smc_step(trie, d, w, st, nd, logp, lw0, G, seed=5, offset=512)
    assert eager[6].any()
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        smc_step(trie, d, w, st, nd, logp, lw0, G, seed=5, offset=512)
    stream.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        out = smc_step(trie, d, w, st, nd, logp, lw0, G, seed=5, offset=512)
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        for have, want in zip(out, eager):
            assert torch.equal(have, want)


@pytest.mark.gpu
def test_sampler_seed_and_offset_give_an_independent_stream():
    G, P, seed, offset = 16, 128, 77, 4096
    lw = skewed(G, P, seed=9)
    for method in METHODS:
        anc = run(lw, method, math.inf, seed, offset)[0]
        want1, *_, near1 = ro.resample(lw, method, math.inf, seed, offset, stream=1)
        want0 = ro.resample(lw, method, math.inf, seed, offset, stream=0)[0]
        check_ancestors(anc, want1, near1)
        assert (anc != want0).any()
    # the oracle's stream 0 is the sampler's: over 8 equal tokens (one 16-byte group per thread, in token order) row b
    # draws token floor(8 u) for the uniform at counter offset + b
    rows = 64
    logp = torch.full((rows, 8), -math.log(8)).cuda()
    tok = smc.masked_logsumexp_sample(logp, seed=seed, offset=offset)[1].cpu().numpy()
    u0 = ro.uniforms(seed, offset + np.arange(rows, dtype=np.uint64), stream=0)
    assert np.array_equal(tok, np.floor(u0 * 8).astype(np.int64))
