"""GPU tests of the fused masked logsumexp + categorical draw (csrc/sampler_kernels.cu).

logZ is pinned against torch.logsumexp in float64 (golden, and the numpy float64 oracle); the draw has no
result-pinning test in the reference ("parity unpinned"), so it is checked by chi-square goodness of fit
against the exact probabilities and by a two-sample chi-square against a stored torch.multinomial histogram.
tests/test_draw_replay.py replays every draw exactly against its Philox uniform and an fp64 inverse CDF.
"""
import numpy as np
import pytest
import torch
from scipy import stats

import oracle
from genlm_backend_b200 import smc
from genlm_backend_b200.synthetic import logsoftmax_rows, bernoulli_log_mask
from helpers import load_golden

pytestmark = pytest.mark.gpu


def test_logZ_matches_torch_float64_golden():
    g = load_golden("sampler")
    logp, mask = torch.tensor(g["logp"]).cuda(), torch.tensor(g["mask"]).cuda()
    logZ, tok = smc.masked_logsumexp_sample(logp, mask, seed=1)
    np.testing.assert_allclose(logZ.cpu().numpy(), g["logZ"], rtol=1e-5, atol=1e-6)
    logZ_T, _ = smc.masked_logsumexp_sample(logp, mask, temperature=0.7, seed=1)
    np.testing.assert_allclose(logZ_T.cpu().numpy(), g["logZ_T07"], rtol=1e-5, atol=1e-6)
    tok = tok.cpu().numpy()
    assert np.isfinite(g["mask"][np.arange(4), tok]).all()  # never a masked-out token


@pytest.mark.parametrize("V", [128256, 151665, 1000, 37])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_logZ_against_oracle(V, dtype):
    B = 6
    logp = torch.tensor(logsoftmax_rows(B, V, seed=V % 97)).to(dtype)
    mask = bernoulli_log_mask(B, V, p=0.3, seed=2)
    as32 = logp.to(torch.float32).numpy()
    want = oracle.masked_logsumexp(as32, mask)
    for kind in ("add", "bool", "bits", "shared", "none"):
        if kind == "add":
            m, w = torch.tensor(mask).cuda(), want
        elif kind == "bool":
            m, w = torch.tensor(np.isfinite(mask)).cuda(), want
        elif kind == "bits":
            keep = np.isfinite(mask)
            pad = np.zeros((B, (V + 31) // 32 * 32), dtype=bool)
            pad[:, :V] = keep
            words = np.packbits(pad.reshape(B, -1, 32), axis=-1, bitorder="little").view(np.uint32).reshape(B, -1)
            m, w = torch.tensor(words.view(np.int32)).cuda(), want
        elif kind == "shared":
            m, w = torch.tensor(mask[0]).cuda(), oracle.masked_logsumexp(as32, mask[0][None, :])
        else:
            m, w = None, oracle.masked_logsumexp(as32)
        logZ, tok = smc.masked_logsumexp_sample(logp.cuda(), m, seed=3)
        got = logZ.cpu().numpy().astype(np.float64)
        # north star: fp32 relative 1e-5.  The unmasked rows have logZ ~ 0 (+- the fp32 rounding of the log-softmax
        # inputs), where only an absolute bound means anything: 1e-6.
        err = np.abs(got - w)
        print(f"logZ V={V} {str(dtype).split('.')[-1]} {kind}: max |dlogZ| = {err.max():.3g}, max rel = {(err / np.maximum(np.abs(w), 1e-30)).max():.3g}")
        np.testing.assert_allclose(got, w, rtol=1e-5, atol=1e-6)
        tok = tok.cpu().numpy()
        assert ((tok >= 0) & (tok < V)).all()
        if kind in ("add", "bool", "bits"):
            assert np.isfinite(mask[np.arange(B), tok]).all()


def test_rows_without_mass_and_nan():
    V = 5000
    logp = torch.tensor(logsoftmax_rows(3, V, seed=1)).cuda()
    mask = torch.zeros((3, V), device="cuda")
    mask[1] = -float("inf")
    logZ, tok = smc.masked_logsumexp_sample(logp, mask, seed=0)
    assert float(logZ[1]) == -float("inf") and int(tok[1]) == -1
    assert int(tok[0]) >= 0 and int(tok[2]) >= 0
    with pytest.raises(RuntimeError, match="invalid multinomial distribution"):
        smc.masked_logsumexp_sample(logp, mask, seed=0, check_valid=True)
    logp[2, 17] = float("nan")
    logZ, tok = smc.masked_logsumexp_sample(logp, None, seed=0)
    assert np.isnan(float(logZ[2])) and int(tok[2]) == -1
    # a NaN at an allowed position of an otherwise fully masked stretch (sparse SMC masks): torch gives logZ = NaN and
    # multinomial raises; so do we, for every mask kind, wherever in the row the NaN sits
    for pos in (17, 2500, V - 1):
        lp = torch.tensor(logsoftmax_rows(2, V, seed=3)).cuda()
        lp[1, pos] = float("nan")
        keep = torch.zeros((2, V), dtype=torch.bool, device="cuda")
        keep[:, pos] = True
        keep[0, 100] = True
        add = torch.where(keep, 0.0, -float("inf"))
        want = (lp.double() + add.double()).logsumexp(-1)
        for m in (add, keep, add[1]):
            logZ, tok = smc.masked_logsumexp_sample(lp, m, seed=1)
            assert np.isnan(float(logZ[1])) and int(tok[1]) == -1, (pos, m.dtype, m.dim())
            if m.dim() == 2:
                assert abs(float(logZ[0]) - float(want[0])) <= 1e-5 * abs(float(want[0])) and int(tok[0]) in (pos, 100)
        with pytest.raises(RuntimeError, match="nan"):
            smc.masked_logsumexp_sample(lp, add, seed=1, check_valid=True)
    # a single allowed token is always drawn
    mask = torch.full((1, V), -float("inf"), device="cuda")
    mask[0, 4321] = 0.0
    logZ, tok = smc.masked_logsumexp_sample(logp[:1], mask, seed=5)
    assert int(tok[0]) == 4321
    np.testing.assert_allclose(float(logZ[0]), float(logp[0, 4321]), rtol=1e-6)


def test_seed_and_offset_discipline():
    V, B = 3000, 64
    logp = torch.tensor(logsoftmax_rows(1, V, seed=4)).cuda().expand(B, V).contiguous()
    _, a = smc.masked_logsumexp_sample(logp, None, seed=11, offset=0)
    _, b = smc.masked_logsumexp_sample(logp, None, seed=11, offset=0)
    _, c = smc.masked_logsumexp_sample(logp, None, seed=12, offset=0)
    _, d = smc.masked_logsumexp_sample(logp[:32], None, seed=11, offset=32)
    assert torch.equal(a, b)            # deterministic
    assert not torch.equal(a, c)        # seed matters
    assert torch.equal(a[32:], d)       # row b of a call uses counter offset + b


def _draws(logp_row, mask_row, n_calls, rows, seed):
    V = logp_row.shape[0]
    logp = torch.tensor(logp_row).cuda().expand(rows, V).contiguous()
    mask = torch.tensor(mask_row).cuda()
    counts = np.zeros(V, dtype=np.int64)
    for k in range(n_calls):
        _, tok = smc.masked_logsumexp_sample(logp, mask, seed=seed, offset=k * rows)
        counts += np.bincount(tok.cpu().numpy(), minlength=V)
    return counts


def test_chi_square_against_exact_probabilities_and_torch_multinomial():
    g = load_golden("sampler")
    logp, mask = g["logp"][0], g["mask"][0]
    n_calls, rows = 50, 4096
    counts = _draws(logp, mask, n_calls, rows, seed=2024)
    n = n_calls * rows
    p = oracle.masked_probs(logp[None, :], mask[None, :])[0]
    assert counts[p == 0].sum() == 0
    # goodness of fit, bins merged to expected >= 5
    order = np.argsort(p)
    exp_sorted, obs_sorted = (p * n)[order], counts[order]
    bins_e, bins_o, ce, co = [], [], 0.0, 0
    for e, o in zip(exp_sorted, obs_sorted):
        ce, co = ce + e, co + o
        if ce >= 5:
            bins_e.append(ce); bins_o.append(co); ce, co = 0.0, 0
    bins_e[-1] += ce; bins_o[-1] += co
    chi, pval = stats.chisquare(bins_o, np.array(bins_e) * (sum(bins_o) / sum(bins_e)))
    assert pval > 1e-4, (chi, pval)
    # two-sample test against torch.multinomial's histogram for the same row (200,000 reference draws)
    ref = g["multinomial_counts_row0"]
    keep = (counts + ref) >= 10
    table = np.stack([np.append(counts[keep], counts[~keep].sum()), np.append(ref[keep], ref[~keep].sum())])
    table = table[:, table.sum(0) > 0]
    chi2, pval2, _, _ = stats.chi2_contingency(table)
    assert pval2 > 1e-4, (chi2, pval2)


def test_full_size_rows_are_sampled_in_proportion():
    """BASELINE config 4 shape (V=128,256): the empirical mass of coarse vocabulary slices matches the oracle."""
    V, rows = 128256, 4096
    logp = logsoftmax_rows(1, V, seed=9)[0]
    mask = bernoulli_log_mask(1, V, p=0.5, seed=10)[0]
    counts = _draws(logp, mask, 8, rows, seed=77)
    p = oracle.masked_probs(logp[None, :], mask[None, :])[0]
    assert counts[p == 0].sum() == 0
    n = counts.sum()
    edges = np.linspace(0, V, 65).astype(int)
    obs = np.add.reduceat(counts, edges[:-1])
    exp = np.add.reduceat(p, edges[:-1]) * n
    chi, pval = stats.chisquare(obs, exp * (obs.sum() / exp.sum()))
    assert pval > 1e-4, (chi, pval)


@pytest.mark.parametrize("V,dtype", [(300_001, torch.float32), (140_003, torch.float64), (600_011, torch.bfloat16)])
def test_rows_longer_than_one_candidate_per_thread(V, dtype):
    """Rows with more 16-byte groups than threads^2: the second pass gives a thread several candidate groups.
    Point masses must be drawn exactly wherever they sit, and a two-point row splits in proportion."""
    rng = np.random.default_rng(V)
    spots = [0, 1, V // 2, V - 5, V - 1] + rng.integers(0, V, 11).tolist()
    logp = torch.full((len(spots) + 1, V), float("-inf"), dtype=dtype)
    for b, i in enumerate(spots):
        logp[b, i] = -0.25
    a, c = V // 3, V - 2  # 1/4 : 3/4
    logp[-1, a], logp[-1, c] = np.log(0.25), np.log(0.75)
    dev = logp.cuda()
    logZ, tok = smc.masked_logsumexp_sample(dev, None, seed=11)
    assert tok.cpu().numpy()[:-1].tolist() == spots
    np.testing.assert_allclose(logZ.cpu().numpy()[:-1], -0.25, atol=2e-3 if dtype == torch.bfloat16 else 1e-6)
    two = dev[-1:].repeat(512, 1)
    draws = np.concatenate([smc.masked_logsumexp_sample(two, None, seed=5, offset=512 * i)[1].cpu().numpy() for i in range(32)])
    assert set(np.unique(draws)) == {a, c}
    frac = (draws == c).mean()
    assert abs(frac - 0.75) < 5 * np.sqrt(0.75 * 0.25 / len(draws))  # 5 sigma
    # a dense row of this length: logZ against the float64 oracle
    dense = torch.tensor(logsoftmax_rows(2, V, seed=3)).to(dtype)
    lz, tk = smc.masked_logsumexp_sample(dense.cuda(), None, seed=1)
    np.testing.assert_allclose(lz.cpu().numpy(), oracle.masked_logsumexp(dense.to(torch.float64).numpy()), rtol=1e-5, atol=2e-5)
    assert ((tk.cpu().numpy() >= 0) & (tk.cpu().numpy() < V)).all()


def test_shared_additive_mask_cache_follows_the_tensor():
    """Shared {0, -inf} additive masks are packed into bit masks once per tensor object and version: a new tensor at a
    recycled address, an in-place edit and a general additive mask must all give the plain additive results."""
    V, B = 4099, 8
    logp = torch.tensor(logsoftmax_rows(B, V, seed=2)).cuda()

    def want(mask):
        return (logp.double() + mask.double()).logsumexp(-1).cpu().numpy()

    for seed in range(6):  # fresh tensors: the caching allocator hands out the same address again
        m = torch.tensor(bernoulli_log_mask(1, V, p=0.4, seed=seed)[0]).cuda()
        for _ in range(2):
            logZ, tok = smc.masked_logsumexp_sample(logp, m, seed=seed)
            np.testing.assert_allclose(logZ.cpu().numpy(), want(m), rtol=1e-5, atol=1e-6)
            assert torch.isfinite(m[tok.long()]).all()
        del m
    m = torch.tensor(bernoulli_log_mask(1, V, p=0.4, seed=9)[0]).cuda()
    smc.masked_logsumexp_sample(logp, m, seed=1)
    m[:2000] = -float("inf")  # in-place edit: version changes, packed again
    logZ, tok = smc.masked_logsumexp_sample(logp, m, seed=1)
    np.testing.assert_allclose(logZ.cpu().numpy(), want(m), rtol=1e-5, atol=1e-6)
    assert int(tok.min()) >= 2000
    soft = torch.where(torch.isfinite(m), 0.0, -3.0)  # not a {0, -inf} mask: stays additive
    logZ, _ = smc.masked_logsumexp_sample(logp, soft, seed=1)
    np.testing.assert_allclose(logZ.cpu().numpy(), want(soft), rtol=1e-5, atol=1e-6)
