"""Exact replay of the draws against the Philox stream and an fp64 inverse CDF (``draw_oracle``).

``gt_lse_sample`` is replayed over its input types, mask kinds (and the scalar / vector mask paths), row phases,
temperatures and rows longer than ``NT**2`` groups: each draw must fall in the drawn token's fp64 CDF interval,
widened by the ``lse_delta`` bound of the kernel's fp32 arithmetic, and ``logZ`` must match fp64.  A chi-square test
at other temperatures stays as the order-independent backstop, and ``+inf`` logits are pinned against
``torch.logsumexp``.  The next-symbol draws are replayed child for child.  The order and the oracle run without a GPU.
"""
import math

import numpy as np
import pytest
import torch

import child_oracle
import draw_oracle
import oracle
import symbol_oracle
from draw_oracle import child_replay, draw_displacement, lse_draw_order, lse_replay, sampler_threads
from genlm_backend_b200 import ParallelTokenCharacterTrie, smc
from genlm_backend_b200.synthetic import dirichlet_rows, logsoftmax_rows
from helpers import depth1_node, golden_vocab, load_golden, trie_layout
from resample_oracle import uniforms


# ---- CPU ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("NT", [256, 512])
@pytest.mark.parametrize("EPV", [2, 4, 8])
def test_lse_draw_order_is_a_permutation(NT, EPV):
    for V in sorted({1, 2, EPV - 1, EPV, EPV + 1, 37, 4099, NT * NT * EPV - 1, NT * NT * EPV + EPV + 1}):
        for phase in range(EPV):
            order = lse_draw_order(V, phase, EPV, NT)
            assert len(order) == V and np.array_equal(np.sort(order), np.arange(V)), (V, phase)
    # the walk of a short row: thread t's groups t, t + NT, ... in increasing order, element by element
    V, phase = 3 * NT * EPV, 1
    order = lse_draw_order(V, phase, EPV, NT)
    first = [g * EPV - phase + k for g in (0, NT, 2 * NT, 3 * NT) for k in range(EPV) if 0 <= g * EPV - phase + k < V]
    assert order[:len(first)].tolist() == first
    # a long row: the picked thread's candidates c go sub-thread by sub-thread (c % NT), then c // NT
    V = (NT * NT + 2 * NT) * EPV
    order = lse_draw_order(V, 0, EPV, NT)
    assert (order[::EPV][:4] // EPV).tolist() == [0, NT * NT, NT, NT * NT + NT]


def test_sampler_threads_follow_the_launch():
    assert sampler_threads(torch.bfloat16, "add") == sampler_threads(np.float16, "add") == 512
    for dt in (np.float32, np.float64, torch.float16, torch.bfloat16):
        for kind in ("none", "bool", "bits"):
            assert sampler_threads(dt, kind) == 256
    assert sampler_threads(torch.float32, "add") == sampler_threads(torch.float64, "add") == 256


def test_replay_reproduces_the_equal_token_pin():
    """Eight equal fp32 tokens are two groups of threads 0 and 1: the draw is token ``floor(8 u)``."""
    rows, seed, offset = 64, 77, 4096
    r = lse_replay(np.full((rows, 8), -math.log(8), dtype=np.float32), seed=seed, offset=offset)
    u = uniforms(seed, offset + np.arange(rows, dtype=np.uint64), stream=0)
    assert np.array_equal(r.tok, np.floor(8 * u).astype(np.int64))
    np.testing.assert_allclose(r.logZ, 0.0, atol=1e-7)  # -log(8) rounded to fp32
    for b in range(rows):
        assert draw_displacement(r.tok[b], u[b], r.cdf[b], r.order[b]) == 0.0
        assert draw_displacement((r.tok[b] + 4) % 8, u[b], r.cdf[b], r.order[b]) >= 0.375 - 1e-12  # 3 tokens away


def test_replay_of_masks_temperature_phases_and_special_rows():
    V = 41
    rng = np.random.default_rng(3)
    logp = rng.normal(0, 3, (5, V)).astype(np.float32)
    keep = rng.random((5, V)) < 0.5
    keep[3] = False
    logp[4, 7] = np.nan
    add = np.where(keep, rng.normal(0, 1, (5, V)), -np.inf).astype(np.float32)
    for kind, mask, T in (("bool", keep, 0.7), ("add", add, 0.05), ("bits", keep, 2.0)):
        r = lse_replay(logp, mask, kind, temperature=T, seed=5, phases=[0, 1, 2, 3, 1], dtype=np.float32)
        x = logp.astype(np.float64) / T + (add if kind == "add" else np.where(keep, 0.0, -np.inf))
        np.testing.assert_allclose(r.logZ[:3], oracle.masked_logsumexp(x[:3]), rtol=1e-14)
        assert r.logZ[3] == -np.inf and r.tok[3] == -1 and np.isnan(r.logZ[4]) == keep[4, 7]
        for b in range(3):
            assert mask[b, r.tok[b]] if kind != "add" else np.isfinite(add[b, r.tok[b]])
            assert sorted(r.order[b].tolist()) == list(range(V))
            assert np.isclose(r.cdf[b][-1], np.exp(x[b] - x[b].max()).sum())


def test_child_replay_matches_searchsorted():
    rng = np.random.default_rng(1)
    for _ in range(200):
        D = int(rng.integers(1, 40))
        q = rng.random(D) * (rng.random(D) < 0.6)
        q[rng.integers(0, D)] = rng.random() + 0.1  # some mass
        u = rng.random()
        j, near = child_replay(q, u)
        c = np.cumsum(q)
        assert j == int(np.searchsorted(c, u * c[-1], side="right"))
        assert q[j] > 0  # a zero-mass child is never the first to exceed u * Z
    # hand-made rows: zero-mass children, the fall-back to the last positive child, no mass, a NaN
    q = np.array([0.0, 1.0, 0.0, 3.0, 0.0])
    assert child_replay(q, 0.0)[0] == 1 and child_replay(q, 0.2499)[0] == 1 and child_replay(q, 0.25)[0] == 3
    assert child_replay(q, 1.0 - 1e-17)[0] == 3
    assert child_replay(np.array([0.5, 0.5, 0.0]), np.nextafter(1.0, 0.0))[0] == 1
    assert child_replay(np.array([1.0, 0.0]), 1.0)[0] == 0  # u * Z past the total: the last positive child
    assert child_replay(np.zeros(4), 0.3) == (-1, False)
    assert child_replay(np.array([1.0, np.nan]), 0.3) == (-1, False)
    assert child_replay(np.array([1.0, np.inf]), 0.3) == (-1, False)
    assert child_replay(q, 0.25)[1] and not child_replay(q, 0.3)[1]


# ---- GPU: gt_lse_sample ------------------------------------------------------------------------------------------
DTYPES = {"f32": torch.float32, "f64": torch.float64, "f16": torch.float16, "bf16": torch.bfloat16}
# mask name -> the kernel's mask kind (a shared {0, -inf} float mask is packed into bits)
MASKS = {"none": "none", "add_rows": "add", "add_shared_soft": "add", "add_shared_01": "bits", "bool_rows": "bool",
         "bool_shared": "bool", "bits_rows": "bits", "bits_shared": "bits"}
LAYOUTS = ("contiguous", "padded", "column_offset")
TEMPS = (1.0, 0.7, 0.05)


def row_phases(t):
    """Element offset of each row of the 2-D device tensor ``t`` inside its 16-byte line (as the kernel computes it)."""
    isz = t.element_size()
    ld = t.stride(0) if t.shape[0] > 1 else t.shape[1]
    return np.array([(t.data_ptr() + b * ld * isz) % 16 // isz for b in range(t.shape[0])], dtype=np.int64)


def pack_bits(keep, extra_words=0, offset=0):
    """bool ``[B, V]`` or ``[V]`` -> int32 keep-bitmask, with the bits past ``V`` of the last word set (the kernel
    must ignore them); 2-D masks as a view at column ``offset`` of a buffer ``extra_words`` wider."""
    keep = np.atleast_2d(keep)
    B, V = keep.shape
    W = (V + 31) // 32
    pad = np.ones((B, W * 32), dtype=bool)
    pad[:, :V] = keep
    words = np.packbits(pad.reshape(B, W, 32), axis=-1, bitorder="little").view(np.uint32).reshape(B, W)
    buf = np.zeros((B, W + extra_words), dtype=np.uint32)
    buf[:, offset:offset + W] = words
    return torch.tensor(buf.view(np.int32)).cuda()[:, offset:offset + W]


def offset_view(values, lead, tail, fill):
    """A CUDA view of ``values`` ``[B, V]`` at column ``lead`` of a buffer ``lead + tail`` columns wider, filled with
    ``fill`` elsewhere (so that a read outside the row shows)."""
    B, V = values.shape
    buf = torch.full((B, lead + V + tail), fill, dtype=values.dtype)
    buf[:, lead:lead + V] = values
    return buf.cuda()[:, lead:lead + V]


def lm_logits(rng, V):
    """Raw LM-head-like logits: Zipf-shaped over a random permutation, up to about +30, not log-softmaxed."""
    rank = rng.permutation(V) + 1
    return 30.0 - rng.uniform(1.0, 3.0) * np.log(rank) + 0.3 * rng.standard_normal(V)


def edge_positions(V, phase, EPV):
    """Elements where the kernel's paths meet: the first and last group of the row, bit-word boundaries, the end."""
    g_hi = (phase + V) // EPV
    cand = [0, 1, EPV - phase - 1, EPV - phase, g_hi * EPV - phase - 1, g_hi * EPV - phase, V - 2, V - 1,
            31, 32, 33, 63, 64, 95, 96]
    return sorted({i for i in cand if 0 <= i < V})


def make_rows(rng, B, V, phases, EPV):
    """float64 ``[B, V]``: LM-like logits, sparse supports of 2-64 tokens on edge groups and word straddles (and
    the row's last element), and every eighth row a dense log-softmax row."""
    rows = np.empty((B, V))
    for b in range(B):
        if b % 8 == 7:
            rows[b] = logsoftmax_rows(1, V, seed=int(rng.integers(1 << 30)))[0]
        elif b % 2 == 0:
            rows[b] = lm_logits(rng, V)
        else:
            k = min(V, int(rng.integers(2, 65)))
            edge = edge_positions(V, int(phases[b]), EPV)
            pick = rng.choice(edge, min(len(edge), k // 2 + 1), replace=False).tolist()
            rest = np.setdiff1d(np.arange(V), pick)
            pick += rng.choice(rest, min(len(rest), k - len(pick)), replace=False).tolist()
            rows[b] = -np.inf
            rows[b, pick] = rng.normal(0.0, 3.0, len(pick))
    return rows


def make_mask(name, rng, B, V, layout):
    """``(device mask for the call, the oracle's mask kind, the oracle's mask)``."""
    keep = rng.random((B, V)) < 0.6
    soft = np.where(keep, rng.normal(0.0, 1.0, (B, V)), -np.inf).astype(np.float32)
    per_row_view = layout == "column_offset"
    if name == "none":
        return None, "none", None
    if name == "add_rows":
        dev = offset_view(torch.tensor(soft), 1, 4, float("nan")) if per_row_view else torch.tensor(soft).cuda()
        return dev, "add", soft
    if name == "add_shared_soft":
        return torch.tensor(soft[0]).cuda(), "add", soft[0]
    if name == "add_shared_01":
        return torch.tensor(np.where(keep[0], 0.0, -np.inf).astype(np.float32)).cuda(), "bits", keep[0]
    if name == "bool_rows":
        dev = offset_view(torch.tensor(keep), 3, 4, True) if per_row_view else torch.tensor(keep).cuda()
        return dev, "bool", keep
    if name == "bool_shared":
        return torch.tensor(keep[0]).cuda(), "bool", keep[0]
    if name == "bits_rows":
        return (pack_bits(keep, 3, 1) if per_row_view else pack_bits(keep)), "bits", keep
    assert name == "bits_shared"
    return pack_bits(keep[0])[0], "bits", keep[0]


def make_logits(values, dtype, layout):
    """The rows on the device in ``layout``: contiguous, padded past ``V`` (an LM head wider than the vocabulary,
    ``ld = V + 271``), or a view three columns into a wider buffer; the padding is NaN."""
    t = torch.tensor(values).to(dtype)
    if layout == "contiguous":
        return t.cuda()
    if layout == "padded":
        return offset_view(t, 0, 271, float("nan"))
    return offset_view(t, 3, 10, float("nan"))


class DrawStats:
    def __init__(self):
        self.n = self.exact = self.big = 0
        self.dlogz = self.disp = self.disp_ratio = 0.0

    def merge(self, o):
        self.n, self.exact, self.big = self.n + o.n, self.exact + o.exact, self.big + o.big
        self.dlogz, self.disp = max(self.dlogz, o.dlogz), max(self.disp, o.disp)
        self.disp_ratio = max(self.disp_ratio, o.disp_ratio)

    def line(self):
        return (f"draws {self.n}, exact {self.exact / max(self.n, 1):.4f}, max |dlogZ| {self.dlogz:.3g}, "
                f"max displacement {self.disp:.3g} Z = {self.disp_ratio:.3f} delta")


def check_call(logits_dev, mask_dev, kind, ormask, T, seed, offset, stats, what):
    """One ``masked_logsumexp_sample`` call against ``lse_replay``: logZ, the interval rule, no masked-out token."""
    logZ, tok = smc.masked_logsumexp_sample(logits_dev, mask_dev, temperature=T, seed=seed, offset=offset)
    logZ, tok = logZ.cpu().numpy().astype(np.float64), tok.cpu().numpy()
    as32 = logits_dev.float().cpu().numpy()
    r = lse_replay(as32, ormask, kind, temperature=T, seed=seed, offset=offset, phases=row_phases(logits_dev),
                   dtype=logits_dev.dtype)
    np.testing.assert_allclose(logZ, r.logZ, rtol=1e-5, atol=1e-6, err_msg=what)
    fin = np.isfinite(r.logZ)
    if fin.any():
        stats.dlogz = max(stats.dlogz, float(np.abs(logZ[fin] - r.logZ[fin]).max()))
    assert (tok[~fin] == -1).all(), what
    x = draw_oracle._working_rows(as32, ormask, kind, T)
    for b in np.flatnonzero(fin):
        t = int(tok[b])
        assert 0 <= t < x.shape[1] and x[b, t] > -np.inf, (what, b, t)  # never a masked-out or -inf token
        d = draw_displacement(t, r.u[b], r.cdf[b], r.order[b])
        assert d <= r.delta[b], (what, b, t, int(r.tok[b]), d, r.delta[b])
        stats.n += 1
        stats.exact += t == r.tok[b]
        stats.disp = max(stats.disp, d)
        stats.disp_ratio = max(stats.disp_ratio, d / r.delta[b])
        stats.big += math.exp(x[b, t] - r.logZ[b]) > 10 * r.delta[b]
    return r, tok


def layout_phases(B, V, itemsize, layout):
    """Row phases of ``make_logits(..., layout)`` (device allocations are aligned to 16 bytes and more)."""
    lead, ld = {"contiguous": (0, V), "padded": (0, V + 271), "column_offset": (3, V + 13)}[layout]
    return np.array([(lead + b * ld) * itemsize % 16 // itemsize for b in range(B)])


@pytest.mark.gpu
@pytest.mark.parametrize("mask", list(MASKS))
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_lse_draws_replay_exactly(dtype, mask):
    """Every (type, mask kind, layout, temperature) at V in {1, 5, 37, 4099} (32 rows), and once at 151,665 (8 rows
    of an LM head padded to 151,936 columns, so that rows 1-3 mod 4 take the scalar mask path)."""
    tdt = DTYPES[dtype]
    EPV = 16 // tdt.itemsize
    rng = np.random.default_rng([EPV, list(MASKS).index(mask)])
    seed, offset = int(rng.integers(1 << 40)), 0
    total = DrawStats()
    for layout in LAYOUTS:
        for T in TEMPS:
            st = DrawStats()
            for V in (1, 5, 37, 4099):
                B = 32
                rows = make_rows(rng, B, V, layout_phases(B, V, tdt.itemsize, layout), EPV)
                dev = make_logits(rows, tdt, layout)
                mdev, kind, om = make_mask(mask, rng, B, V, layout)
                check_call(dev, mdev, kind, om, T, seed, offset, st, (dtype, mask, layout, T, V))
                offset += B
            print(f"lse {dtype} {mask} {layout} T={T}: {st.line()}")
            total.merge(st)
    V, B, T = 151665, 8, TEMPS[EPV % 3]
    st = DrawStats()
    dev = offset_view(torch.tensor(make_rows(rng, B, V, np.zeros(B), EPV)).to(tdt), 0, 151936 - V, float("nan"))
    mdev, kind, om = make_mask(mask, rng, B, V, "padded")
    check_call(dev, mdev, kind, om, T, seed, offset, st, (dtype, mask, V))
    print(f"lse {dtype} {mask} V={V} padded T={T}: {st.line()}")
    total.merge(st)
    # the interval check means something only if most draws land on tokens far wider than the tolerance
    assert total.big >= total.n / 2, (total.big, total.n)
    assert total.n > 500


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,kind", [("f32", "bits"), ("f32", "add"), ("bf16", "add"), ("bf16", "bits"),
                                        ("f64", "add"), ("f16", "bool")])
def test_rows_longer_than_nt_squared_groups_under_masks(dtype, kind):
    """Pass 2 with several candidates per sub-thread: point masses at both ends and on group boundaries, two-point
    rows and dense rows, under per-row masks, replayed draw by draw."""
    tdt = DTYPES[dtype]
    EPV = 16 // tdt.itemsize
    NT = sampler_threads(tdt, kind)
    V = NT * NT * EPV + 3 * EPV + 1
    rng = np.random.default_rng(V)
    B = 12
    rows = np.full((B, V), -np.inf)
    ng = NT * NT + 4
    spots = [0, V - 1, EPV, 2 * EPV - 1, NT * NT * EPV - 1, NT * NT * EPV, NT * EPV - 1, V - EPV - 1]
    for b, i in enumerate(spots):
        rows[b, i] = -0.25
    rows[8, [V // 3, V - 2]] = np.log([0.25, 0.75])
    rows[9, [1, ng // 2 * EPV]] = np.log([0.5, 0.5])
    rows[10] = lm_logits(rng, V)
    rows[11] = logsoftmax_rows(1, V, seed=4)[0]
    keep = rng.random((B, V)) < 0.7
    keep[:10][np.isfinite(rows[:10])] = True  # the point masses stay allowed
    dev = offset_view(torch.tensor(rows).to(tdt), 3, 5, float("nan"))  # phase 3 on every row
    if kind == "add":
        om = np.where(keep, rng.normal(0, 1, (B, V)), -np.inf).astype(np.float32)
        mdev = torch.tensor(om).cuda()
    elif kind == "bits":
        om, mdev = keep, pack_bits(keep)
    else:
        om, mdev = keep, torch.tensor(keep).cuda()
    st = DrawStats()
    for k, T in enumerate((1.0, 0.7)):
        r, tok = check_call(dev, mdev, kind, om, T, 99, k * B, st, (dtype, kind, T))
        assert tok[:8].tolist() == spots and r.tok[:8].tolist() == spots
    print(f"long rows {dtype} {kind} V={V} NT={NT}: {st.line()}")


@pytest.mark.gpu
@pytest.mark.parametrize("T", [0.7, 2.0])
def test_chi_square_at_other_temperatures(T):
    """Order-independent backstop: the golden sampler row at T = 0.7 and 2 under every mask kind."""
    from scipy import stats

    g = load_golden("sampler")
    logp, mask = g["logp"][0], g["mask"][0]
    V, rows, n_calls = logp.shape[0], 4096, 12
    keep = np.isfinite(mask)
    dev = torch.tensor(logp).cuda().expand(rows, V).contiguous()
    masks = {"none": (None, None), "add_rows": (torch.tensor(mask).cuda().expand(rows, V).contiguous(), mask),
             "add_shared_01": (torch.tensor(mask).cuda(), mask),
             "bool_rows": (torch.tensor(keep).cuda().expand(rows, V).contiguous(), mask),
             "bits_shared": (pack_bits(keep)[0], mask)}
    for name, (m, om) in masks.items():
        counts = np.zeros(V, dtype=np.int64)
        for k in range(n_calls):
            tok = smc.masked_logsumexp_sample(dev, m, temperature=T, seed=31, offset=k * rows)[1].cpu().numpy()
            counts += np.bincount(tok, minlength=V)
        p = oracle.masked_probs(logp[None, :], None if om is None else om[None, :], temperature=T)[0]
        assert counts[p == 0].sum() == 0, name
        exp = p * counts.sum()
        order = np.argsort(exp)
        be, bo, ce, co = [], [], 0.0, 0
        for e, o in zip(exp[order], counts[order]):  # bins merged to expected >= 5
            ce, co = ce + e, co + o
            if ce >= 5:
                be.append(ce); bo.append(co); ce, co = 0.0, 0
        be[-1] += ce; bo[-1] += co
        pval = stats.chisquare(bo, np.array(be) * (sum(bo) / sum(be))).pvalue
        print(f"chi-square T={T} {name}: p = {pval:.3g} over {len(be)} bins")
        assert pval > 1e-4, (name, pval)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_infinite_logits_against_torch_logsumexp(dtype):
    """An allowed ``+inf`` logit gives ``logZ = +inf`` (torch.logsumexp) and no draw; with an allowed NaN too, NaN.
    A ``+inf`` at a masked-out position gives NaN under a per-row additive mask (``inf - inf``, as torch) and is
    ignored by a keep-mask (bool, bits, and a shared {0, -inf} mask, which is packed into bits)."""
    tdt = DTYPES[dtype]
    V, B = 4099, 8
    rng = np.random.default_rng(7)
    base = logsoftmax_rows(B, V, seed=5).astype(np.float64)
    keep = np.ones(V, dtype=bool)
    keep[[5, 700, V - 1]] = False
    for layout in ("contiguous", "column_offset"):
        for pos in (0, 13, 2048, V - 2):
            rows = base.copy()
            rows[0, pos] = np.inf                          # allowed +inf
            rows[1, pos] = np.inf; rows[1, 3000] = np.nan  # allowed +inf and an allowed NaN
            rows[2, [pos, 2049]] = np.inf                  # two of them
            rows[3, 700] = np.inf                          # +inf masked out
            rows[4, 700] = np.inf; rows[4, pos] = np.inf   # masked out and allowed
            rows[5, pos] = -np.inf                         # a plain row with a -inf
            rows[6] = -np.inf; rows[6, pos] = np.inf       # only the +inf
            dev = make_logits(rows, tdt, layout)
            x = dev.double()
            add = torch.tensor(np.where(keep, 0.0, -np.inf), dtype=torch.float32).cuda()
            for name, m in (("none", None), ("add_rows", add.expand(B, V).contiguous()), ("add_shared_01", add),
                            ("bool_rows", torch.tensor(keep).cuda().expand(B, V).contiguous()),
                            ("bits_shared", pack_bits(keep)[0])):
                for T in (1.0, 0.7):
                    logZ, tok = smc.masked_logsumexp_sample(dev, m, temperature=T, seed=3)
                    logZ, tok = logZ.cpu().numpy(), tok.cpu().numpy()
                    want = torch.logsumexp(x / T + (0 if m is None else add.double()), -1).cpu().numpy()
                    what = (dtype, layout, pos, name, T)
                    assert (logZ[[0, 2, 6]] == np.inf).all() and (tok[[0, 1, 2, 6]] == -1).all(), what
                    assert np.isnan(logZ[1]), what
                    assert np.isfinite(logZ[5]) and tok[5] >= 0 and tok[5] != pos, what
                    np.testing.assert_allclose(logZ[[0, 1, 2, 5, 6, 7]], want[[0, 1, 2, 5, 6, 7]], rtol=1e-5, atol=1e-6,
                                               err_msg=str(what))
                    if name == "add_rows":  # inf - inf: NaN, as torch
                        assert np.isnan(logZ[[3, 4]]).all() and np.isnan(want[3]) and tok[3] == tok[4] == -1, what
                    elif name == "none":
                        assert logZ[3] == np.inf == want[3] and logZ[4] == np.inf and tok[3] == -1, what
                    else:  # a keep-mask drops the masked-out +inf
                        want3 = torch.logsumexp(torch.where(torch.tensor(keep).cuda(), x[3] / T, -math.inf), -1).item()
                        assert abs(logZ[3] - want3) <= 1e-5 * abs(want3) + 1e-6 and keep[tok[3]], what
                        assert logZ[4] == np.inf and tok[4] == -1, what


# ---- GPU: next-symbol draws --------------------------------------------------------------------------------------
def _child_check(trie, lay, ids, q, m, out, seed, offset, what, weighted):
    """Every row's child against ``child_replay`` outside its near band; logp / logZ / log-mass within 1e-6."""
    if weighted:
        child, sym, logp, logZ, logM = (t.cpu().numpy() for t in out)
    else:
        child, _, logp, logZ = (t.cpu().numpy() for t in out)
    B = len(child)
    u = uniforms(seed, offset + np.arange(B, dtype=np.uint64), stream=0)
    n_near = agree = 0
    for b in range(B):
        j, near = child_replay(q[b], u[b])
        if j < 0:
            assert child[b] == -1, (what, b)
            continue
        if near:
            n_near += 1
            continue
        assert child[b] == ids[b, j], (what, b, int(child[b]), int(ids[b, j]))
        agree += 1
    Z = q.sum(axis=1)
    hm = np.flatnonzero(Z > 0)
    col = np.argmax(ids == child[:, None], axis=1)
    assert (q[hm, col[hm]] > 0).all(), what
    np.testing.assert_allclose(logZ[hm], np.log(Z[hm]), rtol=1e-6, atol=1e-6, err_msg=what)
    np.testing.assert_allclose(logp[hm], np.log(q[hm, col[hm]] / Z[hm]), rtol=1e-6, atol=1e-6, err_msg=what)
    if weighted:
        with np.errstate(divide="ignore"):
            # the root's log-mass is ~0 (rows sum to 1): only an absolute bound means anything there, as for logZ
            np.testing.assert_allclose(logM, np.log(m.sum(axis=1)), rtol=1e-6, atol=1e-6, err_msg=what)
    print(f"next-symbol {what}: {agree} draws equal to the replay, {n_near} in the near band, "
          f"{B - len(hm)} without mass")
    assert agree > 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["synth3000", "sentinel"])
def test_next_symbol_draws_replay_exactly(name):
    dec = golden_vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    lay = trie_layout(trie)
    sym = symbol_oracle.child_symbols(lay, trie.decode)[0]
    N, V, S = len(trie), len(dec), trie.num_symbols
    rng = np.random.default_rng(11)
    internal = np.flatnonzero(np.diff(trie._layout["child_ptr"]) > 0)
    if name == "synth3000":
        nodes = np.concatenate([[trie.root] * 40, [depth1_node(trie)] * 40, rng.choice(internal, 2000)])
    else:
        nodes = np.repeat(internal, 64)
    nodes = nodes.astype(np.int32)
    B = len(nodes)
    ws = dirichlet_rows(B, V, alpha=0.3, seed=12)
    keep = rng.random((B, V)) < 0.7
    ws_kept = np.where(keep, ws, np.float32(0))
    logw = rng.normal(0.0, 1.5, (B, S + 1))
    logw[rng.random((B, S + 1)) < 0.1] = -np.inf
    wdev, ndev, kdev = torch.tensor(ws).cuda(), torch.tensor(nodes).cuda(), torch.tensor(keep).cuda()
    ids = child_oracle.child_ids(lay, nodes)
    for masked in (False, True):
        rows = ws_kept if masked else ws
        kw = dict(mask=kdev) if masked else {}
        m = child_oracle.child_masses(lay, rows, nodes, "sum")
        seed, offset = 5 + masked, 1000 * masked
        out = trie.sample_next_symbol(wdev, ndev, seed=seed, offset=offset, **kw)
        _child_check(trie, lay, ids, m, m, out, seed, offset, (name, "masked" if masked else "plain"), False)
        out = trie.sample_next_symbol_weighted(wdev, ndev, torch.tensor(logw, dtype=torch.float32).cuda(), seed=seed,
                                               offset=offset + 7, **kw)
        # the kernel reads fp32 log-weights: the oracle's terms from the same fp32 values
        _, m2, q = symbol_oracle.weighted_child_masses(lay, sym, rows, nodes, logw.astype(np.float32))
        _child_check(trie, lay, ids, q, m2, out, seed, offset + 7, (name, "weighted masked" if masked else "weighted"),
                     True)
