"""Next-symbol read-outs restricted to the tokens a per-row keep-bitmask allows (``gt_child_masses_masked``,
``gt_child_sample_masked``, ``gt_symbol_masses_masked``, ``gt_symbol_sample_masked``).

The contract: a masked call returns bit for bit what the unmasked call returns on rows whose masked-out weights are 0
(-inf for log inputs).  CPU part: the argument checks of the four entry points in their pinned order, and the Python
mask validation.  GPU part (``-m gpu``): bit-equality with the zeroed rows over vocabularies, input dtypes, flags and
masks; all-ones masks; determinism across batches, chunks and graph replay; exactness against the token-level masked
sampler (the root's mass, and a byte-by-byte walk); and the one-mask-per-token DFA recipe.
"""
import ctypes

import numpy as np
import pytest
import torch

from genlm_backend_b200 import ParallelTokenCharacterTrie, _lib, dfa, smc
from genlm_backend_b200.synthetic import dirichlet_rows, logsoftmax_rows
import dfa_oracle
from helpers import golden_vocab

F32, SUM, MAX = _lib.GT_F32, _lib.GT_OP_SUM, _lib.GT_OP_MAX
NORM, LOG = _lib.GT_CHILD_NORMALIZE, _lib.GT_CHILD_LOG


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_masked_entry_points_reject_bad_arguments_without_a_gpu():
    trie = ParallelTokenCharacterTrie(golden_vocab("synth3000"))
    h = trie._engine._handle
    V, S, D = trie._engine.V, trie.num_symbols, trie.max_children
    W = (V + 31) // 32
    lib = _lib.lib
    p = ctypes.c_void_p(1 << 20)  # stands for a device pointer: never dereferenced by the checks
    work_bytes = lib.gt_child_workspace_bytes(h, 4)
    base = dict(t=h, ws=p, in_type=F32, n=4, ld_ws=V, nodes=p, mask=p, mask_ld=W, flags=0, work=p, work_bytes=work_bytes)

    def child_masses(a):
        return lib.gt_child_masses_masked(a["t"], a["ws"], a["in_type"], a["n"], a["ld_ws"], a["nodes"], a["mask"],
                                          a["mask_ld"], a["ids"], a["s"], a["m"], a["ld_out"], a["ops"], a["flags"],
                                          a["work"], a["work_bytes"], None)

    def child_sample(a):
        return lib.gt_child_sample_masked(a["t"], a["ws"], a["in_type"], a["n"], a["ld_ws"], a["nodes"], a["mask"],
                                          a["mask_ld"], a["flags"], 1, 0, a["c"], a["lp"], a["lz"], a["work"],
                                          a["work_bytes"], None)

    def symbol_masses(a):
        return lib.gt_symbol_masses_masked(a["t"], a["ws"], a["in_type"], a["n"], a["ld_ws"], a["nodes"], a["mask"],
                                           a["mask_ld"], a["s"], a["m"], a["ld_out"], a["ops"], a["flags"], a["work"],
                                           a["work_bytes"], None)

    def symbol_sample(a):
        return lib.gt_symbol_sample_masked(a["t"], a["ws"], a["in_type"], a["n"], a["ld_ws"], a["nodes"], a["mask"],
                                           a["mask_ld"], a["w"], a["ld_w"], a["flags"], 1, 0, a["c"], a["sy"], a["lp"],
                                           a["lz"], a["lm"], a["work"], a["work_bytes"], None)

    calls = [  # (call, its own arguments, its own bad scalars, its own outputs)
        (child_masses, dict(ids=p, s=p, m=p, ld_out=D, ops=SUM | MAX),
         [dict(ops=0), dict(ld_out=D - 1), dict(flags=0x40)], ["ids", "s", "m"]),
        (child_sample, dict(c=p, lp=p, lz=p), [dict(flags=NORM)], ["c", "lp", "lz"]),
        (symbol_masses, dict(s=p, m=p, ld_out=S + 1, ops=SUM | MAX), [dict(ops=4), dict(ld_out=S)], ["s", "m"]),
        (symbol_sample, dict(w=p, ld_w=0, c=p, sy=p, lp=p, lz=p, lm=p), [dict(ld_w=S), dict(ld_w=-1), dict(flags=LOG)],
         ["w", "c", "sy", "lp", "lz"]),
    ]
    for call, own, own_bad, outs in calls:
        def run(**kw):
            a = dict(base, **own)
            a.update(kw)
            return call(a)

        bad_scalars = [dict(t=None), dict(in_type=7), dict(n=-1), dict(ld_ws=V - 1), dict(mask_ld=-1), dict(mask_ld=1),
                       dict(mask_ld=W - 1)] + own_bad
        for bad in bad_scalars + [dict(ws=None), dict(nodes=None), dict(mask=None), dict(work=None),
                                  dict(work=ctypes.c_void_p((1 << 20) + 8))] + [{o: None} for o in outs]:
            assert run(**bad) == 1, (call.__name__, bad)
        assert run(work_bytes=16) == 3 and b"workspace too small" in lib.gt_last_error()
        assert run(mask_ld=0, work_bytes=16) == 3 and run(mask_ld=W + 5, work_bytes=16) == 3  # shared and padded strides
        # the order of the checks: scalars and mask_ld, the early return for no rows, data pointers, the workspace
        nulls = dict(ws=None, nodes=None, mask=None, work=None, **{o: None for o in outs})
        assert run(n=0, **nulls) == 0, call.__name__
        for bad in bad_scalars:
            if "n" not in bad:
                assert run(n=0, **dict(nulls, **bad)) == 1, (call.__name__, bad)
        assert run(mask=None, work=None) == 1 and b"null data pointer" in lib.gt_last_error()
        assert run(mask=None, work_bytes=16) == 1 and b"null data pointer" in lib.gt_last_error()


def test_keep_bits_validation_and_packing():
    trie = ParallelTokenCharacterTrie(golden_vocab("synth3000"))
    eng = trie._engine
    V, W, B = eng.V, (eng.V + 31) // 32, 3
    rng = np.random.default_rng(0)
    keep = torch.tensor(rng.random((B, V)) < 0.3)
    bits, ld = eng.keep_bits(keep, B, "cpu")
    assert bits.dtype == torch.int32 and tuple(bits.shape) == (B, W) and ld == W
    unpacked = ((bits[:, :, None] >> torch.arange(32)) & 1).reshape(B, -1)[:, :V].bool()
    assert torch.equal(unpacked, keep)
    assert ((bits[:, -1] >> (V % 32 or 32)) == 0).all()  # no bit at or above V
    shared, ld = eng.keep_bits(keep[1], B, "cpu")
    assert ld == 0 and torch.equal(shared, bits[1])
    wide = torch.zeros((B, W + 7), dtype=torch.int32)
    wide[:, :W] = bits
    view, ld = eng.keep_bits(wide[:, :W], B, "cpu")  # a row stride above ceil(V/32) is kept
    assert ld == W + 7 and view.data_ptr() == wide.data_ptr()
    for bad in (bits.to(torch.int64), bits.float(), bits.to(torch.uint8), keep.to(torch.uint8), bits[:, :W - 1],
                torch.zeros((B, W + 1), dtype=torch.int32), torch.zeros(W + 1, dtype=torch.int32), bits[:2], keep[:2],
                keep[:, :V - 1], torch.zeros((1, B, W), dtype=torch.int32), torch.zeros((), dtype=torch.int32)):
        with pytest.raises(ValueError):
            eng.keep_bits(bad, B, "cpu")


# ---- GPU ---------------------------------------------------------------------------------------------------------
def bits_of(f):
    """Float tensors as their bit patterns (so that NaN patterns compare too); ints as they are."""
    return f.view(torch.int32) if f.dtype == torch.float32 else f


def assert_same(a, b, what=""):
    for x, y in zip(a, b):
        if x is None:
            assert y is None, what
            continue
        assert torch.equal(bits_of(x), bits_of(y)), what


def random_bits(rng, B, V, density, pad=0):
    """int32 keep-bitmask [B, ceil(V/32) + pad] with each bit set with probability ``density`` (bits at or above V and
    the padding words random too: they must be ignored), and its bool keep-mask [B, V]."""
    W = (V + 31) // 32
    raw = rng.random((B, (W + pad) * 32)) < density
    words = (raw.reshape(B, W + pad, 32).astype(np.uint64) << np.arange(32, dtype=np.uint64)).sum(-1)
    bits = torch.tensor(words.astype(np.uint32).view(np.int32))
    return bits, torch.tensor(raw[:, :V])


def unpack(bits, B, V):
    b = bits.expand(B, -1) if bits.dim() == 1 else bits
    return ((b[:, :, None] >> torch.arange(32, device=b.device)) & 1).reshape(b.shape[0], -1)[:, :V].bool()


def all_calls(trie, ws, nodes, mask, logw, log_input, dfs_order, seed=3, offset=11):
    """Every output of the four read-outs under one mask (None: the unmasked calls)."""
    kw = dict(log_input=log_input, dfs_order=dfs_order, mask=mask)
    out = []
    for normalize, log in ((False, False), (True, True), (True, False)):
        out += trie.batch_child_masses_tensor(ws, nodes, ops=("sum", "max"), normalize=normalize, log=log, **kw)
        out += trie.batch_symbol_masses_tensor(ws, nodes, ops=("sum", "max"), normalize=normalize, log=log, **kw)
    out += trie.batch_child_masses_tensor(ws, nodes, ops=("max",), **kw)
    out += trie.sample_next_symbol(ws, nodes, seed=seed, offset=offset, **kw)
    out += trie.sample_next_symbol_weighted(ws, nodes, logw, seed=seed, offset=offset, **kw)
    return out


def check_bit_equal(trie, nodes, base, rng, dtypes, mask_kinds):
    V, B, S = len(trie.decode), len(nodes), trie.num_symbols
    nt = torch.tensor(nodes).cuda()
    dfs_perm = trie.dfs_token_order.cuda()
    logw = torch.tensor(rng.normal(size=(B, S + 1)).astype(np.float32)).cuda()
    for kind in mask_kinds:
        density, shared, pad = {"d0.5": (0.5, False, 3), "d0.02": (0.02, False, 0), "shared0.5": (0.5, True, 0),
                                "ones": (1.0, True, 0), "zeros": (0.0, False, 0), "bool0.3": (0.3, False, 0)}[kind]
        bits, keep = random_bits(rng, 1 if shared else B, V, density, pad)
        bits = bits.cuda()
        mask = keep.cuda() if kind.startswith("bool") else (bits[0] if shared else bits[:, :(V + 31) // 32])
        keep = unpack(bits[0] if shared else bits, B, V)
        for dtype in dtypes:
            for log_input in (False, True):
                with np.errstate(divide="ignore"):
                    x = torch.tensor(np.log(base) if log_input else base).to(dtype).cuda()
                fill = float("-inf") if log_input else 0.0
                # masked-out positions hold NaN and inf: the masked call never reads them, the reference has them zeroed
                poison = (torch.rand(x.shape, device="cuda") < 0.1) & ~keep
                x = torch.where(poison & (torch.rand(x.shape, device="cuda") < 0.5), float("nan"),
                                torch.where(poison, float("inf"), x))
                ref = torch.where(keep, x, torch.full_like(x, fill))
                for dfs_order in (False, True):
                    xs, rs = (x[:, dfs_perm].contiguous(), ref[:, dfs_perm].contiguous()) if dfs_order else (x, ref)
                    have = all_calls(trie, xs, nt, mask, logw, log_input, dfs_order)
                    want = all_calls(trie, rs, nt, None, logw, log_input, dfs_order)
                    assert_same(have, want, (kind, dtype, log_input, dfs_order))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["toy", "edge", "sentinel", "synth3000"])
def test_bit_equal_to_zeroed_rows_at_every_node(name):
    dec = golden_vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    N, V = len(trie), len(dec)
    nodes = np.concatenate([np.arange(N), [-1, N]]).astype(np.int32)
    base = np.concatenate([dirichlet_rows(3, V, alpha=0.1, seed=11), dirichlet_rows(2, V, alpha=1.0, seed=12)])
    base = base[np.arange(len(nodes)) % len(base)]
    check_bit_equal(trie, nodes, base, np.random.default_rng(1),
                    [torch.float32, torch.float64, torch.float16, torch.bfloat16],
                    ["d0.5", "d0.02", "shared0.5", "ones", "zeros", "bool0.3"])


@pytest.mark.gpu
def test_bit_equal_to_zeroed_rows_at_sampled_nodes_of_128k_tokens():
    trie = ParallelTokenCharacterTrie(golden_vocab("synth128256"))
    N, V = len(trie), len(trie.decode)
    rng = np.random.default_rng(2)
    leaves = trie._layout["leaf_node"]
    nodes = rng.integers(0, N, 96).astype(np.int32)
    nodes[:8] = trie.root
    nodes[8:12] = leaves[rng.integers(0, V, 4)]
    nodes[12:14] = (-1, N)
    nodes[14:30] = rng.choice(trie.jump[trie.root], 16)
    base = dirichlet_rows(len(nodes), V, alpha=0.3, seed=4)
    check_bit_equal(trie, nodes, base, rng, [torch.float32, torch.float64, torch.float16, torch.bfloat16],
                    ["d0.5", "d0.02", "ones", "zeros"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["edge", "synth3000"])
def test_all_ones_mask_equals_unmasked(name):
    dec = golden_vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    N, V, S = len(trie), len(dec), trie.num_symbols
    W = (V + 31) // 32
    nodes = torch.tensor(np.concatenate([np.arange(N), [-1, N]]).astype(np.int32)).cuda()
    B = len(nodes)
    x = torch.tensor(dirichlet_rows(B, V, alpha=0.2, seed=3)).cuda()
    logw = torch.tensor(np.random.default_rng(5).normal(size=(B, S + 1)).astype(np.float32)).cuda()
    ones = torch.full((W,), -1, dtype=torch.int32, device="cuda")
    for dfs_order in (False, True):
        xs = x[:, trie.dfs_token_order.cuda()].contiguous() if dfs_order else x
        want = all_calls(trie, xs, nodes, None, logw, False, dfs_order)
        assert_same(all_calls(trie, xs, nodes, ones, logw, False, dfs_order), want)
        assert_same(all_calls(trie, xs, nodes, ones.expand(B, -1).contiguous(), logw, False, dfs_order), want)
        assert_same(all_calls(trie, xs, nodes, torch.ones(V, dtype=torch.bool), logw, False, dfs_order), want)
    # NaN and inf at masked-out positions change nothing: one item masked out, its weight poisoned, against the row
    # with that weight at 0
    item = int(trie.dfs_token_order[0])
    keep = torch.ones(V, dtype=torch.bool)
    keep[item] = False
    zeroed = x.clone()
    zeroed[:, item] = 0
    want = all_calls(trie, zeroed, nodes, None, logw, False, False)
    for bad in (float("nan"), float("inf")):
        poisoned = x.clone()
        poisoned[:, item] = bad
        assert_same(all_calls(trie, poisoned, nodes, keep, logw, False, False), want)


@pytest.mark.gpu
def test_bit_identical_alone_in_batch_in_chunks_and_in_graphs():
    trie = ParallelTokenCharacterTrie(golden_vocab("synth128256"))
    eng = trie._engine
    V, S, N = len(trie.decode), trie.num_symbols, len(trie)
    W = (V + 31) // 32
    rng = np.random.default_rng(8)
    B = 64
    nodes = np.full(B, trie.root, dtype=np.int32)
    nodes[::3] = rng.integers(0, N, len(nodes[::3]))
    nt = torch.tensor(nodes).cuda()
    ws = torch.tensor(dirichlet_rows(B, V, alpha=0.5, seed=6)).cuda()
    bits = random_bits(rng, B, V, 0.4, pad=2)[0].cuda()
    mask = bits[:, :W]  # row stride W + 2
    logw = torch.tensor(rng.normal(size=(B, S + 1)).astype(np.float32)).cuda()
    sums, maxes = trie.batch_symbol_masses_tensor(ws, nt, ops=("sum", "max"), normalize=True, mask=mask)
    draw = trie.sample_next_symbol_weighted(ws, nt, logw, seed=3, offset=9, mask=mask)
    for r in (0, 1, 31, 63):  # a row alone (its Philox counter is offset + its position)
        one = trie.batch_symbol_masses_tensor(ws[r:r + 1], nt[r:r + 1], ops=("sum", "max"), normalize=True, mask=mask[r:r + 1])
        assert_same(one, (sums[r:r + 1], maxes[r:r + 1]))
        d1 = trie.sample_next_symbol_weighted(ws[r:r + 1], nt[r:r + 1], logw[r:r + 1], seed=3, offset=9 + r, mask=mask[r])
        assert_same(d1, [t[r:r + 1] for t in draw])
    # a one-row workspace through the C ABI: 64 chunks of one row, each with its own mask row
    need = _lib.lib.gt_child_workspace_bytes(eng._handle, 1)
    work = torch.empty(need, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    s1 = torch.empty((B, S + 1), dtype=torch.float32, device="cuda")
    m1 = torch.empty((B, S + 1), dtype=torch.float32, device="cuda")
    _lib.check(_lib.lib.gt_symbol_masses_masked(eng._handle, ws.data_ptr(), F32, B, V, nt.data_ptr(), bits.data_ptr(),
                                                W + 2, s1.data_ptr(), m1.data_ptr(), S + 1, SUM | MAX, NORM,
                                                work.data_ptr(), need, st), "gt_symbol_masses_masked")
    assert_same((s1, m1), (sums, maxes))
    outs = [torch.empty(B, dtype=t, device="cuda") for t in (torch.int32, torch.int32, torch.float32, torch.float32, torch.float32)]
    _lib.check(_lib.lib.gt_symbol_sample_masked(eng._handle, ws.data_ptr(), F32, B, V, nt.data_ptr(), bits.data_ptr(), W + 2,
                                                logw.data_ptr(), S + 1, 0, 3, 9, *[o.data_ptr() for o in outs],
                                                work.data_ptr(), need, st), "gt_symbol_sample_masked")
    assert_same(outs, draw)
    # CUDA graph capture and replay == eager
    cs = torch.cuda.Stream()
    cs.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(cs):  # the workspace of this stream, before capture
        trie.batch_symbol_masses_tensor(ws, nt, ops=("sum", "max"), normalize=True, mask=mask)
    torch.cuda.current_stream().wait_stream(cs)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=cs):
        cap = trie.batch_symbol_masses_tensor(ws, nt, ops=("sum", "max"), normalize=True, mask=mask)
        cap_draw = trie.sample_next_symbol_weighted(ws, nt, logw, seed=3, offset=9, mask=mask)
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        assert_same(cap, (sums, maxes))
        assert_same(cap_draw, draw)


def ascii_words_dfa(S):
    """Lower-case ASCII letters and single spaces between them (state 0: after a letter or at the start, 1: after a
    space); accepts in state 0."""
    d = np.full((2, S), -1, dtype=np.int32)
    d[:, ord("a"):ord("z") + 1] = 0
    d[0, ord(" ")] = 1
    return dfa.trim(d, [0])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["synth3000", "synth128256"])
def test_root_mass_is_the_masked_token_logZ(name):
    dec = golden_vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    V, S = len(dec), trie.num_symbols
    rng = np.random.default_rng(3)
    B = 64
    logp = torch.tensor(logsoftmax_rows(B, V, seed=2)).cuda()
    root = torch.full((B,), trie.root, dtype=torch.int32)
    delta, acc = dfa_oracle.random_dfa(rng, 64, S, p_live=0.6)
    tables = [torch.tensor(ascii_words_dfa(S)).cuda(), torch.tensor(dfa.trim(delta, acc)).cuda()]
    masks = [trie.dfa_token_mask(t, torch.tensor(rng.integers(0, t.shape[0], B).astype(np.int32)).cuda()) for t in tables]
    masks += [random_bits(rng, B, V, d)[0].cuda() for d in (0.5, 0.01)]
    drawn = 0
    for bits in masks:
        want, _ = smc.masked_logsumexp_sample(logp, bits)
        _, _, _, logZ = trie.sample_next_symbol(logp, root, log_input=True, mask=bits)
        _, _, _, wZ, logM = trie.sample_next_symbol_weighted(logp, root, torch.zeros(S + 1), log_input=True, mask=bits)
        sums, _ = trie.batch_symbol_masses_tensor(logp, root, log_input=True, mask=bits)
        w = want.cpu().numpy()
        drawn += int(np.isfinite(w).sum())
        for have in (logZ, wZ, logM, torch.log(sums.double().sum(1)).float()):
            np.testing.assert_allclose(have.cpu().numpy(), w, rtol=1e-5, atol=1e-6)
    assert drawn > len(masks) * B // 2


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["edge", "sentinel"])
def test_byte_walk_from_the_root_draws_the_masked_token_distribution(name):
    from scipy import stats

    dec = golden_vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    V = len(dec)
    row = dirichlet_rows(1, V, alpha=1.0, seed=21)[0]
    keep = np.ones(V, dtype=bool)
    keep[np.random.default_rng(4).permutation(V)[: max(1, V // 3)]] = False
    p = np.where(keep, row, 0.0)
    p /= p.sum()
    n = 40000
    ws = torch.tensor(row).expand(n, -1).cuda()
    bits = smc._pack_keep_bits(torch.tensor(keep).cuda())  # one shared mask, packed once for the token
    nodes = torch.full((n,), trie.root, dtype=torch.int32, device="cuda")
    token = torch.full((n,), -1, dtype=torch.int64, device="cuda")
    walk_logp = torch.zeros(n, dtype=torch.float64, device="cuda")
    for k in range(int(_lib.lib.gt_max_depth(trie._engine._handle)) + 1):  # a token's walk is at most that deep
        live = token < 0
        if not bool(live.any()):
            break
        child, label, logp, _ = trie.sample_next_symbol(ws, nodes, seed=7, offset=k * n, mask=bits)
        assert bool((child[live] >= 0).all())
        walk_logp += torch.where(live, logp.double(), torch.zeros_like(walk_logp))
        ends = live & (label < 0)
        token = torch.where(ends, (-1 - label).long(), token)
        nodes = torch.where(live & ~ends, child, nodes)
    tok = token.cpu().numpy()
    assert (tok >= 0).all() and keep[tok].all()
    counts = np.bincount(tok, minlength=V).astype(np.float64)
    big = p * n >= 5
    obs = np.append(counts[big], counts[~big].sum())
    exp = np.append(p[big] * n, p[~big].sum() * n)
    sel = exp > 0
    assert stats.chisquare(obs[sel], exp[sel] * obs[sel].sum() / exp[sel].sum()).pvalue > 1e-4
    np.testing.assert_allclose(walk_logp.cpu().numpy(), np.log(p[tok]), rtol=1e-5, atol=1e-5)


def path_state(trie, delta, q, node):
    """The DFA state after the symbols of the path root -> node from state q (-1 once rejected)."""
    lay = trie._layout
    syms = []
    n = int(node)
    while n != trie.root:
        syms.append(int(lay["edge_label"][n]))
        n = int(lay["parent"][n])
    for s in reversed(syms):
        if q < 0:
            break
        q = int(delta[q, s])
    return q


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sentinel", "synth3000"])
def test_one_root_mask_per_token_equals_the_mask_at_the_node(name):
    dec = golden_vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    V, S, N = len(dec), trie.num_symbols, len(trie)
    rng = np.random.default_rng(6)
    delta, acc = dfa_oracle.random_dfa(rng, 16, S, p_live=0.7)
    delta = dfa.trim(delta, acc)
    internal = np.flatnonzero(np.diff(trie._layout["child_ptr"]) > 0)
    B = 512
    nodes = rng.choice(internal, B).astype(np.int32)
    q0 = rng.integers(0, delta.shape[0], B).astype(np.int32)
    qn = np.array([path_state(trie, delta, int(q), int(n)) for q, n in zip(q0, nodes)], dtype=np.int32)
    dt = torch.tensor(delta).cuda()
    root_bits = trie.dfa_token_mask(dt, torch.tensor(q0).cuda())
    node_bits = trie.dfa_token_mask(dt, torch.tensor(qn).cuda(), nodes=torch.tensor(nodes).cuda())
    ws = torch.tensor(dirichlet_rows(B, V, alpha=0.3, seed=2)).cuda()
    nt = torch.tensor(nodes).cuda()
    a = trie.batch_symbol_masses_tensor(ws, nt, ops=("sum", "max"), mask=root_bits)
    b = trie.batch_symbol_masses_tensor(ws, nt, ops=("sum", "max"), mask=node_bits)
    assert_same(a, b)
    assert bool((a[0].sum(1) > 0).any())
