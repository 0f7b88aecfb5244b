"""Child masses of one node per row (``gt_child_masses``) and the next-symbol draw (``gt_child_sample``).

CPU part: the reference values of ``child_oracle`` (the oracle's ``weight_sum`` / ``weight_max`` at ``jump[node]``)
pinned to the reference's golden sums, ``gt_max_children`` and the argument checks of the two entry points (they
reject bad arguments before any CUDA call).  GPU part (``-m gpu``): the kernels against the fp64 oracle (sums within
one fp32 ulp, maxes bit-equal to the mass slab), the determinism guarantees of the header, the draw's distribution and
edge cases, and the async wrapper.
"""
import asyncio
import ctypes

import numpy as np
import pytest
import torch

from genlm_backend_b200 import AsyncTokenCharacterTrie, ParallelTokenCharacterTrie, TokenCharacterTrie, _lib
from genlm_backend_b200.synthetic import dirichlet_rows, synth_vocab
import child_oracle
from helpers import assert_within_ulp, depth1_node, golden_layout, golden_vocab, trie_layout

F32, SUM, MAX = _lib.GT_F32, _lib.GT_OP_SUM, _lib.GT_OP_MAX
INT32_MIN = np.iinfo(np.int32).min


# ---- CPU ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["toy", "edge", "sentinel"])
def test_oracle_child_masses_pinned_to_golden(name):
    lay, g = golden_layout(name)
    N, D = lay.n_nodes, int(np.diff(g["jump_ptr"]).max())
    nodes = np.concatenate([np.arange(N), [-1, N]])
    for b in range(g["ws"].shape[0]):
        rows = np.repeat(g["ws"][b:b + 1], len(nodes), axis=0)
        ids = child_oracle.child_ids(lay, nodes)
        assert ids.shape == (len(nodes), D)
        for op, ref in (("sum", g["seq_sum"][b]), ("max", g["seq_max"][b])):
            have = child_oracle.child_masses(lay, rows, nodes, op)
            want = np.where(ids >= 0, ref[np.maximum(ids, 0)], 0.0)
            assert np.array_equal(have, want), (name, op)
        for i, n in enumerate(nodes.tolist()):
            kids = g["jump_idx"][g["jump_ptr"][n]:g["jump_ptr"][n + 1]] if 0 <= n < N else []
            assert ids[i, :len(kids)].tolist() == list(kids) and (ids[i, len(kids):] == -1).all()


@pytest.mark.parametrize("name", ["toy", "synth128256"])
def test_max_children_host_only(name):
    trie = TokenCharacterTrie(golden_vocab(name))
    want = max(len(j) for j in trie.jump)
    assert trie._engine.max_children == want == _lib.lib.gt_max_children(trie._engine._handle)
    assert want == (3 if name == "toy" else 256)
    assert _lib.lib.gt_max_children(None) == -1


def test_child_entry_points_reject_bad_arguments_without_a_gpu():
    trie = TokenCharacterTrie(golden_vocab("edge"))
    h = trie._engine._handle
    V, D = trie._engine.V, trie._engine.max_children
    lib = _lib.lib
    p = ctypes.c_void_p(1 << 20)  # stands for a device pointer: never dereferenced by the checks
    ws_bytes = lib.gt_child_workspace_bytes(h, 4)
    assert lib.gt_child_workspace_bytes(None, 4) == 0 and lib.gt_child_workspace_bytes(h, 0) == 0
    assert 0 < lib.gt_child_workspace_bytes(h, 1) <= ws_bytes < lib.gt_child_workspace_bytes(h, 1024)
    assert lib.gt_child_workspace_bytes(h, 1024) == lib.gt_child_workspace_bytes(h, 10**6)  # capped: larger batches chunk

    def masses(**kw):
        a = dict(t=h, ws=p, in_type=F32, n=4, ld_ws=V, nodes=p, ids=p, s=p, m=p, ld_out=D, ops=SUM | MAX, flags=0,
                 work=p, work_bytes=ws_bytes)
        a.update(kw)
        return lib.gt_child_masses(a["t"], a["ws"], a["in_type"], a["n"], a["ld_ws"], a["nodes"], a["ids"], a["s"], a["m"],
                                   a["ld_out"], a["ops"], a["flags"], a["work"], a["work_bytes"], None)

    for bad in (dict(t=None), dict(ws=None), dict(nodes=None), dict(ids=None), dict(s=None), dict(m=None), dict(ops=0),
                dict(ops=4), dict(flags=0x40), dict(in_type=7), dict(n=-1), dict(ld_ws=V - 1), dict(ld_out=D - 1),
                dict(work=None), dict(work=ctypes.c_void_p((1 << 20) + 8))):
        assert masses(**bad) == 1, bad
    assert masses(ops=SUM, m=None, flags=_lib.GT_CHILD_NORMALIZE | _lib.GT_CHILD_LOG, work_bytes=16) == 3  # too small
    assert b"workspace too small" in lib.gt_last_error()
    assert masses(n=0) == 0
    # the order of the checks: scalars and strides, the early return for no rows, data pointers, the workspace
    nulls = dict(ws=None, nodes=None, ids=None, s=None, m=None, work=None)
    assert masses(n=0, **nulls) == 0
    for bad in (dict(ops=0), dict(flags=0x40), dict(in_type=7), dict(ld_ws=V - 1), dict(ld_out=D - 1)):
        assert masses(n=0, **nulls, **bad) == 1, bad
    assert masses(ids=None, work=None) == 1 and b"null data pointer" in lib.gt_last_error()

    def sample(**kw):
        a = dict(t=h, ws=p, in_type=F32, n=4, ld_ws=V, nodes=p, flags=0, c=p, lp=p, lz=p, work=p, work_bytes=ws_bytes)
        a.update(kw)
        return lib.gt_child_sample(a["t"], a["ws"], a["in_type"], a["n"], a["ld_ws"], a["nodes"], a["flags"], 1, 0, a["c"],
                                   a["lp"], a["lz"], a["work"], a["work_bytes"], None)

    for bad in (dict(t=None), dict(ws=None), dict(nodes=None), dict(c=None), dict(lp=None), dict(lz=None),
                dict(flags=_lib.GT_CHILD_NORMALIZE), dict(in_type=-1), dict(n=-1), dict(ld_ws=V - 1), dict(work=None)):
        assert sample(**bad) == 1, bad
    assert sample(work_bytes=16) == 3
    assert sample(n=0) == 0
    nulls = dict(ws=None, nodes=None, c=None, lp=None, lz=None, work=None)
    assert sample(n=0, **nulls) == 0
    for bad in (dict(flags=_lib.GT_CHILD_NORMALIZE), dict(in_type=-1), dict(ld_ws=V - 1)):
        assert sample(n=0, **nulls, **bad) == 1, bad
    assert sample(lz=None, work=None) == 1 and b"null data pointer" in lib.gt_last_error()


# ---- GPU ---------------------------------------------------------------------------------------------------------
def slab_max_at(trie, ws, ids, **kw):
    mx = trie._engine.reduce(ws, ("max",), **kw)[1].cpu().numpy()
    return np.where(ids >= 0, np.take_along_axis(mx, np.maximum(ids, 0), axis=1), 0.0).astype(np.float32)


def check_all(trie, lay, ws_t, nodes, ws32=None):
    ids, s, m = trie.batch_child_masses(ws_t, torch.tensor(nodes), ops=("sum", "max"))
    ws32 = ws_t.float().cpu().numpy() if ws32 is None else ws32
    assert np.array_equal(ids, child_oracle.child_ids(lay, nodes))
    assert_within_ulp(s, child_oracle.child_masses(lay, ws32, nodes, "sum"))
    assert np.array_equal(m, slab_max_at(trie, ws_t.cuda(), ids))
    return ids, s, m


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["toy", "edge", "sentinel", "synth3000"])
def test_every_node_matches_oracle(name):
    dec = golden_vocab(name)
    trie = ParallelTokenCharacterTrie(dec)
    lay = trie_layout(trie)
    N, V = len(trie), len(dec)
    nodes = np.concatenate([np.arange(N), [-1, N]]).astype(np.int32)
    base = np.concatenate([dirichlet_rows(3, V, alpha=0.1, seed=11), dirichlet_rows(2, V, alpha=1.0, seed=12)])
    ws = base[np.arange(len(nodes)) % len(base)]
    check_all(trie, lay, torch.tensor(ws), nodes)


@pytest.mark.gpu
def test_full_vocabulary_sampled_nodes_and_input_orders():
    V = 128256
    trie = ParallelTokenCharacterTrie(synth_vocab(V))
    lay = trie_layout(trie)
    rng = np.random.default_rng(5)
    nodes = np.concatenate([[trie.root, -1, len(trie)], rng.integers(0, len(trie), 509)]).astype(np.int32)
    base = dirichlet_rows(4, V, alpha=0.1, seed=3)
    ws = torch.tensor(base[np.arange(len(nodes)) % 4]).cuda()
    ids, s, m = check_all(trie, lay, ws, nodes, ws32=base[np.arange(len(nodes)) % 4])
    assert (ids[0] >= 0).sum() == 256 and (ids[1:3] == -1).all()
    # DFS-order rows give the very same bits
    dfs = ws[:, trie.dfs_token_order.cuda()].contiguous()
    ids2, s2, m2 = trie.batch_child_masses(dfs, torch.tensor(nodes), ops=("sum", "max"), dfs_order=True)
    assert np.array_equal(ids, ids2) and np.array_equal(s, s2) and np.array_equal(m, m2)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("log_input", [False, True])
def test_input_types_and_flags(dtype, log_input):
    dec = golden_vocab("synth3000")
    trie = ParallelTokenCharacterTrie(dec)
    lay = trie_layout(trie)
    B = 96
    nodes = np.random.default_rng(1).integers(0, len(trie), B).astype(np.int32)
    nodes[:4] = trie.root
    p = dirichlet_rows(B, len(dec), alpha=0.3, seed=4)
    with np.errstate(divide="ignore"):
        x = torch.tensor(np.log(p) if log_input else p).to(dtype).cuda()
    x32 = x.float().cpu().numpy()  # the kernel's conversion (exact for fp16 / bf16, fp32 rounding for fp64)
    w = np.exp(x32.astype(np.float64)).astype(np.float32) if log_input else x32
    ids, s, m = trie.batch_child_masses(x, torch.tensor(nodes), ops=("sum", "max"), log_input=log_input)
    want = child_oracle.child_masses(lay, w, nodes, "sum")
    if log_input:  # the kernel's expf is not reproducible bit for bit here
        np.testing.assert_allclose(s, want, rtol=1e-6, atol=0)
    else:
        assert_within_ulp(s, want)
    assert np.array_equal(m, slab_max_at(trie, x, ids, log_input=log_input))
    # normalised, logs: against the oracle in fp64
    total = want.sum(axis=1, keepdims=True)
    _, sn, _ = trie.batch_child_masses(x, torch.tensor(nodes), log_input=log_input, normalize=True)
    _, sl, ml = trie.batch_child_masses(x, torch.tensor(nodes), ops=("sum", "max"), log_input=log_input, normalize=True, log=True)
    pad = ids < 0
    assert (sn[pad] == 0).all() and np.isneginf(sl[pad]).all() and np.isneginf(ml[pad]).all()
    with np.errstate(divide="ignore", invalid="ignore"):  # rows at a leaf / invalid id: 0 / 0
        wn, wl = want / total, np.log(want / total)
        ml_want = np.log(m.astype(np.float64))
    rtol = 1e-6 if log_input else 0
    if rtol:
        np.testing.assert_allclose(sn[~pad], wn[~pad], rtol=rtol)
        np.testing.assert_allclose(sl[~pad], wl[~pad], rtol=rtol, atol=1e-6)
    else:
        assert_within_ulp(sn[~pad], wn[~pad])
        fin = np.isfinite(wl[~pad])
        err = np.abs(sl[~pad][fin] - wl[~pad][fin])
        assert (err <= np.spacing(np.abs(wl[~pad][fin]).astype(np.float32)) + 1e-12).all()
        assert np.array_equal(np.isneginf(sl[~pad]), np.isneginf(wl[~pad]))
    assert np.array_equal(ml[~pad], ml_want[~pad].astype(np.float32))


@pytest.mark.gpu
def test_bit_identical_across_batches_calls_workspaces_and_graphs():
    V = 128256
    trie = ParallelTokenCharacterTrie(synth_vocab(V))
    eng = trie._engine
    rng = np.random.default_rng(8)
    B = 1024
    nodes = np.full(B, trie.root, dtype=np.int32)  # mostly at the root
    nodes[::7] = rng.integers(0, len(trie), len(nodes[::7]))
    ws = torch.tensor(dirichlet_rows(B, V, alpha=0.5, seed=6)).cuda()
    nt = torch.tensor(nodes).cuda()
    ids, s, m = trie.batch_child_masses_tensor(ws, nt, ops=("sum", "max"))
    again = trie.batch_child_masses_tensor(ws, nt, ops=("sum", "max"))
    for a, b in zip((ids, s, m), again):
        assert torch.equal(a, b)
    for r in (0, 7, 517, 1023):  # a row alone
        one = trie.batch_child_masses_tensor(ws[r:r + 1], nt[r:r + 1], ops=("sum", "max"))
        for a, b in zip((ids, s, m), one):
            assert torch.equal(a[r:r + 1], b)
    # a one-row workspace through the C ABI: 64 chunks of one row
    Bs = 64
    need = _lib.lib.gt_child_workspace_bytes(eng._handle, 1)
    work = torch.empty(need, dtype=torch.uint8, device="cuda")
    D = eng.max_children
    ids1 = torch.empty((Bs, D), dtype=torch.int32, device="cuda")
    s1 = torch.empty((Bs, D), dtype=torch.float32, device="cuda")
    m1 = torch.empty((Bs, D), dtype=torch.float32, device="cuda")
    _lib.check(_lib.lib.gt_child_masses(eng._handle, ws.data_ptr(), F32, Bs, V, nt.data_ptr(), ids1.data_ptr(), s1.data_ptr(),
                                        m1.data_ptr(), D, SUM | MAX, 0, work.data_ptr(), need,
                                        torch.cuda.current_stream().cuda_stream), "gt_child_masses")
    for a, b in zip((ids, s, m), (ids1, s1, m1)):
        assert torch.equal(a[:Bs], b)
    # CUDA graph replay == eager
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        trie.batch_child_masses_tensor(ws, nt, ops=("sum", "max"))  # workspace of this stream, before capture
        trie.sample_next_symbol(ws, nt, seed=3)
    torch.cuda.current_stream().wait_stream(st)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        cap = trie.batch_child_masses_tensor(ws, nt, ops=("sum", "max"))
        cap_draw = trie._engine.child_sample(ws, nt, seed=3)
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip((ids, s, m), cap):
        assert torch.equal(a, b)
    for a, b in zip(trie._engine.child_sample(ws, nt, seed=3), cap_draw):
        assert torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["root", "depth1"])
def test_draw_distribution_chi_square(where):
    from scipy import stats

    dec = golden_vocab("synth3000")
    trie = ParallelTokenCharacterTrie(dec)
    node = trie.root if where == "root" else depth1_node(trie)
    row = torch.tensor(dirichlet_rows(1, len(dec), alpha=1.0, seed=21))
    n = 20000
    ws = row.expand(n, -1).cuda()
    nodes = torch.full((n,), node, dtype=torch.int32)
    child, label, logp, logZ = trie.sample_next_symbol(ws, nodes, seed=1234, offset=77)
    ids, sums, _ = trie.batch_child_masses(row, [node])
    deg = int((ids[0] >= 0).sum())
    p = sums[0, :deg].astype(np.float64)
    p /= p.sum()
    pos = {int(c): j for j, c in enumerate(ids[0, :deg])}
    c = child.cpu().numpy()
    assert (c >= 0).all()
    counts = np.bincount([pos[int(x)] for x in c], minlength=deg).astype(np.float64)
    exp = p * n
    big = exp >= 5  # pool the small cells
    obs_b = np.append(counts[big], counts[~big].sum())
    exp_b = np.append(exp[big], exp[~big].sum())
    keep = exp_b > 0
    pval = stats.chisquare(obs_b[keep], exp_b[keep] * obs_b[keep].sum() / exp_b[keep].sum()).pvalue
    assert pval > 1e-4, pval
    assert np.array_equal(label.cpu().numpy(), trie.edge_labels[c])


@pytest.mark.gpu
def test_draw_properties():
    dec = golden_vocab("synth3000")
    trie = ParallelTokenCharacterTrie(dec)
    N, V = len(trie), len(dec)
    B = 2000
    rng = np.random.default_rng(2)
    internal = np.flatnonzero(np.diff(trie._layout["child_ptr"]) > 0)
    nodes = rng.choice(internal, B).astype(np.int32)
    nodes[:50] = trie.root
    ws = torch.tensor(dirichlet_rows(B, V, alpha=0.1, seed=9)).cuda()
    nt = torch.tensor(nodes)
    child, label, logp, logZ = trie.sample_next_symbol(ws, nt, seed=5, offset=10)
    ids, sl, _ = trie.batch_child_masses(ws, nt, log=True)
    _, sln, _ = trie.batch_child_masses(ws, nt, normalize=True, log=True)
    c, lp, lz = child.cpu().numpy(), logp.cpu().numpy(), logZ.cpu().numpy()
    has_mass = np.isfinite(lz)
    assert (c[~has_mass] == -1).all() and np.isneginf(lz[~has_mass]).all()
    col = np.argmax(ids == c[:, None], axis=1)
    hm = np.flatnonzero(has_mass)
    assert (ids[hm, col[hm]] == c[hm]).all()
    assert np.isfinite(sl[hm, col[hm]]).all()  # a zero-mass child is never drawn
    with np.errstate(divide="ignore"):
        lz_want = np.log(np.exp(sl.astype(np.float64)).sum(axis=1))
    np.testing.assert_allclose(lz[hm], lz_want[hm], rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(lp[hm], sln[hm, col[hm]], rtol=1e-6, atol=1e-6)
    assert np.array_equal(label.cpu().numpy()[hm], trie.edge_labels[c[hm]])
    # the same (seed, offset) gives the same draw; counters are offset + row
    again = trie.sample_next_symbol(ws, nt, seed=5, offset=10)
    assert torch.equal(child, again[0]) and torch.equal(logp, again[2]) and torch.equal(logZ, again[3])
    shifted = trie.sample_next_symbol(ws[1:], nt[1:], seed=5, offset=11)[0]
    assert torch.equal(child[1:], shifted)
    assert not torch.equal(child, trie.sample_next_symbol(ws, nt, seed=6, offset=10)[0])


@pytest.mark.gpu
def test_draw_edge_cases():
    dec = golden_vocab("synth3000")
    trie = ParallelTokenCharacterTrie(dec)
    V = len(dec)
    leaf = int(trie.idx_to_leaf[5, 1])
    ws = torch.tensor(dirichlet_rows(5, V, alpha=1.0, seed=1)).cuda()
    ws[3].zero_()
    ws[4, trie.dfs_token_order[0]] = float("nan")  # a NaN under the root
    nodes = torch.tensor([leaf, -1, len(trie), trie.root, trie.root], dtype=torch.int32)
    child, label, logp, logZ = trie.sample_next_symbol(ws, nodes, seed=1)
    c, lz = child.cpu().numpy(), logZ.cpu().numpy()
    assert (c == -1).all() and (label.cpu().numpy() == INT32_MIN).all()
    assert np.isneginf(lz[:4]).all() and np.isnan(lz[4]) and np.isnan(logp.cpu().numpy()[4])
    with pytest.raises(RuntimeError, match="sum of probabilities"):
        trie.sample_next_symbol(ws[:4], nodes[:4], check_valid=True)
    with pytest.raises(RuntimeError, match="nan"):
        trie.sample_next_symbol(ws, nodes, check_valid=True)
    ids, s, m = trie.batch_child_masses(ws[:3], nodes[:3], ops=("sum", "max"))
    assert (ids == -1).all() and (s == 0).all() and (m == 0).all()
    # input checks shared with batch_weight_tensor
    with pytest.raises(AssertionError):
        trie.batch_child_masses_tensor(ws[:, :-1], nodes)
    with pytest.raises(ValueError):
        trie.batch_child_masses_tensor(ws, nodes[:4])
    with pytest.raises(ValueError):
        trie.sample_next_symbol(ws, nodes[None, :])


@pytest.mark.gpu
def test_async_child_masses_batch_together():
    dec = golden_vocab("synth3000")
    atrie = AsyncTokenCharacterTrie(ParallelTokenCharacterTrie(dec))
    trie = atrie.trie
    n = 64
    rows = dirichlet_rows(n, len(dec), alpha=0.3, seed=3)
    nodes = np.random.default_rng(4).integers(0, len(trie), n).astype(np.int32)
    nodes[0] = trie.root
    calls = []
    orig = trie.batch_child_masses

    def counting(*a, **kw):
        calls.append(len(a[1]))
        return orig(*a, **kw)

    trie.batch_child_masses = counting

    async def run():
        try:
            return await asyncio.gather(*[atrie.child_masses(torch.tensor(rows[i]), int(nodes[i]), normalize=True) for i in range(n)])
        finally:
            await atrie.cleanup()

    got = asyncio.run(run())
    assert calls == [n]
    ids, s, _ = orig(torch.tensor(rows), nodes, normalize=True)
    for i, (gi, gs) in enumerate(got):
        deg = len(trie.jump[nodes[i]])
        assert gi.dtype == np.int32 and gs.dtype == np.float32 and len(gi) == len(gs) == deg
        assert np.array_equal(gi, ids[i, :deg]) and np.array_equal(gs, s[i, :deg])
