"""Particle resampling: ``smc.resample`` against the torch composition an SMC driver writes today.

Shapes ``G x P`` (groups x particles): 1 x 4096, 1 x 16384, 8 x 512, 64 x 64 and 512 x 8.  Log-weights are seeded normals;
each shape runs at ``tau = inf`` (scale 2: every group resamples) and at ``tau = 0.5`` (per-group scales spread over
[0.2, 1.6], so that about half the groups resample; a single group gets scale 0.9 and resamples).  Times are CUDA-event
medians per call over a CUDA graph of K calls (``child_step_bench.time_graph``); the inputs are a few KB to 256 KB and
stay L2-resident, which is where an SMC driver's weights live.  Routes:

  (a)  ``smc.resample(..., "systematic")``                                   gt_resample
  (a_multinomial), (a_stratified)   the same call under the other two methods
  (b)  the sync-free torch composition: ``amax``, ``exp`` (fp64), ESS from ``sum`` and ``sum`` of squares, ``cumsum``,
       ``searchsorted(right=True)``, ``clamp``, two ``where``; the systematic uniforms are the oracle's Philox stream
       (``tests/resample_oracle.py``), computed once and held on the device, so (b) is timed without drawing them
  (b') (b) run eagerly behind a host ``if (ess < tau * P).any()``: one device-to-host sync per call (no graph; CUDA events
       around K calls)

Before timing, (b) is checked against (a): ESS, resampled flags and ancestors agree except at points within 1e-12 * S of
a CDF value.

``--step``: the weighted-DFA step of DESIGN section 5.12 at 128,256 tokens (``utf8`` table with seeded log-weights, root
nodes), rows in groups of 64, timed as (s) the step alone, (c) the step + ``log_weights += logZ`` + (a) + ``index_select``
of the states and of a token history, and (d) the same with (b): what resampling costs as a share of a step.

Prints one JSON line per (shape, tau, route); ``--out`` also writes them to a file.
"""
import argparse
import json
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from genlm_backend_b200 import smc  # noqa: E402
from child_step_bench import gpu_info, time_graph  # noqa: E402
import resample_oracle as ro  # noqa: E402

SHAPES = [(1, 4096), (1, 16384), (8, 512), (64, 64), (512, 8)]


def weights(G, P, tau, seed):
    rng = np.random.default_rng(seed)
    if tau == math.inf:
        scale = np.full((G, 1), 2.0)
    else:
        scale = np.linspace(0.2, 1.6, G)[:, None] if G > 1 else np.full((1, 1), 0.9)
    return (rng.normal(size=(G, P)) * scale).astype(np.float32)


class TorchResample:
    """The sync-free torch composition of systematic resampling, with the uniforms given."""

    def __init__(self, G, P, u, device):
        self.P = P
        self.j = torch.arange(P, device=device, dtype=torch.float64)
        self.base = (torch.arange(G, device=device, dtype=torch.int64) * P)[:, None]
        self.ident = self.base + torch.arange(P, device=device)
        self.u = u  # [G, 1] float64
        self.logP = math.log(P)

    def __call__(self, lw, tau):
        m = lw.amax(1, keepdim=True)
        w = torch.exp(lw.double() - m.double())
        S = w.sum(1, keepdim=True)
        Q = (w * w).sum(1, keepdim=True)
        ess = S * S / Q
        c = w.cumsum(1)
        t = (self.j + self.u) / self.P * c[:, -1:]
        i = torch.searchsorted(c, t, right=True).clamp_(max=self.P - 1)
        do = ess < tau * self.P
        anc = torch.where(do, i + self.base, self.ident)
        lmw = (m.double() + S.log() - self.logP).float()
        return anc, torch.where(do, lmw, lw), ess.squeeze(1).float(), lmw.squeeze(1), do.squeeze(1)

    def eager_host_if(self, lw, tau):
        m = lw.amax(1, keepdim=True)
        w = torch.exp(lw.double() - m.double())
        S = w.sum(1, keepdim=True)
        ess = S * S / (w * w).sum(1, keepdim=True)
        do = ess < tau * self.P
        if not bool(do.any()):  # the host-side driver's decision: one sync per call
            return self.ident, lw
        c = w.cumsum(1)
        t = (self.j + self.u) / self.P * c[:, -1:]
        i = torch.searchsorted(c, t, right=True).clamp_(max=self.P - 1)
        lmw = (m.double() + S.log() - self.logP).float()
        return torch.where(do, i + self.base, self.ident), torch.where(do, lmw, lw)


def time_eager(fn, args, K, reps):
    for _ in range(3):
        fn(*args)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(reps):
        t0.record()
        for _ in range(K):
            fn(*args)
        t1.record()
        t1.synchronize()
        times.append(t0.elapsed_time(t1) * 1e3 / K)
    return float(np.median(times)), float(np.min(times))


def check_agreement(a, b, lw, u, P):
    anc_a, _, ess_a, _, res_a = [x.cpu().numpy() for x in a]
    anc_b, _, ess_b, _, res_b = [x.cpu().numpy() for x in b]
    assert np.array_equal(res_a, res_b), "resampled flags differ"
    assert np.allclose(ess_a, ess_b, rtol=1e-6), "ESS differs"
    lw64 = lw.double().cpu().numpy()
    c = np.cumsum(np.exp(lw64 - lw64.max(axis=1, keepdims=True)), axis=1)
    t = (np.arange(P) + u.cpu().numpy()) / P * c[:, -1:]
    for g in np.flatnonzero(res_a):  # only points within 1e-12 * S of a CDF value may differ
        diff = anc_a[g] != anc_b[g]
        k = np.clip(np.searchsorted(c[g], t[g, diff]), 1, P - 1)
        gap = np.minimum(np.abs(c[g, k] - t[g, diff]), np.abs(c[g, k - 1] - t[g, diff]))
        assert (gap <= 1e-12 * c[g, -1]).all(), f"group {g}: ancestors differ away from a CDF boundary"


def resample_rows(args, gpu, power, stream):
    lines = []
    for G, P in SHAPES:
        for tau in (math.inf, 0.5):
            lw = torch.tensor(weights(G, P, tau, seed=G * 31 + P)).cuda()
            seed, offset = 5, 0
            u = torch.tensor(ro.uniforms(seed, np.arange(G, dtype=np.uint64) * P + offset)[:, None]).cuda()
            tr = TorchResample(G, P, u, "cuda")
            a = smc.resample(lw, "systematic", tau, seed=seed, offset=offset)
            check_agreement(a, tr(lw, tau), lw, u, P)
            frac = float(a[4].float().mean())
            routes = {
                "a_resample": (lambda x: smc.resample(x, "systematic", tau, seed=seed, offset=offset), True),
                "a_multinomial": (lambda x: smc.resample(x, "multinomial", tau, seed=seed, offset=offset), True),
                "a_stratified": (lambda x: smc.resample(x, "stratified", tau, seed=seed, offset=offset), True),
                "b_torch": (lambda x: tr(x, tau), True),
                "b_torch_eager_host_if": (lambda x: tr.eager_host_if(x, tau), False),
            }
            res = {}
            for name, (fn, graph) in routes.items():
                if graph:
                    res[name] = time_graph(fn, [(lw,)], args.calls, args.reps, stream)
                else:
                    res[name] = time_eager(fn, (lw,), args.calls, args.reps)
            for name, (med, best) in res.items():
                line = {"G": G, "P": P, "tau": "inf" if tau == math.inf else tau, "route": name,
                        "us_per_call": round(med, 2), "us_per_call_min": round(best, 2),
                        "time_vs_a": round(med / res["a_resample"][0], 2), "groups_resampled": round(frac, 3),
                        "calls_per_graph": args.calls, "gpu": gpu, "power_limit": power}
                lines.append(line)
                print(json.dumps(line), flush=True)
    return lines


def step_rows(args, gpu, power, stream):
    from genlm_backend_b200 import ParallelTokenCharacterTrie
    from genlm_backend_b200.synthetic import logsoftmax_rows, synth_vocab
    from child_step_bench import L2_BYTES
    from dfa_step_bench import random_logw, utf8_dfa

    V = 128256
    trie = ParallelTokenCharacterTrie(synth_vocab(V))
    table = utf8_dfa(trie.num_symbols)
    delta = torch.tensor(table).cuda()
    logw = torch.tensor(random_logw(table, seed=10)).cuda()
    lines = []
    for B in (64, 1024):
        G, P = B // 64, 64
        sets = max(2, -(-3 * L2_BYTES // (4 * B * V)))
        logps = [torch.tensor(logsoftmax_rows(B, V, seed=s)).cuda() for s in range(sets)]
        rng = np.random.default_rng(7)
        states = [torch.zeros(B, dtype=torch.int32, device="cuda") for _ in range(sets)]
        lws = [torch.tensor((rng.normal(size=B) * 2).astype(np.float32)).cuda() for _ in range(sets)]
        hist = [torch.zeros((B, 16), dtype=torch.int32, device="cuda") for _ in range(sets)]
        bufs = list(zip(logps, states, lws, hist))
        u = torch.tensor(ro.uniforms(1, np.arange(G, dtype=np.uint64) * P)[:, None]).cuda()
        tr = TorchResample(G, P, u, "cuda")

        def step(lp, q, lw, h):
            tokw = trie.dfa_token_logw(delta, logw, q)
            logZ, tok = smc.masked_logsumexp_sample(lp, tokw, seed=1)
            return logZ, tok, trie.dfa_advance(delta, q, tok)

        def step_a(lp, q, lw, h):
            logZ, tok, q2 = step(lp, q, lw, h)
            anc, lw2, *_ = smc.resample((lw + logZ).view(G, P), "systematic", 0.5, seed=1)
            idx = anc.view(-1)
            return q2.index_select(0, idx), h.index_select(0, idx), lw2.view(-1)

        def step_b(lp, q, lw, h):
            logZ, tok, q2 = step(lp, q, lw, h)
            anc, lw2, *_ = tr((lw + logZ).view(G, P), 0.5)
            idx = anc.view(-1)
            return q2.index_select(0, idx), h.index_select(0, idx), lw2.view(-1)

        for s in range(2):  # the two steps compute the same reindexing and (to rounding) the same log-weights
            (qa, ha, la), (qb, hb, lb) = step_a(*bufs[s]), step_b(*bufs[s])
            assert torch.equal(qa, qb) and torch.equal(ha, hb) and torch.allclose(la, lb, rtol=1e-6, atol=1e-6)
        res = {name: time_graph(fn, bufs, args.steps, args.reps, stream)
               for name, fn in (("s_step", step), ("c_step_resample", step_a), ("d_step_torch_resample", step_b))}
        for name, (med, best) in res.items():
            line = {"B": B, "G": G, "P": P, "dfa": "utf8", "mix": "root", "route": name, "us_per_step": round(med, 2),
                    "us_per_step_min": round(best, 2),
                    "resample_share": round((med - res["s_step"][0]) / med, 3) if name != "s_step" else None,
                    "V": V, "buffer_sets": sets, "steps_per_graph": args.steps, "gpu": gpu, "power_limit": power}
            lines.append(line)
            print(json.dumps(line), flush=True)
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20, help="calls per CUDA graph")
    ap.add_argument("--steps", type=int, default=20, help="steps per CUDA graph (--step)")
    ap.add_argument("--reps", type=int, default=20, help="graph replays timed (median reported)")
    ap.add_argument("--step", action="store_true", help="also time the weighted-DFA step with and without resampling")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "resample_bench.py measures on a GPU"
    gpu, power = gpu_info()
    stream = torch.cuda.Stream()
    lines = resample_rows(args, gpu, power, stream)
    if args.step:
        lines += step_rows(args, gpu, power, stream)
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
