"""bench.py's reference arm runs without a GPU: it must print ONE JSON line with the contract's keys, must not load the
product package, and must use every host thread whatever OMP_NUM_THREADS says (torchrun sets it to 1).  On the GPU,
--dump-outputs must write what the last timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, env=e, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def test_reference_arm_line():
    d = run_bench("--impl", "reference", "--vocab", "3000", "--batch", "16", "--steps", "3", "--warmup", "1", env={"OMP_NUM_THREADS": "1"})
    assert d["impl"] == "reference" and d["unit"] == "distributions/s" and d["higher_is_better"] is True
    assert d["steps"] == 3 and d["warmup"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["product_package_loaded"] is False
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"]
    want = min(16, len(os.sched_getaffinity(0)))  # OpenMP over the 16 rows of a step, OMP_NUM_THREADS ignored
    assert cb["cores"] == want, cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("batch_weight_sum + batch_weight_max") and d["config"]["vocab"] == 3000


def test_reference_arm_other_ranks_and_workloads():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--vocab", "3000"], capture_output=True,
                         text=True, env={**os.environ, "RANK": "1", "WORLD_SIZE": "2"}, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ""  # ranks other than 0 exit without work
    d = run_bench("--impl", "reference", "--workload", "smc4096")
    assert d["impl"] == "reference" and "unavailable" in d


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    """With one timed step the last step is step 0, on the first buffer set: bench.py's rows dirichlet_rows(B, V, alpha=1,
    seed=1).  At this size every node fits the dump, so the files hold the whole [B, N] results."""
    import oracle
    from genlm_backend_b200 import TokenCharacterTrie
    from genlm_backend_b200.synthetic import synth_vocab, dirichlet_rows
    from helpers import rel_err

    V, B = 3000, 16
    d = run_bench("--vocab", str(V), "--batch", str(B), "--steps", "1", "--warmup", "1", "--e2e-steps", "1", "--no-sampler",
                  "--no-cpu-baseline", "--no-reference-gpu", "--dump-outputs", str(tmp_path))
    assert d["steps"] == 1 and d["value"] > 0
    trie = TokenCharacterTrie(synth_vocab(V))  # the host layout only
    N = len(trie)
    ids, s, m = (np.load(tmp_path / f"{n}.npy") for n in ("node_ids", "weight_sum", "weight_max"))
    assert ids.dtype == np.float64 and np.array_equal(ids, np.arange(N))
    assert s.dtype == m.dtype == np.float32 and s.shape == m.shape == (B, N)
    lay = trie._layout
    o = oracle.OracleLayout(trie.idx_to_leaf, lay["child_ptr"], lay["child_idx"])
    ws = dirichlet_rows(B, V, alpha=1.0, seed=1)
    r, z = rel_err(s, o.weight_sum(ws))
    assert r <= 2e-6 and z == 0.0
    assert np.array_equal(m, o.weight_max(ws).astype(np.float32))
