"""GPU model-level parity: the native engine (CUDA graph, fused launches) against the CPU oracle on the same
synthetic weights, against the reference's own Transformer::forward on the same GGUF file (its greedy decode
recorded under tests/golden/ by tests/golden/make_ref_golden.py, see oracle/trace.py), and through the reference's
declared C API (include/ntransformer.h).  Tolerance: max|logit diff| / max|logit| <= 1e-3 (BASELINE.json
north_star) — measured values are ~1e-5 — and greedy token ids identical."""
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from ntransformer_b200 import kernels as K
from ntransformer_b200.engine import Engine, Model
from ntransformer_b200.gguf_write import synthetic_tensors_np, write_gguf
from ntransformer_b200.model_spec import TINY, LlamaConfig
from oracle import oracle as O
from oracle.trace import Trace

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
GOLDEN = ROOT / "tests" / "golden"

MID = LlamaConfig(vocab_size=2048, hidden_size=1024, intermediate_size=3584, n_layers=4, n_heads=16, n_kv_heads=4, head_dim=64,
                  max_seq_len=256, bos_token_id=1, eos_token_id=2)


def rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def write_case(mix, d):
    cfg = TINY if mix != "Q6_K" else MID
    tensors = synthetic_tensors_np(cfg, mix, seed=11)
    path = d / f"{mix}.gguf"
    write_gguf(path, cfg, tensors)
    return cfg, tensors, path


@pytest.fixture(scope="module", params=["Q4_K_M", "Q8_0", "Q6_K", "F16"])
def gguf_case(request, tmp_path_factory):
    mix = request.param
    cfg, tensors, path = write_case(mix, tmp_path_factory.mktemp("m"))
    host = {n: (np.ascontiguousarray(a), int(dt)) for n, (a, dt, r, c) in tensors.items()}
    return cfg, mix, path, host


def test_logits_and_greedy_ids_vs_oracle(gguf_case):
    cfg, mix, path, host = gguf_case
    m = Model.load(path, max_context=cfg.max_seq_len)
    om = O.Model(cfg.dict(), host)
    prompt = [cfg.bos_token_id, 17, 300, 5, 44, 9]
    got = m.forward(prompt, 0).copy()
    want = om.forward(prompt, 0)
    assert rel(got, want) <= 1e-3
    pos, ids_a, ids_b, tok_a, tok_b = len(prompt), [], [], int(np.argmax(got)), int(np.argmax(want))
    for _ in range(24):
        ids_a.append(tok_a)
        ids_b.append(tok_b)
        la = m.forward([tok_a], pos).copy()
        lb = om.forward([tok_b], pos)
        assert tok_a != tok_b or rel(la, lb) <= 1e-3
        assert m.argmax() == int(np.argmax(la))              # GPU argmax == host argmax
        tok_a, tok_b, pos = int(np.argmax(la)), int(np.argmax(lb)), pos + 1
    assert ids_a == ids_b
    m.close()


def test_graph_replay_equals_eager_launches(gguf_case):
    cfg, mix, path, host = gguf_case
    a, b = Model.load(path, cfg.max_seq_len), Model.load(path, cfg.max_seq_len)
    b.use_graph(False)
    toks = [1, 2, 3, 250, 7]
    la, lb = a.forward(toks, 0).copy(), b.forward(toks, 0).copy()
    np.testing.assert_array_equal(la, lb)
    np.testing.assert_array_equal(a.forward([9], 5), b.forward([9], 5))
    a.close(), b.close()


@pytest.mark.parametrize("mix,n_prompt,start", [("F16", 16, 0), ("F16", 97, 0), ("F16", 128, 0), ("F16", 40, 23), ("F16", 200, 0),
                                                ("Q4_K_M", 48, 0), ("Q4_K_M", 130, 17), ("Q8_0", 64, 0), ("Q6_K", 33, 5)])
def test_batched_tensor_core_prefill_vs_oracle_and_per_token(tmp_path, mix, n_prompt, start):
    """The tcgen05 batched prefill (csrc/prefill_gemm.cu; quantised mixes go through csrc/prefill_dequant.cu's hi/lo
    expansion) against the oracle's forward and against the per-token replay path; the KV cache it leaves must
    continue into identical greedy decode."""
    from dataclasses import replace
    cfg = replace(TINY if mix != "Q6_K" else MID, max_seq_len=256)
    tensors = synthetic_tensors_np(cfg, mix, seed=5)
    path = tmp_path / "m.gguf"
    write_gguf(path, cfg, tensors)
    host = {n: (np.ascontiguousarray(a), int(dt)) for n, (a, dt, r, c) in tensors.items()}
    rng = np.random.default_rng(n_prompt)
    warm = [int(t) for t in rng.integers(3, cfg.vocab_size, size=start)]
    prompt = [int(t) for t in rng.integers(3, cfg.vocab_size, size=n_prompt)]
    a, b, om = Model.load(path, cfg.max_seq_len), Model.load(path, cfg.max_seq_len), O.Model(cfg.dict(), host)
    b.set_prefill_min_tokens(0)                      # per-token replay
    a.set_prefill_min_tokens(8)
    if start:
        a.set_prefill_min_tokens(0), a.forward(warm, 0), a.set_prefill_min_tokens(8)
        b.forward(warm, 0), om.forward(warm, 0)
    n0 = K.launch_count()
    la = a.forward(prompt, start).copy()
    batched_launches = K.launch_count() - n0
    lb, lo = b.forward(prompt, start).copy(), om.forward(prompt, start)
    assert batched_launches < 40 * cfg.n_layers          # one pass over the layers, not n_prompt of them
    assert rel(la, lo) <= 1e-3 and rel(la, lb) <= 1e-3
    pos, ta, tb = start + n_prompt, int(np.argmax(la)), int(np.argmax(lo))
    for _ in range(12):
        assert ta == tb
        la, lo = a.forward([ta], pos), om.forward([tb], pos)
        assert rel(la, lo) <= 1e-3
        ta, tb, pos = int(np.argmax(la)), int(np.argmax(lo)), pos + 1
    a.close(), b.close()


REF_PROMPT, REF_STEPS = [1, 17, 300, 5, 44, 9], 32


def test_vs_reference_transformer_forward(gguf_case):
    """The reference's greedy decode of the same GGUF, recorded: its ids and, per step, its logits at the positions oracle/trace.py
    keeps (the largest ones and a fixed sample)."""
    cfg, mix, path, host = gguf_case
    with np.load(GOLDEN / f"ref_forward_{mix}.npz") as g:
        ref = Trace(g)
    assert len(ref) == REF_STEPS + 1
    m = Model.load(path, cfg.max_seq_len)
    prompt = np.array(REF_PROMPT, np.int32)
    ours = m.forward(prompt, 0).copy()
    assert ref.rel_err(0, ours) <= 1e-3
    pos, ta, tb, ida, idb = len(prompt), int(np.argmax(ours)), ref.greedy(0), [], []
    for step in range(1, REF_STEPS + 1):
        ida.append(ta)
        idb.append(tb)
        la = m.forward([ta], pos).copy()
        assert ta != tb or ref.rel_err(step, la) <= 1e-3
        ta, tb, pos = int(np.argmax(la)), ref.greedy(step), pos + 1
    assert ida == idb                                        # greedy ids bit-exact with the reference CUDA path
    m.close()


def test_synthetic_device_tensor_path_matches_oracle():
    m = Model.synthetic(TINY, "Q4_K_M", seed=3)
    host = {n: (v[0].cpu().numpy(), int(v[1])) for n, v in m._keep.items()}
    om = O.Model(TINY.dict(), host)
    toks = [1, 100, 200, 300]
    assert rel(m.forward(toks, 0), om.forward(toks, 0)) <= 1e-3
    assert m.bytes_per_token(10) > 0
    m.close()


def test_c_api_engine_and_cli(gguf_case):
    cfg, mix, path, host = gguf_case
    e = Engine()
    assert e.load(str(path))
    assert (e.vocab_size, e.n_layers, e.hidden_size) == (cfg.vocab_size, cfg.n_layers, cfg.hidden_size)
    text = e.generate("Hello", max_tokens=8, temperature=0.0)
    assert isinstance(text, str)
    assert text == e.generate("Hello", max_tokens=8, temperature=0.0)          # greedy is deterministic
    e.close()
    cli = ROOT / "ntransformer_b200" / "ntransformer"
    r = subprocess.run([str(cli), "-m", str(path), "-p", "Hello", "-n", "8", "-t", "0", "--repeat-penalty", "1.0", "-c", "64"],
                       capture_output=True, text=True, errors="replace", timeout=120)
    assert r.returncode == 0 and "Decode: 7 tokens" in r.stderr, r.stderr[-500:]
    r2 = subprocess.run([str(cli), "-m", str(path), "--streaming"], capture_output=True, text=True, errors="replace", timeout=60)
    assert r2.returncode == 1 and "not supported" in r2.stderr


PARITY_CONFIGS = [
    ("llama3-8b-q4_k_m-decode", 8, 64, ["--oracle-steps", "64"]), ("llama3-8b-q8_0-decode", 8, 64, ["--oracle-steps", "64"]),
    ("llama3-70b-q4_k_m-decode", 4, 48, ["--oracle-steps", "48"]), ("llama3-70b-q6_k-decode", 4, 48, ["--oracle-steps", "48"]),
    ("llama3-8b-q4_k_m-decode", 0, 24, ["--oracle-steps", "3"])]


def parity_trace(workload, layers):
    return GOLDEN / f"ref_check_{workload}_{layers}l.npz"


@pytest.mark.parametrize("workload,layers,steps,extra", PARITY_CONFIGS)
def test_parity_at_the_benchmarked_configs(workload, layers, steps, extra):
    """bench.py --check: the benchmark's own seeded weights (8-layer slices of the 8B shapes, 4-layer slices of the 70B shapes with
    full-width tensors, and the full 32-layer 8B stack) through ours, against the reference's CUDA path on the same GGUF (recorded
    by tests/golden/make_ref_golden.py: bench.py --check --record-reference-trace), the F64 oracle beside them.  Greedy ids must be
    identical; logits within 1e-3 of the reference, or — these stacks of random blocks are ill-conditioned: the reference's own F32
    path drifts up to 2.9e-3 from the F64 result over 128 steps on the 8-layer slice, ours 2.8e-3 (profiles/r02_parity_8b.txt) — our
    distance from the F64 result within twice the reference's (bench.py run_check)."""
    import json
    cmd = [sys.executable, str(ROOT / "bench.py"), "--check", "--workload", workload, "--steps", str(steps),
           "--reference-trace", str(parity_trace(workload, layers))] + extra
    if layers:
        cmd += ["--layers", str(layers)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-3000:])
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["ok"] and d["greedy_ids_identical"], d
