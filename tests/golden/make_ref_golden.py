#!/usr/bin/env python3
"""Records what the original project computes for the inputs of the parity tests, so that they run without it:

    python tests/golden/make_ref_golden.py host DIR      # CPU only: ref_host.json (tokenizer, sampler, GGUF loader)
    python tests/golden/make_ref_golden.py kernels DIR   # one GPU: ref_kernels.npz
    python tests/golden/make_ref_golden.py models DIR    # one GPU: ref_forward_<mix>.npz, ref_check_*.npz

Needs oracle/_ref/libnt_ref.so, which `make -C oracle ref REF=<checkout of the original project>` compiles (build() does it
when NT_REFERENCE_SRC is set), and a built libnt_b200.so.  The files it writes belong in tests/golden/.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]


def ref_lib():
    return C.CDLL(str(ROOT / "oracle" / "_ref" / "libnt_ref.so"))


def host(out: Path, tmp: Path) -> None:
    import test_ref_host as H
    import test_sample_sim as S

    ref = H._setup(ref_lib())
    cfg, _, gpt2, spm = H.write_files(tmp)
    golden = {"tokenizer": {name: H.record_tokenizer(ref, path, cfg.vocab_size) for name, path in (("gpt2", gpt2), ("spm", spm))},
              "sampler": [ref.ref_sample_token(*H.sample_args(c)) for c in H.sampler_cases()],
              "gguf": H.record_gguf(ref, gpt2)}
    ref.ref_sample_token.argtypes = S.SIG
    golden["sample_sim"] = [ref.ref_sample_token(*S.args_for(*c)) for c in S.draw_cases()]
    (out / "ref_host.json").write_text(json.dumps(golden, separators=(",", ":")) + "\n")


def kernels(out: Path, tmp: Path) -> None:
    import torch
    import test_kernels_gpu as T

    ref = ref_lib()
    dev = T.dev
    stream = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)
    g = {}
    for dt in T.REF_GEMV_DT:
        for out_, inn in T.REF_GEMV_SHAPES:
            if dt in (T.DType.Q8_0, T.DType.Q4_0, T.DType.F16) and inn * 4 > 64 * 1024:
                continue                                          # the test skips these (the reference kernel cannot launch)
            raw, x, key = T.ref_gemv_case(dt, (out_, inn))
            W, xd, yr = dev(raw), dev(x), torch.zeros(out_, device="cuda")
            ref.ref_gemv(C.c_void_p(yr.data_ptr()), C.c_void_p(W.data_ptr()), C.c_void_p(xd.data_ptr()), out_, inn, int(dt), stream())
            torch.cuda.synchronize()
            g[key] = yr.cpu().numpy()
    seq, nh, nkv, hd = T.ROPE_SHAPE
    q, k, pos = T.ref_rope_case()
    qb, kb = dev(q), dev(k)
    ref.ref_rope(C.c_void_p(qb.data_ptr()), C.c_void_p(kb.data_ptr()), C.c_void_p(dev(pos).data_ptr()), 1, seq, nh, nkv, hd,
                 C.c_float(500000.0), C.c_float(1.0), 0, stream())
    torch.cuda.synchronize()
    qo, ko = qb.cpu().numpy(), kb.cpu().numpy()
    g.update(rope_q_sha256=T.sha256(qo), rope_k_sha256=T.sha256(ko), rope_q_every16=qo.reshape(-1)[::16],
             rope_k_every16=ko.reshape(-1)[::16])
    for cfg in T.REF_ATTN_CFGS:
        for ctx in T.REF_ATTN_CTX:
            nh, nkv, hd = cfg
            q, kc, vc, key = T.ref_attention_case(cfg, ctx)
            b = torch.zeros(nh, hd, device="cuda")
            qd, kd, vd = dev(q), dev(kc), dev(vc)
            ref.ref_attention_decode(C.c_void_p(b.data_ptr()), C.c_void_p(qd.data_ptr()), C.c_void_p(kd.data_ptr()),
                                     C.c_void_p(vd.data_ptr()), ctx, nh, nkv, hd, 2048, C.c_float(float(1.0 / np.sqrt(hd))), stream())
            torch.cuda.synchronize()
            g[key] = b.cpu().numpy()
    np.savez_compressed(out / "ref_kernels.npz", **g)


def models(out: Path, tmp: Path) -> None:
    import test_model_gpu as M
    from oracle.trace import Recorder

    ref = ref_lib()
    ref.ref_model_load.restype = C.c_void_p
    ref.ref_model_load.argtypes = [C.c_char_p, C.c_int]
    ref.ref_model_forward.restype = C.c_float
    ref.ref_model_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    ref.ref_model_free.argtypes = [C.c_void_p]
    for mix in ("Q4_K_M", "Q8_0", "Q6_K", "F16"):
        cfg, _, path = M.write_case(mix, tmp)
        h = ref.ref_model_load(str(path).encode(), cfg.max_seq_len)
        assert h
        rec, logits = Recorder(cfg.vocab_size), np.empty(cfg.vocab_size, np.float32)
        toks, pos = np.array(M.REF_PROMPT, np.int32), 0
        for _ in range(M.REF_STEPS + 1):
            ref.ref_model_forward(h, toks.ctypes.data_as(C.c_void_p), len(toks), pos, logits.ctypes.data_as(C.c_void_p))
            rec.add(logits)
            pos += len(toks)
            toks = np.array([int(np.argmax(logits))], np.int32)
        ref.ref_model_free(h)
        np.savez_compressed(out / f"ref_forward_{mix}.npz", **rec.arrays())

    for workload, layers, steps, extra in M.PARITY_CONFIGS:
        cmd = [sys.executable, str(ROOT / "bench.py"), "--check", "--workload", workload, "--steps", str(steps),
               "--record-reference-trace", str(out / M.parity_trace(workload, layers).name)] + extra
        if layers:
            cmd += ["--layers", str(layers)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        print(r.stdout.strip().splitlines()[-1] if r.stdout.strip() else r.stderr[-2000:], flush=True)
        assert r.returncode == 0


if __name__ == "__main__":
    import tempfile

    part, out = sys.argv[1], Path(sys.argv[2])
    out.mkdir(parents=True, exist_ok=True)
    with tempfile.TemporaryDirectory() as tmp:
        {"host": host, "kernels": kernels, "models": models}[part](out, Path(tmp))
