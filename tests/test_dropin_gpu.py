"""The drop-in claim, executed: the reference's UNMODIFIED host code — nt::Transformer::forward (src/model/transformer.cpp:604-669),
Attention::forward, FFN::forward, RMSNorm::forward, its GGUF loader and tensor/device core — linked against libnt_b200.so for
every nt::cuda::launch_* it calls (src/cuda/kernels.h:10-74; oracle/Makefile `dropin`, none of the reference's kernels are in
that build) must produce the same greedy ids as the all-reference build (oracle/_ref/libnt_ref.so) on the same GGUF, with logits
within 1e-3 relative, and every kernel it launches must be ours (the library's launch counter moves)."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

from ntransformer_b200 import kernels as K
from ntransformer_b200.gguf_write import synthetic_tensors_np, write_gguf
from ntransformer_b200.model_spec import TINY, LlamaConfig

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
MID = LlamaConfig(vocab_size=2048, hidden_size=1024, intermediate_size=3584, n_layers=4, n_heads=16, n_kv_heads=4, head_dim=64,
                  max_seq_len=256, bos_token_id=1, eos_token_id=2)


def _bind(lib):
    lib.ref_model_load.restype = C.c_void_p
    lib.ref_model_load.argtypes = [C.c_char_p, C.c_int]
    lib.ref_model_forward.restype = C.c_float
    lib.ref_model_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.ref_model_free.argtypes = [C.c_void_p]
    return lib


@pytest.fixture(scope="module")
def dropin_lib():
    p = ROOT / "oracle" / "_ref" / "libnt_dropin.so"
    if not p.exists():
        pytest.skip("oracle/_ref/libnt_dropin.so not built (build() with NT_REFERENCE_SRC set compiles it)")
    return _bind(C.CDLL(str(p)))


def rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


@pytest.mark.parametrize("mix", ["Q4_K_M", "Q8_0", "Q6_K", "F16", "Q4_0"])
def test_reference_host_code_on_our_kernels_matches_the_all_reference_build(ref_lib, dropin_lib, tmp_path, mix):
    cfg = MID if mix in ("Q6_K", "Q4_0") else TINY
    path = tmp_path / f"{mix}.gguf"
    write_gguf(path, cfg, synthetic_tensors_np(cfg, mix, seed=13))
    _bind(ref_lib)
    ha = dropin_lib.ref_model_load(str(path).encode(), cfg.max_seq_len)
    hb = ref_lib.ref_model_load(str(path).encode(), cfg.max_seq_len)
    assert ha and hb
    prompt = np.array([cfg.bos_token_id, 17, 300, 5, 44, 9, 12, 400], np.int32)
    la, lb = np.empty(cfg.vocab_size, np.float32), np.empty(cfg.vocab_size, np.float32)
    n0 = K.launch_count()
    dropin_lib.ref_model_forward(ha, prompt.ctypes.data_as(C.c_void_p), len(prompt), 0, la.ctypes.data_as(C.c_void_p))
    n1 = K.launch_count()
    ref_lib.ref_model_forward(hb, prompt.ctypes.data_as(C.c_void_p), len(prompt), 0, lb.ctypes.data_as(C.c_void_p))
    assert K.launch_count() == n1                                  # the all-reference build never touches our library
    # the reference's host code loops launch_gemv over the prompt's tokens: 7 projections per token per layer, each one OUR launch
    assert n1 - n0 >= len(prompt) * cfg.n_layers * 7
    assert rel(la, lb) <= 1e-3
    pos, ta, tb, ida, idb = len(prompt), int(np.argmax(la)), int(np.argmax(lb)), [], []
    for _ in range(48):
        ida.append(ta)
        idb.append(tb)
        t1, t2 = np.array([ta], np.int32), np.array([tb], np.int32)
        dropin_lib.ref_model_forward(ha, t1.ctypes.data_as(C.c_void_p), 1, pos, la.ctypes.data_as(C.c_void_p))
        ref_lib.ref_model_forward(hb, t2.ctypes.data_as(C.c_void_p), 1, pos, lb.ctypes.data_as(C.c_void_p))
        assert ta != tb or rel(la, lb) <= 1e-3
        ta, tb, pos = int(np.argmax(la)), int(np.argmax(lb)), pos + 1
    assert ida == idb
    dropin_lib.ref_model_free(ha)
    ref_lib.ref_model_free(hb)
