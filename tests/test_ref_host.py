"""Host-side parity against the UNMODIFIED reference code: our GGUF parser, tokenizer and sampler (csrc/engine/{gguf,text}.cpp)
against what the reference's GGUFLoader (src/model/loader.cpp:23-276), Tokenizer (src/inference/tokenizer.cpp:64-314) and Sampler
(src/inference/sampler.cpp:18-117) returned on the same files and inputs, recorded in tests/golden/ref_host.json by
tests/golden/make_ref_golden.py (oracle/_ref/libnt_ref.so, oracle/Makefile `ref`).  No GPU is involved: these are the host rows
(a17, a18) of SURVEY §8, which the reference's own tests do not pin."""
import ctypes as C
import json
from pathlib import Path

import numpy as np
import pytest

from ntransformer_b200._lib import lib
from ntransformer_b200.gguf_write import gpt2_byte_tokens, synthetic_tensors_np, write_gguf
from ntransformer_b200.model_spec import TINY, LlamaConfig

WORDS = ("the quick brown fox jumps over lazy dog hello world how are you today is a good day for inference tokens "
         "quantized decode tensor parallel kernel memory bandwidth roofline").split()


GOLDEN = Path(__file__).resolve().parent / "golden" / "ref_host.json"


@pytest.fixture(scope="module")
def golden():
    return json.loads(GOLDEN.read_text())


def _setup(ref):
    ref.ref_gguf_config.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p]
    ref.ref_gguf_tensor.argtypes = [C.c_char_p, C.c_char_p, C.c_void_p]
    ref.ref_tokenize.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_void_p, C.c_int]
    ref.ref_detokenize.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]
    ref.ref_sample_token.argtypes = [C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_float, C.c_float, C.c_int, C.c_void_p, C.c_int,
                                     C.c_ulonglong]
    return ref


def gpt2_vocab(n):
    """GPT-2 byte-level vocabulary: 256 byte tokens, then words with and without the 'Ġ' space prefix, their prefixes and
    a few multi-byte pieces, padded with placeholders."""
    byte_tok = gpt2_byte_tokens()
    sp = byte_tok[0x20]
    toks = list(byte_tok)
    seen = set(toks)
    for w in WORDS:
        for piece in (w, sp + w, w[:2], w[:3], sp + w[:2], w[-2:], w.capitalize(), sp + w.capitalize()):
            if piece not in seen and len(piece) > 1:
                seen.add(piece)
                toks.append(piece)
    for piece in (sp + sp, sp + sp + sp + sp, byte_tok[0x0A] + byte_tok[0x0A], "".join(byte_tok[b] for b in "é".encode()),
                  "".join(byte_tok[b] for b in "日本".encode())):
        if piece not in seen:
            seen.add(piece)
            toks.append(piece)
    toks += [f"<t{i}>" for i in range(len(toks), n)]
    return toks[:n]


def spm_vocab(n):
    """SentencePiece-style vocabulary: <unk>/<s>/</s>, <0xNN> byte tokens, '▁' word pieces and single characters."""
    toks = ["<unk>", "<s>", "</s>"] + [f"<0x{b:02X}>" for b in range(256)]
    types = [2, 3, 3] + [6] * 256
    seen = set(toks)
    for ch in "abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789.,!?'-\n" + "▁":
        if ch not in seen:
            seen.add(ch); toks.append(ch); types.append(1)
    for w in WORDS:
        for piece in ("▁" + w, w, w[:2], w[:3], "▁" + w[:2], w[-2:], w[-3:]):
            if piece not in seen and len(piece) > 1:
                seen.add(piece); toks.append(piece); types.append(1)
    while len(toks) < n:
        toks.append(f"<t{len(toks)}>"); types.append(1)
    return toks[:n], types[:n]


def write_files(d):
    cfg = LlamaConfig(**{**TINY.dict(), "vocab_size": 1024})
    tensors = synthetic_tensors_np(cfg, "Q4_K_M", seed=3)
    rng = np.random.default_rng(0)
    g = gpt2_vocab(cfg.vocab_size)
    write_gguf(d / "gpt2.gguf", cfg, tensors, vocab_tokens=g, vocab_scores=-np.arange(len(g), dtype=np.float32))
    s, types = spm_vocab(cfg.vocab_size)
    write_gguf(d / "spm.gguf", cfg, tensors, vocab_tokens=s, vocab_scores=rng.standard_normal(len(s)).astype(np.float32) - 5.0,
               vocab_types=types)
    return cfg, tensors, d / "gpt2.gguf", d / "spm.gguf"


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    return write_files(tmp_path_factory.mktemp("refhost"))


TEXTS = ["Hello, how are you?", "hello world", " the quick  brown fox", "The Quick Brown Fox jumps over the lazy dog.", "", " ",
         "a", "tensor parallel kernel\nmemory bandwidth\n\nroofline", "café naïve 日本語 \U0001F600", "1234567890 !@#$%^&*()",
         "today is a good day for inference" * 3, "\t tabs\tand  spaces   ", "x" * 200, "quantizeddecodetokens"]


def ours_tokenize(path, text, add_bos):
    ids = (C.c_int * 4096)()
    n = lib().nt_tokenize(str(path).encode(), text.encode(), int(add_bos), ids, 4096)
    return n, list(ids[: max(n, 0)])


def ref_tokenize(ref, path, text, add_bos):
    ids = (C.c_int * 4096)()
    n = ref.ref_tokenize(str(path).encode(), text.encode(), int(add_bos), ids, 4096)
    return n, list(ids[: max(n, 0)])


def random_id_lists(vocab_size):
    """Arbitrary ids to decode: control / byte / placeholder tokens and out-of-range ids."""
    rng = np.random.default_rng(1)
    return [rng.integers(-2, vocab_size + 3, size=24).astype(np.int32) for _ in range(20)]


def detokenize(fn, path, ids):
    ids = np.ascontiguousarray(ids, dtype=np.int32)
    out = C.create_string_buffer(8192)
    n = fn(str(path).encode(), ids.ctypes.data_as(C.c_void_p), len(ids), out, 8192)
    return [n, out.raw[:max(n, 0)].hex()]


def record_tokenizer(ref, path, vocab_size):
    """The reference's side of test_tokenizer_encode_decode_match_reference (tests/golden/make_ref_golden.py)."""
    encode = [[list(ref_tokenize(ref, path, text, add_bos)) for add_bos in (True, False)] for text in TEXTS]
    decode = [detokenize(ref.ref_detokenize, path, ids) if n > 0 else None for _, (n, ids) in encode]
    return {"encode": encode, "decode": decode,
            "decode_random": [detokenize(ref.ref_detokenize, path, ids) for ids in random_id_lists(vocab_size)]}


@pytest.mark.parametrize("which", ["gpt2", "spm"])
def test_tokenizer_encode_decode_match_reference(golden, files, which, capfd):
    want = golden["tokenizer"][which]
    cfg, _, gpt2, spm = files
    path = gpt2 if which == "gpt2" else spm
    for text, enc, dec in zip(TEXTS, want["encode"], want["decode"]):
        for add_bos, b in zip((True, False), enc):
            a = ours_tokenize(path, text, add_bos)
            assert list(a) == b, (which, text, add_bos, a, b)
        n, ids = ours_tokenize(path, text, False)
        if n == 0:
            continue
        assert detokenize(lib().nt_detokenize, path, ids) == dec, (which, text)
    # decoding arbitrary ids (control / byte / placeholder tokens, out-of-range ids) must agree too
    for ids, dec in zip(random_id_lists(cfg.vocab_size), want["decode_random"]):
        assert detokenize(lib().nt_detokenize, path, ids) == dec, list(ids)
    capfd.readouterr()


def sampler_cases():
    """Arguments of nt_sample_token / ref_sample_token: logits (with ties every 7th), settings and seed."""
    rng = np.random.default_rng(7)
    n = 2048
    for trial in range(60):
        logits = (rng.standard_normal(n) * rng.choice([0.5, 2.0, 6.0])).astype(np.float32)
        if trial % 7 == 0:
            logits[rng.integers(0, n, 5)] = logits.max()                      # ties
        temperature = float(rng.choice([0.0, 0.3, 0.7, 1.0, 1.5]))
        top_k = int(rng.choice([0, 1, 5, 40, n, n + 10]))
        top_p = float(rng.choice([0.0, 0.5, 0.9, 1.0]))
        penalty = float(rng.choice([1.0, 1.1, 1.5]))
        window = int(rng.choice([0, 4, 64]))
        recent = rng.integers(0, n, size=int(rng.integers(0, 80))).astype(np.int32)
        seed = int(rng.integers(0, 2**31))
        yield (logits, n, temperature, top_k, top_p, penalty, window, recent, len(recent), seed)


def sample_args(case):
    logits, n, temperature, top_k, top_p, penalty, window, recent, n_recent, seed = case
    return (logits.ctypes.data_as(C.c_void_p), n, temperature, top_k, top_p, penalty, window,
            recent.ctypes.data_as(C.c_void_p) if n_recent else None, n_recent, seed)


def test_sampler_draws_match_reference(golden):
    for trial, (case, b) in enumerate(zip(sampler_cases(), golden["sampler"], strict=True)):
        a = lib().nt_sample_token(*sample_args(case))
        assert a == b, (trial, case[2:7], case[8], case[9], a, b)


def record_gguf(ref, path):
    """The reference loader's view of the file (tests/golden/make_ref_golden.py)."""
    buf = C.create_string_buffer(4 << 20)
    assert lib().nt_gguf_describe(str(path).encode(), buf, len(buf)) > 0
    out, fout = (C.c_longlong * 12)(), (C.c_float * 2)()
    nt = ref.ref_gguf_config(str(path).encode(), out, fout)
    tensors = {}
    for t in json.loads(buf.value.decode())["tensors"]:
        info = (C.c_longlong * 3)()
        assert ref.ref_gguf_tensor(str(path).encode(), t["name"].encode(), info) == 0
        tensors[t["name"]] = list(info)
    return {"n_tensors": nt, "config": list(out), "norm_eps": fout[0], "rope_theta": fout[1], "tensors": tensors}


def test_gguf_parser_matches_reference_loader(golden, files, capfd):
    cfg, tensors, gpt2, _ = files
    want = golden["gguf"]
    buf = C.create_string_buffer(4 << 20)
    assert lib().nt_gguf_describe(str(gpt2).encode(), buf, len(buf)) > 0
    d = json.loads(buf.value.decode())
    assert want["n_tensors"] == len(d["tensors"]) == len(tensors)
    keys = ("vocab_size", "hidden_size", "intermediate_size", "n_layers", "n_heads", "n_kv_heads", "head_dim", "max_seq_len",
            "bos_token_id", "eos_token_id", "n_vocab_tokens", "data_offset")
    assert [d[k] for k in keys] == want["config"]
    assert abs(d["norm_eps"] - want["norm_eps"]) < 1e-12 and abs(d["rope_theta"] - want["rope_theta"]) < 1e-3
    assert len(want["tensors"]) == len(d["tensors"])
    for t in d["tensors"]:
        assert [t["dtype"], t["offset"], t["nbytes"]] == want["tensors"][t["name"]], t["name"]
    capfd.readouterr()
