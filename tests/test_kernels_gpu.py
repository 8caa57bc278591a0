"""GPU parity tests: every entry point is called through the C-ABI of libnt_b200.so and compared with the CPU
oracle on the same seeded inputs, and with what the reference's own CUDA kernels computed from those inputs
(tests/golden/ref_kernels.npz, recorded by tests/golden/make_ref_golden.py).

Tolerances (floating point, stated per test): GEMV max|d| <= 2e-5 * max|y| against the F64-accumulating
oracle (BASELINE north_star allows 1e-3 on logits); attention 2e-5 abs on O(1) outputs."""
import ctypes as C
import hashlib
from pathlib import Path

import numpy as np
import pytest
import torch

from ntransformer_b200 import kernels as K
from ntransformer_b200.dtypes import DType, dtype_row_size
from ntransformer_b200.synth import random_blocks_np
from oracle import oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
GOLDEN = Path(__file__).resolve().parent / "golden" / "ref_kernels.npz"


@pytest.fixture(scope="module")
def golden():
    with np.load(GOLDEN) as g:
        return dict(g)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def sync():
    torch.cuda.synchronize()


def rel_err(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


GEMV_SHAPES = [(4, 256), (13, 512), (64, 4096), (1024, 8192), (257, 14336), (9, 28672), (100, 3584), (33, 1024)]
ALL_DT = [DType.Q4_K_M, DType.Q5_K, DType.Q6_K, DType.Q8_0, DType.Q4_0, DType.F16, DType.F32]


@pytest.mark.parametrize("dt", ALL_DT)
@pytest.mark.parametrize("shape", GEMV_SHAPES)
def test_gemv_vs_oracle(dt, shape):
    out, inn = shape
    rng = np.random.default_rng(out * 131 + inn + int(dt))
    raw = random_blocks_np(dt, out, inn, rng)
    x = rng.standard_normal(inn).astype(np.float32)
    x[::97] *= 30.0                                    # outlier channels, as real activations have
    W, xd = dev(raw), dev(x)
    y = torch.full((out,), 7.0, device=DEV, dtype=torch.float32)
    K.launch_gemv(y, W, xd, out, inn, dt)
    sync()
    ref = O.gemv(raw, x, out, inn, int(dt))
    assert rel_err(y.cpu().numpy(), ref) <= 2e-5


REF_GEMV_DT = [DType.Q4_K_M, DType.Q5_K, DType.Q6_K, DType.Q8_0, DType.Q4_0, DType.F16]
REF_GEMV_SHAPES = [(64, 4096), (40, 8192), (12, 28672)]


def ref_gemv_case(dt, shape):
    """Inputs of test_gemv_vs_reference_cuda and the key of the reference's output in the golden file."""
    out, inn = shape
    rng = np.random.default_rng(out + inn + 17 * int(dt))
    raw = random_blocks_np(dt, out, inn, rng)
    x = rng.standard_normal(inn).astype(np.float32)
    return raw, x, f"gemv_{dt.name}_{out}x{inn}"


@pytest.mark.parametrize("dt", REF_GEMV_DT)
@pytest.mark.parametrize("shape", REF_GEMV_SHAPES)
def test_gemv_vs_reference_cuda(golden, dt, shape):
    out, inn = shape
    if dt in (DType.Q8_0, DType.Q4_0, DType.F16) and inn * 4 > 64 * 1024:
        pytest.skip("reference kernel needs > 64 KB dynamic smem for this dtype (SURVEY 3.3) and fails to launch")
    raw, x, key = ref_gemv_case(dt, shape)
    y = torch.zeros(out, device=DEV)
    K.launch_gemv(y, dev(raw), dev(x), out, inn, dt)
    sync()
    assert rel_err(y.cpu().numpy(), golden[key]) <= 2e-5


def f16bits(v):
    return int(np.array([v], dtype=np.float16).view(np.uint16)[0])


def test_reference_kats_through_cabi():
    # tests/test_gemm.cpp:26-61, 76-158, 266-393
    W = dev(np.arange(1, 13, dtype=np.float32).reshape(4, 3))
    y = torch.zeros(4, device=DEV)
    K.launch_gemv(y, W, torch.ones(3, device=DEV), 4, 3, DType.F32)
    blk = np.zeros((2, 18), np.uint8)
    blk[:, 0:2] = np.array([f16bits(0.5)], np.uint16).view(np.uint8)
    blk[0, 2:] = (10 << 4) | 10
    blk[1, 2:] = (7 << 4) | 7
    y2 = torch.zeros(2, device=DEV)
    K.launch_gemv(y2, dev(blk), torch.ones(32, device=DEV), 2, 32, DType.Q4_0)
    sync()
    np.testing.assert_allclose(y.cpu().numpy(), [6, 15, 24, 33], atol=1e-3)
    np.testing.assert_allclose(y2.cpu().numpy(), [32.0, -16.0], atol=0.1)
    for Kin, tol in ((256, 0.5), (32768, 1.0)):
        b = np.zeros(210, np.uint8)
        b[192:208] = 1
        b[208:210] = np.array([f16bits(1.0)], np.uint16).view(np.uint8)
        r0, r1 = b.copy(), b.copy()
        r0[0:128], r0[128:192] = 0x11, 0xAA
        r1[0:128], r1[128:192] = 0xFF, 0x55
        Wq = dev(np.stack([np.tile(r0, Kin // 256), np.tile(r1, Kin // 256)]))
        y3 = torch.zeros(2, device=DEV)
        K.launch_gemv(y3, Wq, torch.ones(Kin, device=DEV), 2, Kin, DType.Q6_K)
        sync()
        np.testing.assert_allclose(y3.cpu().numpy(), [Kin, -Kin], atol=tol)


def test_unsupported_dtype_is_a_noop():
    y = torch.full((4,), 3.0, device=DEV)
    K.launch_gemv(y, torch.zeros(1024, device=DEV, dtype=torch.uint8), torch.ones(256, device=DEV), 4, 256, DType.Q2_K)
    sync()
    assert (y == 3.0).all()             # reference: stderr + untouched output (gemm.cu:801-803)


def test_quantize_x_reconstruction():
    rng = np.random.default_rng(2)
    Kn = 4096
    x = (rng.standard_normal(Kn) * np.exp(rng.standard_normal(Kn))).astype(np.float32)
    x[64:96] = 0.0                                               # an all-zero block
    xq = torch.zeros(K.xq_bytes(Kn), device=DEV, dtype=torch.uint8)
    K.quantize_x(dev(x), xq, Kn)
    sync()
    raw = xq.cpu().numpy()
    e = np.arange(Kn)
    swz = e ^ (((e >> 7) & 7) << 4)                             # planes are stored in the GEMV's swizzled order
    q = raw[: 3 * Kn].view(np.int8).reshape(3, Kn)[:, swz].astype(np.float64)
    scale = raw[3 * Kn: 3 * Kn + Kn // 32 * 4].view(np.float32).astype(np.float64)
    sum16 = raw[3 * Kn + Kn // 32 * 4:].view(np.float32)
    xhat = np.repeat(scale, 32) * (q[0] * 16384 + q[1] * 128 + q[2])
    bmax = np.repeat(np.abs(x.reshape(-1, 32)).max(1), 32)
    assert (np.abs(xhat - x) <= bmax * 2.0 ** -21 + 1e-30).all()
    np.testing.assert_allclose(sum16, x.reshape(-1, 16).astype(np.float64).sum(1), rtol=1e-5, atol=1e-5)
    assert np.abs(q[1]).max() <= 64 and np.abs(q[2]).max() <= 64 and np.abs(q[0]).max() <= 127


@pytest.mark.parametrize("inn", [4096, 8192])
def test_gemv_fused_qkv_mixed_dtypes_and_residual(inn):
    rng = np.random.default_rng(inn)
    outs, dts = [inn, 1024, 1024], [DType.Q4_K_M, DType.Q4_K_M, DType.Q6_K]
    raws = [random_blocks_np(d, o, inn, rng) for o, d in zip(outs, dts)]
    x = rng.standard_normal(inn).astype(np.float32)
    xq = torch.zeros(K.xq_bytes(inn), device=DEV, dtype=torch.uint8)
    K.quantize_x(dev(x), xq, inn)
    Ws = [dev(r) for r in raws]
    ys = [torch.zeros(o, device=DEV) for o in outs]
    K.gemv_fused(ys, Ws, outs, dts, inn, xq, epilogue=0)
    sync()
    for y, r, o, d in zip(ys, raws, outs, dts):
        assert rel_err(y.cpu().numpy(), O.gemv(r, x, o, inn, int(d))) <= 2e-5
    # residual epilogue: y += W.x
    base = rng.standard_normal(outs[0]).astype(np.float32)
    yb = dev(base)
    K.gemv_fused([yb], [Ws[0]], [outs[0]], [dts[0]], inn, xq, epilogue=1)
    sync()
    want = base + O.gemv(raws[0], x, outs[0], inn, int(dts[0]))
    assert rel_err(yb.cpu().numpy(), want) <= 2e-5


def test_gemv_fused_swiglu():
    rng = np.random.default_rng(4)
    inn, inter = 4096, 1536 + 3
    g, u = random_blocks_np(DType.Q4_K_M, inter, inn, rng, std=0.05), random_blocks_np(DType.Q4_K_M, inter, inn, rng, std=0.05)
    x = rng.standard_normal(inn).astype(np.float32)
    xq = torch.zeros(K.xq_bytes(inn), device=DEV, dtype=torch.uint8)
    K.quantize_x(dev(x), xq, inn)
    act = torch.zeros(inter, device=DEV)
    dummy = torch.zeros(inter, device=DEV)
    K.gemv_fused([act, dummy], [dev(g), dev(u)], [inter, inter], [DType.Q4_K_M] * 2, inn, xq, epilogue=2)
    sync()
    want = O.silu_mul(O.gemv(g, x, inter, inn, O.Q4_K), O.gemv(u, x, inter, inn, O.Q4_K))
    assert rel_err(act.cpu().numpy(), want) <= 5e-5


@pytest.mark.parametrize("rows,hidden", [(1, 4096), (1, 8192), (3, 1000), (2, 64)])
def test_rmsnorm(rows, hidden, request):
    rng = np.random.default_rng(hidden)
    x = rng.standard_normal((rows, hidden)).astype(np.float32) * 3
    w = (1 + 0.1 * rng.standard_normal(hidden)).astype(np.float32)
    y = torch.zeros(rows, hidden, device=DEV)
    K.launch_rmsnorm(y, dev(x), dev(w), rows, hidden, 1e-5)
    yh = torch.zeros(rows, hidden, device=DEV, dtype=torch.float16)
    K.launch_rmsnorm_f16(yh, dev(x), dev(w), rows, hidden, 1e-5)
    sync()
    want = O.rmsnorm(x, w, 1e-5)
    np.testing.assert_allclose(y.cpu().numpy(), want, rtol=2e-6, atol=1e-6)
    np.testing.assert_allclose(yh.cpu().numpy().astype(np.float32), want, rtol=1e-3, atol=1e-3)


@pytest.mark.parametrize("interleaved", [False, True])
def test_rope_and_kv_cache(interleaved, request):
    rng = np.random.default_rng(8)
    seq, nh, nkv, hd, max_seq = 5, 8, 2, 128, 64
    q = rng.standard_normal((seq, nh, hd)).astype(np.float32)
    k = rng.standard_normal((seq, nkv, hd)).astype(np.float32)
    v = rng.standard_normal((seq, nkv, hd)).astype(np.float32)
    pos = np.array([0, 1, 17, 40, 2047], np.int32)
    qd, kd = dev(q), dev(k)
    K.launch_rope(qd, kd, dev(pos), 1, seq, nh, nkv, hd, 500000.0, 1.0, interleaved)
    kc = torch.zeros(max_seq, nkv, hd, device=DEV, dtype=torch.float16)
    vc = torch.zeros_like(kc)
    K.launch_copy_to_kv_cache(kc, vc, kd, dev(v), seq, nkv, hd, 60, max_seq)     # last token falls off the cache
    sync()
    qo, ko = O.rope(q, k, pos, nh, nkv, hd, 500000.0, 1.0, interleaved)
    # fast-math sin/cos/pow at |angle| up to 2047 rad: ~|angle| * 2^-21 absolute (SURVEY quirk Q2)
    np.testing.assert_allclose(qd.cpu().numpy(), qo, atol=5e-3)
    np.testing.assert_allclose(qd.cpu().numpy()[:4], qo[:4], atol=2e-4)
    kcw = np.zeros((max_seq, nkv, hd), np.uint16)
    vcw = np.zeros_like(kcw)
    O.copy_to_kv_cache(kcw, vcw, kd.cpu().numpy(), v, seq, nkv, hd, 60, max_seq)
    np.testing.assert_array_equal(kc.cpu().numpy().view(np.uint16), kcw)          # bit-exact F16 RN
    np.testing.assert_array_equal(vc.cpu().numpy().view(np.uint16), vcw)


ROPE_SHAPE = (7, 64, 8, 128)                                     # seq, n_heads, n_kv_heads, head_dim


def ref_rope_case():
    rng = np.random.default_rng(80)
    seq, nh, nkv, hd = ROPE_SHAPE
    q = rng.standard_normal((seq, nh, hd)).astype(np.float32)
    k = rng.standard_normal((seq, nkv, hd)).astype(np.float32)
    return q, k, np.array([0, 1, 100, 1000, 2047, 4095, 8191], np.int32)


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def test_rope_matches_reference_cuda_bitwise(golden):
    """The golden file keeps the SHA-256 of the reference's rotated q and k (bit-exact comparison) and every 16th value."""
    seq, nh, nkv, hd = ROPE_SHAPE
    q, k, pos = ref_rope_case()
    qa, ka = dev(q), dev(k)
    K.launch_rope(qa, ka, dev(pos), 1, seq, nh, nkv, hd, 500000.0, 1.0, False)
    sync()
    qo, ko = qa.cpu().numpy(), ka.cpu().numpy()
    np.testing.assert_array_equal(qo.reshape(-1)[::16], golden["rope_q_every16"])
    np.testing.assert_array_equal(ko.reshape(-1)[::16], golden["rope_k_every16"])
    assert (sha256(qo), sha256(ko)) == (str(golden["rope_q_sha256"]), str(golden["rope_k_sha256"]))   # same fast-math instruction sequence


def test_elementwise_ops():
    rng = np.random.default_rng(6)
    n = 28672 + 5
    a, b = rng.standard_normal(n).astype(np.float32) * 4, rng.standard_normal(n).astype(np.float32)
    out = torch.zeros(n, device=DEV)
    K.launch_silu_mul(out, dev(a), dev(b), n)
    sync()
    np.testing.assert_allclose(out.cpu().numpy(), O.silu_mul(a, b), rtol=2e-6, atol=2e-6)
    ad = dev(a)
    K.launch_add_inplace(ad, dev(b), n)
    K.launch_add(out, dev(a), dev(b), n)
    cp = torch.zeros(n, device=DEV)
    K.launch_copy(cp, ad, n)
    yb = dev(a)
    K.launch_add_bias(yb, dev(b), n)
    cos = torch.zeros(1, device=DEV)
    K.launch_cosine_similarity(cos, dev(a), dev(b), n)
    sync()
    np.testing.assert_array_equal(ad.cpu().numpy(), a + b)
    np.testing.assert_array_equal(out.cpu().numpy(), a + b)
    np.testing.assert_array_equal(cp.cpu().numpy(), a + b)
    np.testing.assert_array_equal(yb.cpu().numpy(), a + b)
    want = float(a.astype(np.float64) @ b / (np.linalg.norm(a.astype(np.float64)) * np.linalg.norm(b.astype(np.float64))))
    assert abs(float(cos.item()) - want) < 1e-5


def test_softmax_and_gemm_f32():
    rng = np.random.default_rng(12)
    rows, cols = 5, 3001
    x = rng.standard_normal((rows, cols)).astype(np.float32) * 5
    mask = rng.random((rows, cols)) > 0.3
    o1, o2 = torch.zeros(rows, cols, device=DEV), torch.zeros(rows, cols, device=DEV)
    K.launch_softmax(o1, dev(x), rows, cols)
    K.launch_masked_softmax(o2, dev(x), dev(mask), rows, cols)
    M, N, Kd = 33, 47, 129
    A, B = rng.standard_normal((M, Kd)).astype(np.float32), rng.standard_normal((N, Kd)).astype(np.float32)
    Cm = torch.zeros(M, N, device=DEV)
    K.launch_gemm_f32(Cm, dev(A), dev(B), M, N, Kd)
    sync()
    e = np.exp(x - x.max(1, keepdims=True))
    np.testing.assert_allclose(o1.cpu().numpy(), e / e.sum(1, keepdims=True), rtol=1e-5, atol=1e-8)
    xm = np.where(mask, x, -np.inf)
    em = np.exp(xm - xm.max(1, keepdims=True))
    np.testing.assert_allclose(o2.cpu().numpy(), em / em.sum(1, keepdims=True), rtol=1e-5, atol=1e-8)
    np.testing.assert_allclose(Cm.cpu().numpy(), A @ B.T, rtol=1e-4, atol=1e-4)


ATTN_CFGS = [(32, 8, 128), (64, 8, 128), (8, 8, 128), (4, 2, 64), (6, 2, 128), (16, 1, 256)]


def make_cache(rng, max_seq, nkv, hd):
    kc = (rng.standard_normal((max_seq, nkv, hd)) * 0.7).astype(np.float16)
    vc = rng.standard_normal((max_seq, nkv, hd)).astype(np.float16)
    return kc, vc


@pytest.mark.parametrize("cfg", ATTN_CFGS)
@pytest.mark.parametrize("ctx", [1, 5, 64, 65, 300, 2048])
def test_attention_decode_vs_oracle(cfg, ctx):
    nh, nkv, hd = cfg
    rng = np.random.default_rng(nh * 7 + ctx)
    max_seq = 2048
    kc, vc = make_cache(rng, max_seq, nkv, hd)
    q = rng.standard_normal((nh, hd)).astype(np.float32)
    scale = 1.0 / np.sqrt(hd)
    out = torch.zeros(nh, hd, device=DEV)
    K.launch_attention_decode(out, dev(q), dev(kc), dev(vc), ctx, nh, nkv, hd, max_seq, float(scale))
    sync()
    want = O.attention_decode(q, kc.view(np.uint16), vc.view(np.uint16), ctx, nh, nkv, hd, max_seq, scale)
    np.testing.assert_allclose(out.cpu().numpy(), want, atol=2e-5, rtol=1e-4)


REF_ATTN_CFGS, REF_ATTN_CTX = [(32, 8, 128), (64, 8, 128)], [17, 2048]


def ref_attention_case(cfg, ctx):
    """Inputs of test_attention_decode_vs_reference_cuda and the key of the reference's output in the golden file."""
    nh, nkv, hd = cfg
    rng = np.random.default_rng(nh + ctx)
    kc, vc = make_cache(rng, 2048, nkv, hd)
    q = rng.standard_normal((nh, hd)).astype(np.float32)
    return q, kc, vc, f"attn_{nh}_{nkv}_{hd}_ctx{ctx}"


@pytest.mark.parametrize("cfg", REF_ATTN_CFGS)
@pytest.mark.parametrize("ctx", REF_ATTN_CTX)
def test_attention_decode_vs_reference_cuda(golden, cfg, ctx):
    nh, nkv, hd = cfg
    max_seq = 2048
    q, kc, vc, key = ref_attention_case(cfg, ctx)
    scale = float(1.0 / np.sqrt(hd))
    a = torch.zeros(nh, hd, device=DEV)
    K.launch_attention_decode(a, dev(q), dev(kc), dev(vc), ctx, nh, nkv, hd, max_seq, scale)
    sync()
    np.testing.assert_allclose(a.cpu().numpy(), golden[key], atol=2e-5, rtol=1e-4)


@pytest.mark.parametrize("cfg", [(32, 8, 128), (4, 2, 64)])
@pytest.mark.parametrize("seq,start", [(1, 0), (7, 0), (5, 11), (33, 100), (16, 0), (64, 0), (100, 37), (200, 50), (65, 63)])
def test_attention_prefill_vs_oracle(cfg, seq, start):
    """seq < 16 runs the per-query kernel, seq >= 16 the tiled mma.sync kernel (attention_prefill_mma.cu); the cache is
    random beyond the visible range too (250 rows: the last key tile runs past max_seq), so masking is exercised."""
    nh, nkv, hd = cfg
    rng = np.random.default_rng(seq * 31 + start)
    max_seq = 250
    kc, vc = make_cache(rng, max_seq, nkv, hd)
    Q = rng.standard_normal((seq, nh, hd)).astype(np.float32)
    scale = 1.0 / np.sqrt(hd)
    out = torch.zeros(seq, nh, hd, device=DEV)
    K.launch_attention_prefill(out, dev(Q), dev(kc), dev(vc), seq, start, nh, nkv, hd, max_seq, float(scale))
    sync()
    want = O.attention_prefill(Q, kc.view(np.uint16), vc.view(np.uint16), seq, start, nh, nkv, hd, max_seq, scale)
    np.testing.assert_allclose(out.cpu().numpy(), want, atol=2e-5, rtol=1e-4)


@pytest.mark.parametrize("dt", [DType.F32, DType.F16, DType.Q8_0, DType.Q4_0, DType.Q4_K_M, DType.Q6_K])
def test_embed_rows(dt):
    rng = np.random.default_rng(int(dt))
    vocab, hidden = 50, 512
    raw = random_blocks_np(dt, vocab, hidden, rng)
    toks = np.array([0, 49, 7, 7, 23], np.int32)
    out = torch.zeros(len(toks), hidden, device=DEV)
    K.embed_rows(out, dev(raw), dt, dev(toks), len(toks), hidden)
    sync()
    want = O.dequant_rows(int(dt), raw, vocab, hidden)[toks]
    np.testing.assert_allclose(out.cpu().numpy(), want, rtol=3e-6, atol=1e-9)


def test_launch_counter_counts_our_kernels():
    before = K.launch_count()
    x = torch.ones(256, device=DEV)
    K.launch_add_inplace(x, x, 256)
    sync()
    assert K.launch_count() == before + 1
