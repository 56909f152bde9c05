"""GPU tests of individual kernels through the C ABI (vitb200_test_gemm) against numpy / the oracle's primitives."""
import numpy as np
import pytest

from tests.util import pkg
from oracle import restatement as rs

eng = pkg.engine
pytestmark = pytest.mark.gpu


def _ref(A, W, bias, epi, resid=None):
    ref = A.astype(np.float64) @ W.astype(np.float64).T + bias
    if epi == 2:
        ref = ref + resid
    ref = ref.astype(np.float32)
    if epi == 0:
        ref = ref.astype(np.float16).astype(np.float32)
    if epi == 1:
        ref = rs.gelu_table(ref)  # f16(gelu(f32(f16(x)))) -- ggml.c:1434-1441 table semantics
    return ref


# shapes: single tile; M/N/K tails (TMA zero fill + predicated stores); ViT-tiny/base layer shapes; head N=1000
CASES = [
    (128, 256, 64, 4), (128, 128, 64, 4), (128, 256, 64, 0), (1, 128, 64, 4), (129, 384, 192, 4),
    (300, 576, 192, 0), (300, 576, 192, 1), (300, 576, 192, 2), (197 * 3, 768, 768, 2), (197 * 3, 3072, 768, 1),
    (197 * 2, 768, 3072, 2), (197 * 2, 2304, 768, 0), (256, 1000, 768, 4), (7, 1000, 192, 4), (640, 128, 640, 2),
]


def with_cta_groups(cases):
    """Every case with the default CTA pairs (ids as before) and with VITB200_CTA_GROUP=1 (id suffix -cg1), the 1-CTA
    instantiation of every epilogue."""
    ids = ["-".join(map(str, c)) for c in cases]
    return ([pytest.param(*c, 2, id=i) for c, i in zip(cases, ids)] +
            [pytest.param(*c, 1, id=i + "-cg1") for c, i in zip(cases, ids)])


def set_cta_group(monkeypatch, cta_group):
    if cta_group == 1:
        monkeypatch.setenv("VITB200_CTA_GROUP", "1")
    else:
        monkeypatch.delenv("VITB200_CTA_GROUP", raising=False)


@pytest.mark.parametrize("M,N,K,epi,cta_group", with_cta_groups(CASES))
def test_gemm_against_numpy(M, N, K, epi, cta_group, monkeypatch):
    set_cta_group(monkeypatch, cta_group)
    rng = np.random.default_rng(M * 7 + N * 3 + K + epi)
    A = rng.standard_normal((M, K)).astype(np.float16)
    W = (rng.standard_normal((N, K)) * 0.05).astype(np.float16)
    bias = rng.standard_normal(N).astype(np.float32)
    resid = rng.standard_normal((M, N)).astype(np.float32) if epi == 2 else None
    out = eng.test_gemm(M, N, K, epi, A, W, bias, resid)
    ref = _ref(A, W, bias, epi, resid)
    pre = (A.astype(np.float64) @ W.astype(np.float64).T + bias).astype(np.float32)
    if epi in (2, 4):  # f32 outputs: only fp32 accumulation-order noise
        np.testing.assert_allclose(out, ref, rtol=0, atol=2e-5 * max(1.0, np.abs(ref).max()))
    else:  # f16 outputs: identical except where fp32 noise flips an f16 rounding (<= 1 ulp, rare)
        # bias epilogue: at most one f16 ulp.  GELU: a flipped rounding of the f16 INPUT moves the output by up to
        # |slope| (<= 1.13) input ulps, plus half an output ulp for the final rounding -> 2.5 * 2^-10 * max(|x|, |y|)
        ulp = np.maximum(np.maximum(np.abs(ref), np.abs(pre) * (2.5 if epi == 1 else 0.0)), 2.0 ** -14) * 2.0 ** -10
        noise = 2e-5 * max(1.0, np.abs(ref).max())  # fp32 accumulation noise dominates near zero
        assert (np.abs(out - ref) <= ulp * 1.001 + noise).all()
        assert (out != ref).mean() < 0.02


@pytest.mark.parametrize("M,N,K,cta_group", with_cta_groups([(300, 576, 192), (197 * 3, 2304, 768), (129, 384, 192)]))
def test_gemm_split_precision_epilogue(M, N, K, cta_group, monkeypatch):
    """EPI_BIAS_F16_HILO (the qkv GEMM in front of the tcgen05 attention): hi = f16(x), lo = f16(x - hi); hi + lo must carry the
    f32 result to ~2^-21 relative (2^-24 absolute once lo is subnormal), i.e. only fp32 accumulation-order noise remains."""
    set_cta_group(monkeypatch, cta_group)
    rng = np.random.default_rng(M + N + K)
    A = rng.standard_normal((M, K)).astype(np.float16)
    W = (rng.standard_normal((N, K)) * 0.05).astype(np.float16)
    bias = rng.standard_normal(N).astype(np.float32)
    out = eng.test_gemm(M, N, K, 6, A, W, bias)
    ref = (A.astype(np.float64) @ W.astype(np.float64).T + bias).astype(np.float32)
    hi, lo = eng.split_hi_lo(ref)
    want = hi.astype(np.float32) + lo.astype(np.float32)
    assert np.abs(want - ref).max() <= 2.0 ** -21 * np.abs(ref).max()      # the representation itself
    np.testing.assert_allclose(out, ref, rtol=0, atol=2e-5 * max(1.0, np.abs(ref).max()) * 0.1 + 2.0 ** -20 * np.abs(ref).max())
    # and the hi part alone is exactly what the plain f16 epilogue writes
    plain = eng.test_gemm(M, N, K, 0, A, W, bias)
    assert (np.abs(out - plain) <= 2.0 ** -11 * np.abs(plain) + 2.0 ** -24).all()


def test_gemm_linearity_at_full_size():
    """Size-independent property at the BASELINE batch size (M = 256*197 = 50432): GEMM(A, W1 + W2) with zero bias equals
    GEMM(A, W1) + GEMM(A, W2) up to fp32 rounding, for exactly representable small-integer operands it is EXACT."""
    M, N, K = 256 * 197, 768, 768
    rng = np.random.default_rng(1)
    A = rng.integers(-4, 5, size=(M, K)).astype(np.float16)
    W1 = rng.integers(-3, 4, size=(N, K)).astype(np.float16)
    W2 = rng.integers(-3, 4, size=(N, K)).astype(np.float16)
    z = np.zeros(N, np.float32)
    o1 = eng.test_gemm(M, N, K, 4, A, W1, z)
    o2 = eng.test_gemm(M, N, K, 4, A, W2, z)
    o12 = eng.test_gemm(M, N, K, 4, A, (W1 + W2), z)
    assert np.array_equal(o1 + o2, o12)  # all partial sums are small integers: exact in fp32
    # spot-check rows from the first, a middle and the last M tile against int64 arithmetic
    for r in (0, 127, 128, 25000, M - 1):
        assert np.array_equal(o1[r].astype(np.int64), A[r].astype(np.int64) @ W1.astype(np.int64).T)



def _attention_ref(qkv16, B, N, H):
    """float64 restatement of vit.cpp:826-866 on f16 inputs with the reference soft-max semantics (ggml.c:10533-10558):
    e = f16(exp(f16(s/8 - max))), p = e * (1/sum e); O = P V."""
    D = H * 64
    x = qkv16.astype(np.float64).reshape(B, N, 3, H, 64)
    q, k, v = x[:, :, 0].transpose(0, 2, 1, 3), x[:, :, 1].transpose(0, 2, 1, 3), x[:, :, 2].transpose(0, 2, 1, 3)
    s = np.einsum("bhqd,bhkd->bhqk", q, k).astype(np.float32) * np.float32(0.125)
    z = (s - s.max(-1, keepdims=True)).astype(np.float16).astype(np.float64)
    e = np.exp(z).astype(np.float16).astype(np.float64)
    o = np.einsum("bhqk,bhkd->bhqd", e, v) / e.sum(-1, keepdims=True)
    return o.transpose(0, 2, 1, 3).reshape(B * N, D)


def _attention_ref_f32(qkv32, B, N, H):
    """The same on f32 q, k, v (what the reference's attention mat-muls see, vit.cpp:848,858)."""
    D = H * 64
    x = qkv32.astype(np.float64).reshape(B, N, 3, H, 64)
    q, k, v = x[:, :, 0].transpose(0, 2, 1, 3), x[:, :, 1].transpose(0, 2, 1, 3), x[:, :, 2].transpose(0, 2, 1, 3)
    s = np.einsum("bhqd,bhkd->bhqk", q, k).astype(np.float32) * np.float32(0.125)
    z = (s - s.max(-1, keepdims=True)).astype(np.float16).astype(np.float64)
    e = np.exp(z).astype(np.float16).astype(np.float64)
    o = np.einsum("bhqk,bhkd->bhqd", e, v) / e.sum(-1, keepdims=True)
    return o.transpose(0, 2, 1, 3).reshape(B * N, D), s


@pytest.mark.parametrize("B,N,H", [(3, 17, 2), (2, 197, 3), (1, 224, 1), (40, 197, 12), (2, 50, 1)])
def test_attention_split_precision_against_f32_operand_reference(B, N, H):
    """attention_tc_kernel with hi + lo operands must follow the f32-operand restatement, not the f16-operand one: a score error of
    2^-12 relative (what rounding q or k to f16 costs) moves x - max across f16 rounding boundaries; with split operands the only
    differences left are f32 accumulation order + the f16 roundings the reference makes too.  The last case keeps every CTA looping
    over several (image, head) problems (single-buffered operand groups: empty/full barrier parities)."""
    rng = np.random.default_rng(N * 7 + H)
    qkv = rng.normal(0.0, 1.0, (B * N, 3 * H * 64)).astype(np.float32)
    qkv[:, : H * 64] *= 1.5
    hi, lo = eng.split_hi_lo(qkv)
    q22 = hi.astype(np.float32) + lo.astype(np.float32)   # the 22-bit values the kernel actually sees
    out = eng.test_attention_hilo(qkv, B, N, H)
    ref, _ = _attention_ref_f32(q22, B, N, H)
    ref16, _ = _attention_ref_f32(hi.astype(np.float32), B, N, H)
    assert np.isfinite(out).all()
    err = np.abs(out - ref)
    tol = 2.0 ** -10 * np.abs(ref) + 2e-3 * np.abs(ref).max()
    assert (err <= tol).all(), (err.max(), np.abs(ref).max(), np.unravel_index(err.argmax(), err.shape))
    # closer to the f32-operand result than to the f16-operand one (mean absolute deviation over all outputs)
    assert np.abs(out - ref).mean() < 0.6 * np.abs(out - ref16).mean(), (np.abs(out - ref).mean(), np.abs(out - ref16).mean())


ATTN_CASES = [  # (B, N, H, kernel)
    (3, 17, 2, eng.ATTN_TC), (2, 197, 3, eng.ATTN_TC), (2, 197, 3, eng.ATTN_MMA),
    (2, 577, 2, eng.ATTN_TC_LONG), (2, 577, 2, eng.ATTN_MMA), (1, 225, 1, eng.ATTN_TC_LONG), (3, 384, 1, eng.ATTN_TC_LONG),
    (2, 401, 2, eng.ATTN_TC_LONG), (1, 640, 1, eng.ATTN_TC_LONG), (20, 577, 16, eng.ATTN_TC_LONG),
]


@pytest.mark.parametrize("B,N,H,kernel", ATTN_CASES)
def test_attention_kernels_against_numpy(B, N, H, kernel):
    """Every attention kernel, alone, on random QKV (scores spread over several units so the soft-max is not flat): agreement with
    the float64 restatement to f16 output rounding + f32 accumulation noise; the last case runs every CTA through many
    (image, head) problems (persistent-loop parities, K/V ring reuse)."""
    rng = np.random.default_rng(N * 131 + H)
    qkv = rng.normal(0.0, 1.0, (B * N, 3 * H * 64)).astype(np.float32)
    qkv[:, : H * 64] *= 1.5                       # Q: |s/8| up to ~5
    qkv16 = qkv.astype(np.float16)
    out = eng.test_attention(qkv16, B, N, H, kernel)
    ref = _attention_ref(qkv16, B, N, H)
    assert np.isfinite(out).all()
    err = np.abs(out - ref)
    tol = 2.0 ** -10 * np.abs(ref) + 2e-3 * np.abs(ref).max()
    assert (err <= tol).all(), (err.max(), np.abs(ref).max(), np.unravel_index(err.argmax(), err.shape))


# ---- q8_0 linear layer on the integer tensor cores (prototype, BASELINE.json configs[4]) ---------------------------------------
Q8_CASES = [(128, 128, 128), (1, 128, 128), (300, 576, 768), (197 * 3, 2304, 768), (197 * 2, 768, 3072), (129, 1000, 768), (640, 132, 256)]


@pytest.mark.parametrize("M,N,K", Q8_CASES)
def test_q8_0_gemm_matches_the_reference_integer_dot(M, N, K):
    """tcgen05 kind::i8 GEMM + on-device activation quantisation against the oracle's quantize_row_q8_0 + vec_dot_q8_0_q8_0
    (bit-exact restatements of the reference, tests/test_oracle.py): the quantised activations (integer work) must be bit-identical,
    the f32 outputs within 1e-5 of the row's largest output (same products, same f32 accumulation, different order of the
    reference's eight partial lanes)."""
    rng = np.random.default_rng(M * 7 + N * 3 + K)
    x = (rng.standard_normal((M, K)) * rng.uniform(0.2, 3.0, (M, 1))).astype(np.float32)
    x[0, :32] = 0.0                                  # an all-zero block: d = 0, id = 0 (ggml-quants.c:733)
    if M > 2:
        x[2, 5] = 1e4                                # an outlier squeezing the rest of its block to a few levels
    w = (rng.standard_normal((N, K)) * 0.05).astype(np.float32)
    wb = pkg.convert.quantize_q8_0_reference(w.reshape(-1))  # the file quantiser (roundf variant), as `quantize` writes it
    bias = rng.standard_normal(N).astype(np.float32)
    y_ref, xq_ref, xd_ref = rs.linear_q8_0(x, wb, bias)
    y, xq, xd, _ = eng.test_gemm_q8(x, wb, bias)
    assert np.array_equal(xq, xq_ref), "quantised activations differ from quantize_row_q8_0"
    assert np.array_equal(xd.view(np.uint32), xd_ref.view(np.uint32)), "block scales differ from quantize_row_q8_0"
    scale = np.abs(y_ref).max(axis=1, keepdims=True)
    err = (np.abs(y - y_ref) / scale).max()
    assert err <= 1e-5, f"q8_0 GEMM error {err:.3e}"


# ---- LayerNorm: the persistent bulk-copy kernel (D % 128 == 0, >= 8 rows) and the row-per-warp kernel behind the same launcher -----------
@pytest.mark.parametrize("rows,D", [(1, 768), (7, 768), (8, 768), (9, 768), (591, 768), (1154, 1024), (4097, 128), (34, 128), (50, 192), (2, 384)])
def test_layernorm_matches_the_restatement(rows, D):
    """Row counts around the 8-row block size (partial last block, fewer rows than one block -> row-per-warp kernel), more blocks than
    resident CTAs, hidden sizes of every model in the tests; against the oracle's ggml_norm * w + b rounded to f16 (the GEMM's src1
    conversion): at most one f16 ulp apart (the reference sums in double, the kernel in f32), bit-equal on > 99.5 % of the elements."""
    rng = np.random.default_rng(rows * 131 + D)
    x = (rng.standard_normal((rows, D)) * rng.uniform(0.5, 4.0, (rows, 1)) + rng.uniform(-1, 1, (rows, 1))).astype(np.float32)
    w = rng.uniform(0.5, 1.5, D).astype(np.float32)
    b = rng.uniform(-0.5, 0.5, D).astype(np.float32)
    y = eng.test_layernorm(x, w, b)
    ref = rs.round_f16(rs.layernorm(x, w, b))
    ulp = np.spacing(np.abs(ref).astype(np.float16)).astype(np.float32)
    assert np.isfinite(y).all()
    # one f16 ulp, or -- where (x - mean) * scale * w and b cancel to a result near zero, whose ulp is tiny -- the f32 rounding of the
    # un-cancelled terms (|terms| < 10 here)
    assert (np.abs(y - ref) <= np.maximum(ulp, 4e-6)).all(), float((np.abs(y - ref) / np.maximum(ulp, 4e-6)).max())
    assert (y == ref).mean() > 0.995
