"""GPU parity tests of the tcgen05 contraction (dmm_gemm_bf16_tn) and the fp32 verification
kernel against numpy.  bf16 single pass is compared on bf16-rounded operands (exact products,
fp32 accumulation => tight tolerance); the split-bf16 ("bf16x3") mode against fp64 numpy at the
north-star fp32 tolerance (rel 1e-5 of the row scale)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.fixture(scope="module")
def ops():
    from diffmm_b200 import ops as o
    return o


def _bf16_round(x):
    return torch.from_numpy(x).to(torch.bfloat16).float().numpy()


def _ref(a, b, bias, act, alpha, beta, res):
    v = a.astype(np.float64) @ b.astype(np.float64).T
    if bias is not None:
        v = v + bias
    if act:
        v = np.tanh(v)
    v = alpha * v
    if res is not None:
        v = v + beta * res
    return v


SHAPES = [(128, 256, 64), (128, 64, 64), (128, 128, 128), (200, 300, 210), (1024, 1024, 1000), (300, 7050, 1024),
          (2048, 1024, 7060), (1024, 64, 6710), (77, 40, 50),
          # CTA-pair (cta_group::2) kernel: >= 74 tiles of 256 x 256; tail wave cut into 64-column slices; ragged M and N
          (2048, 2560, 136), (2000, 2500, 136), (5000, 2310, 200),
          # K = batch < 64: the weight-gradient contractions of the fused training step on a small last batch
          (1003, 136, 1), (136, 1003, 17), (1024, 1024, 63)]


@pytest.mark.parametrize("M,N,K", SHAPES)
def test_simt_fp32(ops, M, N, K):
    rng = np.random.default_rng(M + N + K)
    a = rng.standard_normal((M, K)).astype(np.float32)
    b = (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)
    bias = rng.standard_normal(N).astype(np.float32)
    out = torch.empty((M, N), device=DEV)
    ops.gemm_f32_tn(T(a), T(b), M, N, K, bias=T(bias), act=1, out_f32=out)
    np.testing.assert_allclose(out.cpu().numpy(), _ref(a, b, bias, 1, 1.0, 0.0, None), rtol=1e-4, atol=2e-5)


@pytest.mark.parametrize("M,N,K", SHAPES)
@pytest.mark.parametrize("mode", ["bf16", "bf16x3"])
def test_tcgen05(ops, M, N, K, mode):
    rng = np.random.default_rng(M * 3 + N * 5 + K)
    a = rng.standard_normal((M, K)).astype(np.float32)
    b = (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)
    bias = (rng.standard_normal(N) * 0.1).astype(np.float32)
    res = rng.standard_normal((M, N)).astype(np.float32)
    a_hi, a_lo = ops.pack_bf16(T(a))
    b_hi, b_lo = ops.pack_bf16(T(b))
    ldn = ops.pad_to(N, 8)
    res_t = torch.zeros((M, ldn), device=DEV)
    res_t[:, :N] = T(res)
    out = torch.full((M, ldn), float("nan"), device=DEV)
    out_hi = torch.zeros((M, ldn), dtype=torch.bfloat16, device=DEV)
    out_lo = torch.zeros((M, ldn), dtype=torch.bfloat16, device=DEV)
    split = mode == "bf16x3"
    ops.gemm_bf16_tn(a_hi, a_lo if split else None, b_hi, b_lo if split else None, M, N, K, bias=T(bias), act=1,
                     alpha=0.75, beta=0.5, residual=res_t[:, :N], out_f32=out[:, :N], out_hi=out_hi[:, :N],
                     out_lo=out_lo[:, :N])
    torch.cuda.synchronize()
    got = out[:, :N].cpu().numpy()
    if split:
        want = _ref(a, b, bias, 1, 0.75, 0.5, res)
        np.testing.assert_allclose(got, want, rtol=1e-5, atol=5e-5)
    else:
        want = _ref(_bf16_round(a), _bf16_round(b), bias, 1, 0.75, 0.5, res)
        np.testing.assert_allclose(got, want, rtol=1e-5, atol=2e-5)
    rec = (out_hi.float() + out_lo.float())[:, :N].cpu().numpy()
    np.testing.assert_allclose(rec, got, rtol=2 ** -15, atol=1e-30)
    if ldn > N:
        assert torch.isnan(out[:, N:]).all()          # padding columns are never written


@pytest.mark.parametrize("M,N,K", SHAPES + [(19445, 1024, 1024), (640, 1000, 96)])
@pytest.mark.parametrize("pad", [8, 32])
def test_tcgen05_tma_epilogue_hidden_step(ops, M, N, K, pad):
    """Single-pass bf16 with the TMA epilogue: fp32 state updated IN PLACE (z = alpha (acc + bias) + beta z, residual
    prefetch ring + bulk tensor stores) and the post stage h = tanh(z + post_bias) as the bf16 operand copy."""
    rng = np.random.default_rng(M * 7 + N * 3 + K)
    a = rng.standard_normal((M, K)).astype(np.float32)
    b = (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)
    bias = (rng.standard_normal(N) * 0.1).astype(np.float32)
    pbias = (rng.standard_normal(N) * 0.3).astype(np.float32)
    z0 = rng.standard_normal((M, N)).astype(np.float32)
    a_hi, _ = ops.pack_bf16(T(a), split=False)
    b_hi, _ = ops.pack_bf16(T(b), split=False)
    ldn = ops.pad_to(N + (pad - 8), pad)
    z = torch.full((M, ldn), float("nan"), device=DEV)
    z[:, :N] = T(z0)
    h = torch.full((M, ldn), 7.0, dtype=torch.bfloat16, device=DEV)
    ops.gemm_bf16_tn(a_hi, None, b_hi, None, M, N, K, bias=T(bias), alpha=0.75, beta=0.5, residual=z[:, :N],
                     out_f32=z[:, :N], out_hi=h[:, :N], post_bias=T(pbias), post_act=1)
    torch.cuda.synchronize()
    want = _ref(_bf16_round(a), _bf16_round(b), bias, 0, 0.75, 0.5, z0)
    got = z[:, :N].cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=5e-5)      # fp32 accumulation over up to 7060 products, no tanh
    want_h = np.tanh(got.astype(np.float64) + pbias)
    np.testing.assert_allclose(h[:, :N].float().cpu().numpy(), want_h, rtol=2 ** -8, atol=2e-3)   # MUFU tanh + bf16
    # the TMA stores move whole 16-byte units: the padding of a row may be written up to the next 16-byte boundary
    # (4 fp32 / 8 bf16 columns), never beyond
    n4, n8 = ops.pad_to(N, 4), ops.pad_to(N, 8)
    if ldn > n4:
        assert torch.isnan(z[:, n4:]).all()
    if ldn > n8:
        assert (h[:, n8:].float() == 7.0).all()


@pytest.mark.parametrize("M,N,K", [(300, 1024, 1024), (4100, 1000, 520), (19445, 1024, 1024)])
def test_tcgen05_tma_epilogue_last_hidden_step(ops, M, N, K):
    """The last hidden-space step of the chain: the fp32 state is only read (residual), the one output is the bf16
    operand h = tanh(alpha (acc + bias) + beta z + post_bias); z must come back untouched."""
    rng = np.random.default_rng(M + N + K)
    a = rng.standard_normal((M, K)).astype(np.float32)
    b = (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)
    bias = (rng.standard_normal(N) * 0.1).astype(np.float32)
    pbias = (rng.standard_normal(N) * 0.3).astype(np.float32)
    z0 = rng.standard_normal((M, N)).astype(np.float32)
    a_hi, _ = ops.pack_bf16(T(a), split=False)
    b_hi, _ = ops.pack_bf16(T(b), split=False)
    ldn = ops.pad_to(N, 8)
    z = torch.zeros((M, ldn), device=DEV)
    z[:, :N] = T(z0)
    h = torch.full((M, ldn), 7.0, dtype=torch.bfloat16, device=DEV)
    ops.gemm_bf16_tn(a_hi, None, b_hi, None, M, N, K, bias=T(bias), alpha=0.75, beta=0.5, residual=z[:, :N],
                     out_hi=h[:, :N], post_bias=T(pbias), post_act=1)
    torch.cuda.synchronize()
    assert np.array_equal(z[:, :N].cpu().numpy(), z0)
    v = _ref(_bf16_round(a), _bf16_round(b), bias, 0, 0.75, 0.5, z0)
    want_h = np.tanh(v.astype(np.float64) + pbias)
    np.testing.assert_allclose(h[:, :N].float().cpu().numpy(), want_h, rtol=2 ** -8, atol=2e-3)   # MUFU tanh + bf16


@pytest.mark.parametrize("M,N,K", [(200, 300, 210), (77, 40, 50), (2000, 2500, 136), (4100, 1024, 512)])
def test_tcgen05_tma_epilogue_single_outputs(ops, M, N, K):
    """TMA epilogue with one output kind: tanh -> bf16 operand only (dense first layer), and fp32 only with a
    pre-activation fp32 residual."""
    rng = np.random.default_rng(M + N * 11 + K)
    a = rng.standard_normal((M, K)).astype(np.float32)
    b = (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)
    bias = (rng.standard_normal(N) * 0.1).astype(np.float32)
    res = rng.standard_normal((M, N)).astype(np.float32)
    a_hi, _ = ops.pack_bf16(T(a), split=False)
    b_hi, _ = ops.pack_bf16(T(b), split=False)
    ldn = ops.pad_to(N, 8)
    h = torch.zeros((M, ldn), dtype=torch.bfloat16, device=DEV)
    ops.gemm_bf16_tn(a_hi, None, b_hi, None, M, N, K, bias=T(bias), act=1, out_hi=h[:, :N])
    want = _ref(_bf16_round(a), _bf16_round(b), bias, 1, 1.0, 0.0, None)
    np.testing.assert_allclose(h[:, :N].float().cpu().numpy(), want, rtol=2 ** -8, atol=1e-5)
    res_t = torch.zeros((M, ldn), device=DEV)
    res_t[:, :N] = T(res)
    out = torch.full((M, ldn), float("nan"), device=DEV)
    ops.gemm_bf16_tn(a_hi, None, b_hi, None, M, N, K, bias=T(bias), act=1, alpha=1.5, beta=1.0, residual=res_t[:, :N],
                     res_pre_act=True, out_f32=out[:, :N])
    want = 1.5 * np.tanh(_bf16_round(a).astype(np.float64) @ _bf16_round(b).astype(np.float64).T + bias + res)
    np.testing.assert_allclose(out[:, :N].cpu().numpy(), want, rtol=1e-5, atol=2e-5)


def test_tcgen05_k_chunked_pre_activation_residual(ops):
    """res_pre_act: the residual is a partial sum of the same contraction, added before bias-tanh (K in chunks)."""
    rng = np.random.default_rng(12)
    M, N, K, KC = 300, 200, 448, 192
    a = rng.standard_normal((M, K)).astype(np.float32)
    b = (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)
    bias = (rng.standard_normal(N) * 0.1).astype(np.float32)
    a_hi, a_lo = ops.pack_bf16(T(a))
    b_hi, b_lo = ops.pack_bf16(T(b))
    part = torch.empty((M, N), device=DEV)
    out_hi = torch.zeros((M, 208), dtype=torch.bfloat16, device=DEV)
    out_lo = torch.zeros((M, 208), dtype=torch.bfloat16, device=DEV)
    k0 = 0
    while k0 < K:
        kc = min(KC, K - k0)
        sl = slice(k0, k0 + kc)
        res = part if k0 > 0 else None
        if k0 + kc >= K:
            ops.gemm_bf16_tn(a_hi[:, sl], a_lo[:, sl], b_hi[:, sl], b_lo[:, sl], M, N, kc, bias=T(bias), act=1, beta=1.0,
                             residual=res, res_pre_act=True, out_hi=out_hi[:, :N], out_lo=out_lo[:, :N])
        else:
            ops.gemm_bf16_tn(a_hi[:, sl], a_lo[:, sl], b_hi[:, sl], b_lo[:, sl], M, N, kc, beta=1.0, residual=res,
                             out_f32=part)
        k0 += kc
    got = (out_hi.float() + out_lo.float())[:, :N].cpu().numpy()
    want = np.tanh(a.astype(np.float64) @ b.astype(np.float64).T + bias)
    np.testing.assert_allclose(got, want, rtol=2e-5, atol=5e-5)


@pytest.mark.parametrize("M,N,K", [(1024, 1024, 7050), (1024, 1024, 18357), (300, 520, 4100), (256, 256, 70000), (128, 64, 4096),
                                   (19445, 1024, 1024)])
def test_tcgen05_splitk(ops, M, N, K):
    """dmm_gemm_bf16_tn_splitk: fp32 result and its bf16 hi / lo copies against float64 on the bf16-rounded operands (exact
    products; only the fp32 summation order differs), against the plain contraction, and deterministic.  The last two
    shapes do not split (narrow N / tiles fill the machine): the entry point must fall back to the plain contraction."""
    rng = np.random.default_rng(M + N + K)
    a = _bf16_round(rng.standard_normal((M, K)).astype(np.float32) / np.sqrt(K))
    b = _bf16_round(rng.standard_normal((N, K)).astype(np.float32))
    ld = (K + 63) // 64 * 64
    a_d = torch.zeros((M, ld), dtype=torch.bfloat16, device=DEV)
    b_d = torch.zeros((N, ld), dtype=torch.bfloat16, device=DEV)
    a_d[:, :K] = T(a).bfloat16()
    b_d[:, :K] = T(b).bfloat16()
    want = a.astype(np.float64) @ b.astype(np.float64).T
    ldn = (N + 63) // 64 * 64
    out = torch.full((M, (N + 3) // 4 * 4), float("nan"), device=DEV)
    hi = torch.zeros((M, ldn), dtype=torch.bfloat16, device=DEV)
    lo = torch.zeros((M, ldn), dtype=torch.bfloat16, device=DEV)
    ops.gemm_bf16_tn_splitk(a_d[:, :K], b_d[:, :K], M, N, K, out_f32=out[:, :N], out_hi=hi[:, :N], out_lo=lo[:, :N])
    got = out[:, :N].cpu().numpy()
    atol = 2e-5 * max(1.0, np.sqrt(K / 7050))        # test_tcgen05's tolerance (values of order 1), grown with sqrt(K)
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=atol)
    plain = torch.empty_like(out)
    ops.gemm_bf16_tn(a_d[:, :K], None, b_d[:, :K], None, M, N, K, out_f32=plain[:, :N])
    # the plain contraction accumulates K products in ONE fp32 chain of the tensor pipe (its error grows faster than the
    # split sums'): a looser bound, it is not the subject here
    np.testing.assert_allclose(plain[:, :N].cpu().numpy(), want, rtol=1e-5, atol=6 * atol)
    # operand copies: hi = bf16_rn(c), lo = bf16_rn(c - hi), exactly, of the fp32 result the call returned
    g = out[:, :N]
    assert torch.equal(hi[:, :N], g.bfloat16())
    assert torch.equal(lo[:, :N], (g - g.bfloat16().float()).bfloat16())
    out2 = torch.empty_like(out)
    ops.gemm_bf16_tn_splitk(a_d[:, :K], b_d[:, :K], M, N, K, out_f32=out2[:, :N])
    assert torch.equal(out2[:, :N], out[:, :N])
    # bf16 copy only (the rebuild's call)
    hi2 = torch.zeros_like(hi)
    ops.gemm_bf16_tn_splitk(a_d[:, :K], b_d[:, :K], M, N, K, out_hi=hi2[:, :N])
    assert torch.equal(hi2[:, :N], hi[:, :N])


@pytest.mark.parametrize("B,I", [(1, 1003), (1, 7050), (300, 1003), (300, 7050), (1024, 1003), (1024, 7050)])
@pytest.mark.parametrize("mode", ["bf16", "bf16x3"])
def test_tcgen05_bf16_residual_in_place(ops, B, I, mode):
    """The gate add of the fused training step, x_t' = x_t + G F^T, written over its own bf16 residual: out_hi / out_lo
    alias res_hi / res_lo.  The residual is hi + lo in both modes; single-pass mode writes only hi (lo stays the
    residual's).  The columns past N of the same rows (the time-embedding columns of the step's operand) stay as
    they were."""
    rng = np.random.default_rng(B + I + (mode == "bf16x3"))
    split = mode == "bf16x3"
    d = 10
    ld = ops.pad_to(I + d, 64)
    g = (rng.standard_normal((B, 64)) * 0.5).astype(np.float32)
    f = (rng.standard_normal((I, 64)) * 0.1).astype(np.float32)
    x = np.zeros((B, ld), dtype=np.float32)
    x[:, :I] = rng.standard_normal((B, I))
    x[:, I:] = rng.standard_normal((B, ld - I)) * 3.0
    g_hi, g_lo = ops.pack_bf16(T(g))
    f_hi, f_lo = ops.pack_bf16(T(f))
    x_hi, x_lo = ops.pack_bf16(T(x), ld_dst=ld)
    res = (x_hi.double() + x_lo.double())[:, :I].cpu().numpy()
    before_hi, before_lo = x_hi.clone(), x_lo.clone()
    # the same contraction with an fp32 output, out of place: the value the bf16 outputs must split
    want_f32 = torch.empty((B, ops.pad_to(I, 4)), device=DEV)
    ops.gemm_bf16_tn(g_hi, g_lo if split else None, f_hi, f_lo if split else None, B, I, 64, alpha=1.0, beta=1.0,
                     res_hi=before_hi[:, :I], res_lo=before_lo[:, :I], out_f32=want_f32[:, :I])
    ops.gemm_bf16_tn(g_hi, g_lo if split else None, f_hi, f_lo if split else None, B, I, 64, alpha=1.0, beta=1.0,
                     res_hi=x_hi[:, :I], res_lo=x_lo[:, :I], out_hi=x_hi[:, :I], out_lo=x_lo[:, :I] if split else None)
    torch.cuda.synchronize()
    if split:
        a = (g_hi.double() + g_lo.double())[:, :64].cpu().numpy()
        b = (f_hi.double() + f_lo.double())[:, :64].cpu().numpy()
    else:
        a, b = g_hi[:, :64].double().cpu().numpy(), f_hi[:, :64].double().cpu().numpy()
    want = a @ b.T + res
    v = want_f32[:, :I].cpu().numpy()
    got_hi = x_hi[:, :I].double().cpu().numpy()
    if split:
        np.testing.assert_allclose(v, want, rtol=1e-5, atol=5e-5)
        rec = got_hi + x_lo[:, :I].double().cpu().numpy()
        np.testing.assert_allclose(rec, v, rtol=2 ** -15, atol=1e-30)
        np.testing.assert_allclose(rec, want, rtol=1e-5, atol=5e-5)
    else:
        np.testing.assert_allclose(v, want, rtol=1e-5, atol=2e-5)
        np.testing.assert_allclose(got_hi, v, rtol=2 ** -8, atol=1e-30)
        assert torch.equal(x_lo.view(torch.int16), before_lo.view(torch.int16))      # no lo output: untouched
    assert torch.equal(x_hi[:, I:].view(torch.int16), before_hi[:, I:].view(torch.int16))
    assert torch.equal(x_lo[:, I:].view(torch.int16), before_lo[:, I:].view(torch.int16))


def test_tcgen05_no_epilogue_extras(ops):
    rng = np.random.default_rng(9)
    M, N, K = 256, 512, 192
    a = rng.standard_normal((M, K)).astype(np.float32)
    b = rng.standard_normal((N, K)).astype(np.float32)
    a_hi, _ = ops.pack_bf16(T(a), split=False)
    b_hi, _ = ops.pack_bf16(T(b), split=False)
    out = torch.empty((M, N), device=DEV)
    ops.gemm_bf16_tn(a_hi, None, b_hi, None, M, N, K, out_f32=out)
    want = _bf16_round(a).astype(np.float64) @ _bf16_round(b).astype(np.float64).T
    np.testing.assert_allclose(out.cpu().numpy(), want, rtol=1e-5, atol=1e-4)


def test_tcgen05_many_tiles_persistent(ops):
    # more tiles than SMs: exercises the TMEM double buffering and the smem ring phase wrap
    rng = np.random.default_rng(10)
    M, N, K = 128 * 40, 256 * 9, 320
    a = rng.standard_normal((M, K)).astype(np.float32)
    b = rng.standard_normal((N, K)).astype(np.float32)
    a_hi, _ = ops.pack_bf16(T(a), split=False)
    b_hi, _ = ops.pack_bf16(T(b), split=False)
    out = torch.empty((M, N), device=DEV)
    ops.gemm_bf16_tn(a_hi, None, b_hi, None, M, N, K, out_f32=out)
    want = torch.from_numpy(_bf16_round(a)).to(DEV).double() @ torch.from_numpy(_bf16_round(b)).to(DEV).double().T
    assert torch.allclose(out.double(), want, rtol=1e-5, atol=1e-3)


def test_bad_arguments_raise(ops):
    from diffmm_b200._lib import DiffMMError
    a = torch.zeros((128, 60), dtype=torch.bfloat16, device=DEV)       # ld 60 is not a multiple of 8
    out = torch.empty((128, 128), device=DEV)
    with pytest.raises(DiffMMError):
        ops.gemm_bf16_tn(a, None, a, None, 128, 128, 60, out_f32=out)
