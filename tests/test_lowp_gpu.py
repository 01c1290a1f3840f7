"""GPU parity tests for int8 / fp8 / mxfp8 / nvfp4 (quantizers bit-exact vs the oracle; GEMMs vs the
oracle's exact-product result and, where the reference's library kernel exists, vs that kernel)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    import ao_b200  # noqa: F401

    return torch.ops.ao_b200


def _o():
    from oracle import oracle as o

    return o


def sqnr(ref, out):
    ref, out = ref.double(), out.double()
    d = (ref - out).norm()
    return float("inf") if d == 0 else float(20 * torch.log10(ref.norm() / d))


def _x(M, K, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(M, K, device="cuda", generator=g) * torch.logspace(-2, 2, M, device="cuda").unsqueeze(1)
    x = x.to(torch.bfloat16)
    if M >= 5:
        x[2] = 0  # all-zero row: eps clamp (int8) / 0-scale (fp8) / 2^-127 scale (mx)
    return x


@pytest.mark.parametrize("M,K", [(1, 4096), (5, 256), (32, 4096), (130, 512), (32, 14336)])
def test_activation_quantizers_bit_exact(ops, M, K):
    o = _o()
    x = _x(M, K, M + K)
    xb = o.bf16_bits(x)
    q, s = ops.int8_quantize_rowwise(x)
    qo, so = o.int8_quantize_rowwise(xb)
    assert np.array_equal(q.cpu().numpy(), qo) and np.array_equal(s.cpu().numpy().reshape(-1), so)
    q, s = ops.fp8_quantize_rowwise(x)
    qo, so = o.fp8_quantize_rowwise(xb)
    assert np.array_equal(q.view(torch.uint8).cpu().numpy(), qo) and np.array_equal(s.cpu().numpy().reshape(-1), so)
    q, s = ops.mxfp8_quantize(x, False)
    qo, so = o.mxfp8_quantize(xb)
    assert np.array_equal(q.view(torch.uint8).cpu().numpy(), qo) and np.array_equal(s.cpu().numpy(), so)
    q2, s2 = ops.mxfp8_quantize(x, True)
    assert np.array_equal(s2.cpu().numpy().reshape(-1), o.to_blocked(so).reshape(-1))
    q, s = ops.nvfp4_quantize(x, None, False)
    qo, so = o.nvfp4_quantize(xb, None)
    assert np.array_equal(q.cpu().numpy(), qo) and np.array_equal(s.cpu().numpy(), so)
    pts = (x.float().abs().max() / (448.0 * 6.0)).reshape(1)
    q, s = ops.nvfp4_quantize(x, pts, True)
    qo, so = o.nvfp4_quantize(xb, float(pts.item()))
    assert np.array_equal(q.cpu().numpy(), qo) and np.array_equal(s.cpu().numpy().reshape(-1), o.to_blocked(so).reshape(-1))
    # e4m3 "fake quant" used by the nvfp4-weight x fp8-activation path: same codes, as bf16 values
    if M < 5:
        qf, sf = ops.fp8_fakequant_rowwise(x)
        qo, so = o.fp8_quantize_rowwise(xb)
        assert np.array_equal(o.bf16_to_f32(o.bf16_bits(qf)), o.e4m3_to_f32(qo)) and np.array_equal(sf.cpu().numpy().reshape(-1), so)


@pytest.mark.parametrize("M,K", [(2048, 4096), (512, 16384), (300, 14336), (64, 32768)])
def test_rowwise_quantizers_large_sample_vs_torch(ops, M, K):
    """Millions of quotients per case against the reference arithmetic written with torch ops on the GPU (true IEEE
    division, quant_primitives.py:2172-2287 / :1487-1583): the e4m3 kernel forms x / s as x * (1 / s) plus one FMA residual
    correction, which must round exactly like the division; K = 32768 takes the two-pass kernel."""
    g = torch.Generator(device="cuda").manual_seed(M + K)
    x = (torch.randn(M, K, device="cuda", generator=g) * torch.logspace(-3, 3, M, device="cuda").unsqueeze(1)).to(torch.bfloat16)
    q, s = ops.fp8_quantize_rowwise(x)
    amax = x.abs().amax(dim=1, keepdim=True)
    sc = (amax / 448.0).float()            # bf16 division, then f32 (the reference divides in the input dtype)
    ref = (x.float() / sc).clamp(-448.0, 448.0).to(torch.float8_e4m3fn)
    assert torch.equal(s.reshape(-1), sc.reshape(-1))
    assert torch.equal(q.view(torch.uint8), ref.view(torch.uint8))
    q8, s8 = ops.int8_quantize_rowwise(x)
    sc8 = torch.clamp((amax / 127.5).float(), min=torch.finfo(torch.float32).eps)
    ref8 = torch.clamp(torch.round(x.float() * (1.0 / sc8)), -128, 127).to(torch.int8)
    assert torch.equal(s8.reshape(-1), sc8.reshape(-1))
    assert torch.equal(q8, ref8)


SHAPES = [(1, 128, 512), (16, 256, 1024), (32, 4096, 4096), (7, 1024, 4096), (32, 14336, 4096), (32, 4096, 14336),
          (64, 4096, 4096), (128, 1024, 2048), (200, 1024, 4096), (3, 144, 1024)]


@pytest.mark.parametrize("M,N,K", SHAPES)
def test_int8_linear_exact(ops, M, N, K):
    g = torch.Generator(device="cuda").manual_seed(M + N)
    xq = torch.randint(-128, 128, (M, K), device="cuda", dtype=torch.int8, generator=g)
    wq = torch.randint(-128, 128, (N, K), device="cuda", dtype=torch.int8, generator=g)
    acc_ref = (xq.double() @ wq.double().t()).to(torch.int64)
    assert torch.equal(ops.int8_mm_i32(xq, wq).to(torch.int64), acc_ref)  # integer MMA: bit-exact
    sx = torch.rand(M, 1, device="cuda", generator=g) * 0.01 + 1e-3
    sw = torch.rand(N, device="cuda", generator=g) * 0.01 + 1e-3
    b = torch.randn(N, device="cuda", generator=g).to(torch.bfloat16) if M % 2 else None
    y = ops.int8_dyn_linear(xq, sx, wq, sw, b)
    t = (acc_ref.float() * sx).to(torch.bfloat16).float() * sw  # the reference's rounding order
    if b is not None:
        t = t + b.float()
    assert torch.equal(y, t.to(torch.bfloat16))


@pytest.mark.parametrize("M,N,K", SHAPES)
def test_fp8_rowwise_linear(ops, M, N, K):
    x = torch.randn(M, K, device="cuda").to(torch.bfloat16)
    w = (torch.randn(N, K, device="cuda") * 0.05).to(torch.bfloat16)
    xq, sx = ops.fp8_quantize_rowwise(x)
    wq, sw = ops.fp8_quantize_rowwise(w)
    b = torch.randn(N, device="cuda").to(torch.bfloat16) if M % 2 else None
    y = ops.fp8_rowwise_linear(xq, sx, wq, sw.reshape(-1), b)
    ref64 = (xq.double() @ wq.double().t()) * sx.double() * sw.double().reshape(1, -1)
    if b is not None:
        ref64 = ref64 + b.double()
    assert sqnr(ref64, y) > 45.0
    y_t = torch._scaled_mm(xq, wq.t(), scale_a=sx, scale_b=sw.reshape(1, -1), bias=b, out_dtype=torch.bfloat16, use_fast_accum=True)
    assert sqnr(y_t, y) > 70.0  # the reference's own kernel


def _from_blocked(b, H, W):
    return torch.from_numpy(_o().from_blocked(b.cpu().numpy().reshape(-1), H, W)).cuda()


@pytest.mark.parametrize("M,N,K", SHAPES)
def test_mxfp8_linear(ops, M, N, K):
    x = torch.randn(M, K, device="cuda").to(torch.bfloat16)
    w = (torch.randn(N, K, device="cuda") * 0.05).to(torch.bfloat16)
    xq, xs = ops.mxfp8_quantize(x, True)
    wq, ws = ops.mxfp8_quantize(w, True)
    b = torch.randn(N, device="cuda").to(torch.bfloat16) if M % 2 else None
    y = ops.mxfp8_linear(xq, xs, wq, ws, b)
    xd = xq.double() * torch.pow(2.0, _from_blocked(xs, M, K // 32).double() - 127).repeat_interleave(32, 1)
    wd = wq.double() * torch.pow(2.0, _from_blocked(ws, N, K // 32).double() - 127).repeat_interleave(32, 1)
    ref64 = xd @ wd.t() + (b.double() if b is not None else 0)
    assert sqnr(ref64, y) > 45.0  # reference bar for library GEMM vs dequant-matmul: test_mx_mm.py:92-98 (bf16 output)
    assert sqnr(x.double() @ w.double().t() + (b.double() if b is not None else 0), y) > 25.0  # test_inference_workflow.py:123


E2M1 = [0, 0.5, 1, 1.5, 2, 3, 4, 6, -0.0, -0.5, -1, -1.5, -2, -3, -4, -6]


def _fp4_dq(q, s_plain, pts):
    lut = torch.tensor(E2M1, dtype=torch.float64, device=q.device)
    v = torch.stack([lut[(q & 15).long()], lut[(q >> 4).long()]], dim=-1).reshape(q.shape[0], -1)
    sc = s_plain.view(torch.float8_e4m3fn).double().repeat_interleave(16, 1)
    return v * sc * (pts.double() if pts is not None else 1.0)


@pytest.mark.parametrize("M,N,K", [s for s in SHAPES if s[2] % 256 == 0])
def test_nvfp4_linear(ops, M, N, K):
    x = torch.randn(M, K, device="cuda").to(torch.bfloat16)
    w = (torch.randn(N, K, device="cuda") * 0.05).to(torch.bfloat16)
    pa = (x.float().abs().max() / (448.0 * 6.0)).reshape(1)
    pb = (w.float().abs().max() / (448.0 * 6.0)).reshape(1)
    xq, xs = ops.nvfp4_quantize(x, pa, True)
    wq, ws = ops.nvfp4_quantize(w, pb, True)
    b = torch.randn(N, device="cuda").to(torch.bfloat16) if M % 2 else None
    y = ops.nvfp4_linear(xq, xs, pa, wq, ws, pb, b)
    ref64 = _fp4_dq(xq, _from_blocked(xs, M, K // 16), pa) @ _fp4_dq(wq, _from_blocked(ws, N, K // 16), pb).t()
    ref64 = ref64 + (b.double() if b is not None else 0)
    assert sqnr(ref64, y) > 45.0
    assert sqnr(x.double() @ w.double().t() + (b.double() if b is not None else 0), y) > 15.0  # test_inference_workflow.py:224-227


@pytest.mark.parametrize("M,N,K", [(32, 4096, 4096), (128, 1024, 2048), (32, 14336, 4096), (256, 4096, 4096)])
def test_block_scaled_linears_vs_the_library_kernel(ops, M, N, K):
    """mxfp8 and nvfp4 against the kernel the reference calls for them, torch._scaled_mm with blocked e8m0 / e4m3 scales
    (mx_tensor.py:803-810, nvfp4_tensor.py:561-578), on the same quantized operands: both compute exact products with
    fp32 accumulation, so the bf16 outputs may differ by accumulation order only (>= 70 dB, as for the fp8 kernel)."""
    x = torch.randn(M, K, device="cuda").to(torch.bfloat16)
    w = (torch.randn(N, K, device="cuda") * 0.05).to(torch.bfloat16)
    xq, xs = ops.mxfp8_quantize(x, True)
    wq, ws = ops.mxfp8_quantize(w, True)
    y = ops.mxfp8_linear(xq, xs, wq, ws, None)
    y_t = torch._scaled_mm(xq, wq.t(), scale_a=xs.view(torch.float8_e8m0fnu), scale_b=ws.view(torch.float8_e8m0fnu),
                           out_dtype=torch.bfloat16)
    assert sqnr(y_t, y) > 70.0
    xq, xs = ops.nvfp4_quantize(x, None, True)
    wq, ws = ops.nvfp4_quantize(w, None, True)
    y = ops.nvfp4_linear(xq, xs, None, wq, ws, None, None)
    y_t = torch._scaled_mm(xq.view(torch.float4_e2m1fn_x2), wq.view(torch.float4_e2m1fn_x2).t(), scale_a=xs.view(torch.float8_e4m3fn),
                           scale_b=ws.view(torch.float8_e4m3fn), out_dtype=torch.bfloat16)
    assert sqnr(y_t, y) > 70.0


@pytest.mark.parametrize("M,N,K,fp8_act", [(1, 256, 1024, False), (32, 4096, 4096, False), (7, 1024, 4096, True), (32, 8192, 8192, True),
                                           (64, 1024, 2048, False), (130, 512, 1024, True),
                                           (512, 8192, 8192, True), (300, 1024, 4096, False)])
# of the M > 128 shapes only (512, 8192, 8192) is above the prefill crossover and runs the prefill kernel; (130, ...) and
# (300, 1024, 4096) run the decode kernel's 128-token variant
def test_nvfp4_weight_linear(ops, M, N, K, fp8_act):
    x = torch.randn(M, K, device="cuda").to(torch.bfloat16)
    w = (torch.randn(N, K, device="cuda") * 0.05).to(torch.bfloat16)
    pb = (w.float().abs().max() / (448.0 * 6.0)).reshape(1)
    wq, ws = ops.nvfp4_quantize(w, pb, True)
    b = torch.randn(N, device="cuda").to(torch.bfloat16) if M % 2 else None
    wd = _fp4_dq(wq, _from_blocked(ws, N, K // 16), pb)
    if fp8_act:
        xq, sx = ops.fp8_fakequant_rowwise(x)
        y = ops.nvfp4_weight_linear(xq, sx.reshape(-1), wq, ws, pb, b)
        ref64 = (xq.double() * sx.double()) @ wd.t()
    else:
        y = ops.nvfp4_weight_linear(x, None, wq, ws, pb, b)
        ref64 = x.double() @ wd.t()
    ref64 = ref64 + (b.double() if b is not None else 0)
    assert torch.isfinite(y.float()).all()
    assert sqnr(ref64, y) > 45.0


def test_quantize_api_all_formats(ops):
    """quantize_ + nn.Linear forward for every north-star config; SQNR vs the bf16 linear at the reference's bars."""
    from ao_b200.prototype.mx_formats import (MXDynamicActivationMXWeightConfig, MXTensor, NVFP4DynamicActivationNVFP4WeightConfig,
                                              NVFP4Tensor, NVFP4WeightFloat8ActivationConfig, NVFP4WeightOnlyConfig)
    from ao_b200.quantization import (Float8DynamicActivationFloat8WeightConfig, Float8Tensor, Int8DynamicActivationInt8WeightConfig,
                                      Int8Tensor, PerRow, quantize_)

    torch.manual_seed(0)
    cases = [(Int8DynamicActivationInt8WeightConfig(), Int8Tensor, 35.0), (Float8DynamicActivationFloat8WeightConfig(granularity=PerRow()), Float8Tensor, 25.0),
             (MXDynamicActivationMXWeightConfig(), MXTensor, 25.0), (NVFP4DynamicActivationNVFP4WeightConfig(), NVFP4Tensor, 15.0),
             (NVFP4WeightOnlyConfig(), NVFP4Tensor, 18.0), (NVFP4WeightFloat8ActivationConfig(), NVFP4Tensor, 17.0)]
    for cfg, cls, bar in cases:
        lin = torch.nn.Linear(1024, 512, bias=True, device="cuda", dtype=torch.bfloat16)
        ref = torch.nn.Linear(1024, 512, bias=True, device="cuda", dtype=torch.bfloat16)
        ref.load_state_dict(lin.state_dict())
        quantize_(lin, cfg)
        assert isinstance(lin.weight, cls), type(cfg).__name__
        for shape in [(1, 1024), (4, 8, 1024), (0, 1024)]:
            x = torch.randn(*shape, device="cuda", dtype=torch.bfloat16)
            y = lin(x)
            assert y.shape == (*shape[:-1], 512) and y.dtype == torch.bfloat16
            if x.numel():
                s = sqnr(ref(x), y)
                assert s > bar, f"{type(cfg).__name__}: SQNR {s:.1f} dB < {bar}"
        # dequantize() of the stored weight is close to the original
        assert sqnr(ref.weight, lin.weight.dequantize()) > (bar - 3)
