"""GPU parity tests for the int4 tile_packed_to_4d path (call through torch.ops.ao_b200 -> C ABI).

Oracle = oracle/ao_oracle.c (pinned to the reference by tests/test_oracle_golden.py).
Bit-exact: packing, unpacking, qparams, q, scale_and_zero, dequant.  GEMM outputs: SQNR vs the
oracle's exact-product fp64-accumulated result >= 45 dB (bf16 output rounding is ~55 dB) and
>= 80 dB vs aten._weight_int4pack_mm when that op is available (the reference's own kernel).
"""
import os

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


def _mk_q(N, K, g, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    q = torch.randint(0, 16, (N, K), device="cuda", generator=gen, dtype=torch.int32)
    s = (torch.rand(N, K // g, device="cuda", generator=gen) * 0.01 + 0.002).to(torch.bfloat16)
    z = ((torch.rand(N, K // g, device="cuda", generator=gen) - 0.5) * 0.02).to(torch.bfloat16)
    q_u8 = (q[:, ::2] << 4 | q[:, 1::2]).to(torch.uint8).contiguous()
    sz = torch.stack([s, z], dim=-1).transpose(0, 1).contiguous()
    return q, q_u8, sz


@pytest.mark.parametrize("N,K,ikt", [(8, 128, 8), (64, 1024, 8), (4096, 4096, 8), (16, 256, 4), (16, 64, 2)])
def test_pack_matches_oracle_and_aten(ops, N, K, ikt):
    o = _o()
    q, q_u8, _ = _mk_q(N, K, 32, N + K)
    ours = ops.int4_pack_tile4d(q_u8, ikt)
    ref = o.int4_pack_tile4d(q.cpu().numpy().astype(np.uint8), ikt)
    assert np.array_equal(ours.cpu().numpy(), ref)
    aten = torch.ops.aten._convert_weight_to_int4pack(q_u8, ikt)
    assert torch.equal(ours, aten), "layout differs from aten._convert_weight_to_int4pack"
    assert torch.equal(ops.int4_unpack_tile4d(ours), q_u8)


@pytest.mark.parametrize("g", [32, 64, 128, 256])
def test_dequant_bit_exact(ops, g):
    o = _o()
    q, q_u8, sz = _mk_q(256, 1024, g, g)
    qd = ops.int4_pack_tile4d(q_u8, 8)
    w = ops.int4_dequant_tile4d(qd, sz, g)
    ref = o.int4_dequant(q.cpu().numpy().astype(np.uint8), o.bf16_bits(sz), g)
    assert np.array_equal(o.bf16_bits(w), ref)


@pytest.mark.parametrize("impl", [1, 2])
@pytest.mark.parametrize("M,N,K,g,bias", [
    (1, 128, 1024, 32, False), (5, 256, 2048, 32, True), (16, 136, 1024, 64, False), (32, 512, 1024, 128, True),
    (33, 256, 1024, 256, False), (100, 128, 2048, 32, False),
])
def test_linear_vs_oracle(ops, impl, M, N, K, g, bias):
    o = _o()
    q, q_u8, sz = _mk_q(N, K, g, M * 7 + N)
    qd = ops.int4_pack_tile4d(q_u8, 8)
    x = torch.randn(M, K, device="cuda").to(torch.bfloat16)
    b = torch.randn(N, device="cuda").to(torch.bfloat16) if bias else None
    y = ops.int4_tilepacked_linear(x, qd, g, sz, b, N, impl)
    w_hat = o.bf16_to_f32(o.int4_dequant(q.cpu().numpy().astype(np.uint8), o.bf16_bits(sz), g))
    ref = o.linear_f32(o.bf16_to_f32(o.bf16_bits(x)), w_hat, o.bf16_to_f32(o.bf16_bits(b)) if bias else None)
    got = o.bf16_to_f32(o.bf16_bits(y))
    assert np.isfinite(got).all()
    assert o.sqnr_db(ref, got) > 45.0
    # and against the packed-weight oracle (fp32 accumulate, bf16 out)
    ref2 = o.bf16_to_f32(o.int4_linear(o.bf16_bits(x), qd.cpu().numpy(), o.bf16_bits(sz), g, o.bf16_bits(b) if bias else None))
    assert o.sqnr_db(ref2, got) > 45.0


@pytest.mark.parametrize("M,N,K", [(1, 4096, 4096), (32, 4096, 4096), (32, 1024, 4096), (32, 14336, 4096), (8, 4096, 14336)])
def test_linear_full_size_vs_aten_and_linearity(ops, M, N, K):
    """BASELINE sizes: compare with the reference's own kernel and check linearity + one-hot exactness."""
    g = 32
    q, q_u8, sz = _mk_q(N, K, g, 3)
    qd = ops.int4_pack_tile4d(q_u8, 8)
    x = torch.randn(M, K, device="cuda").to(torch.bfloat16)
    y = ops.int4_tilepacked_linear(x, qd, g, sz, None, N, 0)
    y_ref = torch.ops.aten._weight_int4pack_mm(x, qd, g, sz)
    num = y_ref.float().norm()
    den = (y_ref.float() - y.float()).norm()
    assert den == 0 or 20 * torch.log10(num / den) > 70.0
    # determinism
    assert torch.equal(y, ops.int4_tilepacked_linear(x, qd, g, sz, None, N, 0))
    # one-hot activation reads back the dequantised weight column exactly
    k = 1234 % K
    xh = torch.zeros(M, K, device="cuda", dtype=torch.bfloat16)
    xh[0, k] = 1.0
    w = ops.int4_dequant_tile4d(qd, sz, g)
    yh = ops.int4_tilepacked_linear(xh, qd, g, sz, None, N, 0)
    assert torch.equal(yh[0], w[:, k])
    # power-of-two scaling of x is exact
    y2 = ops.int4_tilepacked_linear((x.float() * 2).to(torch.bfloat16), qd, g, sz, None, N, 0)
    assert torch.equal(y2.float(), y.float() * 2)


@pytest.mark.parametrize("M,N,K,g,bias", [
    (129, 256, 1024, 32, False), (200, 136, 2048, 64, True), (256, 512, 1024, 128, False), (257, 384, 1024, 32, True),
    (700, 256, 2048, 256, False),
])
def test_prefill_kernel_vs_oracle(ops, M, N, K, g, bias):
    """M > 128 at small N x K: below the prefill crossover (ts_prefill.cuh `worth_it`), so these run the decode kernel's
    128-token variant over several token blocks (the prefill kernel itself: tests/test_kernel_paths_gpu.py); same
    oracle, same 45 dB bar, ragged token / feature tails included."""
    o = _o()
    q, q_u8, sz = _mk_q(N, K, g, M * 5 + N)
    qd = ops.int4_pack_tile4d(q_u8, 8)
    x = torch.randn(M, K, device="cuda").to(torch.bfloat16)
    b = torch.randn(N, device="cuda").to(torch.bfloat16) if bias else None
    y = ops.int4_tilepacked_linear(x, qd, g, sz, b, N, 1)
    w_hat = o.bf16_to_f32(o.int4_dequant(q.cpu().numpy().astype(np.uint8), o.bf16_bits(sz), g))
    ref = o.linear_f32(o.bf16_to_f32(o.bf16_bits(x)), w_hat, o.bf16_to_f32(o.bf16_bits(b)) if bias else None)
    got = o.bf16_to_f32(o.bf16_bits(y))
    assert np.isfinite(got).all()
    assert o.sqnr_db(ref, got) > 45.0
    # the CUDA-core cross-check kernel (impl = 2) on the same inputs
    y2 = ops.int4_tilepacked_linear(x, qd, g, sz, b, N, 2)
    assert o.sqnr_db(o.bf16_to_f32(o.bf16_bits(y2)), got) > 45.0


@pytest.mark.parametrize("M,N,K", [(512, 4096, 4096), (512, 4096, 14336), (300, 6144, 4096), (2048, 1024, 4096)])
def test_prefill_full_size_vs_aten_and_properties(ops, M, N, K):
    """BASELINE layer shapes at prefill token counts (tiles split across CTAs by the stream-K walk): the reference's own
    kernel, run-to-run determinism, one-hot exactness in rows 0, 255, 256 and M - 1, exact power-of-two scaling.  All
    four shapes are below the prefill crossover (fewer than 50 chunks of 128 x 256 x 128 per SM), so they run the
    decode kernel's 128-token variant with several token blocks; the prefill kernel has its own tests in
    tests/test_kernel_paths_gpu.py."""
    g = 32
    q, q_u8, sz = _mk_q(N, K, g, 11)
    qd = ops.int4_pack_tile4d(q_u8, 8)
    x = torch.randn(M, K, device="cuda").to(torch.bfloat16)
    y = ops.int4_tilepacked_linear(x, qd, g, sz, None, N, 0)
    y_ref = torch.ops.aten._weight_int4pack_mm(x, qd, g, sz)
    num = y_ref.float().norm()
    den = (y_ref.float() - y.float()).norm()
    assert den == 0 or 20 * torch.log10(num / den) > 70.0
    assert torch.equal(y, ops.int4_tilepacked_linear(x, qd, g, sz, None, N, 0))
    w = ops.int4_dequant_tile4d(qd, sz, g)
    xh = torch.zeros(M, K, device="cuda", dtype=torch.bfloat16)
    rows = sorted({0, 255 % M, 256 % M, M - 1})
    ks = [(977 * (i + 1)) % K for i in range(len(rows))]
    for m, k in zip(rows, ks):
        xh[m, k] = 1.0
    yh = ops.int4_tilepacked_linear(xh, qd, g, sz, None, N, 0)
    for m, k in zip(rows, ks):
        assert torch.equal(yh[m], w[:, k])
    y2 = ops.int4_tilepacked_linear((x.float() * 2).to(torch.bfloat16), qd, g, sz, None, N, 0)
    assert torch.equal(y2.float(), y.float() * 2)


@pytest.mark.parametrize("M", [65, 100, 128, 512])
def test_many_token_variants_are_stable_over_repeated_launches(ops, M):
    """Regression (round 2): with 4 weight stages and 3 dequant warpgroups a warpgroup could pass the parity wait for
    chunk i + 4 before chunk i had landed -- sporadic wrong results / launch failures of the 65..128-token variant (and of
    the prefill kernel built on the same ring).  Short per-CTA ranges (a small projection) made it likely."""
    N, K, g = 6144, 4096, 32
    q, q_u8, sz = _mk_q(N, K, g, 5)
    qd = ops.int4_pack_tile4d(q_u8, 8)
    x = torch.randn(M, K, device="cuda").to(torch.bfloat16)
    ref = torch.ops.aten._weight_int4pack_mm(x, qd, g, sz)
    y0 = ops.int4_tilepacked_linear(x, qd, g, sz, None, N, 1)
    for _ in range(40):
        y = ops.int4_tilepacked_linear(x, qd, g, sz, None, N, 1)
    torch.cuda.synchronize()
    assert torch.equal(y, y0)
    d = (ref.float() - y.float()).norm()
    assert d == 0 or 20 * torch.log10(ref.float().norm() / d) > 70.0


def test_quantize_api_end_to_end(ops):
    """quantize_(Int4WeightOnlyConfig tile_packed_to_4d g=32): qparams/qdata bit-exact vs oracle, SQNR vs bf16 linear > 20 dB
    (the reference's own bar, test_int4_tile_packed_to_4d_tensor.py:54-69)."""
    from ao_b200.quantization import Int4TilePackedTo4dTensor, Int4WeightOnlyConfig, quantize_

    o = _o()
    torch.manual_seed(0)
    lin = torch.nn.Linear(1024, 256, bias=True, device="cuda", dtype=torch.bfloat16)
    ref_lin = torch.nn.Linear(1024, 256, bias=True, device="cuda", dtype=torch.bfloat16)
    ref_lin.load_state_dict(lin.state_dict())
    w_bits = o.bf16_bits(lin.weight)
    quantize_(lin, Int4WeightOnlyConfig(group_size=32, int4_packing_format="tile_packed_to_4d"))
    wt = lin.weight
    assert isinstance(wt, Int4TilePackedTo4dTensor)
    s, z = o.int4_choose_qparams(w_bits, 32)
    q = o.int4_quantize(w_bits, 32, s, z)
    assert np.array_equal(o.bf16_bits(wt.scale_and_zero), o.pack_scales_and_zeros(s, z))
    assert np.array_equal(wt.qdata.cpu().numpy(), o.int4_pack_tile4d(q, 8))
    for shape in [(1, 1024), (3, 5, 1024), (0, 1024), (32, 1024)]:
        x = torch.randn(*shape, device="cuda", dtype=torch.bfloat16)
        y = lin(x)
        assert y.shape == (*shape[:-1], 256) and y.dtype == torch.bfloat16
        if x.numel():
            yr = ref_lin(x)
            sq = 20 * torch.log10(yr.float().norm() / (yr.float() - y.float()).norm())
            assert sq > 20.0
    # fp16 activations are cast to bf16 and back (reference :278,:299)
    x = torch.randn(4, 1024, device="cuda", dtype=torch.float16)
    assert lin(x).dtype == torch.float16
    # dequantize() == oracle W^
    w_hat = o.int4_dequant(q, o.pack_scales_and_zeros(s, z), 32)
    assert np.array_equal(o.bf16_bits(wt.dequantize()), w_hat)
    # K not a multiple of 1024 -> padded; N not multiple of 8 -> padded
    lin2 = torch.nn.Linear(1152, 100, bias=False, device="cuda", dtype=torch.bfloat16)
    ref2 = torch.nn.Linear(1152, 100, bias=False, device="cuda", dtype=torch.bfloat16)
    ref2.load_state_dict(lin2.state_dict())
    quantize_(lin2, Int4WeightOnlyConfig(group_size=128, int4_packing_format="tile_packed_to_4d"))
    assert lin2.weight.qdata.shape == (13, 16, 32, 4)
    x = torch.randn(7, 1152, device="cuda", dtype=torch.bfloat16)
    y, yr = lin2(x), ref2(x)
    assert y.shape == (7, 100)
    assert 20 * torch.log10(yr.float().norm() / (yr.float() - y.float()).norm()) > 20.0


def test_prefill_token_counts_through_the_public_api(ops):
    """quantize_ -> nn.Linear.forward with hundreds / thousands of tokens: a gate|up-sized layer takes the prefill-shaped
    kernel (>= 50 chunks of 128 x 256 per SM), a small one the 128-token-block path; both against the linear on the
    dequantised weight (>= 45 dB: bf16 output rounding only) and the bf16 linear (>= 20 dB, the reference's bar), with a
    3-D batch and a bias."""
    from ao_b200.quantization import Int4WeightOnlyConfig, quantize_

    torch.manual_seed(1)
    for (k, n, shapes) in [(4096, 14336, [(2048, 4096), (4, 300, 4096)]), (1024, 512, [(700, 1024)])]:
        lin = torch.nn.Linear(k, n, bias=True, device="cuda", dtype=torch.bfloat16)
        ref_lin = torch.nn.Linear(k, n, bias=True, device="cuda", dtype=torch.bfloat16)
        ref_lin.load_state_dict(lin.state_dict())
        quantize_(lin, Int4WeightOnlyConfig(group_size=32, int4_packing_format="tile_packed_to_4d"))
        w_hat = lin.weight.dequantize()
        for shape in shapes:
            x = torch.randn(*shape, device="cuda", dtype=torch.bfloat16)
            y = lin(x)
            assert y.shape == (*shape[:-1], n) and y.dtype == torch.bfloat16
            yd = torch.nn.functional.linear(x.float(), w_hat.float(), lin.bias.float())
            assert 20 * torch.log10(yd.norm() / (yd - y.float()).norm()) > 45.0
            yr = ref_lin(x).float()
            assert 20 * torch.log10(yr.norm() / (yr - y.float()).norm()) > 20.0


def test_cuda_graph_capture(ops):
    g = 32
    q, q_u8, sz = _mk_q(1024, 4096, g, 9)
    qd = ops.int4_pack_tile4d(q_u8, 8)
    x = torch.randn(8, 4096, device="cuda").to(torch.bfloat16)
    y_eager = ops.int4_tilepacked_linear(x, qd, g, sz, None, 1024, 0)
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        ops.int4_tilepacked_linear(x, qd, g, sz, None, 1024, 0)
    torch.cuda.current_stream().wait_stream(st)
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        y = ops.int4_tilepacked_linear(x, qd, g, sz, None, 1024, 0)
    gr.replay()
    torch.cuda.synchronize()
    assert torch.equal(y, y_eager)


# ---------------------------------------------------------------------------------------------- HQQ (SURVEY §8f-2)
@pytest.mark.gpu
@pytest.mark.parametrize("case", ["g32", "g128", "g64_outlier"])
def test_hqq_quantize_against_reference_fixture_and_oracle(case):
    """The CUDA HQQ solver against (a) the reference's own output on the same weights (golden fixture, CPU fp32 run of
    torchao) and (b) the oracle.  Floating-point iterative solver: bars as in tests/test_oracle_golden.py: scales
    bit-exact, codes at most one step apart and >= 99 % identical, zeros within one step (>= 99 % within 0.01 step),
    mean reconstruction error within 0.1 %."""
    import numpy as np
    import torch

    import ao_b200  # noqa: F401
    from oracle import oracle as o

    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "int4_hqq.npz"))
    w_bits, g = gold[f"{case}__w"], int(gold[f"{case}__g"])
    w = o.bf16_tensor(w_bits).cuda()
    q, s, z = torch.ops.ao_b200.int4_hqq_quantize(w, g)
    torch.cuda.synchronize()
    q = q.cpu().numpy()
    s, z = o.bf16_bits(s), o.bf16_bits(z)
    qo, so, zo, _ = o.int4_hqq(w_bits, g)

    def recon_err(qq, ss, zz):
        wf = o.bf16_to_f32(w_bits).reshape(-1, g)
        deq = (qq.reshape(-1, g).astype(np.float32) - 8.0) * o.bf16_to_f32(ss).reshape(-1, 1) + o.bf16_to_f32(zz).reshape(-1, 1)
        return float(np.abs(wf - deq).mean())

    for name, (qr, sr, zr) in {"reference": (gold[f"{case}__q"], gold[f"{case}__s"], gold[f"{case}__z"]),
                               "oracle": (qo, so, zo)}.items():
        assert np.array_equal(s, sr), f"scale differs from {name}"
        diff = np.abs(q.astype(np.int32) - qr.astype(np.int32))
        assert diff.max() <= 1 and (diff != 0).mean() <= 1e-2, (name, diff.max(), (diff != 0).mean())
        steps = np.abs(o.bf16_to_f32(z) - o.bf16_to_f32(zr)) / o.bf16_to_f32(sr)
        assert (steps > 0.01).mean() <= 0.01 and steps.max() <= 1.0, (name, steps.max())
        e, er = recon_err(q, s, z), recon_err(qr, sr, zr)
        assert abs(e - er) <= 1e-3 * er, (name, e, er)


@pytest.mark.gpu
def test_hqq_through_quantize_api_beats_tinygemm_qparams():
    """Int4WeightOnlyConfig(int4_choose_qparams_algorithm="hqq") end to end (reference test_int4_tile_packed_to_4d_tensor.py
    uses SQNR > 20 dB as its bar; HQQ must also not be worse than the default qparams, which is its purpose)."""
    import torch

    import ao_b200  # noqa: F401
    from ao_b200.quantization import Int4WeightOnlyConfig, quantize_

    torch.manual_seed(0)
    lin = torch.nn.Linear(2048, 512, bias=False, device="cuda", dtype=torch.bfloat16)
    w = lin.weight.detach().clone()
    x = torch.randn(8, 2048, device="cuda", dtype=torch.bfloat16)
    ref = x.float() @ w.float().t()

    def run(algo):
        m = torch.nn.Linear(2048, 512, bias=False, device="cuda", dtype=torch.bfloat16)
        m.weight.data.copy_(w)
        quantize_(m, Int4WeightOnlyConfig(group_size=32, int4_packing_format="tile_packed_to_4d", int4_choose_qparams_algorithm=algo))
        y = m(x).float()
        werr = (m.weight.dequantize().float() - w.float()).abs().mean().item()
        return 20 * torch.log10(ref.norm() / (ref - y).norm()).item(), werr

    sq_t, we_t = run("tinygemm")
    sq_h, we_h = run("hqq")
    assert sq_h > 20.0 and sq_t > 20.0
    assert we_h <= we_t * 1.001, (we_h, we_t)


# ------------------------------------------------------------------ op registration contract (SURVEY §8b)
@pytest.mark.gpu
def test_ops_pass_opcheck_and_survive_fullgraph_tracing():
    """The reference requires its extern ops to pass torch.library.opcheck (schema, fake kernel, functionalisation) and
    to survive torch.compile(fullgraph=True) (test/test_ops.py, test_float8_tensor.py:397).  Tracing uses the
    aot_eager backend: the graph is captured with fake tensors and our Meta kernels, then runs our CUDA ops."""
    import torch

    import ao_b200  # noqa: F401
    from ao_b200.quantization import Int4WeightOnlyConfig, quantize_

    torch.manual_seed(0)
    x = torch.randn(4, 1024, device="cuda", dtype=torch.bfloat16)
    lin = torch.nn.Linear(1024, 256, bias=True, device="cuda", dtype=torch.bfloat16)
    quantize_(lin, Int4WeightOnlyConfig(group_size=32, int4_packing_format="tile_packed_to_4d"))
    w = lin.weight
    tests = ("test_schema", "test_faketensor")
    torch.library.opcheck(torch.ops.ao_b200.int4_tilepacked_linear.default, (x, w.qdata, 32, w.scale_and_zero, lin.bias, 256, 0),
                          test_utils=tests)
    torch.library.opcheck(torch.ops.ao_b200.int8_quantize_rowwise.default, (x,), test_utils=tests)
    torch.library.opcheck(torch.ops.ao_b200.mxfp8_quantize.default, (x, True), test_utils=tests)
    torch.library.opcheck(torch.ops.ao_b200.int4_hqq_quantize.default, (x, 32), test_utils=tests)

    y_eager = lin(x)
    compiled = torch.compile(lin, fullgraph=True, backend="aot_eager")
    y_comp = compiled(x)
    assert torch.equal(y_eager, y_comp)


# ------------------------------------------------------------------ the reference's own tensor-level tests
# (test/quantization/quantize_/workflows/int4/test_int4_tile_packed_to_4d_tensor.py), restated for this package
def _int4_cfg(algo="tinygemm", g=128):
    from ao_b200.quantization import Int4WeightOnlyConfig

    return Int4WeightOnlyConfig(group_size=g, int4_packing_format="tile_packed_to_4d", int4_choose_qparams_algorithm=algo)


def _sqnr(a, b):
    return (20 * torch.log10(a.float().norm() / (a.float() - b.float()).norm())).item()


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["tinygemm", "hqq"])
def test_reference_slice_semantics(algo):
    """reference :90-192: narrow on dim 0 / dim 1 equals narrowing the packed payloads, keeps aliasing, and a linear on
    the (contiguous) slice matches the bf16 linear on the sliced weight (SQNR > 14 dB at g=128)."""
    import ao_b200  # noqa: F401
    from ao_b200.quantization import quantize_

    torch.manual_seed(0)
    dummy = torch.nn.Linear(2048, 2048, bias=False, dtype=torch.bfloat16, device="cuda")
    w_hp = dummy.weight.detach().clone()
    quantize_(dummy, _int4_cfg(algo))
    w = dummy.weight
    w1 = w.narrow(0, 0, 1024)
    assert torch.equal(w1.qdata, w.qdata.narrow(0, 0, 128)) and torch.equal(w1.scale_and_zero, w.scale_and_zero.narrow(1, 0, 1024))
    assert w1.qdata.data_ptr() == w.qdata.data_ptr() and w1.scale_and_zero.data_ptr() == w.scale_and_zero.data_ptr()
    w2 = w.narrow(1, 0, 1024)
    assert torch.equal(w2.qdata, w.qdata.narrow(1, 0, 8)) and torch.equal(w2.scale_and_zero, w.scale_and_zero.narrow(0, 0, 8))
    x1 = torch.randn(2, 2048, dtype=torch.bfloat16, device="cuda")
    l1 = torch.nn.Linear(2048, 1024, bias=False, dtype=torch.bfloat16, device="cuda")
    l1.weight = torch.nn.Parameter(w1.contiguous(), requires_grad=False)
    assert _sqnr(x1 @ w_hp[:1024].t(), l1(x1)) > 14
    x2 = torch.randn(2, 1024, dtype=torch.bfloat16, device="cuda")
    l2 = torch.nn.Linear(1024, 2048, bias=False, dtype=torch.bfloat16, device="cuda")
    l2.weight = torch.nn.Parameter(w2.contiguous(), requires_grad=False)
    assert _sqnr(x2 @ w_hp[:, :1024].t(), l2(x2)) > 14


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["tinygemm", "hqq"])
def test_reference_slice_and_copy_similar_to_vllm(algo):
    """reference torchao/testing/utils.py:471-519 (vLLM's weight loader), plus the write-through the loader relies on."""
    import ao_b200  # noqa: F401
    from ao_b200.quantization import quantize_

    torch.manual_seed(1)
    dst_l = torch.nn.Linear(1024, 1024, device="cuda", dtype=torch.bfloat16)
    quantize_(dst_l, _int4_cfg(algo))
    src_l = torch.nn.Linear(1024, 1024, device="cuda", dtype=torch.bfloat16)
    src_l.weight = torch.nn.Parameter(src_l.weight + 1.0 + 2 * torch.randn(1024, 1024, device="cuda", dtype=torch.bfloat16),
                                      requires_grad=False)
    quantize_(src_l, _int4_cfg(algo))
    for rank in (0, 1):
        pd = dst_l.weight.data.narrow(0, rank * 512, 512)
        lw = src_l.weight.narrow(0, rank * 512, 512)
        assert not torch.equal(pd.qdata[0], lw.qdata[0])
        pd.copy_(lw)
        assert torch.equal(pd.qdata[0], lw.qdata[0]) and torch.equal(pd.scale_and_zero, lw.scale_and_zero)
    assert torch.equal(dst_l.weight.qdata, src_l.weight.qdata) and torch.equal(dst_l.weight.scale_and_zero, src_l.weight.scale_and_zero)


@pytest.mark.gpu
def test_reference_module_path_prescale_to_device_and_cpu_error():
    """reference :72-88 (type path survives state_dict save/load), :242-260 (act_pre_scale), :204-220 (.to(device)),
    :194-202 (CPU init raises NotImplementedError), :298-308 (group sizes 32/64/128)."""
    import io

    import ao_b200  # noqa: F401
    from ao_b200.quantization import quantize_

    lin = torch.nn.Linear(128, 256, dtype=torch.bfloat16, device="cuda")
    quantize_(lin, _int4_cfg())
    assert str(type(lin.weight)) == "<class 'ao_b200.quantization.Int4TilePackedTo4dTensor'>"
    buf = io.BytesIO()
    torch.save(lin.state_dict(), buf)
    buf.seek(0)
    sd = torch.load(buf, weights_only=True)
    assert str(type(sd["weight"])) == "<class 'ao_b200.quantization.Int4TilePackedTo4dTensor'>"
    assert torch.equal(sd["weight"].qdata, lin.weight.qdata)
    lin.to("cuda")
    lin.to(device="cuda")

    x = torch.randn(1, 128, dtype=torch.bfloat16, device="cuda")
    l2 = torch.nn.Linear(128, 256, bias=False, dtype=torch.bfloat16, device="cuda")
    original = l2(x)
    quantize_(l2, _int4_cfg())
    assert l2.weight.act_pre_scale is None
    l2.weight.act_pre_scale = 2
    assert _sqnr(original * 2, l2(x)) > 20

    with pytest.raises(NotImplementedError):
        quantize_(torch.nn.Linear(128, 256, dtype=torch.bfloat16), _int4_cfg())

    for g in (32, 64, 128):
        l3 = torch.nn.Linear(1024, 512, bias=False, dtype=torch.bfloat16, device="cuda")
        ref = l3.weight.detach().clone()
        quantize_(l3, _int4_cfg(g=g))
        assert l3.weight.block_size == [1, g]
        xx = torch.randn(4, 1024, dtype=torch.bfloat16, device="cuda")
        assert _sqnr(xx @ ref.t(), l3(xx)) > 20
