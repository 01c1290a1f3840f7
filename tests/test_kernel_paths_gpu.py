"""Kernel-path tests: every GEMM entry point checked against an fp64 reference, with the kernel that ran asserted by name.

Which kernel serves a call depends on the token count M (16 / 32 / 64 / 128-token variants of the decode kernels), on
the prefill crossover (ts_prefill.cuh `worth_it`: at least 50 chunks of 128 rows x 256 tokens x 128 k per SM) and, for
correctness of the stream-K fix-up, on how many contributor CTAs feed one owner.  Each test here asserts the kernel
(family and token-block template argument) it targets through torch.profiler, so a dispatch change cannot silently turn
a prefill test into a decode test.

Numerics.  Reference: ref = (x_eff @ w_hat^T) * col + bias in fp64, where x_eff and w_hat are the exact operand values
the kernel multiplies (dequantised weights, fake-quantised activations times their scales) and col the per-out-feature
scale.  Every output element must satisfy |y - ref| <= 2^-8 |ref| + C_MAG * mag with mag = |x_eff| @ |w_hat|^T * |col|:
the first term is the bf16 output rounding, the second fp32 accumulation (it scales with the sum of |products|, not
with the result, which can cancel).  Each such comparison carries a self-check: the same bound must FAIL against a
reference with one 128-k chunk dropped from one output tile, in a chunk held by a contributor CTA (not the tile's
owner), so the tolerance provably catches a lost or misplaced partial sum.
"""
import re

import pytest
import torch

pytestmark = pytest.mark.gpu

REL = 2.0 ** -8
# fp32-accumulation term of the bound.  Calibrated on a B200 (148 SMs, 1000 W power limit) over every comparison in
# this file: the largest (|y - ref| - 2^-8 |ref|) / mag observed was 1.5e-7 (about 2^-22.7; int4 fused gate|up, 512
# tokens, K = 4096, prefill kernel), and K = 131072 stayed below it.  2^-18 = 3.8e-6 leaves 25x headroom and is still
# far below what one dropped chunk costs (every self-check fails by a wide margin).  Run with -s to see the ratios.
C_MAG = 2.0 ** -18

FLAG_BYTES = 16 * 1024   # stream-K flag area at the start of the workspace (streamk.cuh WS_FLAGS_BYTES)
E2M1 = [0, 0.5, 1, 1.5, 2, 3, 4, 6, -0.0, -0.5, -1, -1.5, -2, -3, -4, -6]


@pytest.fixture(scope="module")
def ops():
    import ao_b200  # noqa: F401

    return torch.ops.ao_b200


def _sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------------------------------------ which kernel ran
_KERNEL_RE = re.compile(r"\b(ts_gemm_kernel|ts_prefill_kernel|lowp_linear_kernel)\s*<([^>]*)>")


def kernels_launched(fn):
    """Run fn under torch.profiler (CUDA activity only); return (fn's result, names of the kernels launched)."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    events = prof.events()
    names = [e.name for e in events if e.device_type == torch.autograd.DeviceType.CUDA]
    if not names:   # kernels attached to the host events that launched them instead
        names = [k.name for e in events for k in getattr(e, "kernels", [])]
    return out, names


def gemm_kernels(names):
    """(family, N_MMA) of every GEMM kernel in names, in launch order; N_MMA is None for the prefill kernel."""
    out = []
    for n in names:
        m = _KERNEL_RE.search(n)
        if m:
            args = [a.strip() for a in m.group(2).split(",")]
            n_mma = None
            if m.group(1) != "ts_prefill_kernel":
                n_mma = int(re.search(r"(\d+)\s*$", args[1]).group(1))
            out.append((m.group(1), n_mma))
    return out


def run_expecting(fn, family, n_mma=None):
    """fn must launch exactly one GEMM kernel, of `family` (and token block `n_mma`); returns fn's result."""
    out, names = kernels_launched(fn)
    ks = gemm_kernels(names)
    assert ks == [(family, n_mma)], f"expected {family}<N_MMA={n_mma}>, saw {ks} (all kernels: {names})"
    return out


def flags_clear(ops, like):
    ws = ops.debug_workspace(like)
    assert not bool(ws[:FLAG_BYTES].any()), "stream-K flags left raised in the workspace"


# ------------------------------------------------------------------------------------------------ stream-K split
class Split:
    """The stream-K work split the launchers choose (ts_gemm.cuh / ts_prefill.cuh `plan`, lowp_linear.cu `launch`).

    family: "ts" (decode TS kernel: one CTA per SM, >= 4 chunks per CTA), "prefill" (one CTA per SM, >= 8 chunks),
    "lowp" (two CTAs per SM for N_MMA <= 64, >= 8 chunks).  kw = elements of K per chunk."""

    def __init__(self, family, M, N, KT, tok, kw=128):
        self.M, self.N, self.KT, self.tok, self.kw = M, N, KT, tok, kw
        self.n_tiles, self.m_blocks = -(-N // 128), -(-M // tok)
        self.U = self.n_tiles * self.m_blocks * KT
        sm = _sm()
        grid, min_units = {"ts": (sm, 4), "prefill": (sm, 8), "lowp": (sm * (2 if tok <= 64 else 1), 8)}[family]
        if self.U // min_units < grid:
            grid = max(self.U // min_units, 1)
        self.G = grid

    def cta_of_unit(self, u):
        return ((u + 1) * self.G + self.U - 1) // self.U - 1

    def contributors(self, tile):
        """CTAs that publish a partial of `tile` for its owner (the CTA holding chunk 0)."""
        return self.cta_of_unit(tile * self.KT + self.KT - 1) - self.cta_of_unit(tile * self.KT)

    def contributor_chunk(self):
        """(tile, chunk): the last chunk of the most finely split tile (the last such tile) -- held by that tile's last
        contributor CTA, never by its owner."""
        tile = max(range(self.n_tiles * self.m_blocks), key=lambda t: (self.contributors(t), t))
        assert self.contributors(tile) > 0, "no tile of this shape is split: the self-check needs a contributor"
        return tile, self.KT - 1

    def tile_box(self, tile):
        n0, m0 = (tile % self.n_tiles) * 128, (tile // self.n_tiles) * self.tok
        return m0, min(m0 + self.tok, self.M), n0, min(n0 + 128, self.N)


# ------------------------------------------------------------------------------------------------ reference + bound
class Ref:
    """ref = (x_eff @ w_hat^T) * col + bias and mag = |x_eff| @ |w_hat|^T * |col|, in fp64."""

    def __init__(self, x_eff, w_hat, col=None, bias=None):
        self.x, self.w = x_eff.double(), w_hat.double()
        self.col = None if col is None else col.double().reshape(1, -1)
        ref, mag = self.x @ self.w.t(), self.x.abs() @ self.w.abs().t()
        if self.col is not None:
            ref, mag = ref * self.col, mag * self.col.abs()
        if bias is not None:
            ref = ref + bias.double().reshape(1, -1)
        self.ref, self.mag = ref, mag

    def without_chunk(self, split, tile, kc):
        m0, m1, n0, n1 = split.tile_box(tile)
        ks = slice(kc * split.kw, (kc + 1) * split.kw)
        part = self.x[m0:m1, ks] @ self.w[n0:n1, ks].t()
        if self.col is not None:
            part = part * self.col[:, n0:n1]
        bad = self.ref.clone()
        bad[m0:m1, n0:n1] -= part
        return bad


def _within(y, ref, mag):
    return (y.double() - ref).abs() <= REL * ref.abs() + C_MAG * mag


def assert_bound(y, r, split, label=""):
    """Per-element bound against r, and the self-check: the bound fails once one contributor-held chunk is dropped."""
    assert y.shape == r.ref.shape, (y.shape, r.ref.shape)
    assert torch.isfinite(y.float()).all(), f"{label}: non-finite outputs"
    ok = _within(y, r.ref, r.mag)
    slack = ((y.double() - r.ref).abs() - REL * r.ref.abs()) / r.mag.clamp_min(1e-300)
    worst = float(slack.max())
    print(f"[bound] {label}: max (|y - ref| - 2^-8 |ref|) / mag = {worst:.3e} (C_MAG = {C_MAG:.3e})")
    if not bool(ok.all()):
        bad = (~ok).nonzero()[:8].tolist()
        pytest.fail(f"{label}: {int((~ok).sum())} of {ok.numel()} outputs outside the bound, e.g. (m, n) {bad}; "
                    f"worst (|err| - 2^-8|ref|)/mag = {worst:.3e}")
    tile, kc = split.contributor_chunk()
    assert not bool(_within(y, r.without_chunk(split, tile, kc), r.mag).all()), (
        f"{label}: self-check -- the bound also accepts a reference without chunk {kc} of tile {tile}")


def sqnr(ref, out):
    ref, out = ref.double(), out.double()
    d = (ref - out).norm()
    return float("inf") if d == 0 else float(20 * torch.log10(ref.norm() / d))


# ------------------------------------------------------------------------------------------------ operands
def prefill_n(M, K, multiple=8):
    """The smallest number of 128-row output tiles that puts (M, N, K) at the prefill crossover (>= 50 chunks of
    128 x 256 x 128 per SM), as a RAGGED feature count: the last tile has fewer than 128 rows.  Returns (N_out, N)
    with N = N_out rounded up to `multiple` (int4 packs N in multiples of 8; nvfp4 wants N % 16 == 0 and N_out == N)."""
    per_tile = -(-M // 256) * (K // 128)
    tiles = -(-50 * _sm() // per_tile)
    n_out = tiles * 128 - 36 if multiple == 8 else tiles * 128 - 48
    n = -(-n_out // multiple) * multiple
    assert -(-n_out // 128) * per_tile >= 50 * _sm() > (tiles - 1) * per_tile
    return n_out, n


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _int4_weight(ops, N, K, g, seed):
    """Random codes and (scale, zero) pairs as tinygemm stores them; returns (qdata, scale_and_zero, w_hat bf16)."""
    gen = _gen(seed)
    q = torch.randint(0, 16, (N, K), device="cuda", generator=gen, dtype=torch.int32)
    s = (torch.rand(N, K // g, device="cuda", generator=gen) * 0.01 + 0.002).to(torch.bfloat16)
    z = ((torch.rand(N, K // g, device="cuda", generator=gen) - 0.5) * 0.02).to(torch.bfloat16)
    q_u8 = (q[:, ::2] << 4 | q[:, 1::2]).to(torch.uint8).contiguous()
    sz = torch.stack([s, z], dim=-1).transpose(0, 1).contiguous()
    qd = ops.int4_pack_tile4d(q_u8, 8)
    return qd, sz, ops.int4_dequant_tile4d(qd, sz, g)   # dequant: bit-exact vs the oracle (test_int4_gpu.py)


def _fp4_values(q, s_plain):
    """e2m1 codes [rows, K/2] x e4m3 block-16 scales [rows, K/16] -> exact fp64 values."""
    lut = torch.tensor(E2M1, dtype=torch.float64, device=q.device)
    v = torch.stack([lut[(q & 15).long()], lut[(q >> 4).long()]], dim=-1).reshape(q.shape[0], -1)
    return v * s_plain.contiguous().view(torch.float8_e4m3fn).double().repeat_interleave(16, 1)


def _unblock(s, rows, cols):
    from ao_b200.prototype.mx_formats.utils import from_blocked

    return from_blocked(s.reshape(-1), rows, cols)


def _nvfp4_weight(ops, N, K, seed, halves=False):
    """nvfp4 weight with its blocked scales; returns (wq, ws, b_pts, w_values fp64 without b_pts).  halves: the rows
    [0, N1) and [N1, N) are quantized with different per-tensor scales (a fused group) and b_pts has N entries."""
    gen = _gen(seed)
    w = (torch.randn(N, K, device="cuda", generator=gen) * 0.05).to(torch.bfloat16)
    if not halves:
        pts = (w.float().abs().max() / (448.0 * 6.0)).reshape(1)
        wq, ws = ops.nvfp4_quantize(w, pts, True)
        return wq, ws, pts, _fp4_values(wq, _unblock(ws, N, K // 16))
    n1 = 128 * (N // 256)   # a multiple of 128: the blocked scale tiles of the two halves concatenate
    w[n1:] *= 8             # a different amax, so a different per-tensor scale
    parts = []
    for lo, hi in ((0, n1), (n1, N)):
        pts = (w[lo:hi].float().abs().max() / (448.0 * 6.0)).reshape(1)
        wq, ws = ops.nvfp4_quantize(w[lo:hi].contiguous(), pts, True)
        parts.append((wq, ws, pts.expand(hi - lo)))
    wq = torch.cat([p[0] for p in parts]).contiguous()
    ws = torch.cat([p[1].reshape(-1) for p in parts]).contiguous()
    b_pts = torch.cat([p[2] for p in parts]).contiguous()
    assert b_pts.numel() == N and b_pts[0] != b_pts[-1]
    return wq, ws, b_pts, _fp4_values(wq, _unblock(ws, N, K // 16))


def _bf16_ulp(v):
    """One bf16 ulp of each fp64 value (0 for 0)."""
    a = v.abs()
    return torch.where(a > 0, torch.exp2(torch.floor(torch.log2(a.clamp_min(1e-300))) - 7), torch.zeros_like(a))


def _one_hot(M, K, seed):
    """A one-hot x: rows 0, 255, 256 and M - 1 (those < M), each with its 1 in a different 128-k chunk, the last one in
    the last chunk."""
    rows = sorted({r for r in (0, 255, 256, M - 1) if r < M})
    KT = K // 128
    chunks = [KT - 1] + [(KT * (i + 1)) // (len(rows) + 1) for i in range(len(rows) - 1)]
    assert len(set(chunks)) == len(rows)
    ks = [c * 128 + (37 * i + seed) % 128 for i, c in enumerate(chunks)]
    xh = torch.zeros(M, K, device="cuda", dtype=torch.bfloat16)
    for m, k in zip(rows, ks):
        xh[m, k] = 1.0
    return xh, rows, ks


def _other_rows_zero(yh, rows):
    keep = torch.ones(yh.shape[0], dtype=torch.bool, device=yh.device)
    keep[rows] = False
    assert not bool(yh[keep].any()), "a one-hot input produced non-zero outputs in rows whose input is all zero"


# ================================================================================== A. prefill kernel, int4
@pytest.mark.parametrize("M,K,g,bias,pad", [
    (129, 14336, 32, True, 0),     # first M above 128: a one-token tail tile
    (257, 14336, 64, True, 0),     # N_out < N
    (300, 4096, 128, False, 64),   # x a column slice of a wider buffer (row pitch K + 64)
    (1000, 4096, 256, False, 0),   # a scale row spans two 128-k chunks
])
def test_int4_prefill_kernel_vs_fp64(ops, M, K, g, bias, pad):
    """ts_prefill_kernel<Int4Fmt> with ragged feature / token tails, every group size, strided activations."""
    n_out, N = prefill_n(M, K)
    assert n_out < N and n_out % 128
    qd, sz, w_hat = _int4_weight(ops, N, K, g, M + K + g)
    gen = _gen(M)
    wide = torch.randn(M, K + pad, device="cuda", generator=gen).to(torch.bfloat16)
    x = wide[:, :K]
    assert x.is_contiguous() == (pad == 0)
    b = torch.randn(n_out, device="cuda", generator=gen).to(torch.bfloat16) if bias else None
    lin = lambda xx, bb=b: ops.int4_tilepacked_linear(xx, qd, g, sz, bb, n_out, 0)

    y = run_expecting(lambda: lin(x), "ts_prefill_kernel")
    flags_clear(ops, x)
    split = Split("prefill", M, n_out, K // 128, 256)
    assert_bound(y, Ref(x, w_hat[:n_out], None, b), split, f"int4 prefill M={M} K={K} g={g}")
    # the CUDA-core kernel (impl = 2) on the same inputs
    assert sqnr(ops.int4_tilepacked_linear(x, qd, g, sz, b, n_out, 2), y) >= 45.0
    # run to run: bit-identical (split tiles are summed in a fixed order)
    assert torch.equal(lin(x), y)
    flags_clear(ops, x)
    # one-hot rows read back the dequantised weight column bit for bit
    xh, rows, ks = _one_hot(M, K, g)
    yh = lin(xh, None)
    for m, k in zip(rows, ks):
        assert torch.equal(yh[m], w_hat[:n_out, k]), f"one-hot row {m}, k = {k}"
    _other_rows_zero(yh, rows)
    # power-of-two scaling of x is exact (no bias)
    y1 = lin(x, None)
    y2 = lin((wide * 2)[:, :K], None)
    assert torch.equal(y2.float(), y1.float() * 2)
    flags_clear(ops, x)


# ================================================================================== B. prefill kernel, nvfp4 weight
@pytest.mark.parametrize("M,K,act,bias,halves", [
    (129, 14336, "bf16", True, False),
    (300, 4096, "fp8", False, False),
    (257, 8192, "bf16", True, True),   # per-out-feature b_pts (a fused nvfp4 group)
])
def test_nvfp4_weight_prefill_kernel_vs_fp64(ops, M, K, act, bias, halves):
    """ts_prefill_kernel<Nvfp4Fmt>: bf16 and e4m3 fake-quant activations, bias, ragged N, per-out-feature b_pts."""
    _, N = prefill_n(M, K, 16)
    assert N % 128
    wq, ws, b_pts, w_val = _nvfp4_weight(ops, N, K, M + K, halves)
    gen = _gen(M + 1)
    x = torch.randn(M, K, device="cuda", generator=gen).to(torch.bfloat16)
    b = torch.randn(N, device="cuda", generator=gen).to(torch.bfloat16) if bias else None
    if act == "fp8":
        xq, sx = ops.fp8_fakequant_rowwise(x)
        sx = sx.reshape(-1)
        x_eff = xq.double() * sx.double().reshape(-1, 1)
    else:
        xq, sx, x_eff = x, None, x
    lin = lambda xx, bb=b, s=sx: ops.nvfp4_weight_linear(xx, s, wq, ws, b_pts, bb)

    y = run_expecting(lambda: lin(xq), "ts_prefill_kernel")
    flags_clear(ops, x)
    split = Split("prefill", M, N, K // 128, 256)
    r = Ref(x_eff, w_val, b_pts.expand(N) if b_pts.numel() == 1 else b_pts, b)
    assert_bound(y, r, split, f"nvfp4w prefill M={M} K={K} {act}{' b_pts[N]' if halves else ''}")
    # the decode kernel's 128-token variant on the first 128 tokens: the same sums, split differently
    y_dec = run_expecting(lambda: ops.nvfp4_weight_linear(xq[:128], None if sx is None else sx[:128], wq, ws, b_pts, b),
                          "ts_gemm_kernel", 128)
    assert sqnr(y_dec, y[:128]) >= 60.0
    assert torch.equal(lin(xq), y)
    flags_clear(ops, x)
    # one-hot: the weight value times its scales, within one bf16 ulp (the kernel applies them as a chain of fp32
    # multiplies, then rounds to bf16)
    xh, rows, ks = _one_hot(M, K, 7)
    yh = lin(xh, None, None)
    col = r.col.reshape(-1)
    for m, k in zip(rows, ks):
        want = w_val[:, k] * col
        assert bool(((yh[m].double() - want).abs() <= _bf16_ulp(want)).all()), f"one-hot row {m}, k = {k}"
    _other_rows_zero(yh, rows)
    y1 = lin(xq, None)
    assert torch.equal(lin(xq * 2, None).float(), y1.float() * 2)
    flags_clear(ops, x)


# ================================================================================== C. fused projections at prefill size
class _Attn(torch.nn.Module):
    def __init__(self, h, kv, inter):
        super().__init__()
        mk = lambda k, n: torch.nn.Linear(k, n, bias=True, device="cuda", dtype=torch.bfloat16)
        self.q_proj, self.k_proj, self.v_proj = mk(h, h), mk(h, kv), mk(h, kv)
        self.gate_proj, self.up_proj = mk(h, inter), mk(h, inter)

    def forward(self, x):
        return self.q_proj(x), self.k_proj(x), self.v_proj(x), self.gate_proj(x), self.up_proj(x)


def _member_ref(lin, x):
    """fp64 reference operands of a quantized nn.Linear: (x_eff, w_hat, col, bias)."""
    from ao_b200.prototype.mx_formats.nvfp4_tensor import NVFP4Tensor

    w, bias = lin.weight, lin.bias.detach()
    if isinstance(w, NVFP4Tensor):
        N, K = w.shape
        w_val = _fp4_values(w.qdata, _unblock(w.scale.view(torch.uint8), N, K // 16))
        pts = w.per_tensor_scale
        return x, w_val, torch.ones(N, device="cuda", dtype=torch.float64) if pts is None else pts.reshape(1).double().expand(N), bias
    return x, w.dequantize(), torch.ones(w.shape[0], device="cuda", dtype=torch.float64), bias   # int4: the kernel's W^


@pytest.mark.parametrize("fmt", ["int4", "nvfp4w"])
def test_fused_gate_up_runs_the_prefill_kernel(ops, fmt):
    """Llama-3-8B projections at 512 tokens: the fused gate|up (28672 features) is above the prefill crossover, each
    14336-wide member alone is not -- so this compares the prefill kernel with the decode kernel on the same weights."""
    from ao_b200.fusion import fuse_parallel_linears
    from ao_b200.prototype.mx_formats import NVFP4WeightOnlyConfig
    from ao_b200.quantization import Int4WeightOnlyConfig, quantize_

    h, kv, inter, M = 4096, 1024, 14336, 512
    units = lambda n: -(-n // 128) * -(-M // 256) * (h // 128)
    if not (units(2 * inter) >= 50 * _sm() > units(inter)):
        pytest.skip(f"with {_sm()} SMs the crossover does not separate the fused and the separate gate / up")
    torch.manual_seed(0)
    m = _Attn(h, kv, inter)
    cfg = Int4WeightOnlyConfig(group_size=32, int4_packing_format="tile_packed_to_4d") if fmt == "int4" else NVFP4WeightOnlyConfig()
    quantize_(m, cfg)
    x = torch.randn(M, h, device="cuda", dtype=torch.bfloat16)
    with torch.no_grad():
        parts = [_member_ref(getattr(m, n), x) for n in ("gate_proj", "up_proj")]
        refs = {n: Ref(*p) for n, p in zip(("gate_proj", "up_proj"), parts)}
        fused_ref = Ref(x, torch.cat([p[1].double() for p in parts]), torch.cat([p[2] for p in parts]),
                        torch.cat([p[3] for p in parts]))
        del parts
    with torch.no_grad():
        sep, names = kernels_launched(lambda: m(x))
    ks = gemm_kernels(names)
    assert ks == [("ts_gemm_kernel", 128)] * 5, ks
    for i, n in ((3, "gate_proj"), (4, "up_proj")):
        assert_bound(sep[i], refs[n], Split("ts", M, inter, h // 128, 128), f"{fmt} separate {n} (decode kernel)")
    flags_clear(ops, x)

    assert fuse_parallel_linears(m) == 2
    with torch.no_grad():
        got, names = kernels_launched(lambda: m(x))
    ks = gemm_kernels(names)
    assert ks == [("ts_gemm_kernel", 128), ("ts_prefill_kernel", None)], ks   # q|k|v, gate|up
    flags_clear(ops, x)
    for r, g in zip(sep, got):
        assert sqnr(r, g) >= 60.0
    gate_up = torch.cat([got[3], got[4]], dim=1)
    assert_bound(gate_up, fused_ref, Split("prefill", M, 2 * inter, h // 128, 256), f"{fmt} fused gate|up (prefill kernel)")


# ================================================================================== D. token-block boundaries
TOKEN_COUNTS = [1, 15, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257]
ENTRY_POINTS = ["int4", "nvfp4w_bf16", "nvfp4w_fp8", "int8_mm_i32", "fp8", "mxfp8", "nvfp4"]


def _expected_n_mma(op, M):
    first = 32 if op in ("mxfp8", "nvfp4") else 16   # no 16-token variant of the block-scaled kinds
    return next((n for n in (16, 32, 64, 128) if n >= first and M <= n), 128)


def _case(ops, op, M, N, K, seed, bias=True):
    """(launch, reference, Split family, K elements per chunk, exact int64 reference or None) of one entry point."""
    gen = _gen(seed)
    x = torch.randn(M, K, device="cuda", generator=gen).to(torch.bfloat16)
    b = torch.randn(N, device="cuda", generator=gen).to(torch.bfloat16) if bias else None
    if op == "int4":
        qd, sz, w_hat = _int4_weight(ops, N, K, 32, seed)
        return (lambda: ops.int4_tilepacked_linear(x, qd, 32, sz, b, N, 0)), Ref(x, w_hat, None, b), "ts", 128, x
    if op.startswith("nvfp4w"):
        wq, ws, pts, w_val = _nvfp4_weight(ops, N, K, seed)
        if op.endswith("fp8"):
            xq, sx = ops.fp8_fakequant_rowwise(x)
            r = Ref(xq.double() * sx.double(), w_val, pts.expand(N), b)
            return (lambda: ops.nvfp4_weight_linear(xq, sx.reshape(-1), wq, ws, pts, b)), r, "ts", 128, x
        return (lambda: ops.nvfp4_weight_linear(x, None, wq, ws, pts, b)), Ref(x, w_val, pts.expand(N), b), "ts", 128, x
    if op == "int8_mm_i32":
        xq = torch.randint(-128, 128, (M, K), device="cuda", dtype=torch.int8, generator=gen)
        wq = torch.randint(-128, 128, (N, K), device="cuda", dtype=torch.int8, generator=gen)
        return (lambda: ops.int8_mm_i32(xq, wq)), Ref(xq, wq), "lowp", 128, x
    w = (torch.randn(N, K, device="cuda", generator=gen) * 0.05).to(torch.bfloat16)
    if op == "fp8":
        xq, sx = ops.fp8_quantize_rowwise(x)
        wq, sw = ops.fp8_quantize_rowwise(w)
        r = Ref(xq.double() * sx.double(), wq.double(), sw.reshape(-1), b)
        return (lambda: ops.fp8_rowwise_linear(xq, sx, wq, sw.reshape(-1), b)), r, "lowp", 128, x
    if op == "mxfp8":
        xq, xs = ops.mxfp8_quantize(x, True)
        wq, ws = ops.mxfp8_quantize(w, True)
        e8 = lambda q, s, rows: q.double() * torch.exp2(_unblock(s, rows, K // 32).double() - 127).repeat_interleave(32, 1)
        r = Ref(e8(xq, xs, M), e8(wq, ws, N), None, b)
        return (lambda: ops.mxfp8_linear(xq, xs, wq, ws, b)), r, "lowp", 128, x
    assert op == "nvfp4"
    pa = (x.float().abs().max() / (448.0 * 6.0)).reshape(1)
    pb = (w.float().abs().max() / (448.0 * 6.0)).reshape(1)
    xq, xs = ops.nvfp4_quantize(x, pa, True)
    wq, ws = ops.nvfp4_quantize(w, pb, True)
    r = Ref(_fp4_values(xq, _unblock(xs, M, K // 16)) * pa.double(), _fp4_values(wq, _unblock(ws, N, K // 16)), pb.expand(N), b)
    return (lambda: ops.nvfp4_linear(xq, xs, pa, wq, ws, pb, b)), r, "lowp", 256, x


_FAMILY_KERNEL = {"ts": "ts_gemm_kernel", "lowp": "lowp_linear_kernel"}


def _check_case(ops, op, M, N, K, fn, r, fam, kw, like, n_mma):
    y = run_expecting(fn, _FAMILY_KERNEL[fam], n_mma)
    flags_clear(ops, like)
    split = Split(fam, M, N, -(-K // kw), n_mma, kw)
    if op == "int8_mm_i32":
        want = r.ref.to(torch.int64)   # |acc| <= 2^30: exact in fp64 and in int32
        assert torch.equal(y.to(torch.int64), want), f"int8 M={M}: {int((y.to(torch.int64) != want).sum())} values differ"
        tile, kc = split.contributor_chunk()
        assert not torch.equal(y.to(torch.int64), r.without_chunk(split, tile, kc).to(torch.int64))
    else:
        assert_bound(y, r, split, f"{op} M={M} N={N} K={K}")
    return split


@pytest.mark.parametrize("M", TOKEN_COUNTS)
@pytest.mark.parametrize("op", ENTRY_POINTS)
def test_token_block_boundaries(ops, op, M):
    """Every GEMM entry point at the token counts around its variant switches (N = 384: three tiles, K = 2048): the
    N_MMA that ran is the expected one, these shapes never reach the prefill kernel, and the outputs meet the bound
    (int8: bit-exact against an int64 matmul).  nvfp4 takes K = 4096: its 128-byte chunks hold 256 elements, and at
    K = 2048 (8 chunks) every tile would belong to one CTA, with no split for the self-check to probe."""
    N, K = 384, (4096 if op == "nvfp4" else 2048)
    fn, r, fam, kw, like = _case(ops, op, M, N, K, seed=1000 * ENTRY_POINTS.index(op) + M)
    _check_case(ops, op, M, N, K, fn, r, fam, kw, like, _expected_n_mma(op, M))


# ================================================================================== E. deepest stream-K splits
# contributors = grid - 1 for one output tile; grid = chunks / min_units (4 for the TS kernels, 8 for lowp).  K is
# chosen for 63 contributors (the flag polling and re-arming loops take their second pass of 32) or for 37, which is
# not a multiple of 2, 3 or 8: every gather loop (8 / 3 contributors at a time in ts_gemm.cuh, 2 in lowp_linear.cu)
# ends on its remainder path.
DEEP = [
    ("int4", 1, 128, 32768, ">32"), ("int4", 33, 128, 32768, ">32"), ("int4", 33, 256, 32768, ">32"),
    ("int4", 1, 128, 19456, 37), ("int4", 33, 128, 19456, 37),
    ("nvfp4w_bf16", 1, 128, 32768, ">32"), ("nvfp4w_bf16", 40, 128, 32768, ">32"), ("nvfp4w_bf16", 1, 256, 32768, ">32"),
    ("nvfp4w_bf16", 1, 128, 19456, 37), ("nvfp4w_fp8", 40, 128, 19456, 37),
    ("int8_mm_i32", 1, 128, 65536, ">32"), ("int8_mm_i32", 17, 128, 65536, ">32"), ("int8_mm_i32", 100, 128, 65536, ">32"),
    ("int8_mm_i32", 17, 256, 65536, ">32"), ("int8_mm_i32", 100, 128, 38912, 37),
    ("fp8", 1, 128, 65536, ">32"), ("fp8", 40, 128, 65536, ">32"), ("fp8", 100, 256, 65536, ">32"), ("fp8", 1, 128, 38912, 37),
    ("mxfp8", 1, 128, 65536, ">32"), ("mxfp8", 40, 128, 65536, ">32"), ("mxfp8", 40, 128, 38912, 37),
    ("nvfp4", 1, 128, 131072, ">32"), ("nvfp4", 40, 256, 131072, ">32"), ("nvfp4", 100, 128, 77824, 37),
]


@pytest.mark.parametrize("op,M,N,K,contrib", DEEP)
def test_deep_stream_k_splits(ops, op, M, N, K, contrib):
    """One (or two) output tiles over a long K: each owner gathers the partials of more than 32 contributors (or of
    exactly 37); the result meets the bound, and the owners have re-armed every flag when the kernel ends."""
    fn, r, fam, kw, like = _case(ops, op, M, N, K, seed=K + M + N, bias=(M % 2 == 1))
    n_mma = _expected_n_mma(op, M)
    split = Split(fam, M, N, -(-K // kw), n_mma, kw)
    counts = [split.contributors(t) for t in range(split.n_tiles * split.m_blocks)]
    if contrib == ">32":
        assert min(counts) > 32, counts
    else:
        assert counts == [contrib] * len(counts), counts
    _check_case(ops, op, M, N, K, fn, r, fam, kw, like, n_mma)
