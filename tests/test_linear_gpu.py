"""GPU: HQQLinear.forward through hqq_b200_linear_fwd (fused unpack -> dequant -> MMA) against the reference
HQQBackend.PYTORCH outputs (golden) and the oracle.

Stated tolerance (BASELINE north_star "within a stated fp tolerance"): relative L2 error
||y - y_ref|| / ||y_ref|| <= 2e-3 for float16 and <= 1e-2 for bfloat16.  The fused kernels keep the integer levels
exact and apply scale/zero in float32, so they differ from the reference only by the reference's own fp16/bf16
rounding of W_r and by accumulation order.

A norm over a whole output cannot see a fault in a few elements.  tests/test_linear_bounds_gpu.py holds every route, in both
dtypes, to a per-element bound around a float64 reference, |y - y*| <= ulp_T + c * 2^-24 * (accumulation mass), and checks the
exact identities bit for bit: route 2 == dense GEMM over layer.dequantize() without split-K, y(x, b) == y(x, None) + b, and
split-K results independent of the second-pass variant and of the workspace contents.
"""
import numpy as np
import pytest
import torch

from hqq_b200 import ops
from hqq_b200.core.quantize import BaseQuantizeConfig, HQQBackend, HQQLinear, Quantizer

pytestmark = pytest.mark.gpu
DEV = "cuda"
DT = {"float16": torch.float16, "bfloat16": torch.bfloat16}
TOL = {"float16": 2e-3, "bfloat16": 1e-2}


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30)


def make_layer(W_q, scale, zero, shape, nbits, gs, axis, dt, bias=None):
    layer = HQQLinear(None, None, compute_dtype=dt, device=DEV, initialize=False)
    layer.W_q = torch.nn.Parameter(torch.as_tensor(W_q).to(DEV), requires_grad=False)
    layer.meta = {"nbits": nbits, "group_size": gs, "shape": torch.Size(shape), "axis": axis, "packing": Quantizer.bit_to_packing[nbits],
                  "view_as_float": False, "unpack_view_dtype": Quantizer.unpack_view_dtype[Quantizer.bit_to_packing[nbits]],
                  "compute_dtype": dt, "quant_scale": False, "quant_zero": False,
                  "scale": torch.as_tensor(scale).to(DEV).to(dt), "zero": torch.as_tensor(zero).to(DEV).to(dt)}
    layer.bias = None if bias is None else torch.as_tensor(bias).to(DEV).to(dt)
    layer.ready = True
    layer.in_features, layer.out_features = shape[1], shape[0]
    return layer


@pytest.mark.parametrize("nbits", [8, 4, 3, 2, 1])
@pytest.mark.parametrize("dtype", ["float16", "bfloat16"])
def test_golden_small_layer(golden, nbits, dtype):
    """128x256 layer quantised BY THE REFERENCE; outputs of the reference's PYTORCH backend on the same x."""
    q = golden.quant
    key = f"b{nbits}_a1_g64"
    layer = make_layer(q[key + "/W_q"], q[key + "/scale"], q[key + "/zero"], (128, 256), nbits, 64, 1, DT[dtype])
    x = torch.from_numpy(q["x"]).to(DEV).to(DT[dtype])
    y = layer(x)
    assert y.dtype == DT[dtype] and tuple(y.shape) == (4, 128)
    assert rel(y.float().cpu().numpy(), q[f"{key}/y/{dtype}"]) <= TOL[dtype]


def _random_layer(rng, N, K, nbits, gs, oracle):
    R = N * K // gs
    levels = rng.randint(0, 2 ** nbits, size=(R, gs))
    W_q = oracle.PACK[oracle.BIT_TO_PACKING[nbits]](levels)
    scale = (rng.rand(R, 1) * 0.01 + 2e-3).astype(np.float32)
    zero = (rng.rand(R, 1) * (2 ** nbits - 1)).astype(np.float32)
    return W_q, scale, zero


@pytest.mark.parametrize("nbits", [8, 4, 2, 1])
@pytest.mark.parametrize("dtype", ["float16", "bfloat16"])
@pytest.mark.parametrize("gs", [64, 128])
def test_small_m_kernel_vs_oracle(oracle, nbits, dtype, gs):
    """The weight-streaming kernel (route 1): every bit width / group size, M = 1..32, ragged N, bias."""
    if nbits == 8 and dtype == "bfloat16":
        pytest.skip("8-bit bf16 is served by dequantize + GEMM")
    rng = np.random.RandomState(100 * nbits + gs)
    f = 8 // nbits
    N, K = 24 * f, 512  # N/F = 24 packed rows: not a multiple of every tile height -> ragged last tile
    W_q, scale, zero = _random_layer(rng, N, K, nbits, gs, oracle)
    bias = rng.randn(N).astype(np.float32)
    meta_o = {"nbits": nbits, "group_size": gs, "shape": (N, K), "axis": 1, "packing": oracle.BIT_TO_PACKING[nbits], "scale": scale, "zero": zero}
    for M, use_bias in [(1, False), (3, True), (8, False), (9, True), (16, False), (17, False), (32, True)]:
        assert ops.linear_route(M, N, K, gs, nbits, 1, DT[dtype]) == 1
        x = rng.randn(M, K).astype(np.float32)
        layer = make_layer(W_q, scale, zero, (N, K), nbits, gs, 1, DT[dtype], bias if use_bias else None)
        y = layer(torch.from_numpy(x).to(DEV).to(DT[dtype]))
        ref = oracle.linear_forward(x, W_q, meta_o, bias if use_bias else None, dtype)
        assert rel(y.float().cpu().numpy(), ref) <= TOL[dtype], (M, use_bias)


@pytest.mark.parametrize("nbits", [8, 4, 2, 1])
@pytest.mark.parametrize("dtype", ["float16", "bfloat16"])
@pytest.mark.parametrize("gs", [64, 128])
def test_tcgen05_gemm_vs_oracle(oracle, nbits, dtype, gs):
    """The tcgen05/TMA kernel (route 2): every bit width, both group sizes, token counts that exercise every UMMA N
    (64/128/256), partial token tiles, ragged weight tiles, K not a multiple of 256, bias."""
    rng = np.random.RandomState(7 * nbits + gs)
    f = 8 // nbits
    N, K = 40 * f, 512  # 40 packed rows: partial 128-row tile for every bit width; K = 8 k-blocks = 2 register quads
    W_q, scale, zero = _random_layer(rng, N, K, nbits, gs, oracle)
    bias = rng.randn(N).astype(np.float32)
    meta_o = {"nbits": nbits, "group_size": gs, "shape": (N, K), "axis": 1, "packing": oracle.BIT_TO_PACKING[nbits], "scale": scale, "zero": zero}
    for M, use_bias in [(33, False), (64, True), (100, False), (129, True), (300, False)]:
        assert ops.linear_route(M, N, K, gs, nbits, 1, DT[dtype]) == 2
        x = rng.randn(M, K).astype(np.float32)
        layer = make_layer(W_q, scale, zero, (N, K), nbits, gs, 1, DT[dtype], bias if use_bias else None)
        y = layer(torch.from_numpy(x).to(DEV).to(DT[dtype]))
        ref = oracle.linear_forward(x, W_q, meta_o, bias if use_bias else None, dtype)
        assert rel(y.float().cpu().numpy(), ref) <= TOL[dtype], (M, use_bias)


@pytest.mark.parametrize("N,K,M", [(4096, 4096, 4096), (11008, 4096, 1024), (4096, 11008, 512), (14336, 4096, 64), (4096, 4096, 33)])
def test_tcgen05_gemm_full_size(N, K, M):
    """BASELINE sweep sizes: the fused GEMM against an fp32 GEMM over the (bit-exactly tested) dequantised matrix.  The A
    operand the tensor core sees is bit-identical to Quantizer.dequantize, so only the accumulation order differs."""
    torch.manual_seed(N + K + M)
    W = (torch.randn(N, K, device=DEV) * 0.02).half()
    layer = HQQLinear.from_weights(W, None, BaseQuantizeConfig(nbits=4, group_size=64, axis=1), compute_dtype=torch.float16, device=DEV)
    assert ops.linear_route(M, N, K, 64, 4, 1, torch.float16) == 2
    x = torch.randn(M, K, device=DEV).half()
    y = layer(x).float()
    ref = x.float() @ layer.dequantize().float().t()
    assert (y - ref).norm() / ref.norm() <= 5e-4
    assert torch.equal(layer(x), layer(x))


@pytest.mark.parametrize("N,K", [(4096, 4096), (1024, 4096), (14336, 4096), (4096, 14336), (11008, 4096)])
def test_llama_shapes_vs_dequant_gemm(N, K):
    """BASELINE sizes (Llama-3-8B / Llama-2-7B linears), 4-bit gs=64, M=1 and M=16: fused kernel vs fp32 GEMM over the
    (bit-exactly tested) dequantize kernel's output.  Also checks linearity: f(a*x1 + x2) == a*f(x1) + f(x2)."""
    torch.manual_seed(N + K)
    W = (torch.randn(N, K, device=DEV) * 0.02).half()
    layer = HQQLinear.from_weights(W, None, BaseQuantizeConfig(nbits=4, group_size=64, axis=1), compute_dtype=torch.float16, device=DEV)
    W_r = layer.dequantize().float()
    for M in (1, 16):
        assert ops.linear_route(M, N, K, 64, 4, 1, torch.float16) == 1
        x = torch.randn(M, K, device=DEV).half()
        y = layer(x).float()
        ref = x.float() @ W_r.t()
        assert (y - ref).norm() / ref.norm() <= 2e-3
    x1, x2 = torch.randn(1, K, device=DEV).half(), torch.randn(1, K, device=DEV).half()
    lhs = layer((2 * x1 + x2)).float()
    rhs = 2 * layer(x1).float() + layer(x2).float()
    assert (lhs - rhs).norm() / rhs.norm() <= 4e-3


def test_multi_launch_equals_single_launches():
    """q/k/v (and gate/up) share the activation: one stream-K launch over all matrices == separate launches, bit for bit."""
    torch.manual_seed(8)
    K = 2048
    layers = [HQQLinear.from_weights((torch.randn(n, K, device=DEV) * 0.02).half(), None, BaseQuantizeConfig(nbits=4, group_size=64, axis=1),
                                     compute_dtype=torch.float16, device=DEV) for n in (1024, 256, 264, 4096)]
    for M in (1, 7, 24):
        x = torch.randn(M, K, device=DEV).half()
        outs = ops.linear_fwd_multi(x, layers)
        assert outs is not None and len(outs) == 4
        for l, o in zip(layers, outs):
            assert torch.equal(o, l(x))
    # repeated launches reuse the flag workspace: results must not drift
    x = torch.randn(1, K, device=DEV).half()
    first = [o.clone() for o in ops.linear_fwd_multi(x, layers)]
    for _ in range(20):
        again = ops.linear_fwd_multi(x, layers)
        assert all(torch.equal(a, b) for a, b in zip(first, again))


def test_forward_is_deterministic_and_batch_invariant():
    torch.manual_seed(5)
    W = (torch.randn(4096, 4096, device=DEV) * 0.02).half()
    layer = HQQLinear.from_weights(W, None, BaseQuantizeConfig(nbits=4, group_size=64, axis=1), compute_dtype=torch.float16, device=DEV)
    x = torch.randn(8, 4096, device=DEV).half()
    y1, y2 = layer(x), layer(x)
    assert torch.equal(y1, y2)
    assert torch.equal(layer(x[:2]), y1[:2])  # a token's result does not depend on its batch-mates (same kernel variant)
    assert torch.allclose(layer(x[:1]).float(), y1[:1].float(), rtol=2e-3, atol=2e-3)  # M == 1 takes the decode specialisation
    assert tuple(layer(x.reshape(2, 4, 4096)).shape) == (2, 4, 4096)


@pytest.mark.parametrize("cfg", [dict(nbits=4, group_size=64, axis=0), dict(nbits=3, group_size=64, axis=1), dict(nbits=4, group_size=None, axis=1),
                                 dict(nbits=4, group_size=16, axis=1), dict(nbits=2, group_size=64, axis=1)])
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16, torch.float32])
def test_every_config_has_a_forward(cfg, dt):
    """Configurations outside the fused kernels (axis=0, 3-bit, other group sizes) run route 3: our dequantize kernel + the dense
    tcgen05 GEMM (float32 compute: dequantize kernel + library GEMM); results agree with the explicit dequantise-then-matmul
    definition (quantize.py:880-898)."""
    torch.manual_seed(9)
    lin = torch.nn.Linear(256, 128, bias=True)
    layer = HQQLinear(lin, BaseQuantizeConfig(**cfg), compute_dtype=dt, device=DEV)
    for M in (1, 40):
        x = torch.randn(M, 256, device=DEV).to(dt)
        y = layer(x)
        ref = x.float() @ layer.dequantize().float().t() + layer.bias.float()
        tol = 1e-5 if dt == torch.float32 else (4e-3 if dt == torch.float16 else 2e-2)
        assert (y.float() - ref).norm() / ref.norm() <= tol


def test_backend_members_share_one_path():
    torch.manual_seed(2)
    lin = torch.nn.Linear(512, 256, bias=False)
    layer = HQQLinear(lin, BaseQuantizeConfig(nbits=4, group_size=64), compute_dtype=torch.float16, device=DEV)
    x = torch.randn(2, 512, device=DEV).half()
    outs = []
    for b in (HQQBackend.PYTORCH, HQQBackend.PYTORCH_COMPILE, HQQBackend.ATEN, HQQBackend.PYTORCH_FORWARD, HQQBackend.ATEN_FORWARD):
        HQQLinear.set_backend(b)
        outs.append(layer(x))
    HQQLinear.set_backend(HQQBackend.PYTORCH)
    assert all(torch.equal(outs[0], o) for o in outs[1:])


def test_backward_matches_dequant_matmul():
    """quantize.py:322-352: grad_input = grad_out @ W_r, bias grad = sum over tokens."""
    torch.manual_seed(4)
    lin = torch.nn.Linear(512, 256, bias=True)
    layer = HQQLinear(lin, BaseQuantizeConfig(nbits=4, group_size=64), compute_dtype=torch.float16, device=DEV)
    x = torch.randn(3, 512, device=DEV, dtype=torch.float16, requires_grad=True)
    y = layer(x)
    g = torch.randn_like(y)
    y.backward(g)
    ref = g.float() @ layer.dequantize().float()
    assert (x.grad.float() - ref).norm() / ref.norm() <= 2e-3


@pytest.mark.parametrize("M,N,K", [(1, 256, 512), (40, 384, 1000), (300, 130, 72), (1024, 4096, 4096), (257, 11008, 4096)])
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_dense_tcgen05_gemm_vs_fp32_matmul(M, N, K, dt):
    """hqq_b200_dense_gemm (the persistent tcgen05 kernel with both operands on TMA): ragged rows / tokens / K (K % 8 == 0 only),
    bias, against an fp32 matmul of the same 16-bit operands."""
    torch.manual_seed(M + N + K)
    x = torch.randn(M, K, device=DEV).to(dt)
    W = (torch.randn(N, K, device=DEV) * 0.05).to(dt)
    b = torch.randn(N, device=DEV).to(dt)
    y = ops.dense_gemm(x, W, b)
    assert y is not None and y.shape == (M, N)
    ref = x.float() @ W.float().t()
    assert ((y.float() - b.float()) - ref).norm() / ref.norm() <= (1e-3 if dt == torch.float16 else 6e-3)
    assert torch.equal(ops.dense_gemm(x, W, b), y)


@pytest.mark.parametrize("cfg", [dict(nbits=3, group_size=64, axis=1), dict(nbits=4, group_size=64, axis=0), dict(nbits=2, group_size=32, axis=1)])
def test_route3_full_size(cfg):
    """3-bit / axis 0 / other group sizes at a BASELINE sweep size: route 3 (dequantize kernel -> dense tcgen05 GEMM) against an fp32
    GEMM over the (bit-exactly tested) dequantised matrix; the A operand IS that matrix, so only the accumulation order differs."""
    torch.manual_seed(11)
    N, K = 4096, 4096
    layer = HQQLinear.from_weights((torch.randn(N, K, device=DEV) * 0.02).half(), None, BaseQuantizeConfig(**cfg), compute_dtype=torch.float16, device=DEV)
    nb = Quantizer._packing_bits[layer.meta["packing"]]
    for M in (1, 48, 600):
        assert ops.linear_route(M, N, K, layer.meta["group_size"], nb, cfg["axis"], torch.float16) == 3
        x = torch.randn(M, K, device=DEV).half()
        y = layer(x).float()
        ref = x.float() @ layer.dequantize().float().t()
        assert (y - ref).norm() / ref.norm() <= 5e-4


def test_persistent_gemm_schedule_is_result_invariant(monkeypatch):
    """HQQ_B200_GEMM_CTAS caps the persistent grid: 7 CTAs walk 32 x 5 tiles one after another (both TMEM accumulators, epilogue under
    the next main loop, the half-tile round) and must reproduce the full-grid result bit for bit."""
    from hqq_b200 import _lib
    torch.manual_seed(12)
    layer = HQQLinear.from_weights((torch.randn(4096, 1024, device=DEV) * 0.02).half(), torch.randn(4096, device=DEV).half(),
                                   BaseQuantizeConfig(nbits=4, group_size=64, axis=1), compute_dtype=torch.float16, device=DEV)
    x = torch.randn(1100, 1024, device=DEV).half()
    ref = layer(x)
    for cap in ("7", "1", "40"):
        monkeypatch.setenv("HQQ_B200_GEMM_CTAS", cap)
        _lib.load().hqq_b200_reload_env()
        assert torch.equal(layer(x), ref), cap
    monkeypatch.delenv("HQQ_B200_GEMM_CTAS")
    _lib.load().hqq_b200_reload_env()
