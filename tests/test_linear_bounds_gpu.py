"""Every forward route of HQQLinear checked element by element against a float64 reference, in fp16 and bf16.

The other linear tests compare one relative L2 norm over the whole output; a fault that touches a few elements (one ragged row,
one token, one group, one k-slice) hides inside it.  Here every output element y must satisfy

    |y - y*| <= ulp_T(max(|y*|, |y* - b|) + e) + e,        e = c * 2^-24 * A,

where y* is the exact (float64, on the device) value of the route's operation and A the absolute accumulation mass of the route:

  route 1 (linear_small.cu, M <= 32 and the one-token kernel).  The kernel does not round W_r to T: the tensor core contracts the
      raw levels, planted into 16-bit lanes as OFF + q * V, against x, and the affine map is applied per group in fp32
      (s * invV * S_g - s * (OFF / V + z) * X_g, X_g = sum of x over the group).  So
          y* = x @ ((q - z) * s)^T + b          (q from ops.unpack, s and z the T-valued meta as float64)
          A  = sum_k |s_g(k)| |x_k| (OFF_T + 2^nbits + |z_g(k)|),  OFF_T = 1024 (fp16 lanes) or 128 (bf16 lanes)
      The two big terms of every group carry the lane offset and cancel; their fp32 roundings are what A measures.
  routes 2 and 3 (fused tcgen05 GEMM; dequantize kernel + dense GEMM).  The A operand is W_r = layer.dequantize(), so
          y* = x @ W_r^T + b,     A = (|x| @ |W_r|^T) * K / 16   (K / 16 tensor-core accumulation steps)

ulp_T is the spacing of T at that magnitude (fp16: 2^-24 below 2^-14, bf16: 8 significant bits).  The ulp term covers the two
roundings to T of the epilogue, out = T(T(acc) + bias); e covers the fp32 arithmetic before it.  u = 2^-24 is the fp32 unit
roundoff; one tensor-core step (alignment of the products to the largest exponent, then the accumulator update) is counted as
two truncations, 4u, of the magnitude it acts on.

  c2 = c3 = 5.  Routes 2/3: K/16 UMMA steps, 4u each of a running sum bounded by the mass: 4u * mass * K/16.  The split-K second
      pass adds at most 8 fp32 sums of partials, each bounded by the mass, and 8 <= K/16 whenever K is split (K >= 512): +1.
  c1 = 24.  Route 1, per group and relative to A_g (every term below is bounded by the group's share of A):
      2   the two fmaf of the affine correction (one rounding each, of a result bounded by A_g plus the small running total);
      8   the chain of GS/16 <= 8 MMAs into S_g: 4u per step on partial sums of zero-mean terms, which grow like sqrt(steps)
          (4u * sqrt(8) < 12u, counted as 8 + the 2 below);
      12  X_g, a sequential fp32 sum of GS <= 128 activations: one rounding per addition of a partial sum that grows like
          sqrt(k) |x|, i.e. u * sum_k sqrt(k) / GS * sum|x| <= 0.7 * sqrt(128) u * sum|x| < 8u; counted as 12;
      2   the reduction of the eight warps' partial results and the fp32 sum across K units (bounded by the small totals).
  The sqrt(n) growth of the zero-mean inner chains is the one non-worst-case step; every other count is a worst case.

Largest observed |y - y*| / bound on a B200 (whole file): not measured yet.  Each check prints its worst ratio ("[bound]" lines
with pytest -s).

test_the_bound_rejects_planted_faults (no GPU) shows on exact outputs that the bound rejects planted faults, and that it is at
least four times tighter than the single-element error the relative-L2 limits of tests/test_linear_gpu.py let through.

The exact properties the kernels have are checked bit for bit, with no tolerance:
  - route 2 with HQQ_B200_GEMM_KSPLIT=1 == ops.dense_gemm(x, layer.dequantize(), bias): the same MMA sequence (k-blocks in order,
    four UMMA_K = 16 steps each) on an A operand that is bit-identical to Quantizer.dequantize, on the same schedule
    (cdiv(N/F, 128/F) == cdiv(N, 128) row tiles);
  - y(x, b) == y(x, None) + b in torch T arithmetic on every route (fp32 has >= 2p + 2 bits for both T, so rounding the fp32 sum
    to T equals adding in T);
  - split-K: both second-pass variants (4 outputs per thread, or 1 when step % 4 != 0 or y is not 8-byte aligned) give the same
    bits, and a dirty workspace changes nothing.
"""
import math

import pytest
import torch

from hqq_b200 import _lib, ops
from hqq_b200.core.quantize import BaseQuantizeConfig, HQQLinear, Quantizer

DEV = "cuda"
DT = {"float16": torch.float16, "bfloat16": torch.bfloat16}
U = 2.0 ** -24
C1, C2, C3 = 24.0, 5.0, 5.0
OFF = {torch.float16: 1024.0, torch.bfloat16: 128.0}
PREC = {torch.float16: (11, 2.0 ** -24), torch.bfloat16: (8, 2.0 ** -133)}  # significant bits, smallest spacing
TOL = {torch.float16: 2e-3, torch.bfloat16: 1e-2}  # the relative-L2 limits of tests/test_linear_gpu.py


# ----------------------------------------------------------------------------------------------------------- the criterion
def ulp(v: torch.Tensor, dt) -> torch.Tensor:
    """Spacing of `dt` at |v| (float64 in, float64 out)."""
    p, tiny = PREC[dt]
    _, e = torch.frexp(v.abs())  # |v| = m * 2^e, m in [0.5, 1)
    out = torch.ldexp(torch.ones_like(v), e - p)
    return torch.where(v == 0, torch.full_like(v, tiny), out.clamp_min(tiny))


def bound(ystar, bias, mass, c, dt, extra=None):
    e = c * U * mass
    if extra is not None:
        e = e + extra
    b = torch.zeros_like(ystar) if bias is None else bias.double().reshape(1, -1).expand_as(ystar)
    return ulp(torch.maximum(ystar.abs(), (ystar - b).abs()) + e, dt) + e


def ratio(y, ystar, bias, mass, c, dt, extra=None):
    """Per element |y - y*| / bound."""
    return (y.double() - ystar).abs() / bound(ystar, bias, mass, c, dt, extra)


def check(name, y, ystar, bias, mass, c, dt, extra=None):
    r = ratio(y, ystar, bias, mass, c, dt, extra)
    worst = float(r.max())
    print(f"[bound] {name}: max |y - y*| / bound = {worst:.3f}")
    if worst > 1.0:
        i = int(r.flatten().argmax())
        m, n = divmod(i, y.shape[-1])
        raise AssertionError(f"{name}: element (token {m}, row {n}) y={float(y.flatten()[i])!r} y*={float(ystar.flatten()[i])!r} "
                             f"bound={float(bound(ystar, bias, mass, c, dt, extra).flatten()[i])!r}; {int((r > 1).sum())} elements out of bound")
    return worst


# ------------------------------------------------------------------------------------------------ exact references (float64)
def expand_meta(t, N, K, gs):
    """[N*K/gs, 1] group meta -> [N, K] float64."""
    return t.double().reshape(N, K // gs).repeat_interleave(gs, dim=1)


def route1_ref(x, q, s, z, bias, N, K, gs, nbits, dt):
    """y* and A of route 1: W = (q - z) * s, not rounded to T."""
    s64, z64 = expand_meta(s, N, K, gs), expand_meta(z, N, K, gs)
    W = (q.double() - z64) * s64
    x64 = x.double()
    y = x64 @ W.t()
    if bias is not None:
        y = y + bias.double()
    mass = x64.abs() @ (s64.abs() * (OFF[dt] + 2.0 ** nbits + z64.abs())).t()
    return y, mass, W


def dense_ref(x, W_r, bias):
    """y* and A of routes 2 / 3: W_r is the T-valued dequantised matrix."""
    W = W_r.double()
    x64 = x.double()
    y = x64 @ W.t()
    if bias is not None:
        y = y + bias.double()
    mass = (x64.abs() @ W.abs().t()) * (W.shape[1] / 16.0)
    return y, mass


def round_chain(acc, bias, dt):
    """out = T(T(acc) + bias): the epilogue of every route, applied to an exact accumulator."""
    y = acc.to(dt)
    return y if bias is None else y + bias.to(dt)


# ------------------------------------------------------------------------------------------------------------ layers
def make_layer(N, K, nbits, gs, dt, seed, bias=False, device=DEV):
    """A random axis-1 layer: uniform levels, scale in [2e-3, 1.2e-2], zero in [0, 2^nbits - 1], all meta in T."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    R = N * K // gs
    levels = torch.randint(0, 2 ** nbits, (R, gs), generator=g, dtype=torch.uint8)
    scale = (torch.rand(R, 1, generator=g) * 0.01 + 2e-3).to(dt)
    zero = (torch.rand(R, 1, generator=g) * (2 ** nbits - 1)).to(dt)
    b = torch.randn(N, generator=g).to(dt) if bias else None
    if device == "cpu":
        return levels.reshape(N, K), scale, zero, b
    layer = HQQLinear(None, None, compute_dtype=dt, device=device, initialize=False)
    layer.W_q = torch.nn.Parameter(ops.pack(levels.to(device), nbits), requires_grad=False)
    pk = Quantizer.bit_to_packing[nbits]
    layer.meta = {"nbits": nbits, "group_size": gs, "shape": torch.Size((N, K)), "axis": 1, "packing": pk, "view_as_float": False,
                  "unpack_view_dtype": Quantizer.unpack_view_dtype[pk], "compute_dtype": dt, "quant_scale": False, "quant_zero": False,
                  "scale": scale.to(device), "zero": zero.to(device)}
    layer.bias = None if b is None else b.to(device)
    layer.ready = True
    layer.in_features, layer.out_features = K, N
    return layer


def levels_of(layer):
    N, K = layer.meta["shape"]
    return ops.unpack(layer.W_q, layer.meta["nbits"]).reshape(N, K)


def fwd(layer, x, bias="layer", out=None):
    m = layer.meta
    N, K = m["shape"]
    b = layer.bias if bias == "layer" else bias
    return ops.linear_fwd(x, layer.W_q, m["scale"], m["zero"], b, N, K, m["group_size"], m["nbits"], m["axis"], out=out)


def rand_x(M, K, dt, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.randn(M, K, generator=g).to(dt).to(DEV)


def set_knobs(monkeypatch, **knobs):
    """Set (value) or clear (None) HQQ_B200_* knobs and have the library parse them again."""
    for k, v in knobs.items():
        if v is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, str(v))
    _lib.load().hqq_b200_reload_env()


@pytest.fixture
def knobs(monkeypatch):
    """monkeypatch for HQQ_B200_* knobs; the library re-reads the restored environment afterwards."""
    yield lambda **kw: set_knobs(monkeypatch, **kw)
    monkeypatch.undo()
    _lib.load().hqq_b200_reload_env()


# ---------------------------------------------------------------------------------------------------------- (b) route 1
# N is given in packed rows (step = N / F): 1 = a single packed row, 37 = a ragged last tile for every P = 16 / F; else N itself.
ROUTE1_CASES = [
    # M, N (or step), K, nbits, gs, bias     -- what the case is for
    (1, "1", 256, 4, 64, True),        # fewer 256-k units than warps; one packed row
    (1, "37", 768, 4, 128, False),     # K % 512 != 0: the one-token kernel with register meta (MR = 0)
    (1, 14336, 4096, 4, 64, True),     # the one-token kernel with meta on the cp.async ring (MR = 1), a Llama-3-8B gate/up
    (1, "37", 16384, 2, 64, False),    # K = 16384: the one-token kernel's limit
    (1, "37", 16640, 4, 64, True),     # K > 16384: M = 1 on the generic small-M kernel
    (1, 1024, 28672, 4, 64, False),    # K = 28672 (Llama-70B down_proj) on the generic kernel
    (1, "37", 28672, 1, 128, True),
    (1, "37", 4096, 8, 128, True),     # 8-bit one-token kernel
    (2, "37", 2304, 8, 64, True),      # MT = 1, 8-bit lanes, K % 512 != 0
    (7, 14336, 4096, 2, 128, False),   # MT = 1
    (8, "1", 4096, 1, 64, True),       # MT = 1, one packed row of 8 slabs
    (9, "37", 2304, 4, 64, False),     # MT = 2
    (15, "37", 16384, 8, 128, True),   # MT = 2, 8-bit
    (16, 1024, 28672, 2, 64, True),    # MT = 2, long K
    (17, "37", 4096, 4, 64, True),     # MT = 4 (N * K <= 2^24 keeps M = 17..32 on route 1)
    (31, "37", 768, 1, 64, False),     # MT = 4, 1-bit
    (32, 14336, 1024, 4, 128, True),   # MT = 4, 14336 rows
    (32, "37", 256, 2, 128, False),    # one 256-k unit
]


def route1_n(Nspec, nbits):
    F = 8 // nbits
    return F * int(Nspec) if isinstance(Nspec, str) else Nspec


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(ROUTE1_CASES)))
@pytest.mark.parametrize("dtype", ["float16", "bfloat16"])
def test_route1_every_element_within_bound(case, dtype):
    """Route 1 over token counts 1..32 (the one-token kernel, MT = 1 / 2 / 4), K from one 256-k unit to 28672, every width and
    group size, one packed row, ragged last tiles and 14336 rows, with and without bias; plus the bias identity."""
    M, Nspec, K, nbits, gs, use_bias = ROUTE1_CASES[case]
    dt = DT[dtype]
    if nbits == 8 and dt == torch.bfloat16:
        pytest.skip("8-bit levels need the fp16 lanes: 8-bit bf16 runs on route 2")
    N = route1_n(Nspec, nbits)
    assert ops.linear_route(M, N, K, gs, nbits, 1, dt) == 1
    layer = make_layer(N, K, nbits, gs, dt, seed=1000 + case, bias=use_bias)
    x = rand_x(M, K, dt, seed=case)
    y = fwd(layer, x)
    ystar, mass, _ = route1_ref(x, levels_of(layer), layer.meta["scale"], layer.meta["zero"], layer.bias, N, K, gs, nbits, dt)
    check("route 1", y, ystar, layer.bias, mass, C1, dt)
    if use_bias:
        assert torch.equal(y, fwd(layer, x, bias=None) + layer.bias)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float16", "bfloat16"])
def test_route1_one_token_on_the_generic_kernel(dtype, knobs):
    """HQQ_B200_DECODE1=0 sends M = 1 to the generic small-M kernel at every K."""
    dt = DT[dtype]
    knobs(HQQ_B200_DECODE1=0)
    for i, (N, K, nbits, gs) in enumerate([(4096, 4096, 4, 64), (296, 768, 2, 128), (74, 16384, 4, 64)]):
        layer = make_layer(N, K, nbits, gs, dt, seed=2000 + i, bias=True)
        x = rand_x(1, K, dt, seed=50 + i)
        y = fwd(layer, x)
        ystar, mass, _ = route1_ref(x, levels_of(layer), layer.meta["scale"], layer.meta["zero"], layer.bias, N, K, gs, nbits, dt)
        check("route 1", y, ystar, layer.bias, mass, C1, dt)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float16", "bfloat16"])
def test_route1_multi_launch_every_element_within_bound(dtype):
    """linear_fwd_multi with 2-4 matrices of unequal N, one of them smaller than a 16-row tile, at M = 1, 5 and 24; each output
    within the bound and equal to its single-matrix launch."""
    dt = DT[dtype]
    K, nbits, gs = 2048, 4, 64
    sets = [(2, 296), (2, 1024, 74, 14), (4, 2, 512, 1000)]
    for si, Ns in enumerate(sets):
        layers = [make_layer(N, K, nbits, gs, dt, seed=3000 + 10 * si + j, bias=(j % 2 == 0)) for j, N in enumerate(Ns)]
        for M in (1, 5, 24):
            x = rand_x(M, K, dt, seed=70 + M)
            outs = ops.linear_fwd_multi(x, layers)
            assert outs is not None and len(outs) == len(layers)
            for l, y in zip(layers, outs):
                N = l.meta["shape"][0]
                ystar, mass, _ = route1_ref(x, levels_of(l), l.meta["scale"], l.meta["zero"], l.bias, N, K, gs, nbits, dt)
                check("route 1", y, ystar, l.bias, mass, C1, dt)
                assert torch.equal(y, fwd(l, x))


# ------------------------------------------------------------------------------------------- (c) one-token prologues
def rounded_bracket(v, rel, dt, post):
    """The T values a kernel can produce for post(T(v')) when it computes v' within relative `rel` of the exact v: rounding and
    `post` (a product with a fixed factor) are monotone, so they lie between the results at v (1 - rel) and v (1 + rel)."""
    a, b = post((v * (1 - rel)).to(dt)), post((v * (1 + rel)).to(dt))
    return post(v.to(dt)), torch.minimum(a, b), torch.maximum(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [4096, 14336, 16384])
@pytest.mark.parametrize("dtype", ["float16", "bfloat16"])
def test_one_token_prologues_every_element_within_bound(K, dtype):
    """x_op 1 (t = x + x2, h_out = t, x' = T(T(t * inv) * w)) and x_op 2 (x' = T(T(silu(x)) * x2)): h_out bit for bit, the linear
    outputs within the route-1 bound around the exact value for the rounded prologue activation.

    The kernel's inv = rsqrtf(sum(t^2) / K + eps) is an fp32 sum of K squares in its own order (partials of K / 256 <= 64 terms,
    a 5-level shuffle tree, 8 warps: < 80 roundings of positive terms, < 2^-17.6 relative) and rsqrtf (2 ulp): within 2^-16 of
    the exact value.  silu uses __expf and an fp32 division: within 2^-18.  Where that slack can move the rounding of the first
    product to T the activation is known only to a bracket [lo, hi]; the bound then grows by sum_k (hi_k - lo_k) |W_nk|."""
    dt = DT[dtype]
    N, nbits, gs = 1040, 4, 64
    A = make_layer(N, K, nbits, gs, dt, seed=4000 + K, bias=True)
    B = make_layer(N, K, nbits, gs, dt, seed=5000 + K)
    g = torch.Generator(device="cpu").manual_seed(K)
    x = torch.randn(1, K, generator=g).to(dt).to(DEV)
    x2 = (torch.randn(1, K, generator=g) * 0.5).to(dt).to(DEV)
    w = torch.rand(K, generator=g).to(dt).to(DEV)
    eps = 1e-5
    ya, yb, hout = (torch.empty(1, n, device=DEV, dtype=dt) for n in (N, N, K))

    def check_linear(layer, y, act, lo, hi):
        m = layer.meta
        ystar, mass, W = route1_ref(act, levels_of(layer), m["scale"], m["zero"], layer.bias, N, K, gs, nbits, dt)
        mass = torch.maximum(lo.double().abs(), hi.double().abs()) @ ((expand_meta(m["scale"], N, K, gs).abs()
                                                                       * (OFF[dt] + 2.0 ** nbits + expand_meta(m["zero"], N, K, gs).abs())).t())
        slack = (hi.double() - lo.double()) @ W.abs().t()
        check("one-token prologue", y, ystar, layer.bias, mass, C1, dt, extra=slack)

    # x_op 1: residual add + RMSNorm
    assert ops.decode_linear_fwd(x, (A, B), [ya, yb], 1, x2, w, hout, eps)
    t = x + x2
    assert torch.equal(hout, t)
    t64 = t.double()
    inv = 1.0 / math.sqrt(float((t64 * t64).sum()) / K + eps)
    act, lo, hi = rounded_bracket(t64 * inv, 2.0 ** -16, dt, lambda r: (r.double() * w.double()).to(dt))
    check_linear(A, ya, act, lo, hi)
    check_linear(B, yb, act, lo, hi)
    # the paired SiLU * mul epilogue after the same prologue == the two products + the glue kernel
    ref, act_out, u2 = (torch.empty(1, N, device=DEV, dtype=dt) for _ in range(3))
    _lib.check(_lib.load().hqq_b200_glue_silu_mul(_lib.ptr(ya), _lib.ptr(yb), _lib.ptr(ref), N, _lib.DTYPE_CODE[dt], _lib.stream_ptr(x.device)))
    assert ops.decode_linear_fwd(x, (A, B), [act_out, u2], 1 | ops.YOP_SILU_MUL_PAIR, x2, w, hout, eps)
    assert torch.equal(act_out, ref)

    # x_op 2: SiLU(x) * x2
    assert ops.decode_linear_fwd(x, (A,), [ya], 2, x2)
    x64 = x.double()
    act, lo, hi = rounded_bracket(x64 / (1.0 + torch.exp(-x64)), 2.0 ** -18, dt, lambda r: (r.double() * x2.double()).to(dt))
    check_linear(A, ya, act, lo, hi)


# ------------------------------------------------------------------------------------------------------ (d) route 2
def gemm_ws_bytes(M, N, K, gs, nbits, dt):
    return _lib.load().hqq_b200_linear_fwd_workspace_bytes(M, N, K, gs, nbits, 1, _lib.DTYPE_CODE[dt])


BITS_GS = [(nb, gs) for nb in (8, 4, 2, 1) for gs in (64, 128)]


@pytest.mark.gpu
@pytest.mark.parametrize("nbits,gs", BITS_GS)
@pytest.mark.parametrize("dtype", ["float16", "bfloat16"])
def test_route2_equals_dense_gemm_over_dequantize_bit_for_bit(nbits, gs, dtype, knobs):
    """HQQ_B200_GEMM_KSPLIT=1: the fused GEMM == ops.dense_gemm(x, layer.dequantize(), bias), bit for bit, at partial and full
    token tiles (M = 17 .. 1100; HQQ_B200_SMALL_M_MAX=16 sends M = 17 here) and persistent grids of every CTA count (1 and 7: tile
    after tile on both TMEM accumulators; 40 and the SM count: the half-tile round).  N = 42 F (one ragged tile, step % 4 != 0)
    and 42 F + 256 (several row tiles, the last ragged).  Also every element within the route-2 bound, and the bias identity."""
    dt = DT[dtype]
    F = 8 // nbits
    K = 1024
    knobs(HQQ_B200_GEMM_KSPLIT=1, HQQ_B200_SMALL_M_MAX=16)
    for ni, N in enumerate((42 * F, 42 * F + 256)):
        layer = make_layer(N, K, nbits, gs, dt, seed=6000 + 10 * nbits + gs + ni, bias=True)
        W_r = layer.dequantize()
        for cap in (None, 1, 7, 40):
            knobs(HQQ_B200_GEMM_CTAS=cap)
            for M in (17, 33, 64, 128, 129, 255, 256, 257, 384, 512, 513, 1100):
                assert ops.linear_route(M, N, K, gs, nbits, 1, dt) == 2 and gemm_ws_bytes(M, N, K, gs, nbits, dt) == 0
                x = rand_x(M, K, dt, seed=M + ni)
                y = fwd(layer, x)
                assert torch.equal(y, ops.dense_gemm(x, W_r, layer.bias)), (N, cap, M)
                if cap is None:
                    ystar, mass = dense_ref(x, W_r, layer.bias)
                    check("route 2", y, ystar, layer.bias, mass, C2, dt)
                    assert torch.equal(y, fwd(layer, x, bias=None) + layer.bias), (N, M)


def expected_slices(K, cap, full, P):
    quads = K // 256
    S = min(P // full, cap, quads)
    return -(-quads // -(-quads // S))


@pytest.mark.gpu
@pytest.mark.parametrize("nbits,gs", BITS_GS)
@pytest.mark.parametrize("dtype", ["float16", "bfloat16"])
def test_route2_split_k_against_the_unsplit_result(nbits, gs, dtype, knobs):
    """HQQ_B200_GEMM_KSPLIT = 2 / 3 / 5 / 8 on K = 2 / 3 / 5 / 7 / 16 quads of 256 (uneven last slices: 7 quads in 4 slices of
    2, 2, 2, 1; 16 in 3 of 6, 6, 4).  Against the KSPLIT=1 output (bias off): within 1 ulp_T wherever the fp32 reassociation
    cannot move the result by more, i.e. outside the sum of both results' route-2 bounds; every element within the route-2 bound;
    the same bits on a workspace filled with garbage first; the bias identity through the second pass."""
    dt = DT[dtype]
    F = 8 // nbits
    N = 40 * F  # step = 40 packed rows: step % 4 == 0, the 4-wide second pass; 1 .. 3 row tiles of PR = 128 / F
    n_row = -(-40 // (128 // F))
    P = torch.cuda.get_device_properties(0).multi_processor_count
    for quads in (2, 3, 5, 7, 16):
        K = 256 * quads
        if K % gs:
            continue
        layer = make_layer(N, K, nbits, gs, dt, seed=7000 + 10 * nbits + gs + quads, bias=True)
        W_r = layer.dequantize()
        for M in (64, 300):
            x = rand_x(M, K, dt, seed=quads * 1000 + M)
            knobs(HQQ_B200_GEMM_KSPLIT=1)
            y1 = fwd(layer, x, bias=None)
            ystar, mass = dense_ref(x, W_r, None)
            b1 = bound(ystar, None, mass, C2, dt)
            for cap in (2, 3, 5, 8):
                knobs(HQQ_B200_GEMM_KSPLIT=cap)
                n_tok = -(-M // 256)
                S = expected_slices(K, cap, n_row * n_tok, P)
                assert gemm_ws_bytes(M, N, K, gs, nbits, dt) == S * n_row * n_tok * 256 * 128 * 4, (quads, cap)
                ys = fwd(layer, x, bias=None)
                check("route 2 split-K", ys, ystar, None, mass, C2, dt)
                d = (ys.double() - y1.double()).abs()
                one_ulp = ulp(torch.maximum(ys.double().abs(), y1.double().abs()), dt)
                bad = (d > one_ulp) & (d > 2 * b1)
                assert not bool(bad.any()), (quads, cap, M, int(bad.sum()))
                ops._workspace(gemm_ws_bytes(M, N, K, gs, nbits, dt), x.device).fill_(0xCD)
                assert torch.equal(fwd(layer, x, bias=None), ys), (quads, cap, M)
                assert torch.equal(fwd(layer, x), ys + layer.bias), (quads, cap, M)


@pytest.mark.gpu
@pytest.mark.parametrize("nbits,gs", [(8, 64), (4, 128), (2, 64), (1, 128)])
@pytest.mark.parametrize("dtype", ["float16", "bfloat16"])
def test_route2_split_k_one_output_per_thread(nbits, gs, dtype, knobs):
    """The second pass with one output per thread, forced (1) by an output view 2 bytes off 8-byte alignment -- same bits as the
    4-wide pass on the same problem -- and (2) by N = 42 F (step % 4 != 0): within the bound, within 1 ulp of the unsplit result
    as above, bias identity."""
    dt = DT[dtype]
    F = 8 // nbits
    K, M = 1792, 200
    knobs(HQQ_B200_GEMM_KSPLIT=4)
    for N in (40 * F, 42 * F):
        layer = make_layer(N, K, nbits, gs, dt, seed=8000 + 10 * nbits + gs + N, bias=True)
        x = rand_x(M, K, dt, seed=N)
        assert gemm_ws_bytes(M, N, K, gs, nbits, dt) > 0
        y = fwd(layer, x)
        base = torch.empty(M * N + 1, device=DEV, dtype=dt)
        view = base[1:].view(M, N)
        assert view.data_ptr() % 8 != 0
        assert fwd(layer, x, out=view) is view
        assert torch.equal(view, y), N
        ystar, mass = dense_ref(x, layer.dequantize(), layer.bias)
        check("route 2 split-K", y, ystar, layer.bias, mass, C2, dt)
        ynb = fwd(layer, x, bias=None)
        assert torch.equal(y, ynb + layer.bias), N
        knobs(HQQ_B200_GEMM_KSPLIT=1)
        y1 = fwd(layer, x, bias=None)
        knobs(HQQ_B200_GEMM_KSPLIT=4)
        ystar0, _ = dense_ref(x, layer.dequantize(), None)
        d = (ynb.double() - y1.double()).abs()
        slack = 2 * bound(ystar0, None, mass, C2, dt)
        assert not bool(((d > ulp(torch.maximum(ynb.double().abs(), y1.double().abs()), dt)) & (d > slack)).any()), N


# ------------------------------------------------------------------------------------------------------------ route 3
ROUTE3_CFGS = [dict(nbits=3, group_size=64, axis=1), dict(nbits=4, group_size=64, axis=0), dict(nbits=4, group_size=32, axis=1)]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", range(len(ROUTE3_CFGS)))
@pytest.mark.parametrize("dtype", ["float16", "bfloat16"])
def test_route3_every_element_within_bound(cfg, dtype):
    """Route 3 (dequantize kernel + dense GEMM): 3-bit, axis 0 and group size 32, with K = 1000 (not a multiple of 64); within the
    bound around x @ layer.dequantize()^T + b, and the bias identity."""
    dt = DT[dtype]
    c = ROUTE3_CFGS[cfg]
    N, K = 520, 1000
    torch.manual_seed(9000 + cfg)
    layer = HQQLinear.from_weights((torch.randn(N, K, device=DEV) * 0.02).to(dt), torch.randn(N, device=DEV).to(dt), BaseQuantizeConfig(**c),
                                   compute_dtype=dt, device=DEV)
    W_r = layer.dequantize()
    nb = Quantizer._packing_bits[layer.meta["packing"]]
    for M in (1, 9, 40, 300):
        assert ops.linear_route(M, N, K, layer.meta["group_size"], nb, c["axis"], dt) == 3, (c, M)
        x = rand_x(M, K, dt, seed=M + cfg)
        y = layer(x)
        ystar, mass = dense_ref(x, W_r, layer.bias)
        check("route 3", y, ystar, layer.bias, mass, C3, dt)
        m = layer.meta
        ynb = ops.linear_fwd(x, layer.W_q, m["scale"], m["zero"], None, N, K, m["group_size"], nb, m["axis"])
        assert torch.equal(y, ynb + layer.bias)


# ----------------------------------------------------------------------------------------------- misaligned activations
def _route_layers(dt):
    torch.manual_seed(11)
    mk = lambda cfg, N, K: HQQLinear.from_weights((torch.randn(N, K, device=DEV) * 0.02).to(dt), torch.randn(N, device=DEV).to(dt),  # noqa: E731
                                                  BaseQuantizeConfig(**cfg), compute_dtype=dt, device=DEV)
    return [(1, mk(dict(nbits=4, group_size=64, axis=1), 512, 1024), 4), (2, mk(dict(nbits=4, group_size=64, axis=1), 512, 1024), 300),
            (3, mk(dict(nbits=3, group_size=64, axis=1), 512, 1024), 40)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float16", "bfloat16"])
def test_misaligned_activation_view_on_every_route(dtype):
    """A contiguous activation 2 bytes past a 16-byte boundary (x[1:] of a flat buffer) is a valid input: forward and backward
    equal those of its aligned copy, bit for bit, on every route, and linear_fwd_multi / dense_gemm take such views too."""
    dt = DT[dtype]
    for route, layer, M in _route_layers(dt):
        N, K = layer.meta["shape"]
        assert ops.linear_route(M, N, K, layer.meta["group_size"], Quantizer._packing_bits[layer.meta["packing"]], 1, dt) == route
        flat = torch.randn(M * K + 1, device=DEV).to(dt)
        xv = flat[1:].view(M, K)
        assert xv.is_contiguous() and xv.data_ptr() % 16 != 0
        assert torch.equal(layer(xv), layer(xv.clone())), route
        # backward: grad_input = grad @ W_r on the dense GEMM, with a misaligned gradient as well
        leaf_v = flat.clone().requires_grad_()
        leaf_c = xv.clone().requires_grad_()
        gflat = torch.randn(M * N + 1, device=DEV).to(dt)
        gv = gflat[1:].view(M, N)
        layer(leaf_v[1:].view(M, K)).backward(gv)
        layer(leaf_c).backward(gv.clone())
        assert torch.equal(leaf_v.grad[1:].view(M, K), leaf_c.grad), route
    route, layer, M = _route_layers(dt)[0]
    K = layer.meta["shape"][1]
    flat = torch.randn(M * K + 1, device=DEV).to(dt)
    xv = flat[1:].view(M, K)
    outs = ops.linear_fwd_multi(xv, [layer, layer])
    assert all(torch.equal(o, layer(xv.clone())) for o in outs)
    W = layer.dequantize()
    Wflat = torch.empty(W.numel() + 1, device=DEV, dtype=dt)
    Wv = Wflat[1:].view_as(W)
    Wv.copy_(W)
    assert torch.equal(ops.dense_gemm(xv, Wv, layer.bias), ops.dense_gemm(xv.clone(), W, layer.bias))


# ---------------------------------------------------------------------------------------------- (e) the bound itself
SELF_CASES = [  # route, dtype, M, N, K, nbits, gs
    (1, torch.float16, 8, 74, 2304, 4, 64),      # ragged route-1 tile (step 37)
    (1, torch.bfloat16, 9, 148, 768, 2, 128),
    (2, torch.float16, 33, 84, 1024, 4, 64),     # ragged route-2 tile, step % 4 != 0
    (2, torch.bfloat16, 17, 42, 768, 8, 128),
]


def _self_case(route, dt, M, N, K, nbits, gs, seed):
    q, s, z, b = make_layer(N, K, nbits, gs, dt, seed, bias=True, device="cpu")
    g = torch.Generator(device="cpu").manual_seed(seed + 1)
    x = torch.randn(M, K, generator=g).to(dt)
    s64, z64 = expand_meta(s, N, K, gs), expand_meta(z, N, K, gs)
    if route == 1:
        W = (q.double() - z64) * s64
    else:  # Quantizer.dequantize: (q - z) and (.. * s) rounded to T
        W = ((q.to(dt) - z.reshape(N, K // gs).repeat_interleave(gs, dim=1)) * s.reshape(N, K // gs).repeat_interleave(gs, dim=1)).double()
    return q, s64, z64, b, x, W


@pytest.mark.parametrize("case", range(len(SELF_CASES)))
def test_the_bound_rejects_planted_faults(case):
    """The criterion on exact outputs (y = T(T(y* - b) + b)) accepts them and rejects each of five faults: one group's zero one
    level off for one row, one 64-k block dropped for one (row, token), and the neighbouring group's scale for one row -- each
    planted at three seeded places at once --; the bias missing on the last row of the ragged last tile; the last token computed
    from the previous token's x.  The bound is also at least four times below the single-element error that the relative-L2
    limits of tests/test_linear_gpu.py let through at these shapes (and the norm's share of one element shrinks as outputs grow)."""
    route, dt, M, N, K, nbits, gs = SELF_CASES[case]
    q, s64, z64, b, x, W = _self_case(route, dt, M, N, K, nbits, gs, seed=100 + case)
    x64, b64 = x.double(), b.double()
    if route == 1:
        mass = x64.abs() @ (s64.abs() * (OFF[dt] + 2.0 ** nbits + z64.abs())).t()
        c = C1
    else:
        mass = (x64.abs() @ W.abs().t()) * (K / 16.0)
        c = C2
    acc = x64 @ W.t()
    ystar = acc + b64
    assert float(ratio(round_chain(acc, b, dt), ystar, b, mass, c, dt).max()) <= 1.0

    def deq(zz, ss):  # the route's matrix with changed meta
        if route == 1:
            return (q.double() - zz) * ss
        return ((q.to(dt) - zz.to(dt)) * ss.to(dt)).double()

    g = torch.Generator(device="cpu").manual_seed(case)
    pick = lambda hi: [int(v) for v in torch.randint(0, hi, (3,), generator=g)]  # noqa: E731
    Gk = K // gs
    for fault in ("zero", "block", "scale", "bias", "token"):
        rows, toks, grps, blks = pick(N), pick(M), pick(Gk), pick(K // 64)
        bias_used = b
        if fault == "zero":
            zz = z64.clone()
            for n, grp in zip(rows, grps):
                zz[n, grp * gs:(grp + 1) * gs] += 1.0
            acc_f = x64 @ deq(zz, s64).t()
        elif fault == "block":
            acc_f = acc.clone()
            for n, m, blk in zip(rows, toks, blks):
                acc_f[m, n] -= x64[m, blk * 64:(blk + 1) * 64] @ W[n, blk * 64:(blk + 1) * 64]
        elif fault == "scale":
            ss = s64.clone()
            for n, grp in zip(rows, grps):
                other = grp + 1 if grp + 1 < Gk else grp - 1
                ss[n, grp * gs:(grp + 1) * gs] = s64[n, other * gs]
            acc_f = x64 @ deq(z64, ss).t()
        elif fault == "bias":
            acc_f = acc
            bias_used = b.clone()
            bias_used[N - 1] = 0
        else:
            acc_f = acc.clone()
            acc_f[M - 1] = x64[M - 2] @ W.t()
        y_f = round_chain(acc_f, bias_used, dt)
        r = ratio(y_f, ystar, b, mass, c, dt)
        assert float(r.max()) > 1.0, (fault, float(r.max()))
    # the relative-L2 check lets a single element be off by up to TOL * ||y*||; the bound is four times tighter everywhere
    assert 4 * float(bound(ystar, b, mass, c, dt).max()) <= TOL[dt] * float(ystar.norm())
