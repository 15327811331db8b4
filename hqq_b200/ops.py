"""Tensor-level wrappers over the C ABI: marshal torch tensors (device pointers + current stream)
into ``libhqq_b200.so`` calls.  PyTorch is used for allocation and stream plumbing only.
"""
from __future__ import annotations

import math

import torch

from . import _lib
from ._lib import DTYPE_CODE, HQQ_E_UNSUPPORTED, HQQB200Error, check, load, ptr, stream_ptr

FIELDS = {8: 1, 4: 2, 3: 10, 2: 4, 1: 8}


def _as_device(t: torch.Tensor, device=None):
    """Return (tensor on a CUDA device, original device).  CPU tensors are staged onto the GPU:
    the arithmetic always runs in the CUDA library."""
    if t.is_cuda:
        return t, t.device
    if not torch.cuda.is_available():
        raise RuntimeError("hqq_b200: no CUDA device available; this package has no CPU path")
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if dev.type != "cuda":
        dev = torch.device("cuda", torch.cuda.current_device())
    return t.to(dev), t.device


# ----------------------------------------------------------------------------- BitPack
def pack(W_q: torch.Tensor, nbits: int) -> torch.Tensor:
    if W_q.dim() != 2:
        raise ValueError("BitPack.pack expects a 2-D tensor")
    if W_q.dtype not in DTYPE_CODE:
        raise TypeError(f"BitPack.pack: unsupported dtype {W_q.dtype}")
    w, home = _as_device(W_q.contiguous())
    rows, cols = w.shape
    if nbits == 3:
        out = torch.empty((int(math.ceil(rows / 10.0)), cols), dtype=torch.int32, device=w.device)
    else:
        f = FIELDS[nbits]
        if rows % f:
            raise RuntimeError(f"BitPack.pack_{nbits}bit: {rows} rows cannot be split into {f} equal slabs")
        out = torch.empty((rows // f, cols), dtype=torch.uint8, device=w.device)
    with torch.cuda.device(w.device):
        check(load().hqq_b200_pack(nbits, ptr(w), DTYPE_CODE[w.dtype], ptr(out), rows, cols, stream_ptr(w.device)))
    return out if home.type == "cuda" else out.to(home)


def unpack(W_q: torch.Tensor, nbits: int, dtype=torch.uint8) -> torch.Tensor:
    if W_q.dim() != 2:
        raise ValueError("BitPack.unpack expects a 2-D tensor")
    want = torch.int32 if nbits == 3 else torch.uint8
    if W_q.dtype != want:
        raise TypeError(f"BitPack.unpack_{nbits}bit expects a {want} tensor, got {W_q.dtype}")
    if dtype not in DTYPE_CODE:
        raise TypeError(f"BitPack.unpack: unsupported output dtype {dtype}")
    w, home = _as_device(W_q.contiguous())
    prow, cols = w.shape
    out = torch.empty((prow * FIELDS[nbits], cols), dtype=dtype, device=w.device)
    with torch.cuda.device(w.device):
        check(load().hqq_b200_unpack(nbits, ptr(w), ptr(out), DTYPE_CODE[dtype], prow, cols, stream_ptr(w.device)))
    return out if home.type == "cuda" else out.to(home)


# ----------------------------------------------------------------------------- dequantize
def dequantize(W_q: torch.Tensor, scale: torch.Tensor, zero: torch.Tensor, shape, group_size: int, nbits: int,
               axis: int, dtype: torch.dtype) -> torch.Tensor:
    """((unpack(W_q) - zero) * scale).reshape(shape) in `dtype` (quantize.py:184-199)."""
    N, K = int(shape[0]), int(shape[1])
    w, home = _as_device(W_q)
    w = w.contiguous()
    s = scale.to(device=w.device, dtype=dtype).contiguous()
    z = zero.to(device=w.device, dtype=dtype).contiguous()
    out = torch.empty((N, K), dtype=dtype, device=w.device)
    with torch.cuda.device(w.device):
        check(load().hqq_b200_dequantize(ptr(w), ptr(s), ptr(z), ptr(out), N, K, int(group_size), int(nbits), int(axis),
                                         DTYPE_CODE[dtype], stream_ptr(w.device)))
    return out if home.type == "cuda" else out.to(home)


# ----------------------------------------------------------------------------- quantize
def packed_shape(N: int, K: int, group_size: int, nbits: int, axis: int):
    total = N * K
    G = total // group_size
    R, C = (G, group_size) if axis == 1 else (group_size, G)
    prow = int(math.ceil(R / 10.0)) if nbits == 3 else R // FIELDS[nbits]
    return (prow, C), (R, C), G


def quantize(W: torch.Tensor, nbits: int, group_size: int, axis: int, round_zero: bool, optimize: bool,
             lp_norm: float = 0.7, beta: float = 10.0, iters: int = 20, scale_init=None, zero_init=None,
             max_level=None, want_trace: bool = False):
    """Fused min/max init + proximal solver + pack on the device of `W` (must be CUDA).

    Returns (W_q packed, scale [G] f32 (dequantisation form), zero [G] f32, trace-or-None) where trace is a
    dict of device tensors {info int32[4], errors float32[iters]}.
    """
    _lib.require_cuda(W, "the weight passed to quantize")
    if W.dtype not in (torch.float32, torch.float16, torch.bfloat16):
        W = W.float()
    W = W.contiguous()
    if W.dim() != 2:
        W = W.reshape(W.shape[0], -1)
    N, K = W.shape
    lib = load()
    dev = W.device
    pshape, _, G = packed_shape(N, K, group_size, nbits, axis)
    ws_bytes = lib.hqq_b200_quantize_workspace_bytes(N, K, group_size, nbits, axis, iters)
    if ws_bytes == 0:
        # re-run the checks through the real entry point to get the reference-worded message
        check(lib.hqq_b200_quantize(None, 0, N, K, group_size, nbits, axis, 0, 0, lp_norm, beta, iters, None, None, None, None,
                                    None, None, 0, None))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    W_q = torch.empty(pshape, dtype=torch.int32 if nbits == 3 else torch.uint8, device=dev)
    scale = torch.empty(G, dtype=torch.float32, device=dev)
    zero = torch.empty(G, dtype=torch.float32, device=dev)
    info = torch.zeros(4, dtype=torch.int32, device=dev) if want_trace else None
    errs = torch.zeros(max(iters, 1), dtype=torch.float32, device=dev) if want_trace else None
    if max_level is None:
        max_level = (1 << nbits) - 1
    if scale_init is not None:
        scale_init = scale_init.to(device=dev, dtype=torch.float32).contiguous().reshape(-1)
        zero_init = zero_init.to(device=dev, dtype=torch.float32).contiguous().reshape(-1)
    with torch.cuda.device(dev):
        check(lib.hqq_b200_quantize_ex(ptr(W), DTYPE_CODE[W.dtype], N, K, int(group_size), int(nbits), int(max_level), int(axis),
                                       int(bool(round_zero)), int(bool(optimize)), float(lp_norm), float(beta), int(iters),
                                       ptr(scale_init), ptr(zero_init), ptr(W_q), ptr(scale), ptr(zero), ptr(info), ptr(errs),
                                       ptr(ws), ws_bytes, stream_ptr(dev)))
    trace = {"info": info, "errors": errs} if want_trace else None
    return W_q, scale, zero, trace


def quantize_sharded(W_shard: torch.Tensor, nbits: int, group_size: int, axis: int, round_zero: bool, process_group=None,
                     lp_norm: float = 0.7, beta: float = 10.0, iters: int = 20, want_trace: bool = False):
    """`quantize` for ONE shard of a layer whose rows / groups live on several ranks (tensor parallelism), with the unsharded result:
    every rank solves its groups (`hqq_b200_quantize_shard_begin`), the per-iteration error sums and the element count are
    all-reduced over `process_group` (iters x 8 + 8 bytes -- the reference's early stop looks at the WHOLE tensor,
    optimize.py:239-247), then every rank stops at the global iteration, rounds and packs its shard
    (`hqq_b200_quantize_shard_finish`).  Same return value as `quantize`."""
    import torch.distributed as dist
    _lib.require_cuda(W_shard, "the weight passed to quantize_sharded")
    W = W_shard if W_shard.dtype in (torch.float32, torch.float16, torch.bfloat16) else W_shard.float()
    W = W.contiguous()
    N, K = W.shape
    lib = load()
    dev = W.device
    pshape, _, G = packed_shape(N, K, group_size, nbits, axis)
    ws_bytes = lib.hqq_b200_quantize_workspace_bytes(N, K, group_size, nbits, axis, iters)
    if ws_bytes == 0:
        check(lib.hqq_b200_quantize(None, 0, N, K, group_size, nbits, axis, 0, 0, lp_norm, beta, iters, None, None, None, None, None, None, 0, None))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    sums = torch.zeros(iters + 1, dtype=torch.float64, device=dev)  # [iters] error sums + the element count
    args = (ptr(W), DTYPE_CODE[W.dtype], N, K, int(group_size), int(nbits), int(axis), int(bool(round_zero)), float(lp_norm), float(beta), int(iters))
    with torch.cuda.device(dev):
        check(lib.hqq_b200_quantize_shard_begin(*args, ptr(sums), ptr(ws), ws_bytes, stream_ptr(dev)))
    sums[iters] = float(N * K)
    if dist.is_available() and dist.is_initialized():
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=process_group)
    total = int(sums[iters].item())
    W_q = torch.empty(pshape, dtype=torch.int32 if nbits == 3 else torch.uint8, device=dev)
    scale = torch.empty(G, dtype=torch.float32, device=dev)
    zero = torch.empty(G, dtype=torch.float32, device=dev)
    info = torch.zeros(4, dtype=torch.int32, device=dev) if want_trace else None
    errs = torch.zeros(iters, dtype=torch.float32, device=dev) if want_trace else None
    with torch.cuda.device(dev):
        check(lib.hqq_b200_quantize_shard_finish(*args, ptr(sums), total, ptr(W_q), ptr(scale), ptr(zero), ptr(info), ptr(errs), ptr(ws), ws_bytes,
                                                 stream_ptr(dev)))
    return W_q, scale, zero, ({"info": info, "errors": errs} if want_trace else None)


# ----------------------------------------------------------------------------- fused forward
def linear_route(M: int, N: int, K: int, group_size: int, nbits: int, axis: int, dtype: torch.dtype) -> int:
    code = DTYPE_CODE.get(dtype, -1)
    if code < 0 or not isinstance(nbits, int):
        return 0
    return load().hqq_b200_linear_fwd_route(M, N, K, int(group_size), int(nbits), int(axis), code)


_ws_cache: dict = {}


def _workspace(nbytes: int, device) -> torch.Tensor | None:
    """Per-device scratch for the fused forward (the current kernels need none: nbytes == 0).  Allocated once and kept
    alive so a captured CUDA graph never holds a stale pointer."""
    if nbytes == 0:
        return None
    key = device.index if device.index is not None else torch.cuda.current_device()
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("hqq_b200: run one forward outside CUDA-graph capture first (the workspace is allocated lazily)")
        buf = torch.zeros(nbytes, dtype=torch.uint8, device=device)
        _ws_cache.setdefault("keepalive", []).append(buf)
        _ws_cache[key] = buf
    return buf


def _on(dev: torch.device):
    """Make `dev` the current CUDA device around a launch: the C ABI launches on the calling thread's current device (its
    function-attribute / grid caches are per device), while a layer may live on another GPU of the same process."""
    if dev.type != "cuda" or dev.index is None or torch.cuda.current_device() == dev.index:
        import contextlib
        return contextlib.nullcontext()
    return torch.cuda.device(dev)


def _aligned16(t: torch.Tensor) -> torch.Tensor:
    """`t`, or a fresh contiguous copy of it when its data pointer is not 16-byte aligned.  The forward kernels load
    activations (and the dense GEMM its weight) in 16-byte vectors or through TMA and reject other pointers; a contiguous
    view at an element offset (x[1:] of a flat buffer) is still a valid activation, so it is copied instead."""
    return t if t.data_ptr() % 16 == 0 else t.clone(memory_format=torch.contiguous_format)


def linear_fwd(x2d: torch.Tensor, W_q: torch.Tensor, scale: torch.Tensor, zero: torch.Tensor, bias, N: int, K: int,
               group_size: int, nbits: int, axis: int, out: torch.Tensor | None = None) -> torch.Tensor | None:
    """y = x2d @ dequantize(W_q).T (+ bias) through the fused kernels; returns None when no fused kernel covers
    the configuration (caller then uses dequantize + matmul)."""
    x2d = _aligned16(x2d)
    dtype = x2d.dtype
    M = x2d.shape[0]
    lib = load()
    code = DTYPE_CODE.get(dtype, -1)
    if code < 0 or lib.hqq_b200_linear_fwd_route(M, N, K, int(group_size), int(nbits), int(axis), code) == 0:
        return None
    dev = x2d.device
    y = out if out is not None else torch.empty((M, N), dtype=dtype, device=dev)
    ws_bytes = lib.hqq_b200_linear_fwd_workspace_bytes(M, N, K, int(group_size), int(nbits), int(axis), code)
    ws = _workspace(ws_bytes, dev)
    with _on(dev):
        rc = lib.hqq_b200_linear_fwd(ptr(x2d), ptr(W_q), ptr(scale), ptr(zero), ptr(bias), ptr(y), M, N, K, int(group_size),
                                     int(nbits), int(axis), code, ptr(ws), ws_bytes, stream_ptr(dev))
    if rc == HQQ_E_UNSUPPORTED:
        return None
    check(rc)
    return y


def dense_gemm(x2d: torch.Tensor, W: torch.Tensor, bias=None, out: torch.Tensor | None = None) -> torch.Tensor | None:
    """y = x2d @ W.T (+ bias) for an ordinary fp16/bf16 [N, K] matrix through the dense tcgen05 kernel (`hqq_b200_dense_gemm`);
    None when the shape / dtype is outside it (fp32, K not a multiple of 8)."""
    _lib.require_cuda(x2d, "the activation passed to dense_gemm")
    code = DTYPE_CODE.get(x2d.dtype, -1)
    M, K = x2d.shape
    N = W.shape[0]
    if code not in (DTYPE_CODE[torch.float16], DTYPE_CODE[torch.bfloat16]) or W.dtype != x2d.dtype or W.shape[1] != K or K % 8:
        return None
    x2d, W = _aligned16(x2d.contiguous()), _aligned16(W.contiguous())
    y = out if out is not None else torch.empty((M, N), dtype=x2d.dtype, device=x2d.device)
    with _on(x2d.device):
        rc = load().hqq_b200_dense_gemm(ptr(x2d), ptr(W), ptr(bias), ptr(y), M, N, K, code, stream_ptr(x2d.device))
    if rc == HQQ_E_UNSUPPORTED:
        return None
    check(rc)
    return y


def linear_fwd_multi(x2d: torch.Tensor, layers, outs=None):
    """Several HQQLinear layers consuming the same activation (q/k/v, gate/up) in ONE launch of the small-M kernel.
    `layers` are HQQLinear objects with identical K / group_size / nbits / axis=1 / compute dtype; returns a list of
    outputs, or None when the configuration is outside the fused kernel (caller then runs the layers one by one)."""
    import ctypes
    lib = load()
    n = len(layers)
    if not (1 <= n <= 4):
        return None
    m0 = layers[0].meta
    K = int(m0["shape"][1])
    gs, axis = m0["group_size"], m0["axis"]
    packing = m0["packing"]
    nbits = {"8bit_u8": 8, "4bit_u8": 4, "3bit_32": 3, "2bit_u8": 2, "1bit_u8": 1}.get(packing, 0)
    dtype = x2d.dtype
    code = DTYPE_CODE.get(dtype, -1)
    M = x2d.shape[0]
    if code < 0 or gs is None or nbits == 0:
        return None
    Ns = []
    for l in layers:
        m = l.meta
        if (m["packing"] != packing or m["group_size"] != gs or m["axis"] != axis or int(m["shape"][1]) != K or l.compute_dtype != dtype
                or "scale" not in m or "zero" not in m):
            return None
        N = int(m["shape"][0])
        if lib.hqq_b200_linear_fwd_route(M, N, K, int(gs), nbits, int(axis), code) != 1:
            return None
        Ns.append(N)
    dev = x2d.device
    x2d = _aligned16(x2d)
    if outs is None:
        outs = [torch.empty((M, N), dtype=dtype, device=dev) for N in Ns]
    VP = ctypes.c_void_p * n
    arr = lambda ts: VP(*[ptr(t) for t in ts])
    ws_bytes = lib.hqq_b200_linear_fwd_workspace_bytes(M, Ns[0], K, int(gs), nbits, int(axis), code)
    ws = _workspace(ws_bytes, dev)
    Narr = (ctypes.c_int64 * n)(*Ns)
    with _on(dev):
        check(lib.hqq_b200_linear_fwd_multi(ptr(x2d), n, arr([l.W_q for l in layers]), arr([l.meta["scale"] for l in layers]),
                                            arr([l.meta["zero"] for l in layers]), arr([l.bias for l in layers]), arr(outs), Narr,
                                            M, K, int(gs), nbits, int(axis), code, ptr(ws), ws_bytes, stream_ptr(dev)))
    return outs


YOP_SILU_MUL_PAIR = 16  # HQQ_YOP_SILU_MUL_PAIR (include/hqq_b200.h): or-ed into x_op


def decode_linear_fwd(x: torch.Tensor, layers, outs, x_op: int = 0, x2=None, x_weight=None, h_out=None, eps: float = 0.0, tpx=None) -> bool:
    """One-token fused linear(s) with the activation prologue folded in (`hqq_b200_decode_linear_fwd`): x_op 1 =
    residual add + RMSNorm, 2 = SiLU(x) * x2.  `tpx` (dict) switches on the peer-memory exchange of
    `hqq_b200_decode_linear_fwd_desc`: keys tp, rank, step_ctr, x_index, x_per_step and any of peer_data (ctypes array of peer
    pointers), red_data, y_tagged (list of addresses), x_tagged, x2_tagged (addresses).  Returns False when the configuration is
    outside the fused M = 1 kernel."""
    import ctypes
    lib = load()
    n = len(layers)
    m0 = layers[0].meta
    K = int(m0["shape"][1])
    nbits = {"8bit_u8": 8, "4bit_u8": 4, "3bit_32": 3, "2bit_u8": 2, "1bit_u8": 1}.get(m0["packing"], 0)
    code = DTYPE_CODE.get(x.dtype, -1)
    if code < 0 or m0["group_size"] is None or nbits == 0 or m0["axis"] != 1:
        return False
    VP = ctypes.c_void_p * n
    arr = lambda ts: VP(*[ptr(t) for t in ts])
    Narr = (ctypes.c_int64 * n)(*[int(l.meta["shape"][0]) for l in layers])
    with _on(x.device):
        rc = _decode_launch(lib, x, layers, outs, x_op, x2, x_weight, h_out, eps, tpx, n, m0, K, nbits, code, arr, Narr, VP)
    if rc == HQQ_E_UNSUPPORTED:
        return False
    check(rc)
    return True


def _decode_launch(lib, x, layers, outs, x_op, x2, x_weight, h_out, eps, tpx, n, m0, K, nbits, code, arr, Narr, VP):
    import ctypes
    if tpx is None:
        rc = lib.hqq_b200_decode_linear_fwd(ptr(x), int(x_op), ptr(x2), ptr(x_weight), ptr(h_out), float(eps), n, arr([l.W_q for l in layers]),
                                            arr([l.meta["scale"] for l in layers]), arr([l.meta["zero"] for l in layers]),
                                            arr([l.bias for l in layers]), arr(outs), Narr, K, int(m0["group_size"]), nbits, code,
                                            stream_ptr(x.device))
    else:
        cast = lambda a: ctypes.cast(a, ctypes.c_void_p) if a is not None else None
        arrays = [arr([l.W_q for l in layers]), arr([l.meta["scale"] for l in layers]), arr([l.meta["zero"] for l in layers]),
                  arr([l.bias for l in layers]), arr(outs)]
        ytag = tpx.get("y_tagged")
        ytag_arr = VP(*ytag) if ytag is not None else None
        d = _lib.DecodeDesc(x=ptr(x), x_op=int(x_op), x2=ptr(x2), x_weight=ptr(x_weight), h_out=ptr(h_out), eps=float(eps), count=n,
                            W_q=cast(arrays[0]), scale=cast(arrays[1]), zero=cast(arrays[2]), bias=cast(arrays[3]), y=cast(arrays[4]),
                            N=cast(Narr), K=K, group_size=int(m0["group_size"]), nbits=nbits, dtype=code, tp=int(tpx["tp"]), rank=int(tpx["rank"]),
                            peer_data=cast(tpx.get("peer_data")), red_data=tpx.get("red_data"), y_tagged=cast(ytag_arr),
                            x_tagged=tpx.get("x_tagged"), x2_tagged=tpx.get("x2_tagged"), step_ctr=tpx["step_ctr"],
                            x_index=int(tpx["x_index"]), x_per_step=int(tpx["x_per_step"]))
        rc = lib.hqq_b200_decode_linear_fwd_desc(ctypes.byref(d), stream_ptr(x.device))
    return rc


__all__ = ["pack", "unpack", "dequantize", "quantize", "linear_fwd", "linear_fwd_multi", "linear_route", "packed_shape", "HQQB200Error"]
