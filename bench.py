#!/usr/bin/env python
"""bench.py -- Llama-3-8B-shaped 4-bit (gs=64, axis=1) decode tokens/s on B200 through hqq_b200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is one decoded token (bs=1, seq=1) through all 32 blocks + lm_head of a random-init Llama-3-8B-shaped
stack whose 224 block linears are HQQLinear layers quantised on the GPU by this package (synthetic data, BASELINE.json
configs[1]).  `value` is tokens/s with the token fed back on the device (inputs resident in HBM); `e2e` is the same loop
driven from the host through the public API: every step copies the input token from pinned host memory, replays the
decode graph and reads the produced token back.  For N > 1 the same model is tensor-parallel over N GPUs (column-sharded
q/k/v/gate/up, row-sharded o/down whose partial sums are exchanged inside the kernels over NVLink peer memory -- NCCL
all-reduce with HQQ_B200_TP_MODE=nccl), i.e. strong scaling.

`--impl reference` times the reference algorithm's CPU implementation (the oracle port of HQQBackend.PYTORCH:
dequantise -> matmul per linear) on this box's host cores on a bounded sample of the same workload.

`--dump-outputs DIR` writes what the last timed step of the device-resident loop handed its caller: DIR/next_token.npy (the
greedy token of every sequence, float64) and DIR/logits.npy (float32 [batch, vocab]).  The weights come from fixed seeds and
decoding starts from a fixed token, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "llama3_8b_4bit_gs64_decode_tokens_per_s"
UNIT = "tokens/s"
# BASELINE.json configs[1]; both arms print exactly this string as config.workload
WORKLOAD = "Llama-3-8B-shaped decode bs=1 seq=1, 32 blocks x 7 HQQLinear 4-bit gs=64 axis=1, fp16 lm_head (BASELINE configs[1])"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": float(d["hbm_gbs"]), "tensor_tflops": float(d.get("bf16_tflops", 1590.0)), "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tensor_tflops": 1590.0, "source": "fallback (B200_PROFILING.md)"}


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.samples, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- CPU baseline (oracle port)
def host_topology():
    """(physical cores of ONE socket, sockets, logical cpus) from /proc/cpuinfo; falls back to os.cpu_count()."""
    try:
        cores, phys, cur = set(), set(), {}
        for ln in open("/proc/cpuinfo"):
            if ":" in ln:
                k, v = [t.strip() for t in ln.split(":", 1)]
                cur[k] = v
            elif cur:
                if "physical id" in cur and "core id" in cur:
                    cores.add((cur["physical id"], cur["core id"])); phys.add(cur["physical id"])
                cur = {}
        if cores:
            return max(1, len(cores) // max(1, len(phys))), max(1, len(phys)), os.cpu_count() or 1
    except OSError:
        pass
    n = os.cpu_count() or 1
    return n, 1, n


def pin_openmp_env():
    """Called before anything loads libgomp: one thread per physical core, packed (the CPU arm's team stays on one socket's cores)."""
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")


def _cpu_oracle():
    """(forward factory, cores, label, module): the C/OpenMP restatement (oracle/hqq_oracle_c.c) with its team pinned to the physical
    cores of ONE socket -- the same team in `--impl reference` and in the GPU arm's cpu_baseline leg, whatever OMP_NUM_THREADS the
    launcher exported (torchrun sets 1) -- else the numpy port.  bench.py's cpu_baseline / --impl reference legs are the only
    product-side places that may execute oracle/ (it is the thing timed here, never the thing shipped)."""
    try:
        from oracle import hqq_oracle_c as c
        per_socket, sockets, logical = host_topology()
        cores = c.set_threads(per_socket)
        return ((lambda W_q, meta: c.Forward(W_q, meta)), cores,
                f"C/OpenMP port (oracle/hqq_oracle_c.c, {cores} threads = one socket's physical cores of {sockets} x {per_socket}, {logical} logical cpus)", c)
    except Exception:  # noqa: BLE001 -- no C compiler / no OpenMP: the numpy port
        from oracle import hqq_oracle as o
        return (lambda W_q, meta: (lambda x: o.linear_forward_f32_fast(x, W_q, meta))), 1, "numpy port (oracle/hqq_oracle.py; BLAS matmul may use more threads)", None


class CpuReference:
    """HQQBackend.PYTORCH on the host: per linear, dequantise the whole matrix (unpack, subtract, multiply: three passes over an
    N x K float32 matrix) then matmul (quantize.py:184-199, 880-898), float32 compute dtype (the reference's CPU path), through the
    oracle port.  One `step()` = ONE of the 32 blocks (7 linears, bs=1) plus 1/32 of the fp32 lm_head GEMV, i.e. 1/32 of a token."""

    SHAPES = {"q": (4096, 4096), "k": (1024, 4096), "v": (1024, 4096), "o": (4096, 4096), "gate": (14336, 4096), "up": (14336, 4096),
              "down": (4096, 14336)}
    STEPS_PER_TOKEN = 32

    def __init__(self):
        import numpy as np
        make, self.cores, self.label, _ = _cpu_oracle()
        rng = np.random.RandomState(0)
        self.layers = []
        for name, (n, k) in self.SHAPES.items():
            R = n * k // 64
            W_q = rng.randint(0, 256, size=(R // 2, 64)).astype(np.uint8)
            meta = {"nbits": 4, "group_size": 64, "shape": (n, k), "axis": 1, "packing": "4bit_u8",
                    "scale": (rng.rand(R, 1) * 0.01 + 1e-3).astype(np.float32), "zero": (rng.rand(R, 1) * 15).astype(np.float32)}
            self.layers.append((make(W_q, meta), rng.randn(1, k).astype(np.float32)))
        self.lm = rng.randn(128256 // self.STEPS_PER_TOKEN, 4096).astype(np.float32)  # 1/32 of the 128256-row fp32 lm_head
        self.xv = rng.randn(4096).astype(np.float32)
        self.step()  # untimed pass: page the scratch matrices in
        self.lm @ self.xv

    def step(self):
        for f, x in self.layers:
            f(x)

    def lm_share_s(self, reps: int = 5) -> float:
        """Seconds of 1/32 of the fp32 lm_head GEMV (numpy / BLAS), timed apart from the blocks: alternating the OpenMP team of the
        port with the BLAS thread pool inside one step makes both spin against each other (measured: the step then takes twice as long)."""
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            self.lm @ self.xv
            ts.append(time.perf_counter() - t0)
        return statistics.median(ts)

    def run(self, steps: int, warmup: int, budget_s: float):
        """`warmup` untimed + up to `steps` timed steps (stops early once `budget_s` is spent, never before 10 steps); returns
        (tokens/s over the timed steps, info with min / median / max of five chunk means and the stability verdict)."""
        for _ in range(max(0, warmup)):
            self.step()
        times = []
        t_all = time.perf_counter()
        for i in range(max(1, steps)):
            t0 = time.perf_counter()
            self.step()
            times.append(time.perf_counter() - t0)
            if i + 1 >= 10 and time.perf_counter() - t_all > budget_s:
                break
        n = len(times)
        lm = self.lm_share_s()
        times = [t + lm for t in times]  # a step = one block + 1/32 of the lm_head
        tok_s = n / (sum(times) * self.STEPS_PER_TOKEN)
        k = max(1, n // 5)
        chunks = [sum(times[i:i + k]) / len(times[i:i + k]) for i in range(0, n - n % k if n >= 5 else n, k)][:5]
        lo, hi = min(chunks), max(chunks)
        info = {"steps_timed": n, "cores": self.cores, "port": self.label,
                "tokens_per_s_min_median_max": [1.0 / (hi * self.STEPS_PER_TOKEN), 1.0 / (statistics.median(chunks) * self.STEPS_PER_TOKEN),
                                                1.0 / (lo * self.STEPS_PER_TOKEN)],
                "stable": (hi / lo) <= 1.3,
                "sample": f"{n} steps, each ONE block (7 HQQ linears, dequantise+matmul, fp32, bs=1) + 1/32 of the lm_head GEMV (timed apart) = 1/32 token; {self.label}"}
        return tok_s, info


def cpu_quantizer_baseline():
    """Quantizer.quantize on the host cores through the C/OpenMP oracle port: ONE 4096 x 4096 matrix of the quantizer object's
    workload (same distribution, float32 as the reference's CPU path computes), in G weights/s like `quantizer.gweights_per_s`."""
    import numpy as np
    _, cores, label, c = _cpu_oracle()
    if c is None:
        return {"error": "C oracle unavailable (no compiler)"}
    W = (np.random.RandomState(7).randn(4096, 4096) * 0.02).astype(np.float16).astype(np.float32)
    t0 = time.perf_counter()
    _, _, tr = c.quantize(W, nbits=4, group_size=64, axis=1, round_zero=True, optimize=True, return_trace=True)
    dt = time.perf_counter() - t0
    return {"value": W.size / dt / 1e9, "unit": "Gweights/s", "cores": cores, "kind": "port", "seconds": dt, "solver_iterations": tr["iters"],
            "sample": f"one 4096x4096 matrix (of the block's seven), min/max + proximal solver + round + pack; {label}"}


def run_reference(args, rank, world):
    """--impl reference: rank 0 times the reference's CPU path (the oracle port, team pinned to one socket's physical cores) on the
    arm's own --steps / --warmup, a step being 1/32 of a token (one block + 1/32 of the lm_head).  Unstable timings (max/min of five
    chunk means > 1.3) are measured again, up to three times; the line says whether the last attempt was stable."""
    if rank != 0:
        return
    ref = CpuReference()
    for attempt in range(3):
        value, info = ref.run(args.steps, args.warmup if attempt == 0 else 1, budget_s=100.0)
        if info["stable"]:
            break
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": info["steps_timed"],
            "warmup": args.warmup, "ms_per_step": 1000.0 / value / ref.STEPS_PER_TOKEN, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "path": "HQQBackend.PYTORCH data flow (dequantise + matmul) on the host cores: " + info["port"],
                       "step": "1/32 token (one of the 32 blocks + 1/32 of the lm_head); value = steps / (32 x time)", "attempts": attempt + 1},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": info["cores"], "host_cores": os.cpu_count() or 1, "kind": "port",
                             "sample": info["sample"], "min_median_max": info["tokens_per_s_min_median_max"], "stable": info["stable"]},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- GPU arm
def _time_graph(torch, dev, fn, reps):
    """Capture `reps` x fn() into a CUDA graph, replay once untimed, then time one replay with CUDA events on the launching stream."""
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay()
    torch.cuda.synchronize(dev)
    stream = torch.cuda.current_stream(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    g.replay()
    e1.record(stream)
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / reps


def kernel_roofline(model, torch, peaks, reps=4):
    """Average duration of the fused forward kernel for each of the four launch groups a decode step issues per block
    (q+k+v, o, gate+up, down -- the matrices that share an activation go out in ONE launch).  All launches of one group over
    all layers (x reps) are captured into a CUDA graph so the measurement is not bound by Python launch overhead, replayed,
    and timed with CUDA events on the launching stream.  Cycling through every layer's weights means each launch streams cold
    weights (per-group footprint x 32 layers exceeds the 126 MB L2).
    achieved = algorithmic bytes of the 128 launches (224 matrices) of one step / their summed average durations."""
    from hqq_b200 import ops
    dev = model.device
    groups = [("qkv", ("q", "k", "v")), ("o", ("o",)), ("gate_up", ("gate", "up")), ("down", ("down",))]
    per = {}
    tot_bytes = tot_ms = 0.0
    for gname, names in groups:
        sets = [[blk[n] for n in names] for blk in model.blocks]
        K = sets[0][0].meta["shape"][1]
        Ns = [l.meta["shape"][0] for l in sets[0]]
        x = torch.randn(1, K, device=dev).to(model.dtype)
        outs = [torch.empty(1, N, device=dev, dtype=model.dtype) for N in Ns]
        # the MLP launch ships with the silu*mul epilogue (gate and up rows paired per tile, one output vector)
        x_op = ops.YOP_SILU_MUL_PAIR if (gname == "gate_up" and model.nbits < 8) else 0

        def run_all():
            for ls in sets:
                if not ops.decode_linear_fwd(x, ls, outs, x_op):
                    ops.linear_fwd_multi(x, ls, outs)

        ms = _time_graph(torch, dev, run_all, reps) / len(sets)
        nbytes = sum(N * K * 0.5 + 2 * (N * K // 64) * 2 for N in Ns) + (Ns[0] if x_op else sum(Ns)) * 2 + K * 2
        per[gname] = {"N": Ns, "K": K, "us": round(ms * 1e3, 3), "GBps": round(nbytes / ms / 1e6, 1)}
        tot_bytes += nbytes
        tot_ms += ms
    achieved = tot_bytes / tot_ms / 1e6
    # dram bytes per launch (average over the four launch groups) from the committed `ncu --set full` capture of the shipped kernel
    # -- it was taken on the unsharded Llama-3-8B matrices: for any other launch shapes (tensor-parallel shards, the 70B model)
    # there is no capture and `traffic` is null rather than a number that belongs to other launches
    traffic, traffic_src = None, None
    for name in ("r2_decode1_traffic.json", "r1_decode1_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as fh:
                cap = json.load(fh)
            if abs(cap["algorithmic_bytes_per_launch_avg"] / (tot_bytes / len(groups)) - 1.0) < 0.01:
                traffic, traffic_src = cap["traffic_bytes_per_launch_avg"], "profiles/" + name
            break
        except (OSError, KeyError, ValueError, ZeroDivisionError):
            continue
    return {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
            "traffic": traffic, "algorithmic_bytes_per_launch": tot_bytes / len(groups),
            "kernel": "hqq::linear_decode1_kernel<half,4,64,...,MR=1> (scale/zero on the cp.async ring; 4 launches/block, 128/step)",
            "peak_source": peaks["source"], "per_launch_group": per, "linear_us_per_step": round(tot_ms * 1e3 * len(model.blocks), 1),
            "note": "event-timed graph replay of back-to-back launches over all layers (cold weights); traffic: "
                    + (f"{traffic_src} (ncu dram bytes, same launch shapes)" if traffic_src else "no ncu capture for these launch shapes")}


def quantizer_roofline(torch, peaks, dev, reps=3):
    """North-star path (a): Quantizer.quantize (min/max init + proximal solver + round + pack) of ONE Llama-3-8B block's seven
    matrices (218 M weights, fp16 source, 4-bit gs=64 axis=1, 20 iterations max), timed with CUDA events on the launching stream.
    Algorithmic bytes (SURVEY 8d): N*K*(2 + 0.5) + 2*(N*K/64)*4 per matrix.  The solver is bound by instruction issue, not HBM
    (DESIGN.md 3.2: ncu 75 % issue-active), so the HBM fraction is reported as SURVEY 8d asks and explained there."""
    from hqq_b200 import ops
    shapes = [(4096, 4096), (1024, 4096), (1024, 4096), (4096, 4096), (14336, 4096), (14336, 4096), (4096, 14336)]
    g = torch.Generator(device=dev)
    g.manual_seed(7)
    Ws = [(torch.randn(n, k, device=dev, generator=g, dtype=torch.float32) * 0.02).half() for n, k in shapes]
    stream = torch.cuda.current_stream(dev)

    def run():
        for W in Ws:
            ops.quantize(W, 4, 64, 1, True, True)

    run()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        run()
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / reps
    weights = sum(n * k for n, k in shapes)
    nbytes = sum(n * k * 2.5 + 2 * (n * k // 64) * 4 for n, k in shapes)
    achieved = nbytes / ms / 1e6
    return {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
            "ms_per_block": ms, "gweights_per_s": weights / ms / 1e6, "algorithmic_bytes_per_block": nbytes,
            "kernel": "solver_axis1_kernel + stop_kernel + quant_pack_kernel (3 launches per matrix)",
            "workload": "one Llama-3-8B block (7 matrices, 218 M weights) fp16 -> 4-bit gs=64 axis=1, solver + pack"}


def gemm_sweep(torch, peaks, dev, quick=False):
    """BASELINE configs[2] / the second half of `metric`: the fused dequant-GEMM (hqq_b200_linear_fwd, tcgen05 route) on the
    per-linear sweep -- (N, K) in {4096x4096, 11008x4096, 4096x11008} x nbits {8,4,3,2,1}, gs 64, fp16 -- at M = 4096 (tensor
    roofline) and M = 128, event-timed alone, against the measured dense tensor peak; cuBLAS on the pre-dequantised matrix
    beside it.  3-bit has no tcgen05 route yet: its figure is our dequantize kernel + the library GEMM."""
    from hqq_b200 import ops
    from hqq_b200.core.quantize import BaseQuantizeConfig, HQQLinear
    peak_tf = peaks["tensor_tflops"]
    per = {}
    torch.manual_seed(0)
    shapes = [(4096, 4096)] if quick else [(4096, 4096), (11008, 4096), (4096, 11008)]
    stream = torch.cuda.current_stream(dev)

    def timed(fn, reps):
        for _ in range(2):
            fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / reps

    for nbits in ((4,) if quick else (8, 4, 3, 2, 1)):
        for N, K in shapes:
            layer = HQQLinear.from_weights((torch.randn(N, K, device=dev) * 0.02).half(), None, BaseQuantizeConfig(nbits=nbits, group_size=64, axis=1),
                                           compute_dtype=torch.float16, device=str(dev))
            Wd = layer.dequantize()
            for M in (4096, 128):
                x = torch.randn(M, K, device=dev).half()
                y = torch.empty(M, N, device=dev, dtype=torch.float16)
                route = ops.linear_route(M, N, K, 64, nbits, 1, x.dtype)
                if route != 0:
                    fn = lambda: ops.linear_fwd(x, layer.W_q, layer.meta["scale"], layer.meta["zero"], None, N, K, 64, nbits, 1, out=y)
                else:
                    fn = lambda: layer(x)
                with torch.no_grad():
                    ms = timed(fn, 5)
                    ms_lib = timed(lambda: torch.matmul(x, Wd.t(), out=y), 5)
                tf = 2.0 * M * N * K / ms / 1e9
                per[f"b{nbits}_{N}x{K}_M{M}"] = {"us": round(ms * 1e3, 1), "TFLOPs": round(tf, 1), "frac_of_tensor_peak": round(tf / peak_tf, 4), "route": route,
                                               "cublas_on_dequantised_TFLOPs": round(2.0 * M * N * K / ms_lib / 1e9, 1)}
            del layer, Wd
    head = per["b4_4096x4096_M4096"]
    return {"bound": "tensor", "achieved": head["TFLOPs"], "peak": peak_tf, "unit": "TFLOP/s", "frac": head["frac_of_tensor_peak"],
            "shape": "M=4096 N=4096 K=4096 nbits=4 gs=64 fp16", "kernel": "hqq::gemm::linear_gemm_kernel (persistent tcgen05 / TMA / TMEM)",
            "peak_source": peaks["source"] + " bf16_tflops (burst: kernel timed alone)", "per": per,
            "note": "route 2 = fused tcgen05 kernel, 0 = dequantize kernel + library GEMM (3-bit); cuBLAS runs on the 16-bit matrix our dequantize kernel wrote"}


def _finite(o):
    """json.dumps would print NaN / Infinity, which is not JSON: map non-finite floats to None."""
    if isinstance(o, float):
        return o if o == o and abs(o) != float("inf") else None
    if isinstance(o, dict):
        return {k: _finite(v) for k, v in o.items()}
    if isinstance(o, (list, tuple)):
        return [_finite(v) for v in o]
    return o


def tokens_agree(model, torch, n_tokens=16):
    """N > 1, before anything is timed: the fused NVLink exchange ("p2p") against NCCL all-reduces between the kernels ("nccl").
    The mode that will be timed decodes `n_tokens` greedy tokens from the reset state; the other mode is then fed the SAME tokens
    (teacher forcing, so one flipped pick cannot snowball) and must pick the same token at every step.  The two modes add the
    ranks' 16-bit partial sums in different orders, so the logits differ in their last bits; a differing pick is accepted only if
    it is such a near-tie: the timed mode's own margin between the two candidates is within twice the largest logit difference
    of that step, and the logits as a whole differ by less than 5 % of their range (measured: 0.7 % on the 8B model at tp = 8, 2 % on
    the 80-block 70B model).  Anything else is a wrong exchange.
    Leaves the model captured in the mode it came with.  Returns (agree, detail)."""
    import torch.distributed as dist
    want = model.tp_mode
    other = "nccl" if want == "p2p" else "p2p"
    shard = model.vocab_shard

    def run(mode, forced=None):
        if model.tp_mode != mode or model.graph is None:
            model.tp_mode = mode
            model.graph = None
            model.capture(warmup=2)
        model.reset_state(token=1)
        toks, logits = [], []
        for i in range(n_tokens):
            if forced is not None and i > 0:
                model.tok.copy_(forced[i - 1:i])
            model.decode(feed_back=forced is None)
            toks.append(model.next_tok.clone())
            logits.append(model._bufs["logits"].float().view(1, -1).clone())
        torch.cuda.synchronize(model.device)
        return torch.stack(toks).view(-1), torch.cat(logits)

    def gmax(t):
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t

    t_a, l_a = run(want)
    t_b, l_b = run(other, forced=t_a)
    run(want)  # back to the mode that is timed
    diff = gmax((l_a - l_b).abs().amax(dim=1))              # per step, over the whole vocabulary
    scale = float(gmax(l_a.abs().amax().view(1)))
    identical = bool(torch.equal(t_a, t_b))
    ties = []
    explained = True
    if not identical:
        lo = model.rank * shard
        for i in torch.nonzero(t_a != t_b).view(-1).tolist():
            pair = torch.full((2,), float("-inf"), device=model.device)
            for k, tok in enumerate((int(t_a[i]), int(t_b[i]))):
                if lo <= tok < lo + shard:
                    pair[k] = l_a[i, tok - lo]
            pair = gmax(pair)
            margin = float(pair[0] - pair[1])
            ok = 0.0 <= margin <= 2.0 * float(diff[i])
            explained = explained and ok
            ties.append({"step": i, "margin": margin, "max_logit_diff": float(diff[i]), "near_tie": ok})
    dmax = float(diff.max())
    agree = identical or (explained and dmax <= 0.05 * scale)
    flag = torch.tensor([1 if agree else 0], device=model.device)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    detail = {"tokens": n_tokens, "identical": identical, "max_logit_diff": dmax, "logit_absmax": scale, "against": other}
    if ties:
        detail["differing_picks"] = ties
    return bool(flag.item()), detail


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, next_tok, logits, rank, world):
    """--dump-outputs: the greedy tokens [batch] as float64 and the logits [batch, vocab] as float32 in `out_dir`.  With tp > 1 the
    ranks' vocabulary shards are gathered first.  Above DUMP_BYTES only the first sequences are kept (every sequence of the bench
    starts from the same token, so they are a fixed sample of the batch)."""
    import numpy as np
    if world > 1:
        import torch
        import torch.distributed as dist
        parts = [torch.empty_like(logits) for _ in range(world)]
        dist.all_gather(parts, logits.contiguous())
        logits = torch.cat(parts, dim=-1)
    if rank != 0:
        return
    rows = max(1, DUMP_BYTES // (4 * logits.shape[-1]))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "next_token.npy"), next_tok[:rows].cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "logits.npy"), logits[:rows].float().cpu().numpy())


def run_gpu(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    from hqq_b200 import _lib, harness
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    lib = _lib.load()
    big = args.model == "70b"  # BASELINE configs[4]: needs --gpus 8 (4.8 GB of packed weights per rank); not the default line
    shape = harness.LLAMA3_70B if big else harness.LLAMA3_8B
    metric = "llama3_70b_4bit_gs64_decode_tokens_per_s" if big else METRIC
    workload = ("Llama-3-70B-shaped decode bs=1 seq=1, 80 blocks x 7 HQQLinear 4-bit gs=64 axis=1, fp16 lm_head (BASELINE configs[4], bs=1)"
                if big else WORKLOAD)
    n_layers = args.layers or shape.n_layers
    if args.cache_len <= 0:  # every timed loop starts at position 0 and must not wrap inside the cache
        args.cache_len = min(8192, max(256, args.steps + max(args.warmup, 3) + 8))
    B = max(1, args.batch)
    if B > 1:  # BASELINE configs[4] bs = 32 leg: not the default line
        metric += f"_bs{B}"
        workload = workload.replace("bs=1", f"bs={B}")
    lib.hqq_b200_launch_count_reset()
    model = harness.DecodeModel(shape, nbits=4, group_size=64, dtype=torch.float16, device=dev, cache_len=args.cache_len, tp=world,
                                rank=rank, process_group=pg, n_layers=n_layers, batch=B)
    lib.hqq_b200_launch_count_reset()
    model.capture(warmup=3)
    # launches of OUR kernels in one step = those issued while capturing one step (3 warm-up steps + 1 captured)
    launches_per_step = int(lib.hqq_b200_launch_count()) // 4
    agree, token_check = None, None
    if world > 1 and B == 1 and not args.no_token_check:
        agree, token_check = tokens_agree(model, torch)
        if not agree:
            # never time a model whose exchange is in doubt: NCCL all-reduces between the kernels are the correctness reference
            if rank == 0:
                print(f"bench.py: the fused NVLink exchange and the NCCL all-reduce disagree beyond rounding ({json.dumps(token_check)}); "
                      "timing the NCCL mode instead", file=sys.stderr, flush=True)
            token_check["fell_back_to"] = "nccl"
            model.tp_mode = "nccl"
            model.graph = None
            model.capture(warmup=3)
    stream = torch.cuda.current_stream(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident loop -------------------------------------------------------------------
    model.reset_state(token=1)
    for _ in range(max(args.warmup, 3)):
        model.decode()
    model.pos.zero_()
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        model.decode()
    e1.record(stream)
    barrier()
    dev_ms = e0.elapsed_time(e1)
    # the next loop overwrites the step's buffers: keep what the last timed step produced
    last = (model.next_tok.clone(), model._bufs["logits"].clone()) if args.dump_outputs else None

    # ---- end-to-end loop through the public API with host buffers ------------------------------
    h_in = torch.ones(B, dtype=torch.long).pin_memory()
    h_out = torch.zeros(B, dtype=torch.long).pin_memory()
    model.pos.zero_()
    for _ in range(3):
        model.tok.copy_(h_in, non_blocking=True); model.graph.replay(); h_out.copy_(model.next_tok, non_blocking=True); torch.cuda.synchronize(dev)
    model.pos.zero_()
    barrier()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for _ in range(args.steps):
        model.tok.copy_(h_in, non_blocking=True)          # H2D: this step's input token
        model.graph.replay()
        h_out.copy_(model.next_tok, non_blocking=True)    # D2H: the produced token
        stream.synchronize()
        h_in.copy_(h_out)                                 # host-side feedback, as a generation loop would
    t1.record(stream)
    barrier()
    e2e_ms = t0.elapsed_time(t1)
    clocks = sampler.stop() if rank == 0 else None

    if world > 1:
        t = torch.tensor([dev_ms, e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_ms = t.tolist()
    if last is not None:
        dump_outputs(args.dump_outputs, *last, rank, world)

    peaks = load_peaks()
    roof = kernel_roofline(model, torch, peaks) if (rank == 0 and B == 1) else None
    if rank == 0:
        value = args.steps * B / (dev_ms / 1e3)
        e2e = args.steps * B / (e2e_ms / 1e3)
        bytes_rank = model.bytes_per_token()  # per rank: its shard of every block + its vocabulary shard of the lm_head
        line = {"metric": metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16",
                "data": "synthetic",
                "config": {"workload": workload,
                           "path": f"fused sm_100a kernels, kv cache {args.cache_len}, CUDA graph; {bytes_rank / 1e9:.2f} GB streamed per step and rank "
                                   ">> 126 MB L2 (inputs larger than L2, no flush needed)",
                           "parallelism": f"tp{world}", "layers": n_layers, "global_batch": B,
                           "tp_mode": (model.tp_mode if (world > 1 and B == 1) else ("nccl" if world > 1 else None)), "tokens_agree": agree, "token_check": token_check},
                "clocks": clocks,
                "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": 8 * B, "d2h_bytes_per_step": 8 * B},
                "gpu_launches": launches_per_step * args.steps,
                "step_hbm_GBps_per_rank": bytes_rank / (dev_ms / args.steps) / 1e6}
        if n_layers != shape.n_layers:
            line["config"]["note"] = "REDUCED layer count (debug run) -- not the BASELINE configuration"
        if roof is not None:
            roof["step_frac_of_hbm_peak"] = line["step_hbm_GBps_per_rank"] / peaks["hbm_gbs"]
            line["roofline"] = roof
        # Everything below adds objects to the line that is already complete (GEMM sweep, quantizer, CPU baselines).  A watchdog
        # prints the line as it stands if they ever exceed their deadline, so they cannot cost the measurement.
        printed = threading.Event()

        def emit():
            if printed.is_set():
                return
            printed.set()
            for _ in range(5):
                try:
                    print(json.dumps(_finite(dict(line))), flush=True)
                    return
                except RuntimeError:  # the main thread added a key meanwhile
                    time.sleep(0.05)

        def watchdog():
            if not printed.wait(timeout=args.extras_deadline):
                line["extras"] = f"cut off after {args.extras_deadline:.0f} s"
                emit()
                os._exit(0)

        threading.Thread(target=watchdog, daemon=True).start()
        extras = world == 1 and not big and B == 1 and not args.no_extras
        if extras:
            del model
            torch.cuda.empty_cache()
            # the driver keeps `roofline` / `cpu_baseline` / `config` of the line: the second half of BASELINE's metric (fused
            # dequant-GEMM against the tensor roofline) and the quantizer (north-star path a) therefore live INSIDE `roofline`
            try:
                line["roofline"]["gemm"] = gemm_sweep(torch, peaks, dev, quick=args.quick_extras)
            except Exception as e:  # noqa: BLE001 -- an extra object must never cost the bench line
                line["roofline"]["gemm"] = {"error": repr(e)[:200]}
            try:
                line["roofline"]["quantizer"] = quantizer_roofline(torch, peaks, dev)
            except Exception as e:  # noqa: BLE001
                line["roofline"]["quantizer"] = {"error": repr(e)[:200]}
        if extras and not args.no_cpu_baseline:
            try:  # the reference's CPU solver (float32, optimize.py:201-255) beside the quantizer object, on a bounded sample
                if "ms_per_block" in line["roofline"].get("quantizer", {}):
                    line["roofline"]["quantizer"]["cpu_baseline"] = cpu_quantizer_baseline()
            except Exception as e:  # noqa: BLE001
                line["roofline"]["quantizer"]["cpu_baseline"] = {"error": repr(e)[:200]}
            try:
                v, info = CpuReference().run(steps=160, warmup=2, budget_s=20.0)
                line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": info["cores"], "host_cores": os.cpu_count() or 1, "kind": "port",
                                        "sample": info["sample"], "min_median_max": info["tokens_per_s_min_median_max"], "stable": info["stable"]}
            except Exception as e:  # noqa: BLE001
                line["cpu_baseline"] = {"error": repr(e)[:200]}
        emit()
    if world > 1:
        # Tear down without touching NCCL again: destroying a process group while captured graphs still hold its kernels
        # can hang.  Everything is measured and printed; leave through the fast exit on every rank.
        torch.cuda.synchronize(dev)
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="hqq_b200", choices=["hqq_b200", "reference"])
    ap.add_argument("--cache-len", type=int, default=0, help="KV-cache length; 0 = large enough that the timed loops never wrap (>= 256)")
    ap.add_argument("--layers", type=int, default=0, help="debug: fewer blocks (marks the line as reduced)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the GEMM sweep / quantizer / CPU baseline objects (N=1 only anyway)")
    ap.add_argument("--quick-extras", action="store_true", help="GEMM sweep: the 4096^3 4-bit headline only")
    ap.add_argument("--no-token-check", action="store_true", help="N>1: skip the p2p-vs-nccl token agreement check before timing")
    ap.add_argument("--extras-deadline", type=float, default=240.0, help="seconds the objects added after the measurement (GEMM sweep, "
                    "quantizer, CPU baselines) may take before the line is printed without the unfinished ones")
    ap.add_argument("--batch", type=int, default=1, help="sequences decoded in lock-step (BASELINE configs[4]: 32); > 1 runs the small-M / tcgen05 "
                    "kernels between the batched glue kernels, NCCL all-reduce for the tensor-parallel partials")
    ap.add_argument("--model", default="8b", choices=["8b", "70b"], help="70b = BASELINE configs[4] (use with --gpus 8)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the last timed step's tokens and logits to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm (--impl hqq_b200)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # The CPU legs pin their OpenMP team (reproducible reference arm).  Never in a multi-rank GPU run: with OMP_PLACES set, libgomp
    # binds every process's initial thread to the FIRST place, i.e. all ranks' host threads to core 0, and a loop with one host sync
    # per step (e2e) then time-slices the ranks on one core -- measured: e2e 89 tok/s at N = 4 against 774 in the device loop.
    if args.impl == "reference" or (world == 1 and args.gpus <= 1):
        pin_openmp_env()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", os.environ.get("MASTER_PORT", "29533"), os.path.abspath(__file__)] + sys.argv[1:]
        os.execv(sys.executable, cmd)
    run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
