"""CPU: bench.run_gpu's control flow with every GPU-touching piece replaced by a stand-in -- the bench line's objects (roofline with
the GEMM and quantizer objects nested where the driver keeps them, cpu_baseline, clocks, e2e), the launch count and the watchdog /
emit path are assembled by the real code.  (The numbers are fake; this guards the plumbing.)  Also the CPU reference arm's own
logic: steps of 1/32 token, pinned team, stability verdict."""
import argparse
import json
import os
import types

import numpy as np
import pytest
import torch

import bench
from hqq_b200 import harness


class FakeGraph:
    """A replay counts the steps: step n produces token n and logits filled with n."""
    def __init__(self, model):
        self.model = model

    def replay(self):
        m = self.model
        m.replays += 1
        m.next_tok.fill_(m.replays)
        m._bufs["logits"].fill_(m.replays)


class FakeModel:
    built = []

    def __init__(self, shape, **kw):
        self.kw, self.shape = kw, shape
        self.device, self.dtype, self.nbits, self.tp_mode = torch.device("cpu"), torch.float16, 4, "p2p"
        B = kw.get("batch", 1)
        self.tok, self.pos, self.next_tok = torch.zeros(B, dtype=torch.long), torch.zeros(1, dtype=torch.long), torch.zeros(B, dtype=torch.long)
        self._bufs, self.replays = {"logits": torch.zeros(B, 8, dtype=torch.float16)}, 0
        self.graph, self.blocks = FakeGraph(self), []
        FakeModel.built.append(self)

    def capture(self, warmup=3):
        return self.graph

    def reset_state(self, token=1):
        pass

    def decode(self, feed_back=True):
        self.graph.replay()

    def bytes_per_token(self):
        return 4.98e9


class FakeEvent:
    def __init__(self, enable_timing=True):
        pass

    def record(self, stream=None):
        pass

    def elapsed_time(self, other):
        return 400.0


class FakeStream:
    cuda_stream = 0

    def synchronize(self):
        pass


@pytest.fixture
def fake_gpu(monkeypatch):
    FakeModel.built.clear()
    monkeypatch.setattr(harness, "DecodeModel", FakeModel)
    monkeypatch.setattr(torch.cuda, "set_device", lambda d: None)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda d=None: FakeStream())
    monkeypatch.setattr(torch.cuda, "Event", FakeEvent)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda d=None: None)
    monkeypatch.setattr(torch.cuda, "empty_cache", lambda: None)
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self: self)
    monkeypatch.setattr(bench, "ClockSampler", lambda i: types.SimpleNamespace(start=lambda: None, stop=lambda: {"sm_mhz": 1900.0, "sm_max_mhz": 1965.0, "reasons": []}))
    monkeypatch.setattr(bench, "kernel_roofline", lambda model, torch_, peaks: {"bound": "hbm", "achieved": 3000.0, "peak": peaks["hbm_gbs"], "frac": 0.45})
    monkeypatch.setattr(bench, "quantizer_roofline", lambda torch_, peaks, dev, reps=3: {"ms_per_block": 1.5, "frac": 0.07})
    monkeypatch.setattr(bench, "gemm_sweep", lambda torch_, peaks, dev, quick=False: {"bound": "tensor", "achieved": 1300.0, "peak": peaks["tensor_tflops"],
                                                                                      "frac": 1300.0 / peaks["tensor_tflops"], "shape": "fake"})
    monkeypatch.setattr(bench, "cpu_quantizer_baseline", lambda: {"value": 0.01, "unit": "Gweights/s", "cores": 8, "kind": "port"})

    class FakeRef:
        def run(self, steps, warmup, budget_s):
            return 0.3, {"cores": 8, "sample": "fake", "port": "fake", "tokens_per_s_min_median_max": [0.29, 0.3, 0.31], "stable": True, "steps_timed": steps}

    monkeypatch.setattr(bench, "CpuReference", FakeRef)


def _args(**kw):
    d = dict(gpus=1, steps=20, warmup=3, impl="hqq_b200", cache_len=0, layers=0, no_cpu_baseline=False, no_extras=False, quick_extras=False,
             no_token_check=False, extras_deadline=60.0, batch=1, model="8b", dump_outputs=None)
    d.update(kw)
    return argparse.Namespace(**d)


def test_run_gpu_assembles_one_line_with_the_nested_objects(fake_gpu, capsys):
    bench.run_gpu(_args(), 0, 1, 0)
    out = [ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")]
    assert len(out) == 1  # the contract: rank 0 prints ONE JSON line
    d = json.loads(out[0])
    assert d["metric"] == bench.METRIC and d["n_gpus"] == 1 and d["steps"] == 20 and d["higher_is_better"] is True
    assert d["value"] == pytest.approx(20 / 0.4) and d["e2e"]["value"] == pytest.approx(20 / 0.4)
    assert d["e2e"]["h2d_bytes_per_step"] == 8 and d["e2e"]["d2h_bytes_per_step"] == 8
    # the GEMM roofline (second half of BASELINE's metric) and the quantizer live inside `roofline`, which the driver keeps
    assert d["roofline"]["frac"] == 0.45 and d["roofline"]["gemm"]["frac"] == pytest.approx(1300.0 / d["roofline"]["gemm"]["peak"])
    assert d["roofline"]["quantizer"]["ms_per_block"] == 1.5 and d["roofline"]["quantizer"]["cpu_baseline"]["kind"] == "port"
    assert d["cpu_baseline"]["cores"] == 8 and d["cpu_baseline"]["stable"] is True and d["clocks"]["reasons"] == []
    assert d["config"]["workload"] == bench.WORKLOAD and d["config"]["tp_mode"] is None and d["config"]["tokens_agree"] is None
    assert "autotune" not in d["config"] and "experimental" not in d


def test_run_gpu_without_extras(fake_gpu, capsys):
    bench.run_gpu(_args(no_extras=True), 0, 1, 0)
    d = json.loads([ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")][-1])
    assert "gemm" not in d["roofline"] and "cpu_baseline" not in d and d["value"] > 0


def test_run_gpu_keeps_the_line_when_an_extra_object_fails(fake_gpu, capsys, monkeypatch):
    def boom(*a, **k):
        raise RuntimeError("sweep failed")

    monkeypatch.setattr(bench, "gemm_sweep", boom)
    bench.run_gpu(_args(no_cpu_baseline=True), 0, 1, 0)
    d = json.loads([ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")][-1])
    assert "sweep failed" in d["roofline"]["gemm"]["error"] and d["value"] > 0 and d["roofline"]["quantizer"]["ms_per_block"] == 1.5


def test_dump_outputs_holds_the_last_timed_step(fake_gpu, capsys, tmp_path, monkeypatch):
    """3 warm-up + 20 timed steps in the device loop: the dump is step 23, not what the end-to-end loop replays after it."""
    out = tmp_path / "dump"
    bench.run_gpu(_args(no_extras=True, dump_outputs=str(out)), 0, 1, 0)
    tok, logits = np.load(out / "next_token.npy"), np.load(out / "logits.npy")
    assert tok.dtype == np.float64 and tok.tolist() == [23.0]
    assert logits.dtype == np.float32 and logits.shape == (1, 8) and (logits == 23.0).all()
    assert FakeModel.built[-1].replays > 23
    # above the size limit only the first sequences of the batch are kept
    monkeypatch.setattr(bench, "DUMP_BYTES", 2 * 4 * 8)
    bench.run_gpu(_args(no_extras=True, dump_outputs=str(out), batch=3), 0, 1, 0)
    assert np.load(out / "next_token.npy").shape == (2,) and np.load(out / "logits.npy").shape == (2, 8)


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects_arguments_it_cannot_honour(monkeypatch, argv):
    import sys
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    monkeypatch.setattr(bench, "run_gpu", lambda *a: pytest.fail("ran"))
    monkeypatch.setattr(bench, "run_reference", lambda *a: pytest.fail("ran"))
    with pytest.raises(SystemExit):
        bench.main()


def test_host_topology_and_the_reference_step(monkeypatch):
    per_socket, sockets, logical = bench.host_topology()
    assert per_socket >= 1 and sockets >= 1 and logical >= per_socket

    class Tiny(bench.CpuReference):  # the arithmetic of run() without the 0.1 s-per-step workload
        def __init__(self):
            self.cores, self.label, self.n = 4, "tiny", 0

        def step(self):
            self.n += 1

        def lm_share_s(self, reps=5):
            return 1e-6

    r = Tiny()
    v, info = r.run(steps=25, warmup=2, budget_s=10.0)
    assert r.n == 27 and info["steps_timed"] == 25 and v > 0 and len(info["tokens_per_s_min_median_max"]) == 3
    lo, med, hi = info["tokens_per_s_min_median_max"]
    assert lo <= med <= hi and isinstance(info["stable"], bool) and "1/32" in info["sample"]


def test_openmp_pinning_stays_out_of_multi_rank_gpu_runs(monkeypatch):
    """OMP_PLACES / OMP_PROC_BIND belong to the CPU legs: in a torchrun GPU run they would bind every rank's host thread to core 0
    (libgomp binds the initial thread to the first place) and the per-step host sync of the e2e loop would time-slice the ranks."""
    import sys
    seen = {}
    monkeypatch.setenv("OMP_PLACES", "x")      # so that monkeypatch restores both variables to their state before this test
    monkeypatch.setenv("OMP_PROC_BIND", "x")
    monkeypatch.setattr(bench, "run_gpu", lambda args, rank, world, lr: seen.update(gpu=(world, os.environ.get("OMP_PLACES"))))
    monkeypatch.setattr(bench, "run_reference", lambda args, rank, world: seen.update(ref=(world, os.environ.get("OMP_PLACES"))))
    for env_world, argv, key, want in (("2", ["bench.py", "--gpus", "2"], "gpu", None), ("1", ["bench.py"], "gpu", "cores"),
                                       ("2", ["bench.py", "--impl", "reference", "--gpus", "2"], "ref", "cores")):
        monkeypatch.delenv("OMP_PLACES", raising=False)
        monkeypatch.delenv("OMP_PROC_BIND", raising=False)
        monkeypatch.setenv("WORLD_SIZE", env_world)
        monkeypatch.setenv("RANK", "0")
        monkeypatch.setattr(sys, "argv", argv)
        bench.main()
        assert seen[key] == (int(env_world), want), (argv, seen)
