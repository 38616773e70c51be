"""``bench.py``'s own ``main()`` — the file the driver runs at round end — executed on the CPU, at 1 and at 2 ranks.

Everything below ``bench.build()`` is the real code: world set-up, NUMA binding attempt, warm-up until stable (collective
decision), the device-timed arm with per-step events, the end-to-end arm with its static double-buffered inputs, the re-measure
rule, the cross-rank parameter digest, the clock summary and the JSON line.  The model is the package's ResNet cut down to one
stage on 32 x 32 images (``bench.build`` is replaced: the emulator is ~10^5 times slower than a B200), the engine and the fused ops
run over ``_psb200_emu`` (real bindings on emulated kernels, see ``test_model_integration_emulation.py``), ``torch.cuda`` events are
wall-clock fakes, ranks are threads."""
import contextlib
import json
import sys
import threading
import time

import pytest
import torch
import torch.distributed as dist

import pytorch_ps_mpi_b200 as ps
from pytorch_ps_mpi_b200 import runtime
from pytorch_ps_mpi_b200.ops import ext as ops_ext
from pytorch_ps_mpi_b200.parallel import device_engine as de
from tests import _cuda_emu
from tests import test_model_integration_emulation as MI
from tests import test_multirank_engine_emulation as H
from tests.test_device_engine_control_flow import FakeStream


class TimedEvent:
    """``torch.cuda.Event`` stand-in: launches execute synchronously here, so an event is the wall clock at ``record()``."""

    def __init__(self, *a, **k):
        self.t = None

    def record(self, stream=None):
        self.t = time.perf_counter()

    def query(self):
        return True

    def synchronize(self):
        pass

    def elapsed_time(self, other):
        return (other.t - self.t) * 1e3


def _build(args, device, ps_mod):
    from pytorch_ps_mpi_b200.ops.preprocess import normalize_nhwc
    model = MI._tiny_resnet()

    def make_batch(gen):
        return (torch.randint(0, 256, (args.batch, 3, 32, 32), dtype=torch.uint8, generator=gen),
                torch.randint(0, 10, (args.batch,), generator=gen))

    def loss_fn(x, y):
        return torch.nn.functional.cross_entropy(model(normalize_nhwc(x)).float(), y)

    return model, make_batch, loss_fn, {"global_batch": None, "image": "3x32x32 uint8 (CPU dry run)"}


@pytest.fixture
def bench_env(monkeypatch):
    extm = _cuda_emu.build_extension()
    if extm is None:
        pytest.skip("no g++")
    import bench
    nthreads = torch.get_num_threads()
    torch.set_num_threads(1)
    H._EXT = extm
    H._tls.world, H._tls.m = H.World(H.Cluster(extm.emu, 1), 0), None
    monkeypatch.setattr(bench, "build", _build)
    monkeypatch.setattr(runtime, "world", lambda: H._tls.world)
    monkeypatch.setattr(runtime, "init", lambda *a, **k: H._tls.world)
    monkeypatch.setattr(runtime, "shutdown", lambda: None)
    monkeypatch.setattr(ops_ext, "cuda", lambda: H._tls.m)
    monkeypatch.setattr(de, "SymmetricArena", H.SharedArena)
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "Stream", lambda *a, **k: FakeStream())
    monkeypatch.setattr(torch.cuda, "Event", TimedEvent)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: FakeStream())
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(torch.cuda, "stream", lambda s: contextlib.nullcontext())
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self, *a, **k: self)
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))

    def all_reduce(t, op=dist.ReduceOp.SUM, group=None):
        every = H._tls.world.all_gather_object(t.clone())
        red = {dist.ReduceOp.MAX: torch.maximum, dist.ReduceOp.MIN: torch.minimum, dist.ReduceOp.SUM: torch.add}[op]
        acc = every[0]
        for e in every[1:]:
            acc = red(acc, e)
        t.copy_(acc)

    monkeypatch.setattr(dist, "all_reduce", all_reduce)
    monkeypatch.setenv("PSB200_CHUNK_BYTES", str(2048 * 2 * 8))
    yield bench, extm
    H._EXT = None
    torch.set_num_threads(nthreads)


def _run_bench(bench, extm, n, argv, monkeypatch, capsys):
    monkeypatch.setattr(sys, "argv", ["bench.py", "--gpus", str(n)] + argv)
    cluster = H.Cluster(extm.emu, n)
    rcs, errs = [None] * n, []

    def main(rank):
        w = H.World(cluster, rank)
        w.cpu_group = None
        H._tls.world, H._tls.m = w, MI.ModelM(cluster, extm)
        try:
            rcs[rank] = bench.main()
        except BaseException as exc:       # noqa: BLE001
            errs.append(exc)
            cluster.fail(exc)

    ts = [threading.Thread(target=main, args=(r,), daemon=True) for r in range(n)]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=900)
    assert not any(t.is_alive() for t in ts), "a rank thread is stuck"
    if errs:
        real = [e for e in errs if "another rank" not in str(e) and not isinstance(e, threading.BrokenBarrierError)]
        raise (real or errs)[0]
    assert rcs == [0] * n
    cap = capsys.readouterr()
    lines = [ln for ln in cap.out.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, lines                      # rank 0 prints ONE JSON line
    out = json.loads(lines[0])
    out["_stderr"] = cap.err
    return out


CONTRACT = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "clocks", "e2e", "gpu_launches"]


@pytest.mark.parametrize("n", [1, 2])
def test_bench_main_runs_end_to_end_on_the_emulator(bench_env, monkeypatch, capsys, n):
    bench, extm = bench_env
    K = 2
    out = _run_bench(bench, extm, n, ["--steps", str(K), "--warmup", "3", "--batch", "2", "--no-comparators"], monkeypatch, capsys)
    for key in CONTRACT:
        assert key in out, key
    assert out["n_gpus"] == n and out["steps"] == K and out["warmup"] >= 3 and out["higher_is_better"] and out["scaling"] == "weak"
    assert out["dtype"] == "bf16" and out["impl"] == "ours" and out["unit"] == "samples/sec"
    cfg = out["config"]
    assert cfg["model"] == "resnet18" and cfg["global_batch"] == 2 * n and cfg["bcast_gemm"] == "gate"
    assert cfg["worker_wait_kernel"] is False and cfg["update_pipeline_chunks"] >= 2 and "numa_bind" in cfg
    assert out["value"] > 0 and abs(out["value"] - 2 * n * K / (out["ms_per_step"] * K / 1e3)) < 1e-6 * out["value"]
    e2e = out["e2e"]
    assert e2e["inputs"] == "static double buffer" and e2e["h2d_bytes_per_step"] == 2 * 3 * 32 * 32 + 2 * 8
    assert e2e["d2h_bytes_per_step"] == 4 and e2e["value"] > 0 and e2e["last_loss"] == e2e["last_loss"]       # not NaN
    assert out["gpu_launches"] > 10 * K                                   # our kernels inside the timed region, counted in C++
    assert out["check"] == {"params_bit_identical_across_ranks": True, "params_finite": True, "ranks": n}
    assert set(out["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"} and len(out["value_runs_ms"]) in (1, 2)
    assert out["warmup_total_steps"] >= 5 and set(out["step_ms"]) >= {"median", "p90", "min", "max"}


@pytest.mark.parametrize("extra,expect", [
    (["--mode", "async"], dict(mode="async", contributors=1)),
    (["--code", "topk:0.25", "--optim", "adam"], dict(coding="topk:0.25", optimizer="adam")),
    (["--mode", "allgather", "--code", "scale:int8", "--no-pipeline"], dict(coding="scale:int8"))])
def test_bench_other_configurations_at_two_ranks(bench_env, monkeypatch, capsys, extra, expect):
    """The other BASELINE configurations through the same ``main()``: AsySG-InCon (rank 0 only serves; throughput counts the
    workers), a top-k coded wire with Adam, all-gather with an int8 wire and the unpipelined update."""
    bench, extm = bench_env
    out = _run_bench(bench, extm, 2, ["--steps", "2", "--warmup", "3", "--batch", "2", "--no-comparators"] + extra, monkeypatch, capsys)
    cfg = out["config"]
    assert out["value"] > 0 and out["e2e"]["value"] > 0 and out["gpu_launches"] > 0
    if "mode" in expect:
        assert expect["mode"] in cfg["parallelism"] and cfg["global_batch"] == 2 * expect["contributors"] and out["check"] is None
    else:
        assert out["check"]["params_bit_identical_across_ranks"] and out["check"]["params_finite"]
    for k in ("coding", "optimizer"):
        if k in expect:
            assert cfg[k] == expect[k]
    if "--no-pipeline" in extra:
        assert cfg["update_pipeline_chunks"] == 1


def test_bench_profile_flag_reports_device_spans(bench_env, monkeypatch, capsys):
    """``--profile``: the engine's CUDA-event spans (``dev_step_tail_time``, ``dev_gather_update_bcast_time``,
    ``dev_update_pipeline_time``: read one step late, never a sync) reach ``opt.timings`` and the per-rank stderr line."""
    bench, extm = bench_env
    monkeypatch.setattr(sys, "argv", ["bench.py"])
    out = _run_bench(bench, extm, 2, ["--steps", "2", "--warmup", "3", "--batch", "2", "--no-comparators", "--profile"], monkeypatch, capsys)
    assert out["value"] > 0
    spans = [ln for ln in out["_stderr"].splitlines() if ln.startswith("[rank ")]
    assert len(spans) == 2 and all("dev_step_tail_time=" in ln for ln in spans), out["_stderr"][-500:]
    assert any("dev_gather_update_bcast_time=" in ln and "dev_update_pipeline_time=" in ln for ln in spans)     # the server


def test_bench_with_same_invocation_comparators(bench_env, monkeypatch, capsys):
    """The comparator block (NCCL-PS and the stock-tools reference-equivalent path, ``baseline/comparator.py``) after the headline:
    whatever happens in it — here NCCL cannot exist — the headline line is still printed, with a value or an error per comparator."""
    bench, extm = bench_env
    out = _run_bench(bench, extm, 1, ["--steps", "2", "--warmup", "3", "--batch", "2"], monkeypatch, capsys)
    assert out["value"] > 0 and set(out["comparators"]) == {"nccl", "host"}
    for kind, c in out["comparators"].items():
        assert ("value" in c and c["value"] > 0) or "error" in c, (kind, c)
    assert all(k in out["comparators"] and "value" in out["comparators"][k] for k in (out["vs_comparator"] or {}))


def test_bench_dump_outputs_do_not_depend_on_the_timed_steps(bench_env, monkeypatch, capsys, tmp_path):
    """``--dump-outputs``: the timed step once more, from the start state, on the last timed step's batch; its loss, parameters
    and buffers as float32 ``.npy`` files.  Runs whose last timed batch is the same (2 and 6 steps over 4 rotating batches) write
    the same arrays, whatever the timed, warm-up and comparator steps did before (the emulated kernels are deterministic)."""
    import numpy as np
    bench, extm = bench_env
    runs = []
    for k, (steps, extra) in enumerate(((2, ["--no-comparators"]), (6, []))):       # the second run also trains the comparators
        d = tmp_path / str(k)
        out = _run_bench(bench, extm, 1, ["--steps", str(steps), "--warmup", "3", "--batch", "2", "--no-e2e",
                                          "--dump-outputs", str(d)] + extra, monkeypatch, capsys)
        assert out["steps"] == steps
        runs.append({name: np.load(d / f"{name}.npy") for name in ("loss", "params", "buffers")})
    model = MI._tiny_resnet()
    assert runs[0]["loss"].shape == (1,)
    assert runs[0]["params"].shape == (sum(p.numel() for p in model.parameters()),)
    assert runs[0]["buffers"].shape == (sum(b.numel() for b in model.buffers() if b.is_floating_point()),)
    for name, a in runs[0].items():
        assert a.dtype == np.float32 and np.isfinite(a).all(), name
        np.testing.assert_array_equal(a, runs[1][name], err_msg=name)
    assert not np.array_equal(runs[0]["params"], torch.cat([p.detach().reshape(-1).float() for p in model.parameters()]).numpy())


def test_bench_rejects_fewer_than_one_step(monkeypatch):
    import bench
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "0"])
    with pytest.raises(SystemExit):
        bench.parse()


def test_bench_reference_arm_reports_unavailable(monkeypatch, capsys):
    import bench
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--gpus", "1"])
    assert bench.main() == 0
    out = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert out["impl"] == "reference" and "unavailable" in out
