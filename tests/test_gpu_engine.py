"""Device engine end to end on the GPU box.

* single process: ``ps.SGD`` / ``ps.Adam`` (device engine) vs ``torch.optim`` on the same gradients;
* 2-3 ranks sharing ONE GPU (gloo bootstrap; VMM fd exchange, peer pointers, epoch flags all real);
* ``multigpu``: one rank per GPU (multicast / NVLS paths).
"""
import os

import pytest
import torch

import pytorch_ps_mpi_b200 as ps
from pytorch_ps_mpi_b200.launch import spawn
from pytorch_ps_mpi_b200.models import mnist_mlp
from tests import _mp

pytestmark = pytest.mark.gpu
ONE_GPU = {"PSB200_PG_BACKEND": "gloo", "CUDA_VISIBLE_DEVICES": "0", "PSB200_DEVICE_TIMEOUT": "20"}


def _run(opt_factory, dtype=torch.float32, steps=4):
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    model = mnist_mlp(hidden=64).to(dev).to(dtype)
    opt = opt_factory(model)
    for s in range(steps):
        g = torch.Generator().manual_seed(s)
        x, y = torch.randn(8, 784, generator=g).to(dev).to(dtype), torch.randint(0, 10, (8,), generator=g).to(dev)
        opt.zero_grad()
        torch.nn.functional.cross_entropy(model(x).float(), y).backward()
        opt.step()
    torch.cuda.synchronize()
    return [p.detach().float().clone() for p in model.parameters()], opt


@pytest.mark.parametrize("hyper", [dict(lr=0.1), dict(lr=0.05, momentum=0.9, weight_decay=1e-3),
                                   dict(lr=0.05, momentum=0.9, nesterov=True)])
def test_device_sgd_matches_torch(hyper):
    a, opt = _run(lambda m: ps.SGD(m.named_parameters(), m.parameters(), code=ps.Identity(), engine="device", **hyper))
    assert opt._engine is not None and opt._engine.launches > 0
    b, _ = _run(lambda m: torch.optim.SGD(m.parameters(), **hyper))
    for p, q in zip(a, b):
        assert torch.allclose(p, q, rtol=1e-5, atol=1e-6)
    opt._engine.check()
    sd = opt.state_dict()
    if hyper.get("momentum"):
        assert all("momentum_buffer" in s for s in sd["state"].values())
    opt.close()


def test_device_adam_matches_host_engine():
    a, o1 = _run(lambda m: ps.Adam(m.named_parameters(), m.parameters(), lr=1e-3, engine="device"))
    b, o2 = _run(lambda m: ps.Adam(m.named_parameters(), m.parameters(), lr=1e-3, engine="host"))
    for p, q in zip(a, b):
        assert torch.allclose(p, q, rtol=1e-4, atol=1e-6)
    o1.close(), o2.close()


def test_device_bf16_master_weights():
    a, opt = _run(lambda m: ps.SGD(m.named_parameters(), m.parameters(), lr=0.05, momentum=0.9, engine="device"),
                  dtype=torch.bfloat16, steps=6)
    eng = opt._engine
    assert eng.master is not None and eng.master.dtype == torch.float32
    for s in eng.layout.slots:      # published bf16 parameter == round(master)
        m = eng.master[s.offset:s.offset + s.numel]
        assert torch.equal(m.to(torch.bfloat16), s.param.data.reshape(-1))
    opt.close()


def test_unused_parameter_is_skipped():
    dev = torch.device("cuda", 0)
    a = torch.nn.Parameter(torch.randn(3000, device=dev))
    b = torch.nn.Parameter(torch.randn(100, device=dev))
    opt = ps.SGD([("a", a), ("b", b)], [a, b], lr=0.1, weight_decay=0.5, engine="device")
    b0 = b.detach().clone()
    a0 = a.detach().clone()
    a.sum().backward()
    opt.step()
    torch.cuda.synchronize()
    assert torch.equal(b.detach(), b0)                       # p.grad is None → untouched (ps.py:178-179)
    assert torch.allclose(a.detach(), a0 - 0.1 * (1 + 0.5 * a0), rtol=1e-5, atol=1e-6)
    opt.close()


def test_channels_last_conv_weights_keep_layout():
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    conv = torch.nn.Conv2d(8, 16, 3, padding=1).to(dev).to(memory_format=torch.channels_last)
    ref = torch.nn.Conv2d(8, 16, 3, padding=1).to(dev).to(memory_format=torch.channels_last)
    ref.load_state_dict(conv.state_dict())
    opt = ps.SGD(conv.named_parameters(), conv.parameters(), lr=0.1, momentum=0.9, engine="device")
    ropt = torch.optim.SGD(ref.parameters(), lr=0.1, momentum=0.9)
    assert conv.weight.is_contiguous(memory_format=torch.channels_last)
    x = torch.randn(4, 8, 10, 10, device=dev).contiguous(memory_format=torch.channels_last)
    for _ in range(3):
        for m, o in ((conv, opt), (ref, ropt)):
            o.zero_grad()
            m(x).square().mean().backward()
            o.step()
    torch.cuda.synchronize()
    assert torch.allclose(conv.weight, ref.weight, rtol=1e-5, atol=1e-6)
    assert torch.allclose(conv.bias, ref.bias, rtol=1e-5, atol=1e-6)
    opt.close()


def test_symmetric_arena_two_ranks_one_gpu():
    spawn(_mp.symm_arena, 2, env=ONE_GPU, timeout=180)


@pytest.mark.parametrize("mode,optim,coding,dtype", [
    ("ps", "sgd", "identity", "fp32"), ("ps", "adam", "topk", "fp32"), ("allgather", "sgd", "scale", "fp32"),
    ("ps", "sgd", "cast", "bf16"),
])
def test_engine_two_ranks_one_gpu(mode, optim, coding, dtype):
    spawn(_mp.gpu_train, 2, (mode, optim, coding, dtype), env=ONE_GPU, timeout=240)


@pytest.mark.parametrize("mode,optim,coding,dtype", [("ps", "sgd", "identity", "fp32"), ("ps", "adam", "cast", "bf16"),
                                                      ("ps", "sgd", "topk", "bf16"), ("allgather", "sgd", "scale", "fp32"),
                                                      ("allgather", "adam", "topk", "fp32")])
def test_engine_pipelined_chunks_two_ranks_one_gpu(mode, optim, coding, dtype):
    """Per-chunk pipeline: 8 KB chunks split the 4-tensor MLP into several chunks (chunks hold whole parameters), each with
    its own encode launch, progress flag value and update launch (/root/reference/ps.py:140-148,159-162 per chunk)."""
    env = dict(ONE_GPU, PSB200_CHUNK_BYTES="8192", PSB200_EXPECT_CHUNKS="2")
    spawn(_mp.gpu_train, 2, (mode, optim, coding, dtype, "auto", 128), env=env, timeout=240)


def test_engine_unpipelined_two_ranks_one_gpu():
    spawn(_mp.gpu_train, 2, ("ps", "sgd", "identity", "bf16"), env=dict(ONE_GPU, PSB200_PIPELINE="0"), timeout=240)


def test_engine_three_ranks_allgather_one_gpu():
    spawn(_mp.gpu_train, 3, ("allgather", "adam", "identity", "fp32"), env=ONE_GPU, timeout=240)


def test_engine_async_one_gpu():
    spawn(_mp.gpu_async, 3, ("identity",), env=ONE_GPU, timeout=240)


def test_engine_async_consistent_reads_one_gpu():
    """consistent=True on the device engine: staging arena + sequence lock (README.md:79-81)."""
    spawn(_mp.gpu_async, 3, ("identity", 1), env=ONE_GPU, timeout=240)


@pytest.mark.multigpu
@pytest.mark.parametrize("mode,optim,coding,dtype", [("ps", "sgd", "identity", "fp32"), ("ps", "adam", "cast", "bf16"),
                                                      ("allgather", "sgd", "topk", "fp32")])
def test_engine_multi_gpu(mode, optim, coding, dtype):
    n = min(torch.cuda.device_count(), 4)
    spawn(_mp.gpu_train, n, (mode, optim, coding, dtype), env={"PSB200_DEVICE_TIMEOUT": "20"}, timeout=300)


@pytest.mark.multigpu
@pytest.mark.parametrize("reduce", ["auto", "p2p"])
def test_big_bf16_arena_multi_gpu(reduce):
    """>= 50 M-element bf16 arena, many chunks; auto = multimem.ld_reduce at N >= 4 (bf16 wire), p2p = rank-ordered pull."""
    n = min(torch.cuda.device_count(), 8)
    spawn(_mp.gpu_train_big, n, (reduce,), env={"PSB200_DEVICE_TIMEOUT": "30"}, timeout=420)


def test_checkpoint_resume_two_ranks_one_gpu():
    spawn(_mp.gpu_checkpoint, 2, env=ONE_GPU, timeout=240)


def test_dead_peer_times_out_one_gpu():
    spawn(_mp.gpu_dead_peer, 2, env=dict(ONE_GPU, PSB200_DEVICE_TIMEOUT="3"), timeout=120)


@pytest.mark.multigpu
def test_nvls_switch_reduce_multi_gpu():
    n = min(torch.cuda.device_count(), 4)
    spawn(_mp.gpu_train, n, ("ps", "sgd", "identity", "fp32", "nvls"), env={"PSB200_DEVICE_TIMEOUT": "20"}, timeout=300)
    spawn(_mp.gpu_train, n, ("allgather", "adam", "cast", "bf16", "nvls"), env={"PSB200_DEVICE_TIMEOUT": "20"}, timeout=300)


@pytest.mark.parametrize("pull", [0, 1])
def test_bcast_linear_gated_two_ranks_one_gpu(pull):
    spawn(_mp.gpu_bcast_linear, 2, (pull,), env=ONE_GPU, timeout=240)


@pytest.mark.multigpu
@pytest.mark.parametrize("pull", [0, 1])
def test_bcast_linear_gated_multi_gpu(pull):
    spawn(_mp.gpu_bcast_linear, 2, (pull,), env={"PSB200_DEVICE_TIMEOUT": "20"}, timeout=300)


@pytest.mark.multigpu
def test_async_multi_gpu():
    spawn(_mp.gpu_async, min(torch.cuda.device_count(), 4), ("topk",), env={"PSB200_DEVICE_TIMEOUT": "20"}, timeout=300)


def test_device_engine_with_lr_scheduler():
    def run(factory):
        dev = torch.device("cuda", 0)
        torch.manual_seed(0)
        model = mnist_mlp(hidden=32).to(dev)
        opt = factory(model)
        sched = torch.optim.lr_scheduler.StepLR(opt, step_size=2, gamma=0.5)
        for s in range(5):
            g = torch.Generator().manual_seed(s)
            x, y = torch.randn(8, 784, generator=g).to(dev), torch.randint(0, 10, (8,), generator=g).to(dev)
            opt.zero_grad()
            torch.nn.functional.cross_entropy(model(x), y).backward()
            opt.step()
            sched.step()
        torch.cuda.synchronize()
        return [p.detach().clone() for p in model.parameters()], opt

    a, o = run(lambda m: ps.SGD(m.named_parameters(), m.parameters(), lr=0.2, momentum=0.9, engine="device"))
    b, _ = run(lambda m: torch.optim.SGD(m.parameters(), lr=0.2, momentum=0.9))
    for p, q in zip(a, b):
        assert torch.allclose(p, q, rtol=1e-5, atol=1e-6)
    o.close()


def test_direct_gradient_placement_matches_encode_path(monkeypatch):
    """K10: producers we own (fused BN backward, stem implicit wgrad) write their gradients straight into the wire arena;
    the result must match the psb_encode_kernel copy path (the bytes placed are the same; the two RUNS differ in the last bit
    because BatchNorm statistics are summed with float atomics), and the encode batches must shrink."""
    from pytorch_ps_mpi_b200 import models

    def run(direct):
        monkeypatch.setenv("PSB200_DIRECT_GRAD", "1" if direct else "0")
        dev = torch.device("cuda", 0)
        torch.manual_seed(0)
        model = models.resnet18(num_classes=10).to(dev).to(memory_format=torch.channels_last).bfloat16()
        named = list(model.named_parameters())
        opt = ps.SGD(named, [p for _, p in named], lr=0.05, momentum=0.9, weight_decay=1e-4, engine="device")
        g = torch.Generator().manual_seed(1)
        x = torch.randn(8, 3, 64, 64, generator=g).to(dev).bfloat16().contiguous(memory_format=torch.channels_last)
        y = torch.randint(0, 10, (8,), generator=g).to(dev)
        for _ in range(1):           # ONE step: a randomly initialised ResNet at batch 8 is chaotic over several
            opt.zero_grad(set_to_none=True)
            torch.nn.functional.cross_entropy(model(x).float(), y).backward()
            opt.step()
        torch.cuda.synchronize()
        out = [p.detach().float().clone() for _, p in named]
        n_direct = opt._engine.direct_grads
        missing = [n for n, p in named if (".bn" in n or n.startswith("bn") or "downsample.1" in n or n == "conv1.weight")
                   and n not in opt._engine.direct_names]
        assert not direct or not missing, f"not placed directly: {missing}"
        opt.close()
        return out, n_direct

    a, na = run(True)
    a2, _ = run(True)
    b, nb = run(False)
    assert nb == 0 and na >= 41, (na, nb)          # 20 BN layers x (gamma, beta) + the stem weight
    # BatchNorm statistics are summed with float atomics, so two runs of the SAME path already differ in the last bits and a
    # randomly initialised ResNet at batch 8 amplifies that: the encode path must agree with the direct path as well as the
    # direct path agrees with itself.  Such a last-bit difference can flip the rounding of a bf16 parameter by one step even
    # where the two direct runs happened to round alike, so the floor is one bf16 step of the value (and at least 2e-3)
    half_eps = torch.finfo(torch.bfloat16).eps / 2
    for p, p2, q in zip(a, a2, b):
        noise = float((p - p2).abs().max())
        bf16_step = torch.ldexp(torch.full_like(p, half_eps), torch.frexp(p).exponent) * (p != 0)
        assert bool(((p - q).abs() <= 8.0 * noise + bf16_step.clamp(min=2e-3)).all()), (float((p - q).abs().max()), noise)


def test_stem_weight_lives_in_gemm_layout_in_the_arena():
    from pytorch_ps_mpi_b200 import models
    from pytorch_ps_mpi_b200.ops.stem import STEM_STRIDES, in_gemm_layout
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    model = models.resnet18(num_classes=10).to(dev).to(memory_format=torch.channels_last).bfloat16()
    ref = model.conv1.weight.detach().float().clone()
    named = list(model.named_parameters())
    opt = ps.SGD(named, [p for _, p in named], lr=0.0, engine="device")
    w = model.conv1.weight
    assert in_gemm_layout(w) and tuple(w.stride()) == STEM_STRIDES
    assert torch.equal(w.detach().float(), ref)                          # same logical values
    w2d = torch.as_strided(w.detach(), (64, 176), (176, 1))
    assert float(w2d[:, 168:].abs().max()) == 0.0                        # the K padding is zero
    assert float(w2d.reshape(64, 7 * 24 + 8)[:, :168].reshape(64, 7, 24)[:, :, 21:].abs().max()) == 0.0
    sd = opt.state_dict()
    opt.load_state_dict(sd)
    opt.close()
    assert torch.equal(model.conv1.weight.detach().float(), ref)


@pytest.mark.parametrize("optim", ["sgd", "adam"])
def test_late_parameter_keeps_its_own_step_count(optim):
    """ADVICE r1: optimizer state is per PARAMETER (ps.py:178-179,203-205,226-241) — a parameter whose first gradient
    arrives on step 3 starts its momentum with buf = d_p (dampening ignored) and Adam bias-corrects with ITS step count."""
    dev = torch.device("cuda", 0)

    def run(engine):
        torch.manual_seed(0)
        a = torch.nn.Parameter(torch.randn(5000, device=dev))
        b = torch.nn.Parameter(torch.randn(3000, device=dev))
        kw = dict(lr=0.1, momentum=0.9, dampening=0.5) if optim == "sgd" else dict(lr=0.05)
        cls = ps.SGD if optim == "sgd" else ps.Adam
        opt = cls([("a", a), ("b", b)], [a, b], engine=engine, **kw)
        for s in range(6):
            opt.zero_grad(set_to_none=True)
            loss = (a * (s + 1.0)).sum() + ((b * b).sum() * 0.5 if s >= 2 else 0.0)
            loss.backward()
            opt.step()
        torch.cuda.synchronize()
        sd = opt.state_dict()
        steps = [int(st["step"]) for st in sd["state"].values()] if engine == "device" else None
        out = a.detach().clone(), b.detach().clone()
        opt.close()
        return out, steps

    (a1, b1), steps = run("device")
    (a2, b2), _ = run("host")
    assert sorted(steps) == [4, 6], steps
    da, db = float((a1 - a2).abs().max()), float((b1 - b2).abs().max())
    assert torch.allclose(a1, a2, rtol=1e-4, atol=1e-5) and torch.allclose(b1, b2, rtol=1e-4, atol=1e-5), (da, db)
