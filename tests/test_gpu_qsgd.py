"""Block-wise QSGD on a B200: the ``KIND_QSGD`` encode kernel byte for byte against ``codings.qsgd_blockwise`` (computed with
the kernel's Philox keys), the fused gather-update kernel over 1 / 3 / 8 virtual ranks, and the device engine with two ranks on
one GPU in ``ps`` and ``allgather`` mode against the grad-gather oracle."""
import pytest
import torch

import pytorch_ps_mpi_b200 as ps
from pytorch_ps_mpi_b200.codings import KIND_QSGD, TILE, qsgd_blockwise, qsgd_uniform16
from pytorch_ps_mpi_b200.launch import spawn
from tests.test_gpu_kernels import Virtual, sgd_h

pytestmark = pytest.mark.gpu
SEED = 0x5EED_0000_1234_ABCD
ONE_GPU = {"PSB200_PG_BACKEND": "gloo", "CUDA_VISIBLE_DEVICES": "0", "PSB200_DEVICE_TIMEOUT": "20"}
SHAPES = [(TILE + 9,), (60, 41), (TILE,), (TILE + 100,), (300, 41), (3, 3, 16, 32)]


class VirtualQSGD(Virtual):
    def encode(self, r, grads, step=0):
        L = self.L
        order = [(L.by_id[id(p)], g) for p, g in zip(self.params, grads)]
        self.m.encode(self.kind, self.wire, [g.contiguous() for _, g in order], [s.first_tile for s, _ in order],
                      [s.ntiles for s, _ in order], [s.index for s, _ in order], self.tiles.data_ptr(),
                      self.wires[r].data_ptr(), self.scales[r].data_ptr(), self.amax.data_ptr(), 0, self.bpt, self.cap,
                      1.0, levels=self.spec.levels, seed=self.spec.seed, rng_step=step, rank=r)


def _expect_slots(V, grads, rank, step):
    out = torch.zeros(V.L.ntiles, V.bpt, dtype=torch.uint8, device=V.dev)
    for p, g in zip(V.params, grads):
        s = V.L.by_id[id(p)]
        u = qsgd_uniform16(SEED, rank, step, s.offset, s.ntiles * TILE, device=V.dev)
        q, sc = qsgd_blockwise(g.reshape(-1), V.spec.levels, u)
        out[s.first_tile: s.first_tile + s.ntiles, :TILE] = q.view(torch.uint8).view(s.ntiles, TILE)
        out[s.first_tile: s.first_tile + s.ntiles, TILE:TILE + 4] = sc.view(torch.uint8).view(s.ntiles, 4)
    return out


def _grads(shapes, dtype, rank, dev, specials=False):
    gs = [torch.randn(s, device=dev) * (1 + rank) for s in shapes]
    if specials:                                   # an all-zero tile; tiles holding inf / nan travel as zeros
        gs[2] = torch.zeros(shapes[2], device=dev)
        gs[3][5] = float("inf")
        gs[3][TILE + 7] = float("nan")
    return [g.to(dtype) for g in gs]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("levels", [127, 5])
def test_encode_is_bit_exact(dtype, levels):
    torch.manual_seed(0)
    V = VirtualQSGD(SHAPES, dtype, ps.QSGD(levels=levels, blockwise=True, seed=SEED), 1)
    grads = _grads(SHAPES, dtype, 0, V.dev, specials=True)
    V.encode(0, grads, step=7)
    torch.cuda.synchronize()
    got = V.wires[0].view(V.L.ntiles, V.bpt)
    want = _expect_slots(V, grads, 0, 7)
    assert torch.equal(got, want), int((got != want).sum())


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("nranks", [1, 3, 8])
def test_encode_gather_sgd(dtype, nranks):
    torch.manual_seed(0)
    shapes = [(300, 41), (5000,), (64,), (3, 3, 16, 32), (TILE * 2,)]
    code = ps.QSGD(levels=127, blockwise=True, seed=SEED)
    V = VirtualQSGD(shapes, dtype, code, nranks, master=True)
    assert V.kind == KIND_QSGD
    w0 = [p.data.float().clone() for p in V.params]
    grads = [_grads(shapes, dtype, r, V.dev) for r in range(nranks)]
    for r in range(nranks):
        V.encode(r, grads[r], step=3)
    torch.cuda.synchronize()
    for r in range(nranks):
        assert torch.equal(V.wires[r].view(V.L.ntiles, V.bpt), _expect_slots(V, grads[r], r, 3))
    V.update(1, [sgd_h(lr=0.5)])
    for i, p in enumerate(V.params):
        first = V.L.by_id[id(p)].offset
        tot = torch.zeros(shapes[i], device=V.dev)
        for r in range(nranks):
            tot = tot + code.decode(code.encode(grads[r][i], rank=r, step=3, first_elem=first))
        want = (w0[i] - 0.5 * tot).to(dtype)
        for r in range(nranks):
            got = V.param_values(r)[i]
            tol = 1e-5 if dtype == torch.float32 else 1e-2
            assert torch.allclose(got.float(), want.float(), rtol=tol, atol=tol), float((got.float() - want.float()).abs().max())


def gpu_train_qsgd(rank, size, mode, optim, dtype_name):
    """Device engine with block-wise QSGD, one process per rank: every rank's actual gradients are gathered, coded with the
    engine's keys (seed, rank, step, arena offset), summed in rank order and fed to the reference optimizer on fp32 CPU
    shadows; the server's master weights must match and the ranks must agree bit for bit."""
    from pytorch_ps_mpi_b200.models import mnist_mlp
    from tests._mp import _host_oracle, _mlp_data, _world
    ps_, w = _world(rank, size)
    dev = w.device
    dtype = {"fp32": torch.float32, "bf16": torch.bfloat16}[dtype_name]
    hyper = {"lr": 0.05, "momentum": 0.9, "weight_decay": 1e-4} if optim == "sgd" else {"lr": 1e-2, "eps": 1e-8}
    torch.manual_seed(0)
    model = mnist_mlp(hidden=32).to(dev).to(dtype)
    shadow, oracle, groups = _host_oracle(ps_, model, optim, hyper)
    cls = ps_.SGD if optim == "sgd" else ps_.Adam
    opt = cls(model.named_parameters(), model.parameters(), code=ps_.QSGD(levels=31, blockwise=True, seed=SEED), mode=mode,
              engine="device", **hyper)
    eng = opt._engine
    assert eng is not None and eng.kind == KIND_QSGD
    first = [eng.layout.by_id[id(p)].offset for p in model.parameters()]
    code = ps_.QSGD(levels=31, blockwise=True, seed=SEED)
    for s in range(3):
        x, y = _mlp_data(rank, s)
        opt.zero_grad()
        torch.nn.functional.cross_entropy(model(x.to(dev).to(dtype)).float(), y.to(dev)).backward()
        mine = [p.grad.detach().cpu() for p in model.parameters()]
        opt.step()
        allg = w.all_gather_object(mine)
        with torch.no_grad():
            for i, q in enumerate(shadow):
                total = torch.zeros_like(q)
                for r in range(size):
                    total += code.decode(code.encode(allg[r][i], rank=r, step=s, first_elem=first[i])).reshape(q.shape)
                oracle.optim_step(q, total, **oracle._hyper(groups[id(q)]))
    eng.check()
    torch.cuda.synchronize()
    flat = torch.cat([p.detach().float().reshape(-1) for p in model.parameters()]).cpu()
    allp = w.all_gather_object(flat)
    for f in allp:
        assert torch.equal(f, allp[0]), "ranks diverged"
    if eng.is_server:
        for p, q in zip(model.parameters(), shadow):
            got = (opt.state[p]["master_param"] if eng.master is not None else p).detach().float().cpu()
            assert torch.allclose(got, q.detach(), rtol=2e-4, atol=2e-5), (mode, optim, dtype_name, float((got - q).abs().max()))
    opt.close()


@pytest.mark.parametrize("mode,optim,dtype", [("ps", "sgd", "fp32"), ("allgather", "adam", "bf16"), ("ps", "adam", "bf16"),
                                              ("allgather", "sgd", "fp32")])
def test_engine_two_ranks_one_gpu(mode, optim, dtype):
    spawn(gpu_train_qsgd, 2, (mode, optim, dtype), env=ONE_GPU, timeout=240)
