"""Block-wise QSGD (``QSGD(blockwise=True)``, ``KIND_QSGD``) on the CPU: the Philox stream against its known-answer vectors, the
``psb_encode_kernel`` QSGD branch (compiled from ``ps_kernels.cu`` by ``tests/_cuda_emu.py``) byte for byte against
``codings.qsgd_blockwise``, the fused gather-update kernel over virtual ranks, the coding's statistics, and the real device engine
(``bindings.cpp`` linked against the emulated kernels) at 2-3 ranks in every mode, through checkpoint/resume and ``recover()``."""
import contextlib
import copy
import ctypes
import math
import time

import pytest
import torch

import pytorch_ps_mpi_b200 as ps
from pytorch_ps_mpi_b200 import runtime
from pytorch_ps_mpi_b200.codings import KIND_QSGD, TILE, WIRE_I8, qsgd_blockwise, qsgd_uniform16
from pytorch_ps_mpi_b200.parallel import device_engine as de
from tests import _cuda_emu
from tests import test_multirank_engine_emulation as mr
from tests.test_device_engine_control_flow import FakeEvent, FakeStream
from tests.test_ps_kernels_cpu_emulation import VirtualCPU, sgd_h

SEED = 0x5EED_0000_1234_ABCD


@pytest.fixture(autouse=True)
def _single_threaded_torch():
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


# The emulated kernels with one addition to the driver: ``emu_encode_extra(levels, seed, step, rank)`` sets the QSGD arguments of
# the next ``emu_encode`` call (the driver's own ``emu_encode`` leaves them zero), so ``VirtualCPU`` drives the QSGD encode unchanged.
_EXTRA_DECL = """
static int emu_q_levels = 0; static uint64_t emu_q_seed = 0; static uint32_t emu_q_step = 0; static int emu_q_rank = 0;
extern "C" void emu_encode_extra(int levels, uint64_t seed, uint32_t step, int rank) {
  emu_q_levels = levels; emu_q_seed = seed; emu_q_step = step; emu_q_rank = rank;
}
"""
_EXTRA_USE = """  a.levels = emu_q_levels; a.seed = emu_q_seed; a.rng_step = emu_q_step; a.rank = emu_q_rank;
  emu_q_levels = 0; emu_q_seed = 0; emu_q_step = 0; emu_q_rank = 0;
"""


@pytest.fixture(scope="module")
def lib():
    import shutil
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    src = _cuda_emu.kernel_source()
    head, use = 'extern "C" int emu_encode(', "  if (kind == KIND_SCALED) psb_launch_absmax(nullptr, a);\n"
    assert src.count(head) == 1 and src.count(use) == 1
    src = src.replace(head, _EXTRA_DECL + head).replace(use, _EXTRA_USE + use)
    return _cuda_emu.compile_shared(src, "psb_emu_qsgd_")


def _words(u):
    u = [int(x) for x in u]
    return [u[2 * i] | u[2 * i + 1] << 16 for i in range(4)]


def test_philox_known_answers():
    """Philox4x32-10 known-answer vectors (Random123): counter = (group lo, group hi, step, rank), key = seed."""
    assert _words(qsgd_uniform16(0, 0, 0, 0, 8)) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert _words(qsgd_uniform16((1 << 64) - 1, 0xffffffff, 0xffffffff, 8 * ((1 << 64) - 1), 8)) == \
        [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert _words(qsgd_uniform16(0x299f31d0a4093822, 0x03707344, 0x13198a2e, 8 * (0x85a308d3 << 32 | 0x243f6a88), 8)) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]
    # an element range that starts inside a group and crosses the 2**32 group boundary is a slice of the aligned stream
    a = qsgd_uniform16(SEED, 1, 2, 8 * ((1 << 32) - 1) + 3, 10)
    b = qsgd_uniform16(SEED, 1, 2, 8 * ((1 << 32) - 1), 16)
    assert torch.equal(a, b[3:13])


def test_spec_and_validation():
    c = ps.QSGD(levels=127, blockwise=True, seed=5)
    spec = c.device_spec()
    assert (spec.kind, spec.wire, spec.levels, spec.seed) == (KIND_QSGD, WIRE_I8, 127, 5)
    assert spec.bytes_per_tile(torch.bfloat16) == TILE + 16 and spec.tile_capacity() == TILE
    with pytest.raises(ValueError):
        ps.QSGD(levels=200, blockwise=True)
    with pytest.raises(ValueError):
        ps.QSGD(levels=0, blockwise=True)
    assert ps.QSGD().device_spec() is None and ps.QSGD(levels=15).device_spec() is None    # per-tensor QSGD: host engine
    torch.manual_seed(3)
    s1 = ps.QSGD(blockwise=True, levels=8).seed
    torch.manual_seed(3)
    assert ps.QSGD(blockwise=True, levels=8).seed == s1 and 0 <= s1 < 1 << 64                # drawn from torch's CPU generator


def _wire_slots(V, r):
    nt = V.L.ntiles
    return V.wires[r][: nt * V.bpt].view(nt, V.bpt)


def _expect_slots(V, grads, levels, rank, step):
    """Every wire byte of every parameter, from the Python oracle with the kernel's keys."""
    out = torch.zeros(V.L.ntiles, V.bpt, dtype=torch.uint8)
    for p, g in zip(V.params, grads):
        s = V.L.by_id[id(p)]
        u = qsgd_uniform16(SEED, rank, step, s.offset, s.ntiles * TILE)
        q, sc = qsgd_blockwise(g.reshape(-1), levels, u)
        out[s.first_tile: s.first_tile + s.ntiles, :TILE] = q.view(torch.uint8).view(s.ntiles, TILE)
        out[s.first_tile: s.first_tile + s.ntiles, TILE:TILE + 4] = sc.view(torch.uint8).view(s.ntiles, 4)
    return out


def _encode(lib, V, r, grads, levels, step):
    lib.emu_encode_extra(levels, ctypes.c_uint64(SEED), ctypes.c_uint32(step), r)
    V.encode(r, grads)


SHAPES = [(TILE + 9,), (60, 41), (TILE,), (TILE + 100,)]


def _grads(dtype, rank=0):
    torch.manual_seed(10 + rank)
    gs = [torch.randn(s) * (1 + rank) for s in SHAPES]
    gs[2] = torch.zeros(SHAPES[2])                  # an all-zero tile
    gs[3][5] = float("inf")                         # tile 0: inf, tile 1: nan → both travel as zeros
    gs[3][TILE + 7] = float("nan")
    return [g.to(dtype) for g in gs]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("levels", [127, 5])
def test_encode_is_bit_exact(lib, dtype, levels):
    V = VirtualCPU(lib, SHAPES, dtype, ps.QSGD(levels=levels, blockwise=True, seed=SEED), 1)
    grads = _grads(dtype)
    _encode(lib, V, 0, grads, levels, step=7)
    got, want = _wire_slots(V, 0), _expect_slots(V, grads, levels, 0, 7)
    assert torch.equal(got, want), int((got != want).sum())
    s3 = V.L.by_id[id(V.params[3])]
    assert not _wire_slots(V, 0)[s3.first_tile: s3.first_tile + 2].any()       # non-finite tiles: q = 0, scale = 0
    assert not _wire_slots(V, 0)[V.L.by_id[id(V.params[2])].first_tile].any()   # zero tile


@pytest.mark.parametrize("nranks", [1, 3])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_encode_gather_sgd(lib, nranks, dtype):
    levels, step = 127, 3
    torch.manual_seed(0)
    shapes = SHAPES[:2] + [(64,)]
    V = VirtualCPU(lib, shapes, dtype, ps.QSGD(levels=levels, blockwise=True, seed=SEED), nranks)
    w0 = [p.data.float().clone() for p in V.params]
    grads = [[(torch.randn(s) * (1 + r)).to(dtype) for s in shapes] for r in range(nranks)]
    for r in range(nranks):
        _encode(lib, V, r, grads[r], levels, step)
        assert torch.equal(_wire_slots(V, r), _expect_slots(V, grads[r], levels, r, step))
    V.update(1, [sgd_h(lr=0.5)])
    code = ps.QSGD(levels=levels, blockwise=True, seed=SEED)
    for i, p in enumerate(V.params):
        first = V.L.by_id[id(p)].offset
        tot = torch.zeros(shapes[i])
        for r in range(nranks):                   # rank order = the kernel's summation order
            tot = tot + code.decode(code.encode(grads[r][i], rank=r, step=step, first_elem=first))
        want = (w0[i] - 0.5 * tot).to(dtype)
        for r in range(nranks):
            got = V.param_values(r)[i]
            tol = 1e-5 if dtype == torch.float32 else 1e-2
            assert torch.allclose(got.float(), want.float(), rtol=tol, atol=tol), float((got.float() - want.float()).abs().max())


@pytest.mark.parametrize("levels", [1, 4, 127])
def test_statistics(levels):
    """Unbiased up to the 16-bit draw, per-element variance <= scale²/4, QSGD's variance bound per tile, and key sensitivity."""
    torch.manual_seed(0)
    g = torch.cat([torch.randn(TILE), torch.randn(TILE) * torch.rand(TILE) ** 4])
    steps = 512
    dec = torch.zeros(steps, g.numel())
    scale = None
    for s in range(steps):
        q, sc = qsgd_blockwise(g, levels, qsgd_uniform16(SEED, 1, s, TILE * 3, g.numel()))
        scale = sc if scale is None else scale
        assert torch.equal(sc, scale)                                   # the scale does not depend on the draw
        dec[s] = (q.float().view(-1, TILE) * sc[:, None]).reshape(-1)
    per = scale.repeat_interleave(TILE)
    sigma = per / 2 / math.sqrt(steps)
    err = (dec.mean(0) - g).abs()
    assert bool((err <= 5 * sigma + per * 2.0 ** -16 + 1e-6 * per).all()), float((err / sigma).max())
    n = TILE
    for t in range(2):
        gt = g[t * TILE:(t + 1) * TILE]
        mse = ((dec[:, t * TILE:(t + 1) * TILE] - gt) ** 2).sum(1).mean()
        assert mse <= min(n / levels ** 2, math.sqrt(n) / levels) * float((gt ** 2).sum())
    a = qsgd_blockwise(g, levels, qsgd_uniform16(SEED, 1, 9, 0, g.numel()))[0]
    assert torch.equal(a, qsgd_blockwise(g, levels, qsgd_uniform16(SEED, 1, 9, 0, g.numel()))[0])
    assert not torch.equal(a, qsgd_blockwise(g, levels, qsgd_uniform16(SEED, 1, 10, 0, g.numel()))[0])
    assert not torch.equal(a, qsgd_blockwise(g, levels, qsgd_uniform16(SEED, 2, 9, 0, g.numel()))[0])


# ---------------------------------------------------------------------------------------------------------------------
# the real device engine at 2-3 ranks (threads), real bindings over the emulated kernels
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def emu(monkeypatch):
    ext = _cuda_emu.build_extension()
    if ext is None:
        pytest.skip("no g++")
    lib = ext.emu
    lib.emu_set_sm_count(1)
    monkeypatch.setattr(mr, "_EXT", ext)
    mr._tls.world, mr._tls.m = mr.World(mr.Cluster(lib, 1), 0), None
    monkeypatch.setattr(runtime, "world", lambda: mr._tls.world)
    monkeypatch.setattr(de.ext, "cuda", lambda: mr._tls.m)
    monkeypatch.setattr(de, "SymmetricArena", mr.SharedArena)
    monkeypatch.setattr(torch.cuda, "Stream", lambda *a, **k: FakeStream())
    monkeypatch.setattr(torch.cuda, "Event", FakeEvent)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: FakeStream())
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(torch.cuda, "stream", lambda s: contextlib.nullcontext())
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self, *a, **k: self)
    monkeypatch.setenv("PSB200_CHUNK_BYTES", str(2048 * 4))
    return lib


def _qsgd(levels=16):
    return ps.QSGD(levels=levels, blockwise=True, seed=SEED)


@pytest.mark.parametrize("n,mode,optim,dtype", [
    (2, "ps", "sgd", torch.float32), (3, "allgather", "adam", torch.bfloat16), (2, "allgather", "sgd", torch.bfloat16),
    (3, "ps", "adam", torch.float32)])
def test_engine_matches_grad_gather_oracle(emu, n, mode, optim, dtype):
    """Each step every rank's actual gradient is coded with the engine's own keys (seed, rank, step, arena offset), decoded,
    summed in rank order and fed to the reference optimizer on fp32 shadows; masters must match and ranks be bit-identical."""
    hyper = dict(lr=0.05, momentum=0.9, weight_decay=1e-4) if optim == "sgd" else dict(lr=1e-2, eps=1e-8)
    steps = 3

    def rank_main(rank, w):
        model = mr._model(dtype)
        shadow = [torch.nn.Parameter(p.detach().float().clone()) for p in model.parameters()]
        cls = ps.SGD if optim == "sgd" else ps.Adam
        oracle = cls([(f"p{i}", q) for i, q in enumerate(shadow)], shadow, engine="host", use_mpi=False, **hyper)
        for h in oracle._hooks:
            h.remove()
        groups = oracle._group_of()
        opt = cls(model.named_parameters(), model.parameters(), engine="host", mode=mode, code=_qsgd(), **hyper)
        mr._attach(opt)
        eng = opt._engine
        assert eng.kind == KIND_QSGD and eng.bpt == TILE + 16
        first = [eng.layout.by_id[id(p)].offset for p in model.parameters()]
        for s in range(steps):
            opt.zero_grad(set_to_none=True)
            x, y = mr._data(rank, s, dtype)
            mr._loss(model, x, y, skip_head=False).backward()
            mine = [p.grad.detach().clone() for p in model.parameters()]
            opt.step()
            allg = w.all_gather_object(mine)
            code = _qsgd()
            with torch.no_grad():
                for i, q in enumerate(shadow):
                    total = torch.zeros_like(q)
                    for r in range(n):
                        total += code.decode(code.encode(allg[r][i], rank=r, step=s, first_elem=first[i])).reshape(q.shape)
                    oracle.optim_step(q, total, **oracle._hyper(groups[id(q)]))
        eng.check()
        w.barrier()
        got = [(opt.state[p]["master_param"] if eng.master is not None else p).detach().float().clone() for p in model.parameters()]
        pub = [p.detach().clone() for p in model.parameters()]
        opt.close()
        oracle.close()
        return got, pub, [q.detach().clone() for q in shadow], eng.is_server

    res = mr.run_ranks(emu, n, rank_main)
    for got, pub, shadow, is_server in res:
        for a, b in zip(pub, res[0][1]):
            assert torch.equal(a, b)
        if is_server:
            for g, q, p in zip(got, shadow, pub):
                assert torch.allclose(g, q, rtol=2e-4, atol=2e-5), float((g - q).abs().max())
                if dtype != torch.float32:
                    assert torch.equal(g.to(dtype), p)


def test_engine_async_applies_every_gradient_once(emu):
    nsteps, n = 3, 3

    def rank_main(rank, w):
        model = mr._model()
        opt = ps.SGD(model.named_parameters(), model.parameters(), engine="host", mode="async", quota=1, lr=0.05, average=True,
                     code=_qsgd())
        mr._attach(opt)
        eng = opt._engine
        applied = None
        if rank == 0:
            applied = opt.serve()
        else:
            for s in range(nsteps):
                opt.zero_grad(set_to_none=True)
                mr._loss(model, *mr._data(rank, s), skip_head=False).backward()
                opt.step()
                time.sleep(0.002 * rank)
            assert eng.rng_step == nsteps
        opt.close()
        return applied, list(mr._words(eng.arena.local_ptr)), [p.detach().clone() for p in model.parameters()]

    res = mr.run_ranks(emu, n, rank_main)
    assert res[0][0] == nsteps * (n - 1)
    for r in (1, 2):
        assert res[r][1][mr.M.SIG_ACK] == nsteps and res[0][1][mr.M.SIG_GRAD_READY + r] == mr.DONE
    assert all(torch.isfinite(p).all() for p in res[0][2])
    assert not torch.equal(res[0][2][0], next(mr._model().parameters()).detach())


def test_engine_checkpoint_resume_is_bit_exact(emu):
    """2 steps + state_dict + load into fresh objects + 2 steps == 4 straight steps, bit for bit: the RNG step travels in the
    optimizer state on every rank (workers included), so the resumed run draws the same roundings."""
    hyper = dict(lr=0.05, momentum=0.9, weight_decay=1e-4)

    def rank_main(rank, w):
        def make():
            m = mr._model(torch.bfloat16)
            o = ps.SGD(m.named_parameters(), m.parameters(), engine="host", mode="ps", code=_qsgd(), **hyper)
            mr._attach(o)
            return m, o

        def run(m, o, steps, start=0):
            for s in range(start, start + steps):
                o.zero_grad(set_to_none=True)
                x, y = mr._data(rank, s, torch.bfloat16)
                mr._loss(m, x, y, skip_head=False).backward()
                o.step()

        m1, o1 = make()
        run(m1, o1, 4)
        want = [p.detach().clone() for p in m1.parameters()]
        m2, o2 = make()
        run(m2, o2, 2)
        sd_model = {k: v.clone() for k, v in m2.state_dict().items()}
        sd_opt = copy.deepcopy(o2.state_dict())
        assert sd_opt["qsgd_rng_step"] == 2
        m3, o3 = make()
        with torch.no_grad():
            for k, v in m3.state_dict().items():
                v.copy_(sd_model[k])
        o3.load_state_dict(sd_opt)
        assert o3._engine.rng_step == 2
        run(m3, o3, 2, start=2)
        got = [p.detach().clone() for p in m3.parameters()]
        for o in (o1, o2, o3):
            o._engine.check()
        w.barrier()
        for o in (o1, o2, o3):
            o.close()
        return got, want

    for got, want in mr.run_ranks(emu, 2, rank_main):
        for a, b in zip(got, want):
            assert torch.equal(a, b)


def test_recover_does_not_rewind_the_rng_step(emu):
    """``recover()`` restarts the epoch clock but not the RNG step: the next step's wire bytes use step 2, not 0."""

    def rank_main(rank, w):
        model = mr._model()
        opt = ps.SGD(model.named_parameters(), model.parameters(), engine="host", mode="allgather", lr=0.05, code=_qsgd())
        mr._attach(opt)
        eng = opt._engine
        for s in range(2):
            opt.zero_grad(set_to_none=True)
            mr._loss(model, *mr._data(rank, s), skip_head=False).backward()
            opt.step()
        eng.recover()
        assert eng._epoch == 0 and eng.rng_step == 2
        opt.zero_grad(set_to_none=True)
        mr._loss(model, *mr._data(rank, 2), skip_head=False).backward()
        grads = [p.grad.detach().clone() for p in model.parameters()]
        opt.step()
        eng.check()
        wire = eng.wire_arena.clone()
        w.barrier()
        code = _qsgd()
        for p, g in zip(model.parameters(), grads):
            sl = eng.layout.by_id[id(p)]
            q = code.encode(g, rank=rank, step=2, first_elem=sl.offset)["q"]
            got = wire[sl.first_tile * eng.bpt: sl.first_tile * eng.bpt + TILE].view(torch.int8)
            assert torch.equal(got, q[:TILE])
        opt.close()

    mr.run_ranks(emu, 2, rank_main)


def test_nvls_reduce_is_refused(emu):
    def rank_main(rank, w):
        model = mr._model()
        opt = ps.SGD(model.named_parameters(), model.parameters(), engine="host", mode="ps", lr=0.05, code=_qsgd())
        for h in opt._hooks:
            h.remove()
        with pytest.raises(ValueError, match="nvls"):
            de.DeviceEngine(opt, reduce="nvls")
        return True

    assert mr.run_ranks(emu, 2, rank_main, multicast=True) == [True, True]


def test_host_engine_blockwise_qsgd():
    """The host engine runs the block-wise coding too (its per-tile algorithm on the gradient's own device)."""
    model = mr._model()
    w0 = [p.detach().clone() for p in model.parameters()]
    opt = ps.SGD(model.named_parameters(), model.parameters(), engine="host", mode="allgather", lr=0.1,
                 code=ps.QSGD(levels=8, blockwise=True, seed=SEED))
    assert opt._engine is None
    opt.zero_grad(set_to_none=True)
    mr._loss(model, *mr._data(0, 0), skip_head=False).backward()
    grads = [p.grad.detach().clone() for p in model.parameters()]
    opt.step()
    opt.close()
    for p, a, g in zip(model.parameters(), w0, grads):
        assert torch.isfinite(p).all() and not torch.equal(p.detach(), a)
        err = (a - 0.1 * g - p.detach()).abs().max()
        assert err <= 0.1 * float(g.norm()) / 8 + 1e-6              # within one quantum of the exact step
