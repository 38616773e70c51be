"""Worker bodies for the spawned multi-process tests (import-safe: no work at import)."""
import os

import numpy as np
import torch

#: environment of the ranks of the CPU scenarios: no visible GPU, so ``runtime.init()`` builds a CPU / gloo world on any
#: machine (with a GPU visible every rank would pick ``cuda:0`` and NCCL, which refuses two ranks on one device)
CPU_ONLY = {"CUDA_VISIBLE_DEVICES": ""}


def _world(rank, size):
    import pytorch_ps_mpi_b200 as ps
    w = ps.runtime.init()
    assert (w.rank, w.size) == (rank, size)
    return ps, w


# --- reference test_comms.py:9-16 ------------------------------------------------------
def gather_objects(rank, size, transport):
    os.environ["PSB200_TRANSPORT"] = transport
    ps, w = _world(rank, size)
    comms = ps.comms
    obj = {"str": "str", "rank": rank, "list": [rank] * (rank + 1)}
    msg = comms.igather(obj, name=1)
    assert set(msg[2]) == {"pickle_time", "compress_time", "alloc_time", "igather_time", "alloc_bytes"}
    objs = comms.irecv(msg[0], msg[1], name=1)
    sent = [{"str": "str", "rank": r, "list": [r] * (r + 1)} for r in range(size)]
    if rank == 0:
        assert objs == sent
    else:
        assert objs is None
    # tensors of every dtype survive (the reference cast to float32, mpi_comms.py:48)
    t = {"w": torch.arange(6, dtype=torch.float32).view(2, 3).bfloat16() * (rank + 1),
         "i": torch.tensor([rank], dtype=torch.int64), "np": np.full(3, rank, dtype=np.float64)}
    r = comms.irecv(*comms.igather(t, name="t")[:2], name="t")
    if rank == 0:
        for k, o in enumerate(r):
            assert o["w"].dtype == torch.bfloat16 and torch.equal(o["w"], t["w"] / (rank + 1) * (k + 1))
            assert o["i"].item() == k and o["np"].dtype == torch.float64
    comms.barrier()


# --- reference test_comms.py:19-26 -----------------------------------------------------
def bcast_objects(rank, size, transport):
    os.environ["PSB200_TRANSPORT"] = transport
    ps, w = _world(rank, size)
    comms = ps.comms
    obj = {"x": "x", "list": [1]}
    if rank == 0:
        obj = {"a": "a", "list": [0]}
    tmp = comms.ibroadcast(obj)
    recv = comms.irecv1(*tmp)
    assert recv == {"a": "a", "list": [0]}
    big = torch.arange(3_000_000, dtype=torch.float32) if rank == 0 else None   # > ring size: chunked
    got = comms.irecv1(*comms.ibroadcast(big))
    assert torch.equal(got, torch.arange(3_000_000, dtype=torch.float32))
    comms.barrier()


# --- reference test_iallgather.py:37-54 + test_mpi.py:34-96 ------------------------------
def iallgather_objects(rank, size, transport):
    os.environ["PSB200_TRANSPORT"] = transport
    ps, w = _world(rank, size)
    comms = ps.comms

    def make(r):
        return {"rank": r, "list": [r] * (r + 1)}

    ia = comms.Iallgather()
    msgs = [comms.format_for_send(make(rank))[0], comms.format_for_send({"a": "a", "async": [rank] * (rank + 1)})[0]]
    sizes = ia.prepare([len(m) for m in msgs])
    resp = []
    for (req, count), m in zip(sizes, msgs):
        req.Wait()
        assert int(count[rank]) == len(m) and len(count) == size
        resp.append(ia.send(m, count))
    jar = ia.recv(*resp[0])
    assert jar == [make(r) for r in range(size)]
    jar2 = ia.recv(*resp[1])
    assert jar2 == [{"a": "a", "async": [r] * (r + 1)} for r in range(size)]
    comms.barrier()


def p2p_any_source(rank, size, transport):
    os.environ["PSB200_TRANSPORT"] = transport
    ps, w = _world(rank, size)
    comms = ps.comms
    if rank == 0:
        seen = set()
        for _ in range(size - 1):
            req = comms.irecv_obj(src=comms.ANY_SOURCE, tag=3)
            m = req.Wait()
            assert m["rank"] == req.source
            seen.add(req.source)
        assert seen == set(range(1, size))
    else:
        comms.isend_obj({"rank": rank, "t": torch.ones(rank)}, dst=0, tag=3).Wait()
    comms.barrier()


def three_rank_suite(rank, size, transport):
    """Three ranks, one set of processes: (shm only) the synchronous PS oracle run, then ``average=True`` with several parameter
    groups, then AsySG-InCon — in that order (the async protocol's goodbye messages come last)."""
    os.environ["PSB200_TRANSPORT"] = transport
    ps, w = _world(rank, size)
    if transport == "shm":
        _mlp_train_body(ps, w, rank, size, "ps", "sgd", "identity")
        w.barrier()
    mlp_average_and_groups(rank, size, transport)
    w.barrier()
    mlp_async(rank, size, transport)


def comm_suite(rank, size, transport, names):
    """Several of the comm scenarios above in ONE set of processes (a spawn costs far more than the scenarios; and the façade
    must survive being used for one pattern after another: tags, pending requests, ring state)."""
    for name in names:
        globals()[name](rank, size, transport)


# --- BASELINE config 1: 2-layer MLP, MNIST-shaped synthetic, world_size 2 -------------------
def _mlp_data(rank, step, batch=16):
    g = torch.Generator().manual_seed(1000 * step + rank)
    return torch.randn(batch, 1, 28, 28, generator=g), torch.randint(0, 10, (batch,), generator=g)


def _oracle_sum_sgd(size, steps, optim, hyper, coding_factory):
    """Single-process oracle: sum of every rank's (coded) gradient → torch.optim step."""
    from pytorch_ps_mpi_b200.models import mnist_mlp
    torch.manual_seed(0)
    model = mnist_mlp(hidden=32)
    opt = (torch.optim.SGD if optim == "sgd" else torch.optim.Adam)(model.parameters(), **hyper)
    for s in range(steps):
        total = [torch.zeros_like(p) for p in model.parameters()]
        for r in range(size):
            code = coding_factory()
            x, y = _mlp_data(r, s)
            model.zero_grad()
            torch.nn.functional.cross_entropy(model(x), y).backward()
            for t, p in zip(total, model.parameters()):
                t += code.decode(code.encode(p.grad)).reshape(p.shape).to(t.dtype)
        for t, p in zip(total, model.parameters()):
            p.grad = t
        opt.step()
    return [p.detach().clone() for p in model.parameters()]


def mlp_train(rank, size, mode, optim, coding, transport, coalesce=False):
    os.environ["PSB200_TRANSPORT"] = transport
    ps, w = _world(rank, size)
    _mlp_train_body(ps, w, rank, size, mode, optim, coding, coalesce)


def mlp_train_many(rank, size, transport, cases):
    """Several (mode, optim, coding, coalesce) scenarios in ONE set of processes: a spawn costs ~10 s of interpreter start-up and
    ``import torch`` per rank, the scenarios themselves a fraction of a second — and optimizers following each other in one
    process is itself a scenario (transport tags, pools and hooks of a closed optimizer must not leak into the next)."""
    os.environ["PSB200_TRANSPORT"] = transport
    ps, w = _world(rank, size)
    for mode, optim, coding, coalesce in cases:
        _mlp_train_body(ps, w, rank, size, mode, optim, coding, coalesce)
        w.barrier()


def _mlp_train_body(ps, w, rank, size, mode, optim, coding, coalesce=False):
    from pytorch_ps_mpi_b200.models import mnist_mlp
    factory = {"identity": ps.Identity, "cast": lambda: ps.Cast("bf16"), "scale": lambda: ps.Scale("int8"),
               "topk": lambda: ps.TopK(ratio=0.25), "svd": lambda: ps.SVD(rank=2)}[coding]
    hyper = {"lr": 0.05, "momentum": 0.9, "weight_decay": 1e-4} if optim == "sgd" else {"lr": 1e-2, "eps": 1e-12}
    torch.manual_seed(0)
    model = mnist_mlp(hidden=32)
    cls = ps.SGD if optim == "sgd" else ps.Adam
    opt = cls(model.named_parameters(), model.parameters(), code=factory(), mode=mode, coalesce=coalesce, **hyper)
    steps = 3
    for s in range(steps):
        x, y = _mlp_data(rank, s)
        opt.zero_grad()
        loss = torch.nn.functional.cross_entropy(model(x), y)
        loss.backward()
        out = opt.step()
        assert isinstance(out, tuple) and len(out) == 2
        data = out[1]
        for k in ("comm_wait", "optim_step_time", "decode_time", "msg_bytes", "packaged_bytes", "code_wait",
                  "iallgather_prepare_time", "isend_time"):
            assert k in data, k
    assert opt.steps == steps and opt.rank == rank and opt.size == size
    want = _oracle_sum_sgd(size, steps, optim, hyper, factory)
    tol = 1e-5 if optim == "sgd" else 2e-4     # reference Adam: sqrt(v)+eps  vs torch: sqrt(v/bc2)+eps
    for p, q in zip(model.parameters(), want):
        assert torch.allclose(p, q, rtol=tol, atol=tol), (mode, optim, coding, (p - q).abs().max())
    # every rank ends with identical parameters
    flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
    allp = w.all_gather_object(flat)
    for f in allp:
        assert torch.equal(f, allp[0])
    opt.close()


def mlp_async(rank, size, transport):
    os.environ["PSB200_TRANSPORT"] = transport
    ps, w = _world(rank, size)
    from pytorch_ps_mpi_b200.models import mnist_mlp
    torch.manual_seed(0)
    model = mnist_mlp(hidden=32)
    opt = ps.SGD(model.named_parameters(), model.parameters(), lr=0.05, code=ps.Identity(), mode="async", quota=1)
    before = torch.cat([p.detach().reshape(-1) for p in model.parameters()]).clone()
    if rank == 0:
        n = opt.serve()
        assert n == 4 * (size - 1)          # quota 1: one update per gradient message
        st = [d.get("staleness", [0]) for d in opt.timings if d.get("staleness")]
        assert all(s[0] >= 0 for s in st)
    else:
        import time
        for s in range(4):
            x, y = _mlp_data(rank, s)
            opt.zero_grad()
            torch.nn.functional.cross_entropy(model(x), y).backward()
            opt.step()
            time.sleep(0.01 * rank)          # injected delay → staleness
    opt.close()
    after = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
    if rank == 0:
        assert not torch.equal(before, after)


# --- device engine, spawned ranks (1 GPU shared by all ranks, or one GPU per rank) ----------
def _host_oracle(ps, model, optim, hyper):
    """fp32 CPU copies of the model's parameters + the package's reference optimizer math (``ps.py:195-261``)."""
    shadow = [torch.nn.Parameter(p.detach().float().cpu().clone()) for p in model.parameters()]
    cls = ps.SGD if optim == "sgd" else ps.Adam
    o = cls([(f"p{i}", q) for i, q in enumerate(shadow)], shadow, engine="host", use_mpi=False, **hyper)
    return shadow, o, o._group_of()


def gpu_train(rank, size, mode, optim, coding, dtype_name, reduce="auto", hidden=32):
    """Device engine, one process per rank.  Two oracles: (a) every dtype — each step all ranks' ACTUAL gradients are
    gathered, decode(encode(.)) applied per rank, summed in fp32 in rank order and fed to the reference optimizer math on
    fp32 CPU shadows; the engine's fp32 master weights must match (bf16 parameters included: VERDICT r1 #7d);
    (b) fp32 only — a full single-process re-computation of every rank's forward/backward."""
    ps, w = _world(rank, size)
    from pytorch_ps_mpi_b200.models import mnist_mlp
    dev = w.device
    assert dev.type == "cuda"
    dtype = {"fp32": torch.float32, "bf16": torch.bfloat16}[dtype_name]
    factory = {"identity": ps.Identity, "cast": lambda: ps.Cast("bf16"), "scale": lambda: ps.Scale("int8"),
               "topk": lambda: ps.TopK(ratio=0.25)}[coding]
    hyper = {"lr": 0.05, "momentum": 0.9, "weight_decay": 1e-4} if optim == "sgd" else {"lr": 1e-2, "eps": 1e-8}
    torch.manual_seed(0)
    model = mnist_mlp(hidden=hidden).to(dev).to(dtype)
    shadow, oracle, groups = _host_oracle(ps, model, optim, hyper)
    cls = ps.SGD if optim == "sgd" else ps.Adam
    opt = cls(model.named_parameters(), model.parameters(), code=factory(), mode=mode, engine="device", reduce=reduce, **hyper)
    eng = opt._engine
    assert eng is not None and eng.arena.provider in ("native", "torch")
    if reduce == "nvls":
        assert eng.reduce == 1 and eng.arena.has_multicast
    if os.environ.get("PSB200_EXPECT_CHUNKS"):
        assert eng.nchunks >= int(os.environ["PSB200_EXPECT_CHUNKS"]), eng.nchunks
    steps = 3
    sum_mag = 0.0
    for s in range(steps):
        x, y = _mlp_data(rank, s)
        opt.zero_grad()
        loss = torch.nn.functional.cross_entropy(model(x.to(dev).to(dtype)).float(), y.to(dev))
        loss.backward()
        mine = [p.grad.detach().cpu() for p in model.parameters()]       # the gradients the hooks saw
        out = opt.step()
        assert isinstance(out, tuple) and out[1]["engine"] == "device"
        allg = w.all_gather_object(mine)
        with torch.no_grad():
            for i, q in enumerate(shadow):
                total = torch.zeros_like(q)
                for r in range(size):
                    code = factory()
                    total += code.decode(code.encode(allg[r][i], name=f"p{i}")).reshape(q.shape).float()
                sum_mag = max(sum_mag, float(total.abs().max()))
                oracle.optim_step(q, total, **oracle._hyper(groups[id(q)]))
    eng.check()
    torch.cuda.synchronize()
    flat = torch.cat([p.detach().float().reshape(-1) for p in model.parameters()]).cpu()
    allp = w.all_gather_object(flat)
    for f in allp:
        assert torch.equal(f, allp[0]), "ranks diverged"
    if eng.is_server:
        # switch reduction of a bf16 wire returns the fp32-accumulated sum rounded ONCE to bf16: |err| <= 2^-9 |sum| per step
        atol = 2e-5 + (steps * hyper["lr"] * sum_mag * 2.0 ** -8 if (eng.reduce == 1 and dtype != torch.float32) else 0.0)
        rtol = 2e-4 if optim == "sgd" or eng.reduce == 0 or dtype == torch.float32 else 5e-2
        for p, q in zip(model.parameters(), shadow):
            got = opt.state[p]["master_param"] if eng.master is not None else p
            got = got.detach().float().cpu()
            assert torch.allclose(got, q.detach(), rtol=rtol, atol=atol), \
                (mode, optim, coding, dtype_name, eng.reduce, float((got - q).abs().max()))
            if eng.master is not None:     # published parameter == the master rounded to the parameter dtype
                assert torch.equal(got.to(dtype).float(), p.detach().float().cpu())
    if dtype == torch.float32:
        want = _oracle_sum_ref(size, steps, optim, hyper, factory, hidden)
        # int8 abs-max quantisation: a CPU-recomputed gradient that differs in its last bit can land on the other side of a
        # rounding boundary (one step of amax/127, times lr) — oracle (a) above, fed the ACTUAL gradients, stays tight
        atol_b = 2e-4 if coding == "scale" else 2e-5
        for p, q in zip(model.parameters(), want):
            assert torch.allclose(p.detach().cpu(), q, rtol=2e-4, atol=atol_b), (mode, optim, coding, (p.detach().cpu() - q).abs().max())
    info = {"provider": eng.arena.provider, "multicast": eng.arena.has_multicast, "bcast": eng.bcast, "reduce": eng.reduce,
            "chunks": eng.nchunks, "pipeline": eng.pipeline}
    if rank == 0:
        print("gpu_train ok", mode, optim, coding, dtype_name, info, flush=True)
    opt.close()


def gpu_train_big(rank, size, reduce="auto", numel_m=52):
    """VERDICT r1 #7d: a >= 50 M-element bf16 arena on real multi-GPU (many tiles per CTA, many pipeline chunks), checked
    against an fp32 oracle built from the ranks' actual gradients (NCCL all_gather — test-only plumbing)."""
    import torch.distributed as dist
    ps, w = _world(rank, size)
    dev = w.device
    torch.manual_seed(0)
    nl = max(2, numel_m // 8)                       # layers of 8.4 M elements each (chunks are whole parameters)
    dims = [1024 if i % 2 == 0 else 8192 for i in range(nl + 1)]
    layers = []
    for i in range(nl):
        layers += [torch.nn.Linear(dims[i], dims[i + 1], bias=False), torch.nn.ReLU()]
    model = torch.nn.Sequential(*layers, torch.nn.Linear(dims[nl], 16)).to(dev).bfloat16()
    hyper = {"lr": 0.05, "momentum": 0.9, "weight_decay": 1e-4}
    params = list(model.parameters())
    master = [p.detach().float().clone() for p in params]
    mom = [None] * len(params)
    opt = ps.SGD(model.named_parameters(), model.parameters(), code=ps.Identity(), mode="ps", engine="device", reduce=reduce, **hyper)
    eng = opt._engine
    assert eng.layout.numel_padded >= 50_000_000 and eng.nchunks >= 6, (eng.layout.numel_padded, eng.nchunks)
    sum_mag = 0.0
    for s in range(2):
        g = torch.Generator().manual_seed(100 * s + rank)
        x = torch.randn(8, 1024, generator=g).to(dev).bfloat16()
        y = torch.randint(0, 16, (8,), generator=g).to(dev)
        opt.zero_grad()
        torch.nn.functional.cross_entropy(model(x).float(), y).backward()
        grads = [p.grad.detach().clone() for p in params]
        opt.step()
        for i, gi in enumerate(grads):
            bucket = [torch.empty_like(gi) for _ in range(size)]
            dist.all_gather(bucket, gi)
            total = torch.zeros_like(master[i])
            for b in bucket:
                total += b.float()
            sum_mag = max(sum_mag, float(total.abs().max()))
            d = total + hyper["weight_decay"] * master[i]
            mom[i] = d.clone() if mom[i] is None else mom[i].mul_(hyper["momentum"]).add_(d)
            master[i] -= hyper["lr"] * mom[i]
    eng.check()
    torch.cuda.synchronize()
    w.barrier()
    atol = 1e-6 + (2 * hyper["lr"] * sum_mag * 2.0 ** -8 * 2 if eng.reduce == 1 else 0.0)
    for p, q in zip(params, master):
        if rank == 0:
            got = opt.state[p]["master_param"].detach()
            assert torch.allclose(got, q, rtol=1e-5, atol=atol), float((got - q).abs().max())
        pub = q.to(torch.bfloat16)
        diff = (p.detach().float() - pub.float()).abs().max()
        assert float(diff) <= atol + float(pub.float().abs().max()) * 2.0 ** -7, float(diff)
    if rank == 0:
        print("gpu_train_big ok", {"numel": eng.layout.numel_padded, "chunks": eng.nchunks, "reduce": eng.reduce,
                                   "bcast": eng.bcast}, flush=True)
    opt.close()


def _oracle_sum_ref(size, steps, optim, hyper, coding_factory, hidden=32):
    """Single-process oracle using the package's own host-path optimizer math (reference formulas)."""
    import pytorch_ps_mpi_b200 as ps
    from pytorch_ps_mpi_b200.models import mnist_mlp
    torch.manual_seed(0)
    model = mnist_mlp(hidden=hidden)
    cls = ps.SGD if optim == "sgd" else ps.Adam
    opt = cls(model.named_parameters(), model.parameters(), engine="host", use_mpi=False, **hyper)
    groups = opt._group_of()
    for s in range(steps):
        total = [torch.zeros_like(p) for p in model.parameters()]
        for r in range(size):
            code = coding_factory()
            x, y = _mlp_data(r, s)
            model.zero_grad()
            torch.nn.functional.cross_entropy(model(x), y).backward()
            for t, p in zip(total, model.parameters()):
                t += code.decode(code.encode(p.grad)).reshape(p.shape).to(t.dtype)
        opt.futures, opt.names = [], []
        with torch.no_grad():
            for t, p in zip(total, model.parameters()):
                opt.optim_step(p, t, **opt._hyper(groups[id(p)]))
    return [p.detach().clone() for p in model.parameters()]


def gpu_async(rank, size, coding, consistent=0):
    import time
    ps, w = _world(rank, size)
    from pytorch_ps_mpi_b200.models import mnist_mlp
    dev = w.device
    torch.manual_seed(0)
    model = mnist_mlp(hidden=32).to(dev)
    code = ps.Identity() if coding == "identity" else ps.TopK(ratio=0.25)
    opt = ps.SGD(model.named_parameters(), model.parameters(), lr=0.05, code=code, mode="async", quota=1,
                 engine="device", consistent=bool(consistent))
    assert opt._engine.consistent == bool(consistent)
    seen = []
    before = torch.cat([p.detach().reshape(-1) for p in model.parameters()]).clone()
    nsteps = 4
    if rank == 0:
        n = opt.serve()
        assert n == nsteps * (size - 1), n
    else:
        for s in range(nsteps):
            x, y = _mlp_data(rank, s)
            opt.zero_grad()
            torch.nn.functional.cross_entropy(model(x.to(dev)), y.to(dev)).backward()
            _, data = opt.step()
            if consistent:
                seen.append(data["param_version"])
            time.sleep(0.01 * rank)
        if consistent:
            assert seen == sorted(seen) and seen[-1] >= 1, seen     # whole snapshots, monotonically newer
    opt._engine.check()
    opt.close()
    after = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
    assert not torch.equal(before, after)
    # after the drain every rank holds the server's final parameters
    allp = w.all_gather_object(after.cpu())
    for f in allp:
        assert torch.equal(f, allp[0])


def symm_arena(rank, size):
    ps, w = _world(rank, size)
    from pytorch_ps_mpi_b200.parallel.symmetric import SymmetricArena
    A = SymmetricArena(3 << 20, w.device, w)
    mine = A.tensor(0, 1 << 20, torch.float32)
    mine.fill_(float(rank + 1))
    torch.cuda.synchronize()
    w.barrier()
    for r in range(size):
        peer = A.tensor(0, 1 << 20, torch.float32, rank=r)
        assert float(peer[12345]) == float(r + 1), (rank, r, float(peer[12345]))
    w.barrier()
    if rank == 0:
        print("symm_arena ok", A.provider, "multicast" if A.has_multicast else "no-multicast", A.nbytes, flush=True)
    A.close()


def gpu_bcast_linear(rank, size, pull):
    """MLP whose first GEMM is the tcgen05 kernel gated on the PS broadcast (and optionally PULLING the
    weight tiles from the server's arena over NVLink)."""
    ps, w = _world(rank, size)
    from pytorch_ps_mpi_b200.models import mnist_mlp
    from pytorch_ps_mpi_b200.ops.linear import convert_first_linear, BcastLinear
    dev = w.device
    torch.manual_seed(0)
    model = mnist_mlp(hidden=256).to(dev).bfloat16()
    ref = mnist_mlp(hidden=256).to(dev).bfloat16()
    ref.load_state_dict(model.state_dict())
    opt = ps.SGD(model.named_parameters(), model.parameters(), lr=0.05, momentum=0.9, mode="ps", engine="device")
    ropt = torch.optim.SGD(ref.parameters(), lr=0.05, momentum=0.9)
    layer = convert_first_linear(model, opt, relu=True, pull=bool(pull))
    assert isinstance(model.fc1, BcastLinear) and layer is model.fc1 and opt._engine._gates
    for s in range(4):
        xs = [_mlp_data(r, s, batch=128) for r in range(size)]
        x, y = xs[rank]
        opt.zero_grad()
        loss = torch.nn.functional.cross_entropy(model(x.to(dev).bfloat16()).float(), y.to(dev))
        loss.backward()
        opt.step()
        # single-process reference on the summed gradient (stock cuBLAS linear)
        ropt.zero_grad()
        for xr, yr in xs:
            torch.nn.functional.cross_entropy(ref(xr.to(dev).bfloat16()).float(), yr.to(dev)).backward()
        ropt.step()
    opt._engine.check()
    torch.cuda.synchronize()
    assert torch.isfinite(loss).item()
    flat = torch.cat([p.detach().float().reshape(-1) for p in model.parameters()]).cpu()
    allp = w.all_gather_object(flat)
    for f in allp:
        assert torch.equal(f, allp[0]), "ranks diverged"
    want = torch.cat([p.detach().float().reshape(-1) for p in ref.parameters()]).cpu()
    assert torch.allclose(flat, want, rtol=5e-2, atol=2e-2), (flat - want).abs().max()
    if rank == 0:
        print("gpu_bcast_linear ok pull=", pull, flush=True)
    opt.close()



def gpu_checkpoint(rank, size):
    """state_dict()/load_state_dict() of the device engine: resume must continue bit-identically."""
    ps, w = _world(rank, size)
    from pytorch_ps_mpi_b200.models import mnist_mlp
    dev = w.device

    def make():
        torch.manual_seed(0)
        m = mnist_mlp(hidden=32).to(dev).bfloat16()
        o = ps.SGD(m.named_parameters(), m.parameters(), lr=0.05, momentum=0.9, weight_decay=1e-4, mode="ps", engine="device")
        return m, o

    def run(m, o, steps, start=0):
        for s in range(start, start + steps):
            x, y = _mlp_data(rank, s)
            o.zero_grad()
            torch.nn.functional.cross_entropy(m(x.to(dev).bfloat16()).float(), y.to(dev)).backward()
            o.step()
        torch.cuda.synchronize()

    m1, o1 = make()
    run(m1, o1, 4)
    want = torch.cat([p.detach().float().reshape(-1) for p in m1.parameters()]).cpu()
    m2, o2 = make()
    run(m2, o2, 2)
    sd_model = {k: v.clone() for k, v in m2.state_dict().items()}
    sd_opt = o2.state_dict()
    if rank == 0:
        assert any("momentum_buffer" in s and "master_param" in s for s in sd_opt["state"].values())
    m3, o3 = make()
    with torch.no_grad():
        for k, v in m3.state_dict().items():
            v.copy_(sd_model[k])
    o3.load_state_dict(sd_opt)
    run(m3, o3, 2, start=2)
    got = torch.cat([p.detach().float().reshape(-1) for p in m3.parameters()]).cpu()
    assert torch.equal(got, want), (got - want).abs().max()
    for o in (o1, o2, o3):
        o.close()


def gpu_dead_peer(rank, size):
    """Failure detection: a worker that never posts its gradient must surface as an error, not a hang."""
    ps, w = _world(rank, size)
    from pytorch_ps_mpi_b200.models import mnist_mlp
    dev = w.device
    torch.manual_seed(0)
    m = mnist_mlp(hidden=32).to(dev)
    o = ps.SGD(m.named_parameters(), m.parameters(), lr=0.05, mode="ps", engine="device")
    x, y = _mlp_data(rank, 0)
    if rank == 0:
        o.zero_grad()
        torch.nn.functional.cross_entropy(m(x.to(dev)), y.to(dev)).backward()
        o.step()                     # rank 1 never steps: the bounded spin must time out
        try:
            o._engine.check()
            raise AssertionError("expected a device-side timeout")
        except RuntimeError as e:
            assert "timed out" in str(e)
        # ... and WITHOUT an explicit check(): the periodic, sync-free poll of the error slot raises (ADVICE r1)
        o._engine._poll_error()
        torch.cuda.synchronize()
        try:
            o._engine._poll_error()
            raise AssertionError("the error poll did not surface the time-out")
        except RuntimeError as e:
            assert "timed out" in str(e)
    w.barrier()


# --- host-path robustness ---------------------------------------------------------------------------
def shm_dead_peer(rank, size):
    """Failure detection on the CPU transport: a rank that dies must surface as an error on its peers."""
    os.environ["PSB200_TRANSPORT"] = "shm"
    os.environ["PSB200_COMM_TIMEOUT"] = "20"
    ps, w = _world(rank, size)
    from pytorch_ps_mpi_b200.parallel import transport as tp
    tr = tp.get_transport()
    assert isinstance(tr, tp.ShmTransport)
    tr.barrier()
    if rank == 1:
        os._exit(0)                       # vanish without saying goodbye
    import time
    time.sleep(0.5)
    req = tr.irecv(src=1, tag=5)
    try:
        req.Wait()
        raise AssertionError("expected the dead peer to be detected")
    except RuntimeError as e:
        assert "no longer running" in str(e) or "timed out" in str(e), str(e)
    assert tr.dead_peers() == [1]
    os._exit(0)                           # skip the collective teardown: the peer is gone


def mlp_average_and_groups(rank, size, transport):
    """average=True divides by the number of contributions; several param groups keep their own hyper-parameters."""
    os.environ["PSB200_TRANSPORT"] = transport
    ps, w = _world(rank, size)
    torch.manual_seed(0)
    a = torch.nn.Parameter(torch.ones(5))
    b = torch.nn.Parameter(torch.ones(3))
    opt = ps.SGD([("a", a), ("b", b)], [{"params": [a], "lr": 0.1}, {"params": [b], "lr": 1.0}], lr=0.01,
                 mode="ps", average=True)
    ((rank + 1) * a.sum() + 2 * (rank + 1) * b.sum()).backward()
    opt.step()
    mean = sum(r + 1 for r in range(size)) / size
    assert torch.allclose(a.detach(), torch.full((5,), 1 - 0.1 * mean)), a
    assert torch.allclose(b.detach(), torch.full((3,), 1 - 1.0 * 2 * mean)), b
    opt.close()


def mlp_async_consistent(rank, size):
    """consistent=True (README.md:79-81): every worker step adopts a whole parameter snapshot from the server."""
    os.environ["PSB200_TRANSPORT"] = "shm"
    ps, w = _world(rank, size)
    from pytorch_ps_mpi_b200.models import mnist_mlp
    torch.manual_seed(0)
    model = mnist_mlp(hidden=16)
    opt = ps.SGD(model.named_parameters(), model.parameters(), lr=0.05, mode="async", quota=size - 1, consistent=True)
    if rank == 0:
        n = opt.serve()
        assert n == 3
    else:
        versions = []
        for s in range(3):
            x, y = _mlp_data(rank, s)
            opt.zero_grad()
            torch.nn.functional.cross_entropy(model(x), y).backward()
            _, data = opt.step()
            versions.append(data["param_version"])
        assert versions == [1, 2, 3], versions        # blocks for the snapshot that contains its own gradient
    opt.close()
    flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
    allp = w.all_gather_object(flat)
    for f in allp[1:]:
        assert torch.equal(f, allp[1])


def shm_stress(rank, size):
    """Random all-to-all traffic over the native shm rings: messages far larger than a ring, many outstanding
    operations, ANY_SOURCE receives — every byte must arrive intact and in per-pair order."""
    os.environ["PSB200_TRANSPORT"] = "shm"
    os.environ["PSB200_SHM_RING_BYTES"] = str(64 << 10)          # tiny rings: force chunking + flow control
    ps, w = _world(rank, size)
    from pytorch_ps_mpi_b200.parallel import transport as tp
    tr = tp.get_transport()
    rng = np.random.default_rng(1234)                            # same schedule on every rank
    rounds = 30
    plan = [[(int(rng.integers(0, 300_000)) if rng.random() < 0.8 else 0) for _ in range(size * size)] for _ in range(rounds)]

    def payload(src, dst, rnd, n):
        g = np.random.default_rng(src * 1000 + dst * 10 + rnd)
        return g.integers(0, 256, n, dtype=np.uint8).tobytes()

    sends, recvs = [], []
    for rnd in range(rounds):
        for dst in range(size):
            if dst != rank:
                sends.append(tr.isend(dst, payload(rank, dst, rnd, plan[rnd][rank * size + dst]), tag=7))
        for src in range(size):
            if src != rank:
                recvs.append((src, rnd, tr.irecv(src=src, tag=7)))
    for src, rnd, req in recvs:                                    # posted long before they are waited
        msg = req.Wait()
        assert bytes(memoryview(msg)) == payload(src, rank, rnd, plan[rnd][src * size + rank]), (src, rnd)
        assert req.source == src
    for s in sends:
        s.Wait()
    tr.barrier()
    # ANY_SOURCE fan-in with a distinct tag
    if rank == 0:
        got = {}
        for _ in range((size - 1) * 5):
            r = tr.irecv(src=tp.ANY_SOURCE, tag=9)
            m = bytes(memoryview(r.Wait()))
            got.setdefault(r.source, []).append(m)
        for src in range(1, size):
            assert got[src] == [bytes([src, k]) * (1000 * k + 1) for k in range(5)]      # per-source FIFO order
    else:
        for k in range(5):
            tr.isend(0, bytes([rank, k]) * (1000 * k + 1), tag=9).Wait()
    tr.barrier()


# --- the bench's same-invocation comparators (baseline/comparator.py) on CPU / gloo ---------------------------------------
def comparator_host(rank, size):
    """RefEquivalentSGD (the stock-tools re-creation of the reference's per-step algorithm that bench.py times next to the
    product) must produce the summed-gradient SGD update on every rank — and must not hang: same collective sequence everywhere."""
    ps, w = _world(rank, size)
    from baseline.comparator import ComparatorSGD
    from pytorch_ps_mpi_b200.models import mnist_mlp
    torch.manual_seed(0)
    model = mnist_mlp(hidden=32)
    ref = [p.detach().clone() for p in model.parameters()]
    bufs = [None] * len(ref)
    hyper = dict(lr=0.05, momentum=0.9, weight_decay=1e-4)
    opt = ComparatorSGD(model.named_parameters(), kind="host", **hyper)
    for s in range(3):
        x, y = _mlp_data(rank, s)
        opt.zero_grad()
        torch.nn.functional.cross_entropy(model(x), y).backward()
        mine = [p.grad.detach().clone() for p in model.parameters()]
        opt.step()
        allg = w.all_gather_object(mine)
        for i, q in enumerate(ref):
            d = sum(allg[r][i] for r in range(size)) + hyper["weight_decay"] * q
            bufs[i] = d.clone() if bufs[i] is None else bufs[i].mul_(hyper["momentum"]).add_(d)
            q.add_(bufs[i], alpha=-hyper["lr"])
    for p, q in zip(model.parameters(), ref):
        assert torch.allclose(p.detach(), q, rtol=1e-5, atol=1e-6), float((p.detach() - q).abs().max())
    opt.close()
