#!/usr/bin/env python
"""BASELINE.json config 5: PS gather + broadcast over a parameter vector of 1 KB … 1 GB at N = 2 / 4 / 8 GPUs.

For every size the SAME public objects are exercised three ways and device-timed (CUDA events, max over ranks, warm-up,
distinct gradients every iteration).  The vector is a "model" of equal tensors of at most ``--piece-mb`` (a real parameter
vector is many tensors), so the device engine's per-chunk pipeline is on the measured path exactly as in training.

``fused``   this framework's device engine: per chunk, encode → GRAD_READY progress flag → ``psb_update_kernel`` (one
            ``multimem.ld_reduce`` through the switch — or a rank-ordered P2P pull — sum, SGD on fp32 masters,
            ``multimem.st`` publish); workers wait for PARAMS_READY.  Chunk k+1 is encoded while chunk k is gathered.
``nccl``    library baseline: ``dist.reduce`` to rank 0 + one fused axpy + ``dist.broadcast``.
``host``    the reference's PS round (``/root/reference/mpi_comms.py:60-133``): ``igather`` of every rank's gradient
            object to rank 0 (D2H → serialise → frame → host transport → H2D), sum + axpy there, ``ibroadcast`` of the
            parameters, ``irecv1`` — through this repo's façade of those four calls.  Sizes <= 16 MB.

Reported per size: µs per round trip, gather "bus" GB/s = (N-1)·B_wire / t (what a naive PS's server ingress would
need), broadcast GB/s = B_param / t, and the fraction of the NVLink roofline
``max((N-1)·B_wire, B_param) / BW`` for BW = 770 GB/s (measured peer-copy rate per direction, ``B200_PROFILING.md``)
and BW = 900 GB/s (the nominal figure BASELINE.json quotes).  A fraction above 1 means the switch reduced
(``multimem.ld_reduce``: server ingress is 1×, not (N-1)×).  One JSON line per (size, impl) on rank 0.

    python -m torch.distributed.run --nproc-per-node 8 bench/bandwidth_sweep.py --max-mb 1024 --out profiles/bw_sweep_n8.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pytorch_ps_mpi_b200 as ps   # noqa: E402

NVLINK_MEASURED_GBS = 770.0     # peer copy per direction per GPU (B200_PROFILING.md; re-measured by --peer-copy)
NVLINK_NOMINAL_GBS = 900.0      # BASELINE.json


def timed(w, device, fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize(device)
    w.barrier()
    torch.cuda.synchronize(device)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize(device)
    t = torch.tensor([s.elapsed_time(e) / iters], dtype=torch.float64)
    if w.size > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=w.cpu_group)
    return float(t.item()) * 1e3   # µs


def peer_copy_gbs(w, dev, nbytes=256 << 20):
    """The denominator, measured here: rank 0 pulls ``nbytes`` from rank 1's symmetric block with a plain copy kernel."""
    from pytorch_ps_mpi_b200.parallel.symmetric import SymmetricArena
    if w.size < 2:
        return None
    arena = SymmetricArena(nbytes, dev, w)
    local = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    out = None
    if w.rank == 0:
        src = arena.tensor(0, nbytes, torch.uint8, rank=1)
        for _ in range(2):
            local.copy_(src)
        torch.cuda.synchronize(dev)
        best = 1e9
        for _ in range(5):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            local.copy_(src)
            e.record()
            torch.cuda.synchronize(dev)
            best = min(best, s.elapsed_time(e))
        out = nbytes / best / 1e6
    w.barrier()
    arena.close()
    return out


def sweep_code(name):
    kind, _, arg = name.partition(":")
    if kind == "identity":
        return ps.Identity()
    if kind == "topk":
        return ps.TopK(ratio=float(arg), values="bf16")
    if kind == "cast":
        return ps.Cast(arg)
    if kind == "scale":
        return ps.Scale(arg or "int8")
    if kind == "qsgd":
        return ps.QSGD(levels=int(arg or 127), blockwise=True, seed=0)
    raise ValueError(f"unknown --code {name!r}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-kb", type=float, default=1)
    ap.add_argument("--max-mb", type=float, default=256)
    ap.add_argument("--dtype", default="bf16")
    ap.add_argument("--code", default="identity", help="identity | cast:DT | scale:DT | topk:RATIO | qsgd:LEVELS")
    ap.add_argument("--impls", default="fused,nccl,host")
    ap.add_argument("--reduce", default="auto")
    ap.add_argument("--piece-mb", type=float, default=8.0, help="largest tensor of the synthetic parameter vector")
    ap.add_argument("--peer-copy", action="store_true", help="also measure the plain peer-copy rate (the roofline denominator)")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    w = ps.runtime.init()
    dev = w.device
    dtype = {"bf16": torch.bfloat16, "fp32": torch.float32}[a.dtype]
    esz = 2 if dtype == torch.bfloat16 else 4
    sizes = []
    b = a.min_kb * 1024
    while b <= a.max_mb * (1 << 20) + 1:
        sizes.append(int(b))
        b *= 4
    rows = []
    if a.peer_copy:
        g = peer_copy_gbs(w, dev)
        if w.rank == 0:
            rows.append({"peer_copy_GBs": g, "bytes": 256 << 20, "how": "torch copy_ rank1 → rank0 over a VMM peer mapping, best of 5"})
            print(json.dumps(rows[-1]), flush=True)
    for nbytes in sizes:
        n = max(8, nbytes // esz)
        piece = max(8, int(a.piece_mb * (1 << 20)) // esz)
        shapes = [piece] * (n // piece) + ([n % piece] if n % piece else [])
        iters = 200 if nbytes < (1 << 20) else (50 if nbytes < (64 << 20) else 10)
        for impl in a.impls.split(","):
            if impl == "host" and nbytes > (16 << 20):
                continue
            torch.manual_seed(0)
            params = [torch.nn.Parameter(torch.zeros(m, device=dev, dtype=dtype)) for m in shapes]
            grads = [[torch.randn(m, device=dev).to(dtype) for m in shapes] for _ in range(2)]
            k = [0]
            opt = eng = None
            wire = n * esz
            if impl == "fused":
                code = sweep_code(a.code)
                named = [(f"v{i}", p) for i, p in enumerate(params)]
                opt = ps.SGD(named, params, lr=1e-3, code=code, mode="ps", engine="device", reduce=a.reduce, cuda=True)
                eng = opt._engine
                order = [(s.param, s.name, next(i for i, q in enumerate(params) if q is s.param)) for s in eng.layout.slots]

                def fn():
                    k[0] ^= 1
                    for p, name, i in order:             # hooks fire in arena (= backward) order
                        eng.on_grad(grads[k[0]][i], name, p)
                    opt.step()
                wire = eng.bpt * eng.layout.ntiles
            elif impl == "host":
                from pytorch_ps_mpi_b200 import mpi_comms as comms

                def fn():
                    k[0] ^= 1
                    recv, req, _ = comms.igather({"g": grads[k[0]]}, name="sweep")           # mpi_comms.py:60-93
                    objs = comms.irecv(recv, req, name="sweep", cuda=True)                    # :107-117 (rank 0 only)
                    if w.rank == 0:
                        for i, p in enumerate(params):
                            p.data.add_(sum(o["g"][i] for o in objs), alpha=-1e-3)
                    send, req = comms.ibroadcast({"p": [p.data for p in params]})             # :127-133
                    new = comms.irecv1(send, req, cuda=True)                                  # :120-124
                    if w.rank != 0:
                        for p, q in zip(params, new["p"]):
                            p.data.copy_(q)
            else:
                bufs = [torch.zeros(m, device=dev, dtype=dtype) for m in shapes]

                def fn():
                    k[0] ^= 1
                    works = []
                    for i, buf in enumerate(bufs):
                        buf.copy_(grads[k[0]][i])
                        if w.size > 1:
                            works.append(dist.reduce(buf, dst=0, async_op=True))
                    for wk in works:
                        wk.wait()
                    if w.rank == 0:
                        torch._foreach_add_([p.data for p in params], bufs, alpha=-1e-3)
                    if w.size > 1:
                        works = [dist.broadcast(p.data, src=0, async_op=True) for p in params]
                        for wk in works:
                            wk.wait()
            us = timed(w, dev, fn, iters if impl != "host" else max(3, iters // 10))
            gather_b = (w.size - 1) * wire
            bcast_b = n * esz
            need = max(gather_b, bcast_b) if w.size > 1 else 0
            row = {"bytes": n * esz, "impl": impl, "n_gpus": w.size, "us": us, "tensors": len(shapes),
                   "gather_GBs": gather_b / us / 1e3 if w.size > 1 else None,
                   "bcast_GBs": bcast_b / us / 1e3,
                   "roofline_us_770": need / (NVLINK_MEASURED_GBS * 1e3) if need else None,
                   "roofline_frac_770": need / (NVLINK_MEASURED_GBS * 1e3) / us if need else None,
                   "roofline_frac_900": need / (NVLINK_NOMINAL_GBS * 1e3) / us if need else None,
                   "wire_bytes": wire, "dtype": a.dtype, "code": a.code,
                   "multicast": bool(eng is not None and eng.arena.has_multicast),
                   "reduce": {0: "p2p", 1: "multimem.ld_reduce"}.get(getattr(eng, "reduce", None)),
                   "chunks": getattr(eng, "nchunks", None)}
            if opt is not None:
                eng.check()
                opt.close()
            rows.append(row)
            if w.rank == 0:
                print(json.dumps(row), flush=True)
            w.barrier()
    if w.rank == 0 and a.out:
        with open(a.out, "w") as f:
            json.dump(rows, f, indent=1)
    ps.runtime.shutdown()


if __name__ == "__main__":
    main()
