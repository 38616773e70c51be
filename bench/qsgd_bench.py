#!/usr/bin/env python
"""Block-wise QSGD on one GPU: (1) the encode kernel alone on a bf16 gradient larger than L2, alternated in the same process
with the int8 abs-max ``Scale`` encode (abs-max pass + encode) and the ``Cast('bf16')`` encode; (2) the ResNet-18 training
step at N = 1 with ``qsgd:127`` / ``scale:int8`` / ``identity`` through ``bench.main()`` (``bench.py`` knows no QSGD, so its
``make_code`` is wrapped here).  Prints one JSON object; the GPU name and power limit are read in the same run.

    python bench/qsgd_bench.py --mb 512 --launches 20 --rounds 5 --steps 20 --warmup 5
"""
import argparse
import contextlib
import io
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pytorch_ps_mpi_b200 as ps   # noqa: E402
from pytorch_ps_mpi_b200.codings import TILE   # noqa: E402
from pytorch_ps_mpi_b200.ops import ext   # noqa: E402
from pytorch_ps_mpi_b200.parallel.layout import FlatLayout   # noqa: E402

HBM_TBPS = 7.7     # HGX B200 data sheet, per GPU


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() if q.returncode == 0 else None}


def encode_bench(mb, launches, rounds):
    dev = torch.device("cuda", 0)
    m = ext.cuda()
    n = int(mb * (1 << 20)) // 2
    n = n // TILE * TILE
    p = torch.nn.Parameter(torch.empty(n, device=dev, dtype=torch.bfloat16))
    L = FlatLayout([{"params": [p]}], {id(p): "g"})
    tiles = L.tile_table_fast().to(dev)
    g = torch.randn(n, device=dev).to(torch.bfloat16)
    scales = torch.zeros(1, device=dev)
    amax = torch.zeros(1, dtype=torch.int32, device=dev)
    codes = {"qsgd:127": ps.QSGD(levels=127, blockwise=True, seed=1), "scale:int8": ps.Scale("int8"), "cast:bf16": ps.Cast("bf16")}
    runs = {}
    for name, code in codes.items():
        spec = code.device_spec()
        wire = spec.resolved_wire(torch.bfloat16)
        bpt = spec.bytes_per_tile(torch.bfloat16)
        buf = torch.empty(L.ntiles * bpt, dtype=torch.uint8, device=dev)
        kw = dict(levels=spec.levels, seed=spec.seed, rng_step=0, rank=0) if name.startswith("qsgd") else {}
        # bytes the algorithm must move: the gradient once per pass over it (abs-max scale reads it twice) + the wire slots
        reads = 2 * n * (2 if name.startswith("scale") else 1)
        runs[name] = (lambda spec=spec, wire=wire, bpt=bpt, buf=buf, kw=kw: m.encode(
            spec.kind, wire, [g], [0], [L.ntiles], [0], tiles.data_ptr(), buf.data_ptr(), scales.data_ptr(), amax.data_ptr(), 0,
            bpt, spec.tile_capacity(), float(spec.ratio), **kw), reads + L.ntiles * bpt)
    for fn, _ in runs.values():          # warm-up: module load, first launch of every instantiation
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in runs}
    for _ in range(rounds):              # alternate the codings so that drift on a shared host hits all of them
        for name, (fn, _) in runs.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(launches):
                fn()
            b.record()
            b.synchronize()
            times[name].append(a.elapsed_time(b) / launches * 1e-3)
    out = {}
    for name, (_, nbytes) in runs.items():
        t = statistics.median(times[name])
        out[name] = {"us_median": t * 1e6, "us_min": min(times[name]) * 1e6, "bytes": nbytes, "GBps": nbytes / t / 1e9,
                     "share_of_hbm_peak": nbytes / t / (HBM_TBPS * 1e12)}
    out["gradient"] = {"elements": n, "dtype": "bf16", "MB": 2 * n / (1 << 20), "tiles": L.ntiles}
    return out


def step_bench(codes, steps, warmup):
    import bench
    orig = bench.make_code

    def make_code(ps_, name):
        if name.startswith("qsgd"):
            return ps_.QSGD(levels=int(name.split(":")[1]), blockwise=True, seed=0)
        return orig(ps_, name)

    bench.make_code = make_code
    res = {}
    for c in codes:
        sys.argv = ["bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup), "--code", c, "--no-comparators"]
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            bench.main()
        lines = [ln for ln in buf.getvalue().splitlines() if ln.startswith("{")]
        res[c] = json.loads(lines[-1]) if lines else {"error": buf.getvalue()[-2000:]}
    bench.make_code = orig
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mb", type=float, default=512, help="bf16 gradient size (larger than the 126 MB L2)")
    ap.add_argument("--launches", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--codes", default="qsgd:127,scale:int8,identity")
    ap.add_argument("--no-step", action="store_true")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device"}))
        return 1
    out = {"hardware": gpu_info(), "encode": encode_bench(a.mb, a.launches, a.rounds)}
    if not a.no_step:
        out["resnet18_step_n1"] = step_bench(a.codes.split(","), a.steps, a.warmup)
    print(json.dumps(out))
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    return 0


if __name__ == "__main__":
    sys.exit(main())
