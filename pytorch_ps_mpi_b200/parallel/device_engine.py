"""Device engine: the B200 hot path behind ``MPI_PS.step()``.

Per step, per rank (nothing on this path touches the host after the launches are queued, and
nothing goes through NCCL/MPI):

1. **backward hooks** (``ps.py:65-66,98-101`` in the reference: encode on a thread pool) collect
   gradients into buckets; each full bucket is encoded by ONE ``psb_encode_kernel`` launch on a
   side stream straight into this rank's *symmetric wire arena* (cast / abs-max scale /
   block-wise top-k), overlapping with the rest of backward;
2. ``step()`` raises this rank's ``GRAD_READY`` epoch flag (``st.release.sys`` into the server's
   signal pad — the ``Igatherv`` post of ``mpi_comms.py:88``);
3. the server (rank 0 in ``mode='ps'``; every rank in ``mode='allgather'``) launches
   ``psb_update_kernel`` once: wait flags → pull every rank's wire tiles over NVLink (or one
   ``multimem.ld_reduce`` through the switch) → decode + rank-ordered fp32 sum → SGD/Adam on fp32
   master state → publish the new parameter tiles into every rank's *symmetric parameter
   arena* (``multimem.st`` or peer stores) → raise ``PARAMS_READY``;
4. workers queue a one-thread wait kernel on their compute stream (the ``req.Wait()`` of
   ``mpi_comms.py:121``); the model's parameters ARE views of the parameter arena, so the next
   forward reads the fresh weights with no copy.

``mode='async'`` (AsySG-InCon, ``README.md:56-81``): rank 0 is a dedicated server; a device-side
``select`` kernel waits until ``quota`` workers (ANY source) have posted a gradient, the update
kernel sums exactly those, publishes parameters + version and acknowledges the contributors;
workers never wait for parameters (inconsistent reads) — only for the ack of their previous
gradient before overwriting their wire arena.
"""
from __future__ import annotations

import math
import os
import time
from typing import Dict, List, Optional

import torch

from .. import runtime
from ..codings import KIND_DENSE, KIND_QSGD, KIND_SCALED, KIND_TOPK, TILE, WIRE_BF16, WIRE_F16, WIRE_F32, wire_code_of
from ..ops import ext
from ..utils.misc import CudaStepTimer
from .layout import FlatLayout
from .symmetric import SymmetricArena

_DT = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}
_DONE_EPOCH = 1 << 62


def _align(n: int, a: int = 256) -> int:
    return (n + a - 1) // a * a


def _dense(t: torch.Tensor) -> bool:
    """True if ``t``'s strides describe a dense, non-overlapping permutation of its shape."""
    if t.is_contiguous():
        return True
    dims = sorted(((st, sz) for st, sz in zip(t.stride(), t.shape) if sz > 1), key=lambda x: x[0])
    expect = 1
    for st, sz in dims:
        if st != expect:
            return False
        expect *= sz
    return True


class DeviceEngine:
    def __init__(self, opt, master_fp32: bool = True, reduce: str = "auto"):
        self.opt = opt
        self.m = ext.cuda()
        self.world = runtime.world()
        self.rank, self.size = opt.rank, opt.size
        if self.size > self.m.MAX_RANKS:
            raise ValueError(f"device engine supports up to {self.m.MAX_RANKS} ranks per server")
        if len(opt.param_groups) > self.m.MAX_GROUPS:
            raise ValueError(f"device engine supports up to {self.m.MAX_GROUPS} param groups")
        self.mode = opt.mode
        names = {id(p): n for n, p in opt._named.items()}
        self.layout = FlatLayout(opt.param_groups, names)
        p0 = self.layout.slots[0].param
        self.device, self.dtype = p0.device, p0.dtype
        self.dt = _DT[self.dtype]
        self.psz = p0.element_size()
        self.spec = opt.code.device_spec()
        self.kind = self.spec.kind
        self.wire = self.spec.resolved_wire(self.dtype)
        self.bpt = self.spec.bytes_per_tile(self.dtype)
        self.cap = self.spec.tile_capacity()
        # bounded device spins: a dead peer must never hang the GPU, but an honest stall (rank-0 validation, a
        # checkpoint, a slow data loader) must not poison the flags either — hence a long default, surfaced by
        # _poll_error() every few steps instead of silently disabling synchronisation
        self.timeout_s = float(os.environ.get("PSB200_DEVICE_TIMEOUT", "900"))
        self.chunk_bytes = int(os.environ.get("PSB200_CHUNK_BYTES", os.environ.get("PSB200_BUCKET_BYTES", 4 << 20)))
        self.pipeline = bool(getattr(opt, "pipeline", True)) and os.environ.get("PSB200_PIPELINE", "1") != "0" \
            and self.mode in ("ps", "allgather")
        L = self.layout
        nt, n_pad = L.ntiles, L.numel_padded
        self._check_same_layout_everywhere()

        # ---- symmetric block: [signal pad | scales | wire arena | parameter arena] ----
        self.off_signal = 0
        self.off_scales = _align(self.m.SIGNAL_SLOTS * 8)
        self.off_wire = self.off_scales + _align(max(L.nparams, 1) * 4)
        self.off_param = self.off_wire + _align(nt * self.bpt)
        total = self.off_param + _align(n_pad * self.psz)
        # consistent reads (README.md:79-81 "a buffered broadcast"): the server publishes into a STAGING copy of
        # the parameter arena; workers adopt whole snapshots from it under a sequence lock (see _snapshot)
        self.consistent = bool(getattr(opt, "consistent", False)) and self.mode == "async" and self.size > 1
        self.off_stage = total
        if self.consistent:
            total += _align(n_pad * self.psz)
        self.arena = SymmetricArena(total, self.device, self.world)
        A = self.arena
        self.signal = A.tensor(self.off_signal, self.m.SIGNAL_SLOTS * 8, torch.int64)
        self.scales = A.tensor(self.off_scales, max(L.nparams, 1) * 4, torch.float32)
        self.wire_arena = A.tensor(self.off_wire, nt * self.bpt, torch.uint8)
        self.param_arena = A.tensor(self.off_param, n_pad * self.psz, self.dtype)
        self.stage_arena = A.tensor(self.off_stage, n_pad * self.psz, self.dtype) if self.consistent else None

        # ---- move the model's parameters into the parameter arena (zero-copy from now on) ----
        with torch.no_grad():
            self.wire_arena.zero_()          # tile padding must be (and then stays) zero: see grad_out()
            self.param_arena.zero_()
            for s in L.slots:
                flat = self.param_arena[s.offset: s.offset + s.numel]
                pd = s.param.data
                if s.strides is not None:   # custom placement requested by the module (layout.py): padding stays zero
                    view = torch.as_strided(flat, pd.shape, s.strides)
                elif pd.is_contiguous() or not _dense(pd):
                    view = flat.view(pd.shape)
                else:   # e.g. channels_last conv weights: keep the physical layout cuDNN wants
                    view = torch.as_strided(flat, pd.shape, pd.stride())
                view.copy_(pd)
                s.param.data = view
        torch.cuda.synchronize(self.device)
        self.world.barrier()
        # identical start on every rank: adopt rank 0's weights (the reference silently relies on
        # equal seeds — there is no initial synchronisation anywhere in ps.py)
        if self.size > 1 and self.rank != 0 and os.environ.get("PSB200_SYNC_INIT", "1") == "1":
            src = A.tensor(self.off_param, n_pad * self.psz, self.dtype, rank=0)
            self.param_arena.copy_(src)
            torch.cuda.synchronize(self.device)
        self.world.barrier()

        if self.consistent:
            self.stage_arena.copy_(self.param_arena)
            torch.cuda.synchronize(self.device)
            self.world.barrier()

        # ---- server-side state ----
        self.is_server = (self.mode == "allgather") or self.rank == 0 or self.size == 1
        self.tiles = L.tile_table_fast().to(self.device)
        self.amax = torch.zeros(max(L.nparams, 1), dtype=torch.int32, device=self.device)
        self.active_dev = torch.ones(max(L.nparams, 1), dtype=torch.uint8, device=self.device)
        self.active_host = torch.ones(max(L.nparams, 1), dtype=torch.uint8).pin_memory()
        self._active_all = True
        self._last_fired = None
        self.counters = torch.zeros(8, dtype=torch.int32, device=self.device)   # [0] done, [1] stats
        self.residual = None
        if self.kind == KIND_TOPK and self.spec.error_feedback:
            self.residual = torch.zeros(n_pad, dtype=torch.float32, device=self.device)
        self.master = self.buf0 = self.buf1 = self.buf2 = None
        if self.is_server:
            if self.dtype != torch.float32 and master_fp32:
                self.master = self.param_arena.float()
            need_b0 = opt.optim == "adam" or any(g.get("momentum", 0) != 0 for g in opt.param_groups)
            if need_b0:
                self.buf0 = torch.zeros(n_pad, dtype=torch.float32, device=self.device)
            if opt.optim == "adam":
                self.buf1 = torch.zeros(n_pad, dtype=torch.float32, device=self.device)
                if any(g.get("amsgrad", False) for g in opt.param_groups):
                    self.buf2 = torch.zeros(n_pad, dtype=torch.float32, device=self.device)
            self._expose_state()
        self._group_steps = [0] * len(opt.param_groups)
        self._hyper_cache = None
        # per-parameter step counts (the reference keeps optimizer state per parameter and skips p.grad is None,
        # ps.py:178-179,203-205,226-241).  While every parameter has fired on every step they all equal the group's count and
        # the kernel uses the group tuple; after the first step that skipped a parameter a per-parameter table is uploaded.
        self._param_steps = [0] * max(L.nparams, 1)
        self._uniform_steps = True
        # (a ring: the async H2D copy of step e may still be queued when the host fills the table of step e+1)
        self._phyper_host = [torch.zeros(max(L.nparams, 1), 2, dtype=torch.float32).pin_memory() for _ in range(4)]
        self._phyper_dev = [torch.zeros(max(L.nparams, 1), 2, dtype=torch.float32, device=self.device) for _ in range(4)]

        # ---- publication / reduction strategy ----
        mc = A.has_multicast
        if self.mode == "allgather" or self.size == 1:
            self.bcast = 0                                  # BCAST_LOCAL
        else:
            self.bcast = 2 if (mc and os.environ.get("PSB200_BCAST", "auto") != "unicast") else 1
        nvls_ok = mc and self.kind == KIND_DENSE and self.wire in (WIRE_F32, WIRE_BF16, WIRE_F16) and self.size > 1
        if reduce == "nvls" and not nvls_ok:
            raise ValueError("reduce='nvls' needs multicast memory and a dense fp32/bf16/fp16 wire")
        if reduce == "nvls" and self.mode == "async":
            # multimem.ld_reduce sums EVERY bound rank's wire tile; async sums only the device-selected contributors
            # (quota < N-1), so the switch reduction would re-apply stale / torn gradients of the others
            raise ValueError("reduce='nvls' cannot be combined with mode='async' (the contributor set is a subset)")
        # 'auto': the switch reduces (multimem.ld_reduce: server ingress 1x instead of (N-1)x, 1.9-2x faster than
        # the P2P pull at 16-64 MB on 8 GPUs) for dense fp32 / bf16 / fp16 wires when there is ONE reducer whose
        # contributor set is always every rank (mode='ps') and N >= 4.  bf16/fp16 wires: the switch accumulates in
        # fp32 and returns the sum rounded once to the wire type (|rel err| <= 2^-9 for bf16) before the fp32 master
        # update.  allgather keeps the rank-ordered P2P sum (every rank must produce bit-identical sums), async keeps
        # it because only the selected contributors may be summed.  'nvls' / 'p2p' force either.
        auto_nvls = (nvls_ok and self.mode == "ps" and self.size >= 4
                     and os.environ.get("PSB200_REDUCE", "") != "p2p")
        if reduce == "p2p":
            self.reduce = 0
        else:
            self.reduce = 1 if (reduce == "nvls" or (reduce == "auto" and (auto_nvls or (
                nvls_ok and os.environ.get("PSB200_REDUCE", "") == "nvls")))) else 0

        # ---- the launch plan ----
        self.plan = None
        if self.is_server:
            P = self.m.UpdatePlan()
            P.kind, P.wire, P.opt = self.kind, self.wire, (0 if opt.optim == "sgd" else 1)
            P.grid = min(nt, self.m.update_max_grid(self.kind, self.wire, P.opt))
            pub = self.off_stage if self.consistent else self.off_param      # where fresh parameters are published
            for r in range(self.size):
                base = A.ptrs[r]
                P.set_rank_ptrs(r, base + self.off_wire, base + self.off_scales, base + pub,
                                base + self.off_signal)
            P.configure(self.size, self.rank, nt, self.bpt, self.cap, self.dt, self.bcast, self.reduce,
                        (A.mc_ptr + pub) if mc else 0, (A.mc_ptr + self.off_wire) if mc else 0,
                        A.local_ptr + pub,
                        self.master.data_ptr() if self.master is not None else 0,
                        self.buf0.data_ptr() if self.buf0 is not None else 0,
                        self.buf1.data_ptr() if self.buf1 is not None else 0,
                        self.buf2.data_ptr() if self.buf2 is not None else 0,
                        self.tiles.data_ptr(), A.local_ptr + self.off_signal,
                        self.counters.data_ptr(), self.counters.data_ptr() + 4)
            self.plan = P
        self.comm_stream = torch.cuda.Stream(device=self.device)
        self._cs = self.comm_stream.cuda_stream            # raw handle for explicit-stream launches
        self._ev_pool = [torch.cuda.Event() for _ in range(64)]
        self._ev_i = 0
        self._tiles_ptr = self.tiles.data_ptr()
        self._wire_ptr = self.arena.local_ptr + self.off_wire
        self._scales_ptr = self.arena.local_ptr + self.off_scales
        self._amax_ptr = self.amax.data_ptr()
        self._residual_ptr = self.residual.data_ptr() if self.residual is not None else 0
        self._sigctr_ptr = self.counters.data_ptr() + 8
        self._ratio = float(self.spec.ratio)
        self._sig_base = [p + self.off_signal for p in self.arena.ptrs]
        # ---- the pipeline chunks: contiguous runs of whole parameters in arena (= backward) order ----
        self._make_chunks()
        self._fired: set = set()
        self._keep: List[torch.Tensor] = []
        self._keep_prev: List[torch.Tensor] = []   # last step's gradients: freed one step late (see _flush)
        self._prev_done = None                      # comm-stream completion of the last step
        self._raw_bytes = 0
        self._first_flush_done = False
        self.launches = 0                     # kernels of OURS launched (bench 'gpu_launches')
        self._closed = False
        self._gates: list = []
        self._prof = CudaStepTimer(bool(getattr(opt, "profile", False)))
        self._epoch = 0                       # completed engine steps (the epoch-flag clock)
        # block-wise QSGD: the step word of the Philox counter.  Counts every step of the run and is never rewound (recover()
        # restarts the epoch clock, not this), so no (seed, rank, step) key repeats; checkpoints carry it (MPI_PS.state_dict)
        self.rng_step = 0
        # async bookkeeping
        self.version = 0
        self._consumed = torch.zeros(64, dtype=torch.int64, device=self.device)
        self._select_out = torch.zeros(64, dtype=torch.int64, device=self.device)
        self._select_host = torch.zeros(64, dtype=torch.int64).pin_memory()
        self._async_done_workers: set = set()
        self._async_depth = max(1, int(os.environ.get("PSB200_ASYNC_DEPTH", "4")))
        self._async_ring = [{"host": torch.zeros(64, dtype=torch.int64).pin_memory(), "event": torch.cuda.Event(), "version": 0}
                            for _ in range(self._async_depth + 1)]
        self._async_pending: list = []
        self._async_i = 0
        self._async_applied = 0
        self._async_last = {"contributors": [], "param_version": 0, "staleness": {}, "updates_applied": 0}
        # K10 "no separate serialization pass": producers we own (our BN / stem / linear backward kernels) write their
        # gradient straight into this rank's wire arena when the wire layout IS the gradient layout
        self._direct_ok = (self.kind == KIND_DENSE and self.wire == wire_code_of(self.dtype) and self.mode == "ps"
                           and os.environ.get("PSB200_DIRECT_GRAD", "1") != "0")
        self.direct_grads = 0
        self.direct_names: set = set()
        if self._direct_ok:
            import functools
            for sl in self.layout.slots:
                sl.param.ps_grad_out = functools.partial(self.grad_out, sl.param)
        self._snap_version = 0
        self._snap_shadow = None
        self._step_hyp = None
        self._phyper_ptr = 0
        self._update_spans: list = []
        # device-timeout surfacing: an async copy of SIG_ERROR into pinned memory every few steps, read one poll late
        self._err_host = torch.zeros(1, dtype=torch.int64).pin_memory()
        self._err_event = None
        self._err_every = max(1, int(os.environ.get("PSB200_ERROR_POLL", "16")))
        self.world.barrier()

    def _check_same_layout_everywhere(self):
        """Every rank must describe the SAME flat arena (the kernels address peers' arenas by tile number): compare a fingerprint
        of mode / optimizer / dtype / wire format / parameter names and shapes across ranks and fail on all of them with the first
        difference.  The reference silently assumes identical models on every rank; a mismatch there hangs or corrupts."""
        if self.size == 1 or os.environ.get("PSB200_CHECK_LAYOUT", "1") == "0":
            return
        L = self.layout
        mine = (self.mode, self.opt.optim, str(self.dtype), int(self.kind), int(self.wire), int(self.bpt), L.nparams, L.ntiles,
                tuple((s.name, tuple(s.param.shape)) for s in L.slots))
        every = self.world.all_gather_object(mine)
        for r, other in enumerate(every):
            if other != every[0]:
                what = ["mode", "optimizer", "parameter dtype", "coding kind", "wire dtype", "bytes per tile", "number of parameters",
                        "number of tiles", "parameter names / shapes"]
                k = next(i for i in range(len(mine)) if other[i] != every[0][i])
                detail = ""
                if k == 8:
                    diff = [(a, b) for a, b in zip(every[0][8], other[8]) if a != b][:1]
                    detail = f": first difference {diff[0] if diff else (len(every[0][8]), len(other[8]))}"
                raise ValueError(f"rank {r} and rank 0 disagree on the {what[k]} ({other[k] if k < 8 else '...'} vs "
                                 f"{every[0][k] if k < 8 else '...'}){detail} — every rank must build the same model, coding and mode")

    def _make_chunks(self):
        """Static chunks of the update pipeline (identical on every rank: they depend on the layout only).

        Chunk ``k`` = arena tiles ``[lo, hi)`` holding whole parameters, at least ``chunk_bytes`` of parameter bytes
        each (the last one takes the remainder).  A chunk is encoded — and, on the server, gathered / updated /
        broadcast — as soon as every parameter in it AND in all earlier chunks has produced its gradient, while
        backward keeps running on the later chunks (``/root/reference/ps.py:140-148,159-162``: one collective per
        parameter, consumed as each completes)."""
        L = self.layout
        chunks = L.plan_chunks(self.psz, self.chunk_bytes, single=(not self.pipeline and self.mode != "async"))
        self.chunks = chunks
        self.nchunks = len(chunks)
        self.chunk_tiles = [(c[0].first_tile, c[-1].first_tile + c[-1].ntiles) for c in chunks]
        self._chunk_of = [0] * L.nparams
        for k, c in enumerate(chunks):
            for sl in c:
                self._chunk_of[sl.index] = k
        self._chunk_items: List[list] = [[] for _ in chunks]
        self._chunk_left = [len(c) for c in chunks]
        self._next_chunk = 0

    def _progress(self, epoch: int, chunk: int) -> int:
        """Monotone GRAD_READY value meaning "chunks 0..chunk of step ``epoch`` are in my wire arena"."""
        return (epoch - 1) * self.nchunks + chunk + 1

    # ---------------------------------------------------------------------------------- state
    @staticmethod
    def _like(flat: torch.Tensor, param: torch.Tensor) -> torch.Tensor:
        """View a flat arena slice with the parameter's shape AND physical layout."""
        if flat.numel() != param.numel():          # custom placement (layout.py): same strides over the same span
            return torch.as_strided(flat, param.shape, param.stride())
        if param.is_contiguous() or not _dense(param):
            return flat.view(param.shape)
        return torch.as_strided(flat, param.shape, param.stride())

    def _expose_state(self):
        """Make ``opt.state[p]`` views of the flat fp32 state (checkpoint parity, SURVEY §5)."""
        o = self.opt
        for s in self.layout.slots:
            st = o.state[s.param]
            sl = slice(s.offset, s.offset + s.numel)
            if o.optim == "sgd":
                if self.buf0 is not None:
                    st["momentum_buffer"] = self._like(self.buf0[sl], s.param)
            else:
                st.setdefault("step", 0)
                st["exp_avg"] = self._like(self.buf0[sl], s.param)
                st["exp_avg_sq"] = self._like(self.buf1[sl], s.param)
                if self.buf2 is not None:
                    st["max_exp_avg_sq"] = self._like(self.buf2[sl], s.param)
            if self.master is not None:
                st["master_param"] = self._like(self.master[sl], s.param)

    def sync_state_to_torch(self):
        if not self.is_server:
            return
        o = self.opt
        for s in self.layout.slots:   # SGD too: the first-step momentum rule (ps.py:203-205) needs it on resume
            o.state[s.param]["step"] = self._param_steps[s.index] if self.mode != "async" else self._group_steps[s.group]

    def sync_state_from_torch(self, original=None):
        """After ``load_state_dict``: copy loaded tensors back into the flat (fp32) state.

        ``original`` maps ``id(param)`` → the un-cast saved state of that parameter."""
        if not self.is_server:
            return
        o = self.opt
        with torch.no_grad():
            for s in self.layout.slots:
                st = o.state.get(s.param, {})
                if original is not None and id(s.param) in original:
                    st = original[id(s.param)]
                sl = slice(s.offset, s.offset + s.numel)
                for key, buf in (("momentum_buffer", self.buf0 if o.optim == "sgd" else None),
                                 ("exp_avg", self.buf0 if o.optim == "adam" else None),
                                 ("exp_avg_sq", self.buf1), ("max_exp_avg_sq", self.buf2),
                                 ("master_param", self.master)):
                    if buf is not None and key in st and st[key] is not None:
                        if st[key].data_ptr() != buf[sl].data_ptr():
                            self._like(buf[sl], s.param).copy_(st[key].to(buf.dtype))
                if "step" in st:
                    self._group_steps[s.group] = max(self._group_steps[s.group], int(st["step"]))
                    self._param_steps[s.index] = int(st["step"])
            if self.master is not None:
                # parameters may have been re-loaded by the user: re-seed masters that lack a saved copy
                for s in self.layout.slots:
                    src = original.get(id(s.param), {}) if original is not None else o.state.get(s.param, {})
                    if "master_param" not in src:
                        self._like(self.master[s.offset: s.offset + s.numel], s.param).copy_(s.param.data.float())
        if any(self._param_steps[s.index] != self._group_steps[s.group] for s in self.layout.slots):
            self._uniform_steps = False
        self._expose_state()

    # ------------------------------------------------------------------------------- backward
    def grad_out(self, param: torch.nn.Parameter) -> Optional[torch.Tensor]:
        """Where the producer of ``param``'s gradient may write it DIRECTLY: a view of this rank's wire arena with the
        parameter's shape and physical layout — or ``None`` (coded wires, other modes).

        With Identity / same-dtype wires the wire tile of a parameter is bit-for-bit its gradient, so a kernel we own
        (fused BN backward, the stem's implicit weight gradient, ``BcastLinear``'s dW GEMM with ``out=``) can skip the
        ``psb_encode_kernel`` copy: ``on_grad`` recognises the pointer and only counts the parameter as arrived.  Safe in
        ``mode='ps'`` only: a worker's backward starts after it observed PARAMS_READY (the server finished reading the
        previous wire tiles); in ``allgather`` mode peers may still be reading them (CONSUMED is awaited on the comm stream)."""
        if not self._direct_ok or self._closed:
            return None
        sl = self.layout.by_id.get(id(param))
        if sl is None:
            return None
        flat = self.wire_arena[sl.first_tile * self.bpt: sl.first_tile * self.bpt + sl.numel * self.psz].view(self.dtype)
        return self._like(flat, param) if sl.strides is None else torch.as_strided(flat, param.shape, sl.strides)

    def on_grad(self, grad: torch.Tensor, name: str, param: torch.nn.Parameter):
        """Backward hook (``ps.py:98-101``): file the gradient under its chunk; every chunk that is now complete (in
        arena order) is encoded — and on the server gathered / updated / broadcast — right away, under backward."""
        s = self.layout.by_id[id(param)]
        g = grad.detach()
        if self._direct_ok and g.data_ptr() == self._wire_ptr + s.first_tile * self.bpt and g.dtype == self.dtype \
                and g.stride() == param.stride():
            # the producer already wrote this gradient into the wire arena (grad_out): nothing to encode
            if s.index in self._fired:
                raise RuntimeError(f"parameter {name!r} produced two gradients before step()")
            self._fired.add(s.index)
            k = self._chunk_of[s.index]
            self._chunk_left[k] -= 1
            self._raw_bytes += s.numel * self.psz
            self.direct_grads += 1
            self.direct_names.add(name)
            if param.grad is not None:
                # AccumulateGrad would add the incoming gradient INTO param.grad in place — and both may alias the same wire
                # tile (zero_grad(set_to_none=False)): drop the old one so the new gradient is assigned, not accumulated
                param.grad = None
            while self._next_chunk < self.nchunks and self._chunk_left[self._next_chunk] == 0:
                self._flush_chunk(self._next_chunk)
            return
        if g.dtype != self.dtype:
            g = g.to(self.dtype)
        if s.strides is not None:
            # custom placement: the encode kernel reads the whole span, padding included (it must be zero)
            if not (g.stride() == param.stride() and g.data_ptr() % 16 == 0 and g.storage_offset() * g.element_size() +
                    s.numel * g.element_size() <= g.untyped_storage().nbytes()):
                span = torch.zeros(s.numel, dtype=g.dtype, device=g.device)
                torch.as_strided(span, param.shape, s.strides).copy_(g)
                g = span
            else:
                g = torch.as_strided(g, (s.numel,), (1,))
        elif g.stride() != param.stride() or g.data_ptr() % 16:
            # the arena is in the parameter's physical order: bring the gradient into it
            g = torch.empty_strided(param.shape, param.stride(), dtype=g.dtype, device=g.device).copy_(g)
        if s.index in self._fired:           # gradient accumulation: later micro-batches add up
            raise RuntimeError(f"parameter {name!r} produced two gradients before step(); "
                               "call step() after every backward (the reference encodes per backward)")
        self._fired.add(s.index)
        k = self._chunk_of[s.index]
        self._chunk_items[k].append((s, g))
        self._chunk_left[k] -= 1
        self._raw_bytes += s.numel * self.psz
        while self._next_chunk < self.nchunks and self._chunk_left[self._next_chunk] == 0:
            self._flush_chunk(self._next_chunk)

    def _event(self, timing: bool = False):
        """A pooled CUDA event (creating one costs more than recording one)."""
        if timing:
            return torch.cuda.Event(enable_timing=True)
        self._ev_i = (self._ev_i + 1) % len(self._ev_pool)
        return self._ev_pool[self._ev_i]

    def _flush_chunk(self, k: int, joined: bool = False, active_ptr: int = 0):
        """Everything chunk ``k`` needs, queued on the comm stream (explicit stream handle: no Python-side stream
        switching): encode its gradients into the wire arena, raise this rank's GRAD_READY progress flag from the
        last encode CTA, and — on the server — launch the fused gather/update/broadcast kernel for exactly these tiles.

        Must be called in chunk order.  ``joined``: the caller already made the comm stream wait for the compute stream."""
        assert k == self._next_chunk
        self._next_chunk = k + 1
        m, cs, csh = self.m, self.comm_stream, self._cs
        cur = torch.cuda.current_stream(self.device)
        if not joined:
            ev = self._event()
            ev.record(cur)
            cs.wait_event(ev)
        if not self._first_flush_done:
            if self._prev_done is not None:
                # Bound the comm stream's lag to one step: gradients are kept alive (not record_stream'ed, which
                # would make the caching allocator grow and cudaMalloc for several steps) until the step after
                # they were encoded, so the compute stream must not run further ahead than that.
                cur.wait_event(self._prev_done)
            self._first_flush_done = True
            self._before_first_encode()
        epoch = self._epoch + 1
        last = k == self.nchunks - 1
        n = self.size
        sync = self.mode != "async"                   # async posts its flag from _step_async
        # the launching rank's own gradient is ordered by the stream, so the server neither signals nor waits itself
        must_signal = sync and n > 1 and not (self.mode == "ps" and self.rank == 0) and (self.pipeline or last)
        sig = None
        if must_signal:
            sb = self._sig_base
            targets = [sb[0]] if self.mode == "ps" else [b for r, b in enumerate(sb) if r != self.rank]
            sig = (targets, m.SIG_GRAD_READY + self.rank, self._progress(epoch, k))
        items, self._chunk_items[k] = self._chunk_items[k], []
        if items:
            grads = [g for _, g in items]
            qsgd = {}
            if self.kind == KIND_QSGD:
                qsgd = dict(levels=self.spec.levels, seed=self.spec.seed, rng_step=self.rng_step & 0xFFFFFFFF, rank=self.rank)
            m.encode(self.kind, self.wire, grads, [s.first_tile for s, _ in items],
                     [s.ntiles for s, _ in items], [s.index for s, _ in items],
                     self._tiles_ptr, self._wire_ptr, self._scales_ptr, self._amax_ptr, self._residual_ptr,
                     self.bpt, self.cap, self._ratio,
                     *((sig[0], sig[1], sig[2], self._sigctr_ptr) if sig else ([], 0, 0, 0)),
                     csh, **qsgd)
            nb = (len(items) + 63) // 64
            self.launches += nb * (2 if self.kind == KIND_SCALED else 1)
            self._keep.extend(grads)
        elif sig:                                     # nothing fired in this chunk: the flag alone
            m.signal(sig[0], sig[1], sig[2], -1, 0, csh)
            self.launches += 1
        if sync and self.is_server and (self.pipeline or last):
            lo, hi = self.chunk_tiles[k] if self.pipeline else (0, self.layout.ntiles)
            inv = (1.0 / n) if self.opt.average else 1.0
            prof = self._prof.enabled
            ev_a = self._prof.mark(cs) if prof else None
            wait_mask = ((1 << n) - 1) & ~(1 << self.rank)
            if n > 1:
                # The req.Wait() for this chunk is a ONE-WARP kernel, not the update grid: 444 update CTAs spinning on the
                # peers' flags would hold every SM's register file (3 x 256 threads x 77 registers) while this rank's own
                # backward still has chunks k+1.. to produce — the skew between ranks would land on the critical path.
                m.wait_flags(self.arena.local_ptr + self.off_signal, m.SIG_GRAD_READY, wait_mask, self._progress(epoch, k),
                             self.timeout_s, csh)
                self.launches += 1
            self.plan.launch(epoch, self._get_hypers(), (1 << n) - 1, inv, 0,
                             (0 if n == 1 else (1 if self.mode == "ps" else 2)) if last else 0,
                             active_ptr=active_ptr, timeout_s=self.timeout_s,
                             wait_mask=wait_mask, stream=csh,
                             tile_begin=lo, tile_end=hi, wait_value=self._progress(epoch, k),
                             param_hyper=self._phyper_ptr)
            self.launches += 1
            if prof:
                self._update_spans.append((ev_a, self._prof.mark(cs)))

    def _before_first_encode(self):
        """Queued on the comm stream before this step's first write into the wire arena."""
        epoch = self._epoch + 1              # the step these gradients belong to
        if self.kind == KIND_SCALED:
            with torch.cuda.stream(self.comm_stream):
                self.amax.zero_()
        if self.size == 1:
            return
        sig = self.arena.local_ptr + self.off_signal
        if self.mode == "allgather" and epoch > 1:
            # every peer must have finished READING our previous wire tiles
            self.m.wait_flags(sig, self.m.SIG_CONSUMED, ((1 << self.size) - 1) & ~(1 << self.rank), epoch - 1,
                              self.timeout_s, self._cs)
            self.launches += 1
        elif self.mode == "async" and self.rank != 0 and epoch > 1:
            self.m.wait_flags(sig, self.m.SIG_ACK, 1, epoch - 1, self.timeout_s, self._cs)
            self.launches += 1

    # ----------------------------------------------------------------------------------- step
    def _get_hypers(self):
        """This step's per-group hyper-parameter tuples (sampled once per step, at the first chunk that needs them)."""
        if self._step_hyp is None:
            self._step_hyp = self._hypers()
            self._phyper_ptr = 0
            if not self._uniform_steps and self.is_server:
                self._phyper_ptr = self._upload_param_hypers()
        return self._step_hyp

    def _upload_param_hypers(self) -> int:
        """Per-parameter {step_size, first_step} for THIS step, assuming the parameter fires (tiles of parameters that do not
        are skipped through the active mask, so their entries are never read)."""
        o = self.opt
        slot = self._epoch % len(self._phyper_host)       # the comm stream lags the host by at most one step
        h, dev = self._phyper_host[slot], self._phyper_dev[slot]
        for sl in self.layout.slots:
            t = self._param_steps[sl.index] + 1
            g = o.param_groups[sl.group]
            if o.optim == "adam":
                b1, b2 = g["betas"]
                h[sl.index, 0] = float(g["lr"]) * math.sqrt(1 - b2 ** t) / (1 - b1 ** t)
            else:
                h[sl.index, 0] = 0.0
            h[sl.index, 1] = 1.0 if t == 1 else 0.0
        with torch.cuda.stream(self.comm_stream):
            dev.copy_(h, non_blocking=True)
        return dev.data_ptr()

    def _hypers(self) -> List[List[float]]:
        o = self.opt
        out = []
        if o.optim == "sgd":
            # SGD's tuple only changes with lr schedules / the first step: reuse the cached list otherwise
            key = tuple((g["lr"], g["weight_decay"], g["momentum"], g["dampening"], g["nesterov"]) for g in o.param_groups)
            for gi in range(len(o.param_groups)):
                self._group_steps[gi] += 1
            first = any(t == 1 for t in self._group_steps)
            if not first and self._hyper_cache is not None and self._hyper_cache[0] == key:
                return self._hyper_cache[1]
        for gi, g in enumerate(o.param_groups):
            if o.optim != "sgd":
                self._group_steps[gi] += 1
            t = self._group_steps[gi]
            if o.optim == "sgd":
                out.append([float(g["lr"]), float(g["weight_decay"]), float(g["momentum"]), float(g["dampening"]),
                            0.0, 0.0, 0.0, 0.0, float(bool(g["nesterov"])), 0.0, float(t == 1)])
            else:
                b1, b2 = g["betas"]
                step_size = float(g["lr"]) * math.sqrt(1 - b2 ** t) / (1 - b1 ** t)     # ps.py:257-259
                out.append([float(g["lr"]), float(g["weight_decay"]), 0.0, 0.0, float(b1), float(b2),
                            float(g["eps"]), step_size, 0.0, float(bool(g.get("amsgrad", False))), float(t == 1)])
        if o.optim == "sgd" and not any(t == 1 for t in self._group_steps):
            self._hyper_cache = (key, out)
        return out

    def _handle_inactive(self):
        """Parameters whose hook did not fire this step (``p.grad is None``, ``ps.py:178-179``)."""
        L = self.layout
        if len(self._fired) == L.nparams:
            if not self._active_all:
                self.active_host.fill_(1)
                self.active_dev.copy_(self.active_host, non_blocking=True)
                self._active_all = True
                self._last_fired = None
            return 0
        fired = frozenset(self._fired)
        if fired == self._last_fired:        # same frozen / unused set as last step: mask and zeroed tiles still valid
            return self.active_dev.data_ptr()
        self._last_fired = fired
        self.active_host.zero_()
        for i in self._fired:
            self.active_host[i] = 1
        self.active_dev.copy_(self.active_host, non_blocking=True)
        self._active_all = False
        # a tile the server will read must not carry last step's payload
        for s in L.slots:
            if s.index not in self._fired:
                self.wire_arena[s.first_tile * self.bpt: (s.first_tile + s.ntiles) * self.bpt].zero_()
        return self.active_dev.data_ptr()

    def _flush_rest(self, cs, joined: bool):
        """step(): chunks that did not complete during backward (always the last one's tail when every parameter
        fired from the final hook; all of them when some parameter got no gradient, ``ps.py:178-179``)."""
        if self._next_chunk >= self.nchunks:
            if not self._active_all:                  # every parameter fired again: forget the frozen-set cache
                self._active_all, self._last_fired = True, None
            return
        if len(self._fired) == self.layout.nparams and self._active_all:
            active_ptr = 0                            # the common case: every parameter got a gradient
        else:
            with torch.cuda.stream(cs):
                active_ptr = self._handle_inactive()  # before the flag: a tile the server reads must be final
        while self._next_chunk < self.nchunks:
            self._flush_chunk(self._next_chunk, joined=joined, active_ptr=active_ptr)

    def step(self) -> Dict[str, float]:
        t0 = time.time()
        data = {"comm_wait": 0.0, "optim_step_time": 0.0, "decode_time": 0.0,
                "iallgather_prepare_time": 0.0, "isend_time": 0.0}
        if self.mode == "async" and self.size > 1:
            return self._step_async(data)
        epoch = self._epoch + 1
        m, cs = self.m, self.comm_stream
        prof = self._prof.enabled
        cur = torch.cuda.current_stream(self.device)
        ev = self._event(timing=prof)
        ev.record(cur)                       # backward is complete up to here
        pending = self._next_chunk < self.nchunks
        if pending:
            cs.wait_event(ev)
        data["code_wait"] = time.time() - t0
        t2 = time.time()
        self._flush_rest(cs, joined=True)
        self._get_hypers()                   # workers too: keeps the per-group step counters aligned with the server
        data["optim_step_time"] = time.time() - t2
        data["isend_time"] = 0.0
        done = self._event()
        done.record(cs)
        t3 = time.time()
        if self.size > 1 and self.mode == "ps" and self.rank != 0:
            if not self._gates:
                # the req.Wait() of mpi_comms.py:121 — a one-thread kernel on the compute stream
                m.wait_flags(self._sig_base[self.rank], m.SIG_PARAMS_READY, 1, epoch, self.timeout_s)
                self.launches += 1
            # else: the first forward GEMM (BcastLinear / the stem) acquires the flag inside its TMA producer
        else:
            cur.wait_event(done)
        data["comm_wait"] = time.time() - t3
        data["chunks"] = self.nchunks
        if prof:
            ev_d = self._prof.mark(cur)
            self._prof.span("dev_step_tail_time", ev, ev_d)     # backward-done → parameters usable, on the compute stream
            if self._update_spans:
                self._prof.span("dev_gather_update_bcast_time", *self._update_spans[-1])   # the LAST chunk's kernel
                self._prof.span("dev_update_pipeline_time", self._update_spans[0][0], self._update_spans[-1][1])
            self._update_spans = []
            data.update(self._prof.harvest())                   # device timings of the most recent COMPLETED step
        self._end_of_step(data, done)
        return data

    def _end_of_step(self, data, done=None):
        L = self.layout
        nfired = max(len(self._fired), 1)
        data["msg_bytes"] = self._raw_bytes / nfired
        wire_bytes = sum(L.slots[i].ntiles for i in self._fired) * self.bpt if self._fired else 0
        data["packaged_bytes"] = wire_bytes / nfired
        data["engine"] = "device"
        self._epoch += 1
        self.rng_step += 1
        if len(self._fired) != L.nparams:
            self._uniform_steps = False              # some parameter sat this step out: per-parameter counts diverge from now on
        for i in self._fired:
            self._param_steps[i] += 1
        self._fired = set()
        self._keep_prev, self._keep = self._keep, []
        if done is None:                     # comm-stream completion marker of this step (see _flush)
            done = self._event()
            done.record(self.comm_stream)
        self._prev_done = done
        self._raw_bytes = 0
        self._first_flush_done = False
        self._step_hyp = None
        self._next_chunk = 0
        self._chunk_left = [len(c) for c in self.chunks]
        for it in self._chunk_items:
            it.clear()
        if os.environ.get("PSB200_CHECK") == "1":
            self.check()
        elif self.size > 1 and self._epoch % self._err_every == 0:
            self._poll_error()

    def _poll_error(self):
        """Surface device-side time-outs WITHOUT a sync: every ``PSB200_ERROR_POLL`` steps an async copy of SIG_ERROR
        lands in pinned memory; the previous poll's value is read once its event has completed."""
        if self._err_event is not None and self._err_event.query():
            err = int(self._err_host[0])
            if err:
                raise RuntimeError(f"rank {self.rank}: a device-side wait timed out (code {err}) — a peer is stalled or "
                                   f"dead; synchronisation is disabled until recover() (PSB200_DEVICE_TIMEOUT="
                                   f"{self.timeout_s:.0f} s)")
            self._err_event = None
        if self._err_event is None:
            with torch.cuda.stream(self.comm_stream):
                self._err_host.copy_(self.signal[self.m.SIG_ERROR: self.m.SIG_ERROR + 1], non_blocking=True)
                self._err_event = torch.cuda.Event()
                self._err_event.record(self.comm_stream)

    def recover(self):
        """Collective recovery after a surfaced time-out: bring every rank back to a common, clean protocol state so that
        training can continue (the reference has no failure handling at all; a dead rank hangs ``mpirun`` for good).

        A timed-out step leaves the ranks' epoch clocks and progress flags misaligned (the stalled rank never posted its
        chunks; chunks gathered before the stall may already have been applied and published).  So: quiesce, clear every
        rank's signal pad and error slot, restart the epoch / chunk clocks at zero, re-adopt rank 0's parameters (and, in
        ``allgather`` mode where optimizer state is replicated, rank 0's state and step counts — through the slow object
        path: this is a rare event), and re-open.  Optimizer step counts keep counting the failed step, and so does the QSGD
        RNG step (a rounding draw is never reused)."""
        torch.cuda.synchronize(self.device)
        self.world.barrier()                  # every rank is here: nobody launches into the old epoch any more
        with torch.no_grad():
            self.signal.zero_()               # peers only ever store flags into this pad, and all of them are quiescent
            self.counters.zero_()
            self._consumed.zero_()
            self._select_out.zero_()
        self._err_host.zero_()
        self._err_event = None
        self._epoch = 0
        self._fired = set()
        self._keep, self._keep_prev = [], []
        self._prev_done = None
        self._raw_bytes = 0
        self._first_flush_done = False
        self._step_hyp = None
        self._next_chunk = 0
        self._chunk_left = [len(c) for c in self.chunks]
        for it in self._chunk_items:
            it.clear()
        self._gate_epoch = -1
        self.version = 0
        self._async_pending, self._async_done_workers = [], set()
        self._snap_version = 0
        if self._snap_shadow is not None:
            self._snap_scratch.copy_(torch.tensor([0, -1, 0, 0, 0, 0], dtype=torch.int64))
            self._snap_event = None
        torch.cuda.synchronize(self.device)
        self.world.barrier()                  # all pads are clean before anybody reads a peer's memory
        if self.size > 1:
            L = self.layout
            nbytes = L.numel_padded * self.psz
            with torch.no_grad():
                src = self.arena.tensor(self.off_stage if self.consistent else self.off_param, nbytes, self.dtype, rank=0)
                if self.rank != 0 or self.consistent:
                    self.param_arena.copy_(src)
                if self.consistent and self.rank != 0:
                    self.stage_arena.copy_(src)
                if self.mode == "allgather":
                    bufs = [b for b in (self.master, self.buf0, self.buf1, self.buf2) if b is not None]
                    state = self.world.broadcast_object(
                        ([b.cpu() for b in bufs], self._group_steps, self._param_steps, self._uniform_steps)
                        if self.rank == 0 else None, src=0)
                    if self.rank != 0:
                        for b, v in zip(bufs, state[0]):
                            b.copy_(v)
                        self._group_steps, self._param_steps = list(state[1]), list(state[2])
                        self._uniform_steps = bool(state[3])
                        self._hyper_cache = None
            torch.cuda.synchronize(self.device)
            self.world.barrier()

    def resync_master(self):
        """Re-seed the fp32 master weights from the (bf16/fp16) parameters — call after changing parameters in place
        behind the optimizer's back (``model.load_state_dict`` without ``opt.load_state_dict``, manual re-init, EMA
        swaps): every update writes master → parameters, so un-synced edits would be overwritten."""
        if self.master is not None:
            torch.cuda.current_stream(self.device).wait_stream(self.comm_stream)
            with torch.no_grad():
                self.master.copy_(self.param_arena)

    # ------------------------------------------------------------------------------ async mode
    def _step_async(self, data):
        o = self.opt
        sig_base = [p + self.off_signal for p in self.arena.ptrs]
        cs = self.comm_stream
        cur = torch.cuda.current_stream(self.device)
        if self.rank != 0:
            epoch = self._epoch + 1
            ev = torch.cuda.Event()
            ev.record(cur)
            cs.wait_event(ev)
            self._flush_rest(cs, joined=True)        # chunks not yet encoded during backward (+ inactive parameters)
            with torch.cuda.stream(cs):
                if not self._first_flush_done:       # no parameter produced a gradient at all
                    self._first_flush_done = True
                    self._before_first_encode()
                # publish "gradient `epoch` is in my arena" + the parameter version it was computed on (staleness accounting)
                self.m.signal([sig_base[0]], self.m.SIG_GRAD_READY + self.rank, epoch, -1, 0, 0,
                              self.arena.local_ptr + self.off_signal, self.m.SIG_GRAD_VERSION + self.rank)
                self.launches += 1
            if self.consistent:
                data["param_version"] = self._snapshot()
            self._end_of_step(data)
            return data                      # never waits for NEW parameters (inconsistent reads unless consistent=True)
        # ---- rank 0: the server — device-resident: select → (open sequence lock) → update → ack are all queued without
        # looking at their result; results come back through a ring of pinned slots, read when their event has completed.
        # The host only blocks when it is `_async_depth` iterations AHEAD of the GPU (never the other way round). ----
        self._fired = set()
        self._keep = []
        self._next_chunk = 0
        self._chunk_left = [len(c) for c in self.chunks]
        for it in self._chunk_items:
            it.clear()
        n = self.size
        self._async_harvest(block=False)
        cand = ((1 << n) - 1) & ~1
        for r in self._async_done_workers:
            cand &= ~(1 << r)
        if cand == 0:
            self._async_harvest(block=True, everything=True)
            data.update(self._async_last)
            data["ps_done"] = True
            data["engine"] = "device"
            return data
        quota = max(1, min(o.quota, bin(cand).count("1")))
        t0 = time.time()
        slot = self._async_ring[self._async_i % len(self._async_ring)]
        self._async_i += 1
        self.version += 1
        hyp = self._hypers()
        self.m.select_ready(sig_base[0], self._consumed.data_ptr(), cand, quota, self._select_out.data_ptr(),
                            self.timeout_s, self.version, sig_base if self.consistent else [], self._cs)
        self.plan.launch(o.steps, hyp, 0, 1.0, 0, 1, 0, self.version, self._select_out.data_ptr(),
                         1 if o.average else 0, 0, self.timeout_s, stream=self._cs)
        self.launches += 2
        with torch.cuda.stream(cs):
            slot["host"].copy_(self._select_out, non_blocking=True)
        slot["event"].record(cs)
        slot["version"] = self.version
        self._async_pending.append(slot)
        if len(self._async_pending) >= self._async_depth:
            self._async_harvest(block=True)          # the host is a full ring ahead of the device: wait for the oldest
        data["comm_wait"] = time.time() - t0
        data.update(self._async_last)                # contributors / staleness / version of the latest COMPLETED update
        data["param_version_queued"] = self.version
        data["ps_done"] = False
        self._epoch += 1
        data["engine"] = "device"
        return data

    def _async_harvest(self, block: bool, everything: bool = False):
        """Consume completed server iterations in order (``block``: wait for the oldest; ``everything``: drain)."""
        n = self.size
        while self._async_pending:
            slot = self._async_pending[0]
            if not slot["event"].query():
                if not block:
                    return
                slot["event"].synchronize()
            self._async_pending.pop(0)
            h = slot["host"]
            mask, cnt, finished = int(h[0]), int(h[1]), int(h[40])
            for r in range(n):
                if finished >> r & 1:
                    self._async_done_workers.add(r)
            contributors = [r for r in range(n) if mask >> r & 1]
            if cnt == 0:
                # nothing was applied (every worker finished, or the select timed out): the kernels returned early, the
                # sequence lock was never opened, no version was published — take the host-side prediction back
                self.version -= 1
                for gi in range(len(self._group_steps)):
                    self._group_steps[gi] -= 1
            else:
                self._async_applied += 1
                self._async_last = {"contributors": contributors, "param_version": slot["version"],
                                    "staleness": {r: int(h[44 + r]) for r in contributors},
                                    "updates_applied": self._async_applied}
            if not everything:
                block = False                        # at most one blocking wait per call

    # ------------------------------------------------------------------ consistent reads (async)
    def _snapshot(self, block: bool = False) -> int:
        """Adopt the newest COMPLETE parameter version from the staging copy — entirely on the device.

        The server writes ``BEGIN = v`` before and ``VERSION = v`` after publishing version ``v`` into the staging arena.
        ``psb_snapshot_fetch`` copies staging → a local shadow buffer iff ``BEGIN == VERSION`` before and ``BEGIN`` is unchanged
        after (every CTA must agree); ``psb_snapshot_commit`` then copies shadow → the live parameter arena.  A vetoed attempt
        leaves the parameters on the previous whole version, so the model never reads a torn set.  No host reads: the adopted
        version comes back through an async copy into pinned memory and is reported one call late (``block=True``: wait)."""
        m = self.m
        cur = torch.cuda.current_stream(self.device)
        if self._snap_shadow is None:
            self._snap_shadow = torch.empty_like(self.param_arena)
            self._snap_scratch = torch.tensor([0, -1, 0, 0, 0, 0], dtype=torch.int64, device=self.device)
            self._snap_host = torch.zeros(1, dtype=torch.int64).pin_memory()
            self._snap_event = None
        nbytes = self.param_arena.numel() * self.psz
        m.snapshot(self.arena.local_ptr + self.off_signal, self.stage_arena.data_ptr(), self._snap_shadow.data_ptr(),
                   self.param_arena.data_ptr(), nbytes, self._snap_scratch.data_ptr(),
                   int(os.environ.get("PSB200_SNAPSHOT_ATTEMPTS", "2")), cur.cuda_stream)
        self.launches += 4
        if self._snap_event is None or self._snap_event.query() or block:
            if self._snap_event is not None and self._snap_event.query():
                self._snap_version = int(self._snap_host[0])
            self._snap_host.copy_(self._snap_scratch[5:6], non_blocking=True)
            self._snap_event = torch.cuda.Event()
            self._snap_event.record(cur)
        if block:
            self._snap_event.synchronize()
            self._snap_version = int(self._snap_host[0])
        return self._snap_version

    # -------------------------------------------------------------- broadcast-gated GEMM support
    def register_gate(self, layer) -> None:
        """A :class:`~pytorch_ps_mpi_b200.ops.linear.BcastLinear` will acquire ``PARAMS_READY`` itself,
        so worker ``step()`` stops queueing the separate wait kernel (the GEMM is the Wait)."""
        self._gates.append(layer)

    def gate(self):
        """``(flag_ptr, epoch)`` the next forward must observe before reading broadcast weights.  Taking it marks the
        current epoch's broadcast as acquired by a gated kernel (see :meth:`ensure_params`)."""
        if self.size == 1 or self.mode != "ps" or self.rank == 0 or self._epoch == 0:
            return 0, 0
        self._gate_epoch = self._epoch
        return self.arena.local_ptr + self.off_signal + 8 * self.m.SIG_PARAMS_READY, self._epoch

    def ensure_params(self):
        """For forwards that bypass the gated kernel (eval mode, unsupported shapes) while a gate is registered: queue
        the plain wait kernel on the current stream unless this epoch's broadcast was already acquired."""
        if self.size == 1 or self.mode != "ps" or self.rank == 0 or self._epoch == 0 or not self._gates:
            return
        if getattr(self, "_gate_epoch", -1) == self._epoch:
            return
        self._gate_epoch = self._epoch
        self.m.wait_flags(self._sig_base[self.rank], self.m.SIG_PARAMS_READY, 1, self._epoch, self.timeout_s)
        self.launches += 1

    def peer_param_ptr(self, param: torch.Tensor, rank: int) -> int:
        """Address of ``param`` inside rank ``rank``'s parameter arena as mapped in this process."""
        return self.arena.ptrs[rank] + (param.data_ptr() - self.arena.local_ptr)

    # ------------------------------------------------------------------------------ diagnostics
    def check(self):
        """Raise if any bounded spin timed out (forces a device sync; off the hot path)."""
        torch.cuda.synchronize(self.device)
        err = int(self.signal[self.m.SIG_ERROR].item())
        if err:
            raise RuntimeError(f"rank {self.rank}: a device-side wait timed out (code {err}); "
                               "a peer is stalled or dead")

    def close(self):
        if self._closed:
            return
        self._closed = True
        try:
            if self.mode == "async" and self.size > 1 and self.rank != 0:
                with torch.cuda.stream(self.comm_stream):
                    if self._epoch > 0:      # the server must have consumed our last gradient first
                        self.m.wait_flags(self.arena.local_ptr + self.off_signal, self.m.SIG_ACK, 1,
                                          self._epoch, self.timeout_s)
                    self.m.signal([self.arena.ptrs[0] + self.off_signal],
                                  self.m.SIG_GRAD_READY + self.rank, _DONE_EPOCH)
            torch.cuda.synchronize(self.device)
            self.world.barrier()
            if self.consistent:              # everybody leaves with the server's final parameters
                self._snapshot(block=True)
        finally:
            # parameters keep their arena views alive; detach them so the block can be freed
            with torch.no_grad():
                for s in self.layout.slots:
                    s.param.data = s.param.data.clone()
                    if hasattr(s.param, "ps_grad_out"):
                        del s.param.ps_grad_out
                    if s.param.grad is not None and self._direct_ok:
                        s.param.grad = None          # may alias the wire arena that is about to be unmapped
            self.arena.close()
