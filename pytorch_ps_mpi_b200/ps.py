"""L4 public API: ``MPI_PS`` optimizer wrapper and its ``SGD`` / ``Adam`` subclasses.

Contract kept from ``/root/reference/ps.py``:

* ``SGD(model.named_parameters(), model.parameters(), lr=…, code=coder, optim='sgd', cuda=…)``
  — first positional is the *named* parameters, the rest is forwarded to the real torch
  optimizer constructor through the MRO (``ps.py:54-59,76``);
* every parameter is tagged with ``.name`` and gets a backward hook that encodes its gradient
  the moment autograd produces it, overlapping encode with the rest of backward
  (``ps.py:63-66,92-101``);
* ``loss, data = opt.step(closure=None)`` returns a **tuple** — ``data`` is the timing / byte
  accounting dict with the reference's keys (``ps.py:116,135-148,162,168,191,193``);
* gradients of all ranks are **summed**, not averaged (``ps.py:176``); parameters are processed
  in reverse registration (= backward) order and messages are paired to parameters by
  hook-firing order (``ps.py:121-123,155-156``);
* ``SGD.optim_step`` / ``Adam.optim_step`` implement the reference's update math
  (``ps.py:197-214,218-261``).

What is new (see DESIGN.md): three *modes* — ``'ps'`` (rank-0 parameter server: gather → sum →
step → broadcast, the README plan ``README.md:37-46``), ``'allgather'`` (the replicated scheme
the reference actually wires, ``ps.py:140-190``) and ``'async'`` (AsySG-InCon,
``README.md:56-81``) — and two *engines*: the device engine
(:mod:`pytorch_ps_mpi_b200.parallel.device_engine`: symmetric-memory arenas + fused sm_100a
kernels, used automatically for CUDA parameters with a built-in coding) and the host engine
below (generic Python objects / user codings over the shm / gloo transport; also the CPU
plumbing configuration).
"""
from __future__ import annotations

import math
import os
import pickle
import time
import weakref
from collections import OrderedDict
from concurrent.futures import Future, ThreadPoolExecutor
from functools import partial
from typing import Any, Dict, List, Optional

import torch

from . import codings as _codings
from . import mpi_comms as comms
from . import runtime
from .utils.misc import _bytes_of, find_param  # noqa: F401  (reference helpers, ps.py:25-50)

__all__ = ["MPI_PS", "SGD", "Adam", "_bytes_of", "find_param"]

_MODES = ("ps", "allgather", "async")
_QSGD_RNG_KEY = "qsgd_rng_step"      # extra top-level key of MPI_PS.state_dict() with a block-wise QSGD device engine
_TAG_GRAD, _TAG_PARAM = 11, 12


def _tag_name(param: torch.Tensor, name: str) -> None:
    """Tag a parameter with its name (``param.name = name``, ``ps.py:64``).

    ``torch.Tensor.name`` became a read-only C attribute in torch 2.x, so the tag lives in
    ``param.ps_name`` (and in ``param.__dict__['name']`` for introspection); :func:`find_param`
    reads ``ps_name``.
    """
    param.ps_name = name
    try:
        param.name = name
    except AttributeError:
        param.__dict__["name"] = name


def _accepts_name(fn) -> bool:
    """Does ``encode`` take a ``name=`` keyword (user codings written against the reference's ``encode(grad, **kw)`` do;
    a bare ``encode(grad)`` must keep working)?"""
    target = getattr(fn, "func", fn)
    cached = getattr(target, "_psb_accepts_name", None)
    if cached is not None:
        return cached
    import inspect
    try:
        params = inspect.signature(fn).parameters
        ok = "name" in params or any(p.kind is inspect.Parameter.VAR_KEYWORD for p in params.values())
    except (TypeError, ValueError):
        ok = False
    try:
        target.__dict__["_psb_accepts_name"] = ok
    except Exception:
        pass
    return ok


class MPI_PS(torch.optim.Optimizer):
    """Parameter-server data-parallel optimizer wrapper (``/root/reference/ps.py:53-193``).

    Parameters beyond the reference's (all keyword-only, all optional):

    mode : ``'ps'`` | ``'allgather'`` | ``'async'``
    average : divide the summed gradient by the number of contributions (default ``False`` =
        the reference's sum semantics, ``ps.py:176``)
    quota : async mode — gradients the PS consumes per update (``README.md:67-70``; default
        ``size - 1``)
    engine : ``'auto'`` | ``'device'`` | ``'host'``
    master_fp32 : device engine — keep fp32 master weights on the PS for bf16/fp16 parameters
    consistent : async mode — workers take whole-model snapshots instead of inconsistent reads
        (``README.md:79-81``)
    level : host engine byte-compression level (0 = framing only, as the reference's default)
    profile : device engine — record CUDA-event section timings into ``data`` (one step late)
    pipeline : device engine, sync modes — gather / update / broadcast each CHUNK of the arena as soon as its
        gradients exist, under the rest of backward (the reference posts one non-blocking collective per parameter and
        consumes each as it completes, ``ps.py:140-148,159-162``).  Parameters of finished chunks are therefore
        rewritten DURING ``backward()`` and the hyper-parameters are sampled at the first chunk: set the learning rate
        before ``backward()``, and do not read parameters between ``backward()`` and ``step()``.  ``pipeline=False``
        restores one fused launch inside ``step()``.
    coalesce : host engine — ship all parameters' messages of a step as ONE framed message instead of one
        collective per parameter (the reference's behaviour, ``ps.py:140-148``); same numerics, far fewer round trips
    """

    _default_optim = "sgd"

    def __init__(self, named_params, *args,
                 names=[],
                 optim=None,
                 code=None,
                 use_mpi=True, cuda=False,
                 mode: str = "ps",
                 average: bool = False,
                 quota: Optional[int] = None,
                 engine: str = "auto",
                 master_fp32: bool = True,
                 consistent: bool = False,
                 level: int = 0,
                 profile: bool = False,
                 reduce: str = "auto",
                 coalesce: bool = False,
                 pipeline: bool = True,
                 **kwargs):
        if mode not in _MODES:
            raise ValueError(f"mode must be one of {_MODES}")
        self.code = code if code is not None else _codings.Identity()
        self.optim = optim if optim is not None else self._default_optim
        self.mode, self.average, self.level = mode, bool(average), int(level)
        self.consistent, self.profile = bool(consistent), bool(profile)
        self.coalesce = bool(coalesce)
        self.pipeline = bool(pipeline)

        named_params = list(named_params)
        self._named = OrderedDict()
        for i, (name, param) in enumerate(named_params):
            _tag_name(param, name)
            if name in self._named:
                raise ValueError(f"names not unique. Repeated names = {{{name!r}}}")
            self._named[name] = param
        self.use_mpi = use_mpi
        self.cuda = cuda

        w = runtime.world()
        self.comm = comms.comm
        self.rank = w.rank
        self.size = w.size if use_mpi else 1
        self.steps = 0
        self.iallgather = comms.Iallgather()
        if not args and "params" not in kwargs:
            args = ([p for _, p in named_params],)
        super(MPI_PS, self).__init__(*args, **kwargs)

        self.quota = int(quota) if quota is not None else max(1, self.size - 1)
        self.recv_msgs: Dict[str, Any] = {}
        self.msgs: Dict[str, Any] = {}
        self.timings: List[Dict[str, float]] = []
        self.futures: List[Any] = []
        self.names: List[str] = []
        self.pool = ThreadPoolExecutor(max_workers=int(os.environ.get("PSB200_ENCODE_THREADS", "8")))
        self._inline_encode_bytes = int(os.environ.get("PSB200_INLINE_ENCODE_BYTES", 1 << 20))
        self._finalizer = weakref.finalize(self, self.pool.shutdown, False)

        # async (host engine) bookkeeping
        self._param_version = 0
        self._async_done = set()
        self._async_param_req = None
        self._async_send_req = None
        self._async_param_sends: List[Any] = []
        self._async_bye = False
        self._closed = False

        # which engine drives step()
        self._engine = None
        dev_ok = self._device_engine_possible(engine)
        if dev_ok:
            from .parallel.device_engine import DeviceEngine
            self._engine = DeviceEngine(self, master_fp32=master_fp32, reduce=reduce)
        self._hooks = []
        for name, param in self._named.items():
            if not param.requires_grad:
                continue
            if self._engine is not None:
                fn = partial(self._engine.on_grad, name=name, param=param)
            else:
                fn = partial(self.async_code, name=name, encode=self.code.encode)
            self._hooks.append(param.register_hook(fn))

    # ------------------------------------------------------------------------------- setup
    def _device_engine_possible(self, engine: str) -> bool:
        if engine == "host":
            return False
        params = [p for g in self.param_groups for p in g["params"]]
        all_cuda = bool(params) and all(p.is_cuda for p in params)
        spec = getattr(self.code, "device_spec", lambda: None)()
        ok = all_cuda and spec is not None and self.optim in ("sgd", "adam")
        if ok:
            dts = {p.dtype for p in params}
            ok = len(dts) == 1 and next(iter(dts)) in (torch.float32, torch.bfloat16, torch.float16)
        if engine == "device" and not ok:
            raise ValueError("engine='device' needs CUDA parameters of one float dtype and a built-in "
                             "coding with a device_spec() (Identity / Cast / Scale / block-wise TopK / block-wise QSGD)")
        return ok

    def close(self):
        """Release hooks, threads and (device engine) symmetric memory.  Idempotent."""
        if self._closed:
            return
        self._closed = True
        if self.mode == "async" and self._engine is None and self.size > 1:
            self._async_close()
        if self._engine is not None:
            self._engine.close()
        for h in self._hooks:
            h.remove()
        self._hooks = []
        self.pool.shutdown(wait=False)

    def __exit(self):   # the reference's (name-mangled, never called) pool shutdown, ps.py:89-90
        self.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False

    # -------------------------------------------------------------- encode pipeline (C5)
    def format_for_send(self, grad, encode=None, format=None, **kwargs):
        """Pool-thread body: ``encode`` then serialise + frame (``ps.py:92-96``)."""
        name = kwargs.pop("name", None)
        if name is not None and _accepts_name(encode):
            kwargs["name"] = name          # stateful codings (TopK error feedback) key their residual by parameter
        code = encode(grad.data, **kwargs)
        fmt = format if format is not None else partial(comms.format_for_send, level=self.level)
        msg, data = fmt(code)
        return msg, data

    def async_code(self, grad, *args, name=None, **kwargs):
        """Backward hook: queue the encode on the pool and remember hook-firing order (``ps.py:98-101``)."""
        if (not grad.is_cuda and grad.numel() * grad.element_size() <= self._inline_encode_bytes
                and getattr(self.code, "cheap", False)):
            # small host gradient, trivial coding (identity / cast / scale): the pool hand-off (a GIL round trip per future,
            # ~0.6 ms for four 100 KB messages against 0.08 ms of actual work) costs more than encoding right here
            future = Future()
            try:
                future.set_result(self.format_for_send(grad, *args, name=name, **kwargs))
            except BaseException as exc:       # noqa: BLE001 - surfaced by step(), like a pool failure
                future.set_exception(exc)
        else:
            future = self.pool.submit(self.format_for_send, grad, *args, name=name, **kwargs)
        self.futures += [future]
        self.names += [name]

    # ------------------------------------------------------------------------------- step
    def step(self, closure=None):
        """Perform one optimization step; returns ``(loss, data)`` (``ps.py:103-193``)."""
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        self.steps += 1
        if self._engine is not None:
            data = self._engine.step()
        elif self.mode == "allgather" or self.size == 1:
            data = self._step_allgather()
        elif self.mode == "ps":
            data = self._step_ps()
        else:
            data = self._step_async()
        self.timings.append(data)
        if len(self.timings) > 1024:
            del self.timings[:512]
        return loss, data

    # -- shared host-engine pieces ---------------------------------------------------------
    def _hyper(self, group) -> Dict[str, Any]:
        if self.optim == "sgd":
            return {k: group[k] for k in ["weight_decay", "momentum", "dampening", "nesterov", "lr"]}
        if self.optim == "adam":
            kw = {k: group[k] for k in ["betas", "weight_decay", "eps", "lr"]}
            kw["amsgrad"] = group.get("amsgrad", False)     # the reference forgot this (ps.py:185-186)
            return kw
        raise ValueError("self.optim not in [sgd, adam]")

    def _collect_encoded(self, data):
        """Join the encode pool; returns ``(names, msgs)`` in hook-firing order (``ps.py:128-138``)."""
        start = time.time()
        msgs_and_data = [future.result() for future in self.futures]
        names = list(self.names)
        self.names, self.futures = [], []
        msgs = [m for m, _ in msgs_and_data]
        meta = [d for _, d in msgs_and_data]
        for key in ["msg_bytes", "packaged_bytes"]:
            data[key] = (sum(d[key] for d in meta) / len(meta)) if meta else 0
        data["code_wait"] = time.time() - start
        if len(names) != len(set(names)):
            repeated = set(x for x in names if names.count(x) > 1)
            raise ValueError(f"names not unique. Repeated names = {repeated}")
        return names, msgs

    def _group_of(self):
        m = {}
        for g in self.param_groups:
            for p in g["params"]:
                m[id(p)] = g
        return m

    def _check_hooks(self, names):
        expect = [p for g in self.param_groups for p in g["params"] if p.requires_grad]
        if len(set(names)) != len(expect):
            # the reference raises here (ps.py:118-119); parameters that got no gradient this
            # step (unused branches) are legitimate, so only *extra* / unknown names are fatal
            unknown = set(names) - set(self._named)
            if unknown or len(set(names)) > len(expect):
                raise ValueError("len(set(names)) != len(params)")

    def _apply(self, name, grads, data, groups, scale_by: int):
        """Shape check, sum, optimizer step for one parameter (``ps.py:172-190``)."""
        p = self._named[name]
        start = time.time()
        if not all(g.shape == grads[0].shape for g in grads):
            print("  !!", self.rank, name, [tuple(g.shape) for g in grads])
            raise ValueError("shapes not the same")
        if p.grad is None:
            return
        # rank-ordered sum (ps.py:180) with one allocation and no dead passes: the first pair is added out of place
        # (the decoded gradients may be views of received messages), the rest accumulate in place
        if len(grads) == 1:
            d_p = grads[0].clone()
        else:
            d_p = torch.add(grads[0], grads[1])
            for g in grads[2:]:
                d_p.add_(g)
        d_p = d_p.to(device=p.device).reshape(p.shape)
        if d_p.dtype != p.dtype:
            d_p = d_p.to(p.dtype)
        if self.average and scale_by > 1:
            d_p.div_(scale_by)
        with torch.no_grad():
            self.optim_step(p, d_p, **self._hyper(groups[id(p)]))
        data["optim_step_time"] += time.time() - start

    def _decode_all(self, codes, data):
        start = time.time()
        self.code.codes = codes
        grads = [comms.to_torch(self.code.decode(c, cuda=self.cuda), cuda=self.cuda) for c in codes]
        data["decode_time"] += time.time() - start
        return grads

    # -- mode 'allgather': the reference's wired path (ps.py:117-191) -----------------------
    def _step_allgather(self):
        data = {"comm_wait": 0, "optim_step_time": 0, "decode_time": 0}
        names, msgs = self._collect_encoded(data)
        self._check_hooks(names)
        groups = self._group_of()

        if self.coalesce and self.size > 1:
            return self._step_allgather_coalesced(data, names, msgs, groups)

        start = time.time()
        sizes = self.iallgather.prepare(list(map(len, msgs)))
        data["iallgather_prepare_time"] = time.time() - start

        start = time.time()
        responses = []
        for (req, count), msg in zip(sizes, msgs):
            req.Wait()
            responses += [self.iallgather.send(msg, count)]
        data["isend_time"] = time.time() - start

        for name, msg, response in zip(names, msgs, responses):
            start = time.time()
            codes = self.iallgather.recv(*response, cuda=self.cuda)
            data["comm_wait"] += time.time() - start
            grads = self._decode_all(codes, data)
            self._apply(name, grads, data, groups, scale_by=len(grads))
        return data

    def _step_allgather_coalesced(self, data, names, msgs, groups):
        """One all-gather for the whole step: ``{"names": [...], "msgs": [framed bytes per parameter]}``."""
        start = time.time()
        bundle, _ = comms.format_for_send({"names": names, "msgs": [pickle.PickleBuffer(m) for m in msgs]})
        data["iallgather_prepare_time"] = 0.0
        resp = self.iallgather.send(bundle, None)
        data["isend_time"] = time.time() - start
        start = time.time()
        bundles = self.iallgather.recv(*resp, cuda=self.cuda)
        data["comm_wait"] += time.time() - start
        for b in bundles:
            if list(b["names"]) != names:
                raise ValueError("ranks disagree on the parameter order of this step")
        for i, name in enumerate(names):
            codes = [comms._unpack(b["msgs"][i], numpy=True) for b in bundles]
            grads = self._decode_all(codes, data)
            self._apply(name, grads, data, groups, scale_by=len(grads))
        return data

    # -- mode 'ps': rank-0 parameter server (README.md:37-46; mpi_comms.py:60-133) ----------
    def _step_ps(self):
        data = {"comm_wait": 0, "optim_step_time": 0, "decode_time": 0,
                "iallgather_prepare_time": 0.0}
        names, msgs = self._collect_encoded(data)
        self._check_hooks(names)
        groups = self._group_of()

        start = time.time()
        if self.coalesce:
            # the encoded messages travel out of band (protocol-5 buffers): no second copy into the bundle's pickle
            recv, req, _t = comms.igather({"names": names, "msgs": [pickle.PickleBuffer(m) for m in msgs]},
                                          name="__step__", level=-1)
            data["isend_time"] = time.time() - start
            start = time.time()
            bundles = comms.irecv(recv, req, name="__step__")
            data["comm_wait"] += time.time() - start
            if self.rank == 0:
                for b in bundles:
                    if list(b["names"]) != names:
                        raise ValueError("ranks disagree on the parameter order of this step")
                for i, n in enumerate(names):
                    codes = [comms._unpack(b["msgs"][i], numpy=True) for b in bundles]
                    grads = self._decode_all(codes, data)
                    self._apply(n, grads, data, groups, scale_by=len(grads))
            posted = []
        else:
            # one gather per parameter, all posted before any is waited (the reference's pipelining)
            posted = [comms.igather({"name": n, "msg": pickle.PickleBuffer(m)}, name=n, level=-1)
                      for n, m in zip(names, msgs)]
            data["isend_time"] = time.time() - start

        for n, (recv, req, _t) in zip(names, posted):
            start = time.time()
            objs = comms.irecv(recv, req, name=n)
            data["comm_wait"] += time.time() - start
            if self.rank != 0:
                continue
            if any(o["name"] != n for o in objs):
                raise ValueError(f"gather order mismatch for {n}: {[o['name'] for o in objs]}")
            codes = [comms._unpack(o["msg"], numpy=True) for o in objs]
            grads = self._decode_all(codes, data)
            self._apply(n, grads, data, groups, scale_by=len(grads))

        # PS → workers: fresh parameters (one framed message; receivers overwrite in place)
        start = time.time()
        plist = [p for p in self._named.values()]
        payload = [p.data for p in plist] if self.rank == 0 else None
        send, req = comms.ibroadcast(payload, root=0, level=self.level)
        fresh = comms.irecv1(send, req)
        if self.rank != 0:
            with torch.no_grad():
                for p, q in zip(plist, fresh):
                    p.data.copy_(q.to(p.device), non_blocking=True)
        data["bcast_time"] = time.time() - start
        data["comm_wait"] += data["bcast_time"]
        return data

    # -- mode 'async': AsySG-InCon (README.md:56-81) ------------------------------------------
    def _async_post_param_recv(self):
        self._async_param_req = comms.irecv_obj(src=0, tag=_TAG_PARAM)

    def _async_apply_params_if_any(self, block: bool, data):
        """Worker: adopt the newest parameter message (if any has arrived)."""
        got = 0
        while True:
            if self._async_param_req is None:
                self._async_post_param_recv()
            if not block and not self._async_param_req.Test():
                break
            msg = self._async_param_req.Wait()
            self._async_param_req = None
            block = False
            if msg.get("kind") == "bye":
                self._async_bye = True
                break
            got += 1
            with torch.no_grad():
                for p, q in zip(self._named.values(), msg["params"]):
                    p.data.copy_(q.to(p.device), non_blocking=True)
            self._param_version = int(msg["version"])
        data["param_msgs"] = got
        data["param_version"] = self._param_version

    def _step_async(self):
        data = {"comm_wait": 0, "optim_step_time": 0, "decode_time": 0,
                "iallgather_prepare_time": 0.0, "isend_time": 0.0}
        names, msgs = self._collect_encoded(data)
        groups = self._group_of()
        if self.rank != 0:
            # worker: ship the encoded gradients, never wait for a consistent snapshot
            start = time.time()
            if self._async_send_req is not None:
                self._async_send_req.Wait()
            self._async_send_req = comms.isend_obj(
                {"kind": "grad", "names": names, "msgs": [pickle.PickleBuffer(m) for m in msgs],
                 "version": self._param_version, "rank": self.rank}, dst=0, tag=_TAG_GRAD)
            data["isend_time"] = time.time() - start
            start = time.time()
            self._async_apply_params_if_any(block=self.consistent, data=data)
            data["comm_wait"] = time.time() - start
            return data

        # rank 0 is the parameter server: consume `quota` gradients from ANY source
        n_workers = self.size - 1
        contrib: List[dict] = []
        start = time.time()
        while len(contrib) < self.quota and len(self._async_done) < n_workers:
            req = comms.irecv_obj(src=comms.ANY_SOURCE, tag=_TAG_GRAD)
            m = req.Wait()
            if m["kind"] == "done":
                self._async_done.add(int(m["rank"]))
                continue
            contrib.append(m)
        data["comm_wait"] = time.time() - start
        data["ps_done"] = len(self._async_done) >= n_workers and not contrib
        data["contributors"] = [int(m["rank"]) for m in contrib]
        data["staleness"] = [self._param_version - int(m["version"]) for m in contrib]
        if not contrib:
            return data
        per_name: Dict[str, list] = OrderedDict()
        for m in contrib:
            for n, blob in zip(m["names"], m["msgs"]):
                per_name.setdefault(n, []).append(comms._unpack(blob, numpy=True))
        for n, codes in per_name.items():
            p = self._named[n]
            if p.grad is None:            # the PS never ran backward: give _apply something to see
                p.grad = torch.zeros_like(p)
            grads = self._decode_all(codes, data)
            self._apply(n, grads, data, groups, scale_by=len(grads))
        self._param_version += 1
        start = time.time()
        payload = {"kind": "params", "params": [p.data for p in self._named.values()],
                   "version": self._param_version}
        # fire and forget (the ibcast of README.md:76 is never waited): completion is polled later
        self._async_param_sends = [r for r in self._async_param_sends if not r.Test()]
        self._async_param_sends += [comms.isend_obj(payload, dst=r, tag=_TAG_PARAM, level=self.level)
                                    for r in range(1, self.size) if r not in self._async_done]
        data["bcast_time"] = time.time() - start
        data["param_version"] = self._param_version
        return data

    def _async_close(self):
        """Drain protocol: workers say ``done``; the PS answers ``bye`` once all are done; workers
        keep consuming parameter messages until ``bye`` so no send is left unmatched."""
        if self.rank != 0:
            if self._async_send_req is not None:
                self._async_send_req.Wait()
            done = comms.isend_obj({"kind": "done", "rank": self.rank}, dst=0, tag=_TAG_GRAD)
            scratch = {}
            while not self._async_bye:
                self._async_apply_params_if_any(block=True, data=scratch)
            done.Wait()
        else:
            while len(self._async_done) < self.size - 1:
                m = comms.irecv_obj(src=comms.ANY_SOURCE, tag=_TAG_GRAD).Wait()
                if m["kind"] == "done":
                    self._async_done.add(int(m["rank"]))
            byes = [comms.isend_obj({"kind": "bye"}, dst=r, tag=_TAG_PARAM) for r in range(1, self.size)]
            for r in self._async_param_sends + byes:
                r.Wait()
            self._async_param_sends = []

    def serve(self, max_updates: Optional[int] = None) -> int:
        """Async PS loop for rank 0: apply updates until every worker called ``close()``; returns the number of updates
        APPLIED (the device engine queues server iterations ahead of the GPU, so that is not the number of ``step()`` calls)."""
        n = 0
        while True:
            _, data = self.step()
            if "updates_applied" in data:
                n = data["updates_applied"]
            elif not data.get("ps_done"):
                n += 1
            if data.get("ps_done") or (max_updates is not None and n >= max_updates):
                break
        return n

    # --------------------------------------------------------------------- checkpointing
    def state_dict(self):
        if self._engine is not None:
            self._engine.sync_state_to_torch()
        sd = super().state_dict()
        if self._engine is not None and self._engine.kind == _codings.KIND_QSGD:
            # every rank's RNG step: a resumed run draws the same roundings as the uninterrupted one
            sd[_QSGD_RNG_KEY] = self._engine.rng_step
        return sd

    def load_state_dict(self, state_dict):
        rng_step = state_dict.get(_QSGD_RNG_KEY)
        if rng_step is not None:
            state_dict = {k: v for k, v in state_dict.items() if k != _QSGD_RNG_KEY}
            if self._engine is not None and self._engine.kind == _codings.KIND_QSGD:
                self._engine.rng_step = int(rng_step)
        super().load_state_dict(state_dict)
        if self._engine is not None:
            # torch casts loaded state to the parameter dtype (bf16); the engine's state is fp32, so hand
            # it the ORIGINAL tensors, keyed by parameter position
            params = [p for g in self.param_groups for p in g["params"]]
            saved = state_dict.get("state", {})
            original = {id(params[int(i)]): st for i, st in saved.items() if int(i) < len(params)}
            self._engine.sync_state_from_torch(original)


# ---------------------------------------------------------------------------------------
class SGD(MPI_PS, torch.optim.SGD):
    """SGD with the reference's update rule (``/root/reference/ps.py:195-214``)."""

    _default_optim = "sgd"

    def optim_step(self, p, d_p, weight_decay=0, momentum=0, dampening=0,
                   nesterov=0, lr=0):
        if weight_decay != 0:
            d_p = d_p.add(p.data, alpha=weight_decay)
        if momentum != 0:
            param_state = self.state[p]
            if "momentum_buffer" not in param_state or param_state["momentum_buffer"] is None:
                buf = param_state["momentum_buffer"] = torch.zeros_like(p.data)
                buf.mul_(momentum).add_(d_p)                 # first step: buf = d_p
            else:
                buf = param_state["momentum_buffer"]
                buf.mul_(momentum).add_(d_p, alpha=1 - dampening)
            if nesterov:
                d_p = d_p.add(buf, alpha=momentum)
            else:
                d_p = buf
        p.data.add_(d_p, alpha=-lr)


class Adam(MPI_PS, torch.optim.Adam):
    """Adam with the reference's update rule (``/root/reference/ps.py:217-261``).

    ``optim='adam'`` is implied (the reference made the user pass it, ``ps.py:181-188``) and
    ``amsgrad`` is honoured (the reference never forwarded it, ``ps.py:185-186``).
    """

    _default_optim = "adam"

    def optim_step(self, p, grad, amsgrad=False, betas=(0.9, 0.999), weight_decay=0,
                   eps=1e-8, lr=1e-3):
        if grad.is_sparse:
            raise RuntimeError("Adam does not support sparse gradients, please consider SparseAdam instead")
        state = self.state[p]
        if len(state) == 0 or "exp_avg" not in state:
            state["step"] = 0
            state["exp_avg"] = torch.zeros_like(p.data)
            state["exp_avg_sq"] = torch.zeros_like(p.data)
            if amsgrad:
                state["max_exp_avg_sq"] = torch.zeros_like(p.data)
        exp_avg, exp_avg_sq = state["exp_avg"], state["exp_avg_sq"]
        beta1, beta2 = betas
        state["step"] += 1
        step = int(state["step"])
        if weight_decay != 0:
            grad = grad.add(p.data, alpha=weight_decay)
        exp_avg.mul_(beta1).add_(grad, alpha=1 - beta1)
        exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
        if amsgrad:
            if "max_exp_avg_sq" not in state:
                state["max_exp_avg_sq"] = torch.zeros_like(p.data)
            max_exp_avg_sq = state["max_exp_avg_sq"]
            torch.maximum(max_exp_avg_sq, exp_avg_sq, out=max_exp_avg_sq)
            denom = max_exp_avg_sq.sqrt().add_(eps)
        else:
            denom = exp_avg_sq.sqrt().add_(eps)
        bias_correction1 = 1 - beta1 ** step
        bias_correction2 = 1 - beta2 ** step
        step_size = lr * math.sqrt(bias_correction2) / bias_correction1
        p.data.addcdiv_(exp_avg, denom, value=-step_size)
