"""L3 gradient codings: the ``encode`` / ``decode`` / ``codes`` plug-in contract and built-ins.

The reference imports an *external* ``codings`` module (``/root/reference/ps.py:16-18``) and
uses exactly three members of the object passed as ``code=``:

* ``code.encode(grad.data, **kw)`` in the backward hook (``ps.py:65-66,94``),
* ``code.decode(code_obj, cuda=bool)`` per rank's message (``ps.py:166``),
* ``code.codes = [...]`` — every rank's code for the current parameter, assigned before
  decoding (``ps.py:165``).

This module ships that contract as :class:`Coding` plus the built-ins the framework fuses into
its sm_100a kernels: :class:`Identity`, :class:`Cast`, :class:`Scale`, :class:`TopK` and block-wise
:class:`QSGD`.  Each
built-in has

* a pure-PyTorch ``encode``/``decode`` (host slow path **and** the numerical oracle every CUDA
  kernel is tested against), and
* a :meth:`Coding.device_spec` describing the fixed binary wire layout the device path uses
  (no pickle, no size exchange — ``/root/reference/mpi_comms.py:150-158`` is eliminated).

Arbitrary user codings (any object with ``encode``/``decode``) keep working on the host path.
"""
from __future__ import annotations

import itertools
import math
from dataclasses import dataclass
from typing import Any, List, Optional

import torch

__all__ = [
    "Coding", "Identity", "Cast", "Scale", "TopK", "QSGD", "SVD", "DeviceCodeSpec", "TILE",
    "WIRE_F32", "WIRE_BF16", "WIRE_F16", "WIRE_E4M3", "WIRE_E5M2", "WIRE_I8",
    "KIND_DENSE", "KIND_SCALED", "KIND_TOPK", "KIND_QSGD", "wire_dtype_of", "wire_code_of", "tile_k",
    "qsgd_uniform16", "qsgd_blockwise",
]

#: elements per tile of the flat arena; every parameter starts on a tile boundary and the
#: block-wise top-k selects inside one tile.  Must match ``PSB_TILE`` in csrc/kernels/common.cuh.
TILE = 2048

# wire element types (must match csrc/kernels/common.cuh)
WIRE_F32, WIRE_BF16, WIRE_F16, WIRE_E4M3, WIRE_E5M2, WIRE_I8 = 0, 1, 2, 3, 4, 5
# coding kinds
KIND_DENSE, KIND_SCALED, KIND_TOPK, KIND_QSGD = 0, 1, 2, 3

_WIRE_TORCH = {
    WIRE_F32: torch.float32, WIRE_BF16: torch.bfloat16, WIRE_F16: torch.float16,
    WIRE_E4M3: torch.float8_e4m3fn, WIRE_E5M2: torch.float8_e5m2, WIRE_I8: torch.int8,
}
_WIRE_NAMES = {
    "fp32": WIRE_F32, "float32": WIRE_F32, "f32": WIRE_F32,
    "bf16": WIRE_BF16, "bfloat16": WIRE_BF16,
    "fp16": WIRE_F16, "float16": WIRE_F16, "half": WIRE_F16,
    "fp8": WIRE_E4M3, "fp8_e4m3": WIRE_E4M3, "e4m3": WIRE_E4M3, "float8_e4m3fn": WIRE_E4M3,
    "fp8_e5m2": WIRE_E5M2, "e5m2": WIRE_E5M2, "float8_e5m2": WIRE_E5M2,
    "int8": WIRE_I8, "i8": WIRE_I8,
}
_WIRE_MAX = {WIRE_E4M3: 448.0, WIRE_E5M2: 57344.0, WIRE_I8: 127.0, WIRE_F16: 65504.0}


def wire_code_of(dtype) -> int:
    """Map a torch dtype / string to a wire element code."""
    if isinstance(dtype, int):
        return dtype
    if isinstance(dtype, str):
        return _WIRE_NAMES[dtype.lower()]
    for k, v in _WIRE_TORCH.items():
        if v == dtype:
            return k
    raise ValueError(f"unsupported wire dtype {dtype!r}")


def wire_dtype_of(code: int) -> torch.dtype:
    return _WIRE_TORCH[code]


def tile_k(ratio: float, valid: int) -> int:
    """Entries kept in a tile that holds ``valid`` real elements (block-wise top-k)."""
    return max(1, min(valid, int(math.ceil(ratio * valid - 1e-9))))


@dataclass(frozen=True)
class DeviceCodeSpec:
    """Fixed binary wire layout of a built-in coding (consumed by the CUDA kernels)."""

    kind: int                 # KIND_DENSE | KIND_SCALED | KIND_TOPK | KIND_QSGD
    wire: int                 # WIRE_* element type of the payload values (-1 = same as grad)
    ratio: float = 1.0        # top-k keep ratio (KIND_TOPK)
    error_feedback: bool = False
    levels: int = 0           # quantisation levels (KIND_QSGD)
    seed: int = 0             # 64-bit Philox key (KIND_QSGD)

    def resolved_wire(self, grad_dtype: torch.dtype) -> int:
        return wire_code_of(grad_dtype) if self.wire < 0 else self.wire

    def tile_capacity(self) -> int:
        """Entries reserved per tile on the wire (KIND_TOPK)."""
        return tile_k(self.ratio, TILE) if self.kind == KIND_TOPK else TILE

    def bytes_per_tile(self, grad_dtype: torch.dtype) -> int:
        w = self.resolved_wire(grad_dtype)
        esz = torch.empty((), dtype=_WIRE_TORCH[w]).element_size()
        if self.kind == KIND_TOPK:
            # entry = value + index packed to 2x the value width (bf16+u16 / f32+u32)
            esz = 4 if esz <= 2 else 8
            n = self.tile_capacity() * esz
        elif self.kind == KIND_QSGD:
            n = TILE * esz + 4            # int8 payload + the tile's fp32 scale (trailer zero-padded to 16 bytes)
        else:
            n = TILE * esz
        return (n + 15) // 16 * 16


class Coding:
    """Base class of the coding plug-in interface (``ps.py:57,60,65-66,94,165-166``)."""

    #: every rank's code for the parameter being decoded, set by the optimizer (``ps.py:165``)
    codes: Optional[List[Any]] = None
    #: encode is a view / one elementwise pass: the host engine encodes small gradients inside the hook instead of on its pool
    cheap: bool = False

    def encode(self, grad: torch.Tensor, **kwargs) -> Any:   # pragma: no cover - interface
        raise NotImplementedError

    def decode(self, code: Any, cuda: bool = False) -> torch.Tensor:   # pragma: no cover
        raise NotImplementedError

    def device_spec(self) -> Optional[DeviceCodeSpec]:
        """Binary layout for the fused kernels, or ``None`` → host (pickle) slow path."""
        return None

    # helpers shared by built-ins ----------------------------------------------------
    @staticmethod
    def _place(t: torch.Tensor, cuda: bool) -> torch.Tensor:
        if cuda and torch.cuda.is_available() and not t.is_cuda:
            return t.cuda(non_blocking=True)
        return t

    def __repr__(self) -> str:
        return f"{type(self).__name__}()"


def _as_tensor(x) -> torch.Tensor:
    if isinstance(x, torch.Tensor):
        return x
    return torch.as_tensor(x)


class Identity(Coding):
    """Send the gradient as it is (dtype preserved)."""

    cheap = True

    def encode(self, grad, **kwargs):
        return {"grad": grad.detach()}

    def decode(self, code, cuda=False):
        g = _as_tensor(code["grad"])
        return self._place(g, cuda)

    def device_spec(self):
        return DeviceCodeSpec(KIND_DENSE, -1)


def _sat_cast(x: torch.Tensor, wire: int) -> torch.Tensor:
    """Round-to-nearest-even cast with saturation to the finite range (``cvt.rn.satfinite``)."""
    dt = _WIRE_TORCH[wire]
    if wire in (WIRE_E4M3, WIRE_E5M2, WIRE_F16):
        m = _WIRE_MAX[wire]
        x = x.float().clamp(-m, m)
        return x.to(dt)
    if wire == WIRE_I8:
        return x.float().round().clamp(-127, 127).to(torch.int8)
    return x.to(dt)


class Cast(Coding):
    """Down-cast the gradient to a narrower float on the wire (bf16 / fp16 / fp8)."""

    cheap = True

    def __init__(self, dtype="bf16"):
        self.wire = wire_code_of(dtype)
        if self.wire == WIRE_I8:
            raise ValueError("Cast to int8 needs a scale: use Scale('int8')")

    def encode(self, grad, **kwargs):
        return {"v": _sat_cast(grad.detach(), self.wire), "dtype": str(grad.dtype)}

    def decode(self, code, cuda=False):
        v = _as_tensor(code["v"])
        return self._place(v, cuda).float()

    def device_spec(self):
        return DeviceCodeSpec(KIND_DENSE, self.wire)

    def __repr__(self):
        return f"Cast({_WIRE_TORCH[self.wire]})"


class Scale(Coding):
    """Per-tensor abs-max scaling into a narrow type (int8 / fp8 / fp16).

    ``wire = cast(grad * qmax / absmax)``; the fp32 ``inv = absmax / qmax`` travels with the
    message and ``decode = wire * inv``.
    """

    def __init__(self, dtype="int8"):
        self.wire = wire_code_of(dtype)
        if self.wire not in _WIRE_MAX:
            raise ValueError("Scale supports int8 / fp8_e4m3 / fp8_e5m2 / fp16")

    def encode(self, grad, **kwargs):
        g = grad.detach().float()
        qmax = _WIRE_MAX[self.wire]
        amax = g.abs().max() if g.numel() else g.new_zeros(())
        amax = torch.where(torch.isfinite(amax) & (amax > 0), amax, torch.ones_like(amax))
        inv = amax / torch.full_like(amax, qmax)   # IEEE fp32 division (a Python-scalar divisor is a
        #                                            reciprocal-multiply on CUDA and differs by 1 ulp)
        q = _sat_cast(g / inv, self.wire)       # == g * (qmax/amax) up to fp32 rounding
        return {"q": q, "inv": inv.reshape(1)}

    def decode(self, code, cuda=False):
        q = self._place(_as_tensor(code["q"]), cuda)
        inv = self._place(_as_tensor(code["inv"]), cuda).float()
        return q.float() * inv

    def device_spec(self):
        return DeviceCodeSpec(KIND_SCALED, self.wire)

    def __repr__(self):
        return f"Scale({_WIRE_TORCH[self.wire]})"


class TopK(Coding):
    """Magnitude top-k sparsification.

    Two flavours:

    * ``exact=False`` (default, fused on device): **block-wise** top-k — the flattened tensor is
      cut into ``TILE``-element blocks and each block keeps its ``ceil(ratio * valid)`` largest
      magnitudes (ties → lower index).  Fixed per-block capacity means a fixed-size wire slot —
      no size exchange round (``mpi_comms.py:150-158``) — and the PS decodes a block entirely in
      shared memory.
    * ``exact=True``: classic per-tensor ``k`` / ``ratio`` (host path only).

    ``values`` picks the payload float type (``bf16`` → 4-byte ``(u16 idx, bf16 val)`` entries,
    ``fp32`` → 8-byte ``(u32 idx, f32 val)`` entries).
    """

    def __init__(self, ratio: Optional[float] = None, k: Optional[int] = None,
                 values="fp32", exact: bool = False, error_feedback: bool = False):
        if (ratio is None) == (k is None):
            raise ValueError("give exactly one of ratio= or k=")
        if k is not None and not exact:
            raise ValueError("k= needs exact=True (block-wise top-k is ratio based)")
        if ratio is not None and not (0.0 < ratio <= 1.0):
            raise ValueError("ratio must be in (0, 1]")
        self.ratio, self.k, self.exact = ratio, k, exact
        self.wire = wire_code_of(values)
        if self.wire not in (WIRE_F32, WIRE_BF16):
            raise ValueError("TopK values must be fp32 or bf16")
        self.error_feedback = bool(error_feedback)
        self._residual = {}

    # -- oracle / host path -------------------------------------------------------------
    def _select_blockwise(self, flat: torch.Tensor):
        n = flat.numel()
        nt = (n + TILE - 1) // TILE
        pad = nt * TILE - n
        x = torch.cat([flat, flat.new_zeros(pad)]) if pad else flat
        x = x.view(nt, TILE)
        mag = x.abs().float()
        if pad:  # padded lanes must never win
            mag = mag.clone()
            mag.view(-1)[n:] = -1.0
        order = torch.sort(mag, dim=1, descending=True, stable=True).indices
        idx_parts, val_parts = [], []
        for t in range(nt):
            valid = min(TILE, n - t * TILE)
            kt = tile_k(self.ratio, valid)
            sel = torch.sort(order[t, :kt]).values
            idx_parts.append(sel + t * TILE)
            val_parts.append(x[t, sel])
        return torch.cat(idx_parts), torch.cat(val_parts)

    def encode(self, grad, name=None, **kwargs):
        g = grad.detach()
        flat = g.reshape(-1)
        if self.error_feedback:
            if name is None:
                # id(grad) of a temporary is recycled across parameters and steps: it would mix residuals
                raise ValueError("TopK(error_feedback=True).encode needs name= (the parameter the residual belongs to)")
            key = name
            res = self._residual.get(key)
            work = flat.float() if res is None else flat.float() + res
        else:
            work = flat
        if self.exact:
            k = self.k if self.k is not None else max(1, int(math.ceil(self.ratio * flat.numel())))
            k = min(k, flat.numel())
            idx = torch.sort(torch.topk(work.abs().float(), k, sorted=False).indices).values
            val = work[idx]
        else:
            idx, val = self._select_blockwise(work)
        val = val.to(_WIRE_TORCH[self.wire])
        if self.error_feedback:
            res = work.float().clone()
            res[idx] -= val.float()
            self._residual[key] = res
        return {"idx": idx.to(torch.int32), "val": val, "shape": tuple(g.shape)}

    def decode(self, code, cuda=False):
        idx = self._place(_as_tensor(code["idx"]), cuda).long()
        val = self._place(_as_tensor(code["val"]), cuda).float()
        shape = tuple(int(s) for s in code["shape"])
        out = torch.zeros(int(math.prod(shape)) if shape else 1, dtype=torch.float32, device=val.device)
        out.index_add_(0, idx, val)
        return out.view(shape)

    def device_spec(self):
        if self.exact:
            return None
        return DeviceCodeSpec(KIND_TOPK, self.wire, float(self.ratio), self.error_feedback)

    def __repr__(self):
        what = f"k={self.k}" if self.k is not None else f"ratio={self.ratio}"
        return f"TopK({what}, values={_WIRE_TORCH[self.wire]}, exact={self.exact})"


_PHILOX_M0, _PHILOX_M1, _PHILOX_W0, _PHILOX_W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
_U32 = 0xFFFFFFFF


def _mulhilo32(a: int, b: torch.Tensor):
    """``(hi, lo)`` 32-bit halves of the 64-bit product of the constant ``a`` and int64 tensor ``b`` (values < 2**32), in
    int64 arithmetic that never overflows: ``a`` is split into 16-bit halves."""
    t_lo, t_hi = b * (a & 0xFFFF), b * (a >> 16)          # each < 2**48
    s = t_lo + ((t_hi & 0xFFFF) << 16)                     # < 2**49
    return (t_hi >> 16) + (s >> 32), s & _U32


def qsgd_uniform16(seed: int, rank: int, step: int, first_elem: int, n: int, device=None) -> torch.Tensor:
    """The 16-bit uniforms the block-wise QSGD kernel draws for arena elements ``[first_elem, first_elem + n)`` (int32 tensor).

    Philox4x32-10 with the Random123 constants, one call per 8 consecutive elements ``e0 .. e0 + 7`` (``e0 % 8 == 0``):
    counter = ``(e0 / 8 low 32 bits, e0 / 8 high 32 bits, step, rank)``, key = ``(seed low 32 bits, seed high 32 bits)``;
    element ``e0 + j`` takes 16 bits of output word ``j >> 1`` (low half for even ``j``).  Runs on ``device`` in int64 ops."""
    g0 = int(first_elem) // 8
    k = torch.arange((int(first_elem) + n + 7) // 8 - g0, dtype=torch.int64, device=device)
    lo = (g0 & _U32) + k                                   # the 64-bit group index as two words (any index, no int64 overflow)
    c0, c1 = lo & _U32, ((g0 >> 32) + (lo >> 32)) & _U32
    c2 = torch.full_like(c0, int(step) & _U32)
    c3 = torch.full_like(c0, int(rank) & _U32)
    k0, k1 = int(seed) & _U32, (int(seed) >> 32) & _U32
    for _ in range(10):
        hi0, lo0 = _mulhilo32(_PHILOX_M0, c0)
        hi1, lo1 = _mulhilo32(_PHILOX_M1, c2)
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        k0, k1 = (k0 + _PHILOX_W0) & _U32, (k1 + _PHILOX_W1) & _U32
    words = torch.stack([c0, c1, c2, c3], dim=1)                              # [groups, 4]
    u = torch.stack([words & 0xFFFF, words >> 16], dim=2).reshape(-1)       # [groups * 8] in element order
    off = int(first_elem) - 8 * g0
    return u[off: off + n].to(torch.int32)


def qsgd_blockwise(flat: torch.Tensor, levels: int, u16: torch.Tensor):
    """Block-wise QSGD of a flat tensor with the given 16-bit uniforms: ``(q int8 [ntiles * TILE], scale fp32 [ntiles])``.

    The bit-exact oracle of the ``KIND_QSGD`` encode kernel.  Per ``TILE``-element tile: ``norm = sqrt(sum of squares)``
    summed in the kernel's order (a thread's 8 elements in sequence, an xor butterfly over the 32 lanes of a warp, then the 8
    warp sums in order), ``x = min(|g| * (levels / norm), levels)``, ``q = sign(g) * (floor(x) + [u16 < frac(x) * 2**16])``
    and ``scale = norm / levels``.  A tile whose norm is zero or not finite gets ``q = 0`` and ``scale = 0``."""
    g = flat.reshape(-1).float()
    n = g.numel()
    nt = max(1, -(-n // TILE))
    pad = nt * TILE - n
    u = u16.reshape(-1)[: nt * TILE]
    if pad:
        g = torch.cat([g, g.new_zeros(pad)])
    if u.numel() < nt * TILE:
        u = torch.cat([u, u.new_zeros(nt * TILE - u.numel())])
    sq = (g * g).view(nt, TILE // 8, 8)
    s = sq[:, :, 0]
    for j in range(1, 8):
        s = s + sq[:, :, j]
    s = s.reshape(nt, TILE // 256, 32)
    lanes = torch.arange(32, device=g.device)
    for off in (16, 8, 4, 2, 1):
        s = s + s[:, :, lanes ^ off]
    tot = s[:, 0, 0]
    for w in range(1, TILE // 256):
        tot = tot + s[:, w, 0]
    norm = _sqrt_rn(tot)
    live = (norm > 0) & torch.isfinite(norm)
    lv = torch.full_like(norm, float(levels))
    r = lv / norm                                   # tensor / tensor: IEEE division on every device
    x = torch.minimum(g.view(nt, TILE).abs() * r[:, None], lv[:, None])
    low = torch.floor(x)
    up = u.view(nt, TILE).float() < (x - low) * 65536.0
    q = torch.copysign(low + up.float(), g.view(nt, TILE))
    q = torch.where(live[:, None], q, torch.zeros_like(q))
    scale = torch.where(live, norm / lv, torch.zeros_like(norm))
    return q.to(torch.int8).reshape(-1), scale


def _sqrt_rn(x: torch.Tensor) -> torch.Tensor:
    """Correctly rounded fp32 square root (``__fsqrt_rn``) on any device: torch's vectorised CPU ``sqrt`` is not.  A
    neighbour of ``r`` is taken when the exact square of the midpoint between them (25-bit operands, exact in fp64) lies on
    the other side of ``x``."""
    r = torch.sqrt(x.double()).float()
    xd = x.double()
    for _ in range(2):
        up, dn = torch.nextafter(r, torch.full_like(r, math.inf)), torch.nextafter(r, torch.zeros_like(r))
        r = torch.where(((r.double() + up.double()) / 2) ** 2 < xd, up, r)
        r = torch.where(((r.double() + dn.double()) / 2) ** 2 > xd, dn, r)
    return r


def _host_rank() -> int:
    from . import runtime
    return runtime.world().rank if runtime.is_initialized() else 0


class QSGD(Coding):
    """QSGD-style stochastic quantisation (Alistarh et al. 2017): ``sign · ‖g‖₂ · ξ/levels`` with ``ξ`` drawn so
    the code is an unbiased estimate of the gradient.

    * ``blockwise=False`` (default): one norm per tensor, ``torch.rand`` rounding.  Host (generic-object) path — the kind of
      user coding the reference's external ``codings`` module carried (SURVEY §2.2).
    * ``blockwise=True``: one norm per ``TILE``-element tile of the flat arena ("bucketed" QSGD with bucket size ``TILE``),
      ``1 <= levels <= 127`` on an int8 wire.  Fused on device (``KIND_QSGD``): each tile travels as ``TILE`` int8 codes plus
      its fp32 ``scale = norm / levels``; there is no abs-max pre-pass and no size exchange.  The rounding draws come from
      Philox4x32-10 keyed by ``(seed, rank, step, arena element)`` (:func:`qsgd_uniform16`), so a seeded run is reproducible.
      A draw has 16 bits, which biases each rounding by at most 2⁻¹⁶ of one quantum (``scale``); otherwise
      ``E[decode(encode(g))] = g``.  ``seed=None`` draws a 64-bit seed once, here, from torch's global CPU generator; ranks
      need not agree on it because the rank is part of the Philox counter.  The host ``encode`` runs the same per-tile
      algorithm on the gradient's own device (``rank`` / ``step`` / ``first_elem`` default to this process's rank, a
      per-instance call counter and 0).
    """

    def __init__(self, levels: int = 255, seed: Optional[int] = None, blockwise: bool = False):
        if not 1 <= levels <= 32767:
            raise ValueError("levels must be in [1, 32767]")
        self.levels = int(levels)
        self.blockwise = bool(blockwise)
        if self.blockwise:
            if self.levels > 127:
                raise ValueError("QSGD(blockwise=True) needs 1 <= levels <= 127 (the wire is int8)")
            if seed is None:
                lo, hi = torch.randint(0, 1 << 32, (2,), dtype=torch.int64).tolist()
                seed = lo | hi << 32
            self.seed = int(seed) & ((1 << 64) - 1)
            self._calls = itertools.count()
        else:
            self._gen = torch.Generator().manual_seed(seed) if seed is not None else None

    def encode(self, grad, rank=None, step=None, first_elem=0, **kwargs):
        if self.blockwise:
            g = grad.detach()
            rank = _host_rank() if rank is None else rank
            step = next(self._calls) if step is None else step
            u = qsgd_uniform16(self.seed, rank, step, first_elem, g.numel(), device=g.device)
            q, scale = qsgd_blockwise(g, self.levels, u)
            return {"q": q, "scale": scale, "shape": tuple(g.shape)}
        g = grad.detach().float().cpu()
        norm = g.norm()
        if float(norm) == 0.0 or not torch.isfinite(norm):
            q = torch.zeros(g.shape, dtype=torch.int16)
            return {"q": q, "norm": torch.zeros(1), "levels": self.levels, "shape": tuple(g.shape)}
        x = g.abs() / norm * self.levels                      # in [0, levels]
        low = x.floor()
        up = torch.rand(x.shape, generator=self._gen) < (x - low)      # stochastic rounding → unbiased
        q = (low + up.float()) * g.sign()
        dt = torch.int8 if self.levels <= 127 else torch.int16
        return {"q": q.to(dt), "norm": norm.reshape(1), "levels": self.levels, "shape": tuple(g.shape)}

    def decode(self, code, cuda=False):
        shape = tuple(int(d) for d in code["shape"])
        if "scale" in code:                                   # block-wise: one scale per tile
            q = self._place(_as_tensor(code["q"]), cuda).float()
            scale = self._place(_as_tensor(code["scale"]), cuda).float()
            return (q.view(-1, TILE) * scale[:, None]).reshape(-1)[: math.prod(shape)].reshape(shape)
        q = self._place(_as_tensor(code["q"]), cuda).float()
        norm = self._place(_as_tensor(code["norm"]), cuda).float()
        return (q * (norm / float(code["levels"]))).reshape(shape)

    def device_spec(self):
        if not self.blockwise:
            return None
        return DeviceCodeSpec(KIND_QSGD, WIRE_I8, levels=self.levels, seed=self.seed)

    def __repr__(self):
        return f"QSGD(levels={self.levels}, blockwise=True)" if self.blockwise else f"QSGD(levels={self.levels})"


class SVD(Coding):
    """Rank-``r`` truncated SVD of every ≥2-D gradient (sent as ``U·S`` and ``Vᵀ``); 1-D gradients travel as is.
    Host path (ATOMO / PowerSGD family of the reference author's coding experiments, SURVEY §2.2)."""

    def __init__(self, rank: int = 4):
        if rank < 1:
            raise ValueError("rank must be >= 1")
        self.rank = int(rank)

    def encode(self, grad, **kwargs):
        g = grad.detach().float().cpu()
        if g.dim() < 2 or min(g.shape[0], g[0].numel()) <= self.rank:
            return {"dense": g, "shape": tuple(g.shape)}
        m = g.reshape(g.shape[0], -1)
        u, s, vh = torch.linalg.svd(m, full_matrices=False)
        r = self.rank
        return {"us": (u[:, :r] * s[:r]).contiguous(), "vh": vh[:r].contiguous(), "shape": tuple(g.shape)}

    def decode(self, code, cuda=False):
        shape = tuple(int(d) for d in code["shape"])
        if "dense" in code:
            return self._place(_as_tensor(code["dense"]), cuda).float().reshape(shape)
        us = self._place(_as_tensor(code["us"]), cuda).float()
        vh = self._place(_as_tensor(code["vh"]), cuda).float()
        return (us @ vh).reshape(shape)

    def __repr__(self):
        return f"SVD(rank={self.rank})"
