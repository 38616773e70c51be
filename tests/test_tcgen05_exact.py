"""Bit-exact tests of the tcgen05 / TMEM / TMA kernels: ``psb_bcast_gemm_kernel`` (1-CTA), ``psb_bcast_gemm2_kernel``
(cta_group::2, every epilogue), the fused stem forward ``psb_stem_fwd_kernel`` with its BatchNorm Σy / Σy² epilogue, and the
implicit stem weight gradient ``psb_stem_wgrad_kernel`` + ``psb_stem_wgrad_finalize_kernel``.

These kernels have no CPU model, so the tests pick inputs that leave no room for rounding:

* **exact-small** — operands in {-1, 0, 1}.  Every product is exact, every partial sum is an integer far below 2^24 and so exact
  in fp32 in any order and any tiling, and every output is representable in bf16: the kernel's output must EQUAL the fp64
  reference.
* **exact-rounding** — non-negative integers sized so that outputs land where bf16 spacing is 2 to 16.  The fp32 accumulator is
  still exact, so the output must be the fp64 reference rounded once to nearest-even; the helpers assert that exact ties occurred.
* **random** — N(0,1)/sqrt(K) data against the derived bound |y - ref| <= 2^-8 |ref| + (1 + 2^-8) (K + 1) 2^-24 sum_k |a_k b_k|
  (bf16 output rounding + worst-case fp32 accumulation): catches a bf16 / fp16 accumulator, which integer data cannot show.

References are fp64 on the same device (``@``, ``F.conv2d``, ``torch.nn.grad.conv2d_weight``) and call no repository kernel.
Every helper asserts its own premise (sums below 2^24, outputs representable, ties present, tiles per CTA), so a shape cannot
silently leave its regime.  Inputs sit inside NaN-filled buffers (the weight at a 16-byte, non-zero offset, as in the parameter
arena): a read outside a tensor map's bounds shows up as NaN in the output.

``backend`` ``cuda`` runs the real kernels (marked ``gpu``); ``emu`` runs a small-shape subset through the CPU emulation of the
extension (``tests/_cuda_emu.py``: the real bindings, im2col and wgrad finalize, ATen stand-ins for the tcgen05 entry points), which
proves references, layouts, premises and moats in every CPU run.  The discrimination tests at the end feed plausible wrong
kernels (a few lines of torch each) to the same helpers and assert that each is rejected, and that the loose tolerances the
older GPU tests use accept some of them.
"""
from __future__ import annotations

import math

import pytest
import torch
import torch.nn.functional as F

from pytorch_ps_mpi_b200.ops.stem import _w2d

BF16 = torch.bfloat16
U32 = 2.0 ** -24          # fp32 unit roundoff
UB = 2.0 ** -8            # bf16 unit roundoff
EXACT = 2.0 ** 24         # integers below this are exact in fp32
NAN = float("nan")


# ================================================================ backends
class Backend:
    def __init__(self, name: str):
        self.name = name
        if name == "cuda":
            from pytorch_ps_mpi_b200.ops import ext
            self.m = ext.cuda()
            self.dev = torch.device("cuda", 0)
            self.sms = torch.cuda.get_device_properties(0).multi_processor_count
        else:
            from tests import _cuda_emu
            self.m = _cuda_emu.build_extension()
            if self.m is None:
                pytest.skip("no g++")
            self.dev = torch.device("cpu")
            self.sms = None               # the stand-ins have no grid
        self.emu = name == "emu"

    def sync(self):
        if not self.emu:
            torch.cuda.synchronize()


_BACKENDS = {}


def backend_of(name: str) -> Backend:
    if name not in _BACKENDS:
        _BACKENDS[name] = Backend(name)
    return _BACKENDS[name]


def cases(gpu, emu=()):
    """``(backend, *case)`` parameters: every case on the GPU (marked ``gpu``), the small ones also on the emulator."""
    out = [pytest.param("cuda", *c, marks=pytest.mark.gpu, id="cuda-" + "-".join(map(str, c))) for c in gpu]
    out += [pytest.param("emu", *c, id="emu-" + "-".join(map(str, c))) for c in emu]
    return out


# ================================================================ data
def _gen(dev, seed):
    return torch.Generator(device=dev).manual_seed(seed)


def ternary(shape, p, g, dev):
    """Values in {-1, 0, 1}: non-zero with probability ``p``, then ±1 with equal odds."""
    nz = torch.rand(shape, generator=g, device=dev) < p
    sign = torch.randint(0, 2, shape, generator=g, device=dev) * 2 - 1
    return (nz * sign).to(BF16)


def uints(shape, hi, g, dev):
    return torch.randint(0, hi + 1, shape, generator=g, device=dev).to(BF16)


def sints(shape, h, g, dev):
    return torch.randint(-h, h + 1, shape, generator=g, device=dev).to(BF16)


def in_moat(t: torch.Tensor, lead: int, trail: int = 64) -> torch.Tensor:
    """A copy of ``t`` (same logical shape and strides order) inside a NaN-filled buffer, ``lead`` elements from its start."""
    flat_src = t.permute(*_dim_order(t)).reshape(-1)
    buf = torch.full((lead + flat_src.numel() + trail,), NAN, dtype=t.dtype, device=t.device)
    buf[lead:lead + flat_src.numel()].copy_(flat_src)
    v = torch.as_strided(buf, t.shape, t.stride(), lead)
    v._moat = (buf, lead, flat_src.numel())
    return v


def _dim_order(t):
    """Dimensions of ``t`` from outermost to innermost in memory (channels-last aware)."""
    return sorted(range(t.dim()), key=lambda d: -t.stride(d))


def moat_intact(v: torch.Tensor):
    buf, lead, n = v._moat
    assert torch.isnan(buf[:lead].float()).all() and torch.isnan(buf[lead + n:].float()).all(), "a kernel wrote into its input moat"


# ================================================================ comparison helpers
def _where(idx, fn):
    return "" if fn is None else " " + fn(idx)


def assert_exact(y: torch.Tensor, ref64: torch.Tensor, where=None, what="y"):
    """``y`` (bf16) equals ``ref64`` rounded once to bf16 (nearest-even), element for element (up to the sign of zero)."""
    assert y.shape == ref64.shape, (y.shape, ref64.shape)
    want = ref64.to(BF16).float()
    got = y.float()
    nan = torch.isnan(got)
    bad = nan | (got != want)
    if bool(bad.any()):
        idx = tuple(int(i) for i in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements differ ({int(nan.sum())} NaN); first at {idx}"
                             f"{_where(idx, where)}: got {float(got[idx])}, want {float(want[idx])} (exact {float(ref64[idx])})")


def assert_bounded(y: torch.Tensor, ref64: torch.Tensor, absdot64: torch.Tensor, k: int, where=None, what="y"):
    """Random regime: |y - ref| <= 2^-8 |ref| + (1 + 2^-8) (k + 1) 2^-24 sum|a b| (output rounding + fp32 accumulation)."""
    err = (y.double() - ref64).abs()
    lim = UB * ref64.abs() + (1 + UB) * (k + 1) * U32 * absdot64
    bad = torch.isnan(err) | (err > lim)
    if bool(bad.any()):
        idx = tuple(int(i) for i in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} elements outside the fp32-accumulation bound; first at {idx}"
                             f"{_where(idx, where)}: got {float(y[idx])}, want {float(ref64[idx])} ± {float(lim[idx])}")


def premise_exact(ref64: torch.Tensor, absdot64: torch.Tensor, representable: bool):
    """Every partial sum (bounded by sum|a b|) is an integer below 2^24 → exact in fp32 in any order; optionally every output
    is a bf16 value."""
    assert float(absdot64.max()) < EXACT, "premise: partial sums may exceed 2^24"
    assert bool((ref64 == ref64.round()).all()), "premise: integer data"
    if representable:
        assert bool((ref64.to(BF16).double() == ref64).all()), "premise: every output representable in bf16"


def ties(ref64: torch.Tensor) -> int:
    """Number of exact bf16 rounding ties (ref64 exact in fp32, low 16 bits == 0x8000)."""
    bits = ref64.float().contiguous().view(torch.int32)
    return int(((bits & 0xFFFF) == 0x8000).sum())


def premise_rounding(ref64: torch.Tensor):
    assert ties(ref64) > 0, "premise: the rounding regime must produce exact ties"


def assert_bits_equal(a: torch.Tensor, b: torch.Tensor, what):
    assert a.shape == b.shape and torch.equal(a.contiguous().view(torch.int16), b.contiguous().view(torch.int16)), what


# ================================================================ bcast_gemm
M_SET = [1, 8, 127, 128, 129, 255, 256, 257, 513]
N_SET = [8, 10, 64, 65, 72, 128, 129, 136, 256, 257, 330]       # 64 / 65 and 128 / 129: both sides of the BNT switch
K_SET = [8, 16, 56, 64, 72, 120, 176, 264, 784, 3072]            # K < 64, partial last K block, long K
ACTS = ["none", "bias", "relu", "both"]
# a covering set: value i of each list meets several partners (cyclic indices of co-prime lengths 9 / 11 / 10 / 4)
GEMM_CASES = [(M_SET[i % 9], N_SET[i % 11], K_SET[i % 10], ACTS[i % 4]) for i in range(22)]
REGIMES = ["small", "round", "random"]


def gemm_variants(N):
    """auto, forced 1-CTA, forced 2-CTA with the staged / row-strided / TMA-store epilogue (the last needs N % 8 == 0)."""
    v = [0, 1, 2 | 1 << 4, 2 | 4 << 4]
    return v + ([2 | 3 << 4] if N % 8 == 0 else [])


def gemm_data(regime, M, N, K, act, dev, seed):
    g = _gen(dev, seed)
    if regime == "small":
        p = min(2 / 3, math.sqrt(900.0 / K))           # var(y) = K p² <= 900: |y| < 256 with overwhelming margin
        x, w = ternary((M, K), p, g, dev), ternary((N, K), p, g, dev)
        b = torch.randint(-4, 5, (N,), generator=g, device=dev).float()
    elif regime == "round":
        hi = max(1, min(15, round(math.sqrt(4000.0 / K))))   # typical y ~ 1000: bf16 spacing 4..8
        x, w = uints((M, K), hi, g, dev), uints((N, K), hi, g, dev)
        b = torch.randint(-600, 601, (N,), generator=g, device=dev).float()   # integers bf16 cannot hold
    else:
        x = (torch.randn(M, K, generator=g, device=dev) / math.sqrt(K)).to(BF16)
        w = torch.randn(N, K, generator=g, device=dev).to(BF16)
        b = torch.randn(N, generator=g, device=dev)
    bias = b if act in ("bias", "both") else None
    relu = act in ("relu", "both")
    return x, w, bias, relu


def gemm_ref(x, w, bias, relu):
    acc = x.double() @ w.double().t()
    absdot = x.double().abs() @ w.double().abs().t()
    if bias is not None:
        acc = acc + bias.double()
        absdot = absdot + bias.double().abs()
    return (acc.relu() if relu else acc), absdot


def gemm_where(M, N, variant, sms):
    """(m, n) → its output tile, cluster / CTA and which kernel produced it (for mismatch reports)."""
    two = (variant & 15) == 2 or ((variant & 15) == 0 and M >= 256)

    def fn(idx):
        m, n = idx
        if two:
            bnt = 64 if N <= 64 else (128 if N <= 128 else 256)
            tn = (N + bnt - 1) // bnt
            tile = (m // 256) * tn + n // bnt
            ncl = min(sms // 2, ((M + 255) // 256) * tn) if sms else 1
            return f"[2-CTA BNT={bnt} tile {tile} (rows {m // 256 * 256}.., cols {n // bnt * bnt}..) cluster {tile % ncl} cta {(m % 256) // 128}]"
        tn = (N + 255) // 256
        tile = (m // 128) * tn + n // 256
        grid = min(sms, ((M + 127) // 128) * tn) if sms else 1
        return f"[1-CTA tile {tile} (rows {m // 128 * 128}.., cols {n // 256 * 256}..) cta {tile % grid}]"
    return fn


def run_gemm(be: Backend, x, w, bias, relu, variant, flag_ptr=0, epoch=0):
    """``bcast_gemm`` with x and the weight inside NaN moats (weight 16 bytes into its buffer, as in the parameter arena)."""
    M, K = x.shape
    N = w.shape[0]
    xm, wm = in_moat(x, 64), in_moat(w, 8)
    y = be.m.bcast_gemm(xm, wm.data_ptr(), N, K, bias, relu, flag_ptr, epoch, 30.0, variant)
    be.sync()
    moat_intact(xm)
    moat_intact(wm)
    assert y.dtype == BF16 and y.shape == (M, N)
    return y


def check_gemm(be, regime, M, N, K, act, variants, seed=0):
    x, w, bias, relu = gemm_data(regime, M, N, K, act, be.dev, seed)
    ref, absdot = gemm_ref(x, w, bias, relu)
    if regime != "random":
        premise_exact(ref, absdot, representable=regime == "small")
    if regime == "round":
        premise_rounding(ref)
    for v in variants:
        y = run_gemm(be, x, w, bias, relu, v)
        what = f"bcast_gemm M={M} N={N} K={K} {act} variant={v:#x}"
        if regime == "random":
            assert_bounded(y, ref, absdot, K, gemm_where(M, N, v, be.sms), what)
        else:
            assert_exact(y, ref, gemm_where(M, N, v, be.sms), what)


@pytest.mark.parametrize("backend,M,N,K,act", cases(GEMM_CASES, GEMM_CASES))
@pytest.mark.parametrize("regime", REGIMES)
def test_bcast_gemm_exact(backend, M, N, K, act, regime):
    be = backend_of(backend)
    check_gemm(be, regime, M, N, K, act, gemm_variants(N), seed=M * 7919 + N * 104729 + K)


# persistent loops that wrap: every CTA (cluster) takes >= 3 tiles, so the smem ring and the 2-deep accumulator ring wrap
WRAP_CASES = [("2cta", 8192, 2048, 264), ("1cta", 8192, 2048, 120)]


@pytest.mark.parametrize("backend,kernel,M,N,K", cases(WRAP_CASES))
@pytest.mark.parametrize("regime", REGIMES)
def test_bcast_gemm_persistent_wrap(backend, kernel, M, N, K, regime):
    be = backend_of(backend)
    if kernel == "2cta":
        bnt = 256
        tiles, grid = ((M + 255) // 256) * ((N + bnt - 1) // bnt), be.sms // 2
        variants = [0, 2 | 1 << 4, 2 | 3 << 4]
    else:
        tiles, grid = ((M + 127) // 128) * ((N + 255) // 256), be.sms
        variants = [1]
    assert tiles >= 3 * grid, f"premise: {tiles} tiles on {grid} {'clusters' if kernel == '2cta' else 'CTAs'} do not wrap"
    check_gemm(be, regime, M, N, K, "both", variants, seed=17)


FLAG_CASES = [(128, 128, 64, 1), (512, 256, 128, 0), (300, 72, 176, 2 | 1 << 4), (257, 136, 72, 2 | 3 << 4)]


@pytest.mark.parametrize("backend,M,N,K,variant", cases(FLAG_CASES, FLAG_CASES))
def test_bcast_gemm_gate_already_published_is_transparent(backend, M, N, K, variant):
    """With the PARAMS_READY epoch already published, the gated kernel computes the ungated result bit for bit."""
    be = backend_of(backend)
    x, w, bias, relu = gemm_data("round", M, N, K, "both", be.dev, 5)
    sig = torch.zeros(512, dtype=torch.int64, device=be.dev)
    sig[be.m.SIG_PARAMS_READY] = 9
    flag = sig.data_ptr() + 8 * be.m.SIG_PARAMS_READY
    y0 = run_gemm(be, x, w, bias, relu, variant)
    y1 = run_gemm(be, x, w, bias, relu, variant, flag, 9)
    assert int(sig[be.m.SIG_ERROR]) == 0
    assert_bits_equal(y0, y1, "gated and ungated GEMM differ")
    assert_exact(y1, gemm_ref(x, w, bias, relu)[0], what="gated GEMM")


# ================================================================ fused stem forward + BN sums
def cl(t):
    return t.contiguous(memory_format=torch.channels_last)


def out_hw(h, w):
    return (h - 1) // 2 + 1, (w - 1) // 2 + 1


# (N, H, W, relation of the N*OH output-row tiles to the B200's 148 SMs)
STEM_SHAPES = [
    (1, 1, 8, "few"),          # OW 4, one tile
    (147, 2, 16, "below"),     # 147 tiles: one per CTA, one SM idle
    (148, 1, 32, "equal"),
    (149, 2, 40, "above"),     # 149 tiles: per = 2 → 74 CTAs get 2, one gets 1, the last 73 none (t0 >= t1)
    (74, 3, 248, "equal"),     # OW 124
    (75, 4, 256, "above"),     # OW 128 (the full UMMA M), 150 tiles → 73 empty CTAs
    (297, 1, 16, "above"),     # per = 3 → 99 busy CTAs, 49 empty
    (37, 7, 40, "equal"),
    (23, 13, 8, "above"),      # 161 tiles
    (2, 224, 32, "above"),     # 224 tiles
    (3, 225, 256, "above"),    # 339 tiles, OH 113: odd-H bottom border
]
STEM_EMU = [(1, 1, 8, "few"), (2, 13, 16, "few"), (3, 7, 40, "few"), (1, 4, 256, "few"), (1, 3, 248, "few")]


def check_tiles(be, n, h, rel):
    if be.sms is None or rel == "few":
        return
    tiles = n * out_hw(h, 8)[0]
    want = {"below": tiles < be.sms, "equal": tiles == be.sms, "above": tiles > be.sms, "many": tiles >= 20 * be.sms}[rel]
    assert want, f"premise: {tiles} tiles should be '{rel}' the {be.sms} SMs"


def stem_data(regime, n, h, w, dev, seed, p=2 / 3):
    g = _gen(dev, seed)
    if regime == "small":
        x, wt = ternary((n, 3, h, w), p, g, dev), ternary((64, 3, 7, 7), p, g, dev)
    elif regime == "round":               # interior y ~ 3800: bf16 spacing 16, ties where y = 8 mod 16
        x, wt = uints((n, 3, h, w), 7, g, dev), uints((64, 3, 7, 7), 15, g, dev)
    else:
        x = torch.randn(n, 3, h, w, generator=g, device=dev).to(BF16)
        wt = (torch.randn(64, 3, 7, 7, generator=g, device=dev) * 0.05).to(BF16)
    return cl(x), wt


def small_density(pixels):
    """Operand density of exact-small data keeping E[Σy²] = 147 p² pixels near 2^22 (sums exact in fp32)."""
    return min(2 / 3, (2.0 ** 22 / (147.0 * pixels)) ** 0.5)


def conv_ref(x, wt):
    ref = F.conv2d(x.double(), wt.double(), stride=2, padding=3)
    absdot = F.conv2d(x.double().abs(), wt.double().abs(), stride=2, padding=3)
    return ref, absdot


def stem_where(n, h, sms):
    oh = out_hw(h, 8)[0]
    tiles = n * oh
    grid = min(tiles, sms) if sms else 1
    per = -(-tiles // grid)

    def fn(idx):
        t = idx[0] * oh + idx[2]
        return f"[tile {t} (image {idx[0]}, output row {idx[2]}) cta {t // per} of {grid}, channel {idx[1]}, column {idx[3]}]"
    return fn


def sums_depth(n, h, w, sms):
    """Longest chain of fp32 additions behind one sum of the kernel: a thread adds ceil(OW/2) rows of each of its CTA's
    tiles, then one atomic per CTA."""
    oh, ow = out_hw(h, w)
    tiles = n * oh
    grid = min(tiles, sms) if sms else tiles
    return (ow + 1) // 2 * -(-tiles // grid) + grid + 1


def assert_sums(sums, y, exact, depth):
    """Σy | Σy² of the kernel against the fp64 sums of its OWN bf16 output: equal when every partial sum is an integer below
    2^24 (exact regime), else within depth · 2^-24 · Σ|term| (fp32 recursive summation)."""
    yd = y.detach().double()
    want = torch.cat([yd.sum((0, 2, 3)), (yd * yd).sum((0, 2, 3))])
    mag = torch.cat([yd.abs().sum((0, 2, 3)), (yd * yd).sum((0, 2, 3))])
    assert sums is not None and sums.shape == (128,) and sums.dtype == torch.float32
    got = sums.double()
    if exact:
        assert float(mag.max()) < EXACT, "premise: Σ|y| and Σy² below 2^24"
        bad = got != want
    else:
        bad = torch.isnan(got) | ((got - want).abs() > depth * U32 * mag)
    if bool(bad.any()):
        c = int(bad.nonzero()[0])
        raise AssertionError(f"BN sums: {int(bad.sum())} of 128 differ; first {'Σy' if c < 64 else 'Σy²'}[{c % 64}]: "
                             f"got {float(got[c])}, want {float(want[c])}")


def run_stem_fwd(be, x, wt, want_sums):
    xm, wm = in_moat(x, 64), in_moat(_w2d(wt), 8)
    y, sums = be.m.stem_fwd(xm, wm, want_sums)
    be.sync()
    moat_intact(xm)
    moat_intact(wm)
    return y, (sums if want_sums else None)


def check_stem_fwd(be, regime, n, h, w, p=None, sums_exact=None):
    pixels = n * out_hw(h, w)[0] * out_hw(h, w)[1]
    x, wt = stem_data(regime, n, h, w, be.dev, n * 1009 + h * 31 + w, p if p is not None else small_density(pixels))
    ref, absdot = conv_ref(x, wt)
    if regime != "random":
        premise_exact(ref, absdot, representable=regime == "small")
    if regime == "round":
        premise_rounding(ref)
    y, sums = run_stem_fwd(be, x, wt, True)
    y2, none = run_stem_fwd(be, x, wt, False)
    assert y.shape == ref.shape and y.is_contiguous(memory_format=torch.channels_last)
    what = f"stem_fwd N={n} H={h} W={w} {regime}"
    if regime == "random":
        assert_bounded(y, ref, absdot, 147, stem_where(n, h, be.sms), what)
    else:
        assert_exact(y, ref, stem_where(n, h, be.sms), what)
    assert_bits_equal(y, y2, "want_sums=False changed y")
    if sums_exact is None:
        sums_exact = regime == "small"
    assert_sums(sums, y, sums_exact, sums_depth(n, h, w, be.sms))


@pytest.mark.parametrize("backend,n,h,w,rel", cases(STEM_SHAPES, STEM_EMU))
@pytest.mark.parametrize("regime", REGIMES)
def test_stem_fwd_exact(backend, n, h, w, rel, regime):
    be = backend_of(backend)
    check_tiles(be, n, h, rel)
    check_stem_fwd(be, regime, n, h, w)


@pytest.mark.gpu
def test_stem_fwd_production_batch_32():
    """ResNet input, batch 32: 3584 tiles, about 25 per CTA — exact y and exact sums."""
    be = backend_of("cuda")
    check_tiles(be, 32, 224, "many")
    check_stem_fwd(be, "small", 32, 224, 224)


@pytest.mark.gpu
def test_stem_fwd_batch_256():
    """bench.py's batch: about 194 tiles per CTA.  y exact at full density; Σy² exceeds 2^24, so the sums are held to the
    fp32 summation bound."""
    be = backend_of("cuda")
    check_tiles(be, 256, 224, "many")
    check_stem_fwd(be, "small", 256, 224, 224, p=2 / 3, sums_exact=False)


STEM_AUTOGRAD = [(2, 13, 16), (1, 30, 40), (3, 64, 64), (2, 225, 256)]
STEM_AUTOGRAD_EMU = [(2, 13, 16), (1, 9, 40)]


@pytest.fixture
def ops_on(monkeypatch):
    """Route ``ops.ext.cuda()`` (and, for the emulator, ``Tensor.is_cuda``) to the backend under test."""
    def use(be):
        from pytorch_ps_mpi_b200.ops import ext as ops_ext
        from pytorch_ps_mpi_b200.ops import stem as stem_mod
        monkeypatch.setattr(ops_ext, "cuda", lambda: be.m)
        monkeypatch.setattr(stem_mod, "_IMPLICIT_WGRAD", True)
        if be.emu:
            monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
        return stem_mod
    return use


@pytest.mark.parametrize("backend,n,h,w", cases(STEM_AUTOGRAD, STEM_AUTOGRAD_EMU))
def test_stem_conv_fused_autograd_exact(backend, n, h, w, ops_on):
    """``stem_conv_fused`` forward and ``_StemFused.backward`` (implicit wgrad → finalize → GEMM-layout view)."""
    be = backend_of(backend)
    stem_mod = ops_on(be)
    x, wt = stem_data("small", n, h, w, be.dev, 3)
    gy = cl(sints((n, 64) + out_hw(h, w), 2, _gen(be.dev, 4), be.dev))
    wv = wt.clone().requires_grad_(True)
    y, sums = stem_mod.stem_conv_fused(x, wv)
    ref, absdot = conv_ref(x, wt)
    premise_exact(ref, absdot, representable=True)
    assert_exact(y, ref, what="stem_conv_fused y")
    assert_sums(sums, y, True, sums_depth(n, h, w, be.sms))
    y.backward(gy)
    gref = torch.nn.grad.conv2d_weight(x.double(), wt.shape, gy.double(), stride=2, padding=3)
    premise_exact(gref, torch.nn.grad.conv2d_weight(x.double().abs(), wt.shape, gy.double().abs(), stride=2, padding=3), False)
    assert_exact(wv.grad, gref, what="_StemFused.backward dW")


@pytest.mark.parametrize("backend,n,h,w", cases(STEM_AUTOGRAD, STEM_AUTOGRAD_EMU))
def test_stem_conv_im2col_fallback_exact(backend, n, h, w, ops_on):
    """``stem_conv``: im2col patch matrix + ``bcast_gemm`` (the path for widths the fused kernel does not take)."""
    be = backend_of(backend)
    stem_mod = ops_on(be)
    for regime in ("small", "round"):
        x, wt = stem_data(regime, n, h, w, be.dev, 6)
        ref, absdot = conv_ref(x, wt)
        premise_exact(ref, absdot, representable=regime == "small")
        y = stem_mod.stem_conv(x, wt)
        assert_exact(y, ref, what=f"stem_conv {regime}")


# ================================================================ stem weight gradient
def wgrad_data(regime, n, h, w, dev, seed):
    g = _gen(dev, seed)
    oh, ow = out_hw(h, w)
    if regime == "small":
        x, gy = ternary((n, 3, h, w), 2 / 3, g, dev), ternary((n, 64, oh, ow), 2 / 3, g, dev)
    else:
        # x in {0..3}, gy signed with |dW| ~ 800 (bf16 spacing 4): rounding with ties at every size
        hg = 800.0 / (1.87 * math.sqrt(n * oh * ow))
        hg = max(1, min(256, round(math.sqrt(3 * hg * hg + 0.25) - 0.5)))
        x, gy = uints((n, 3, h, w), 3, g, dev), sints((n, 64, oh, ow), hg, g, dev)
    return cl(x), cl(gy)


def wgrad_ref(x, gy):
    """dW2d [64,176] in the kernel's GEMM layout (pad columns 21-23 of each kernel row and 168-175 zero)."""
    gref = torch.nn.grad.conv2d_weight(x.double(), (64, 3, 7, 7), gy.double(), stride=2, padding=3)
    gabs = torch.nn.grad.conv2d_weight(x.double().abs(), (64, 3, 7, 7), gy.double().abs(), stride=2, padding=3)
    return _w2d(gref), _w2d(gabs)


PAD_COLS = [kh * 24 + c for kh in range(7) for c in (21, 22, 23)] + list(range(168, 176))


def wgrad_where(idx):
    co, k = idx
    return f"[co {co}, k {k} = kernel row {k // 24}, column {k % 24} (kw {k % 24 // 3}, c {k % 3})]"


def check_wgrad(be, regime, n, h, w):
    x, gy = wgrad_data(regime, n, h, w, be.dev, n * 131 + h * 7 + w)
    ref, gabs = wgrad_ref(x, gy)
    premise_exact(ref, gabs, representable=False)
    if regime == "round":
        premise_rounding(ref)
    xm, gm = in_moat(x, 64), in_moat(gy, 64)
    partial = be.m.stem_wgrad(xm, gm)
    if be.sms is not None:
        oh = out_hw(h, w)[0]
        tiles = n * oh
        grid = min(tiles, be.sms)
        per = -(-tiles // grid)
        assert partial.shape == (grid, 176, 64)
        empty = [c for c in range(grid) if c * per >= tiles]
        if empty:                         # CTAs without tiles write zero partials
            assert bool((partial[empty] == 0).all()), "an empty CTA's partial is not zero"
    d = be.m.stem_wgrad_finalize(partial)
    # out= inside a sentinel buffer, 16 bytes in: the result lands there and nothing around it changes
    sentinel = torch.full((8 + 64 * 176 + 64,), -7.0, dtype=BF16, device=be.dev)
    before = sentinel.clone()
    out = sentinel[8:8 + 64 * 176]
    d2 = be.m.stem_wgrad_finalize(partial, out)
    be.sync()
    moat_intact(xm)
    moat_intact(gm)
    what = f"stem wgrad N={n} H={h} W={w} {regime}"
    assert_exact(d, ref, wgrad_where, what)
    assert bool((d[:, PAD_COLS] == 0).all()), "pad columns of dW2d must be exactly zero"
    assert d2.data_ptr() == out.data_ptr()
    assert_bits_equal(d2, d, "finalize with out= differs")
    assert torch.equal(sentinel[:8].view(torch.int16), before[:8].view(torch.int16))
    assert torch.equal(sentinel[8 + 64 * 176:].view(torch.int16), before[8 + 64 * 176:].view(torch.int16))


@pytest.mark.parametrize("backend,n,h,w,rel", cases(STEM_SHAPES, STEM_EMU))
@pytest.mark.parametrize("regime", ["small", "round"])
def test_stem_wgrad_exact(backend, n, h, w, rel, regime):
    be = backend_of(backend)
    check_tiles(be, n, h, rel)
    check_wgrad(be, regime, n, h, w)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [32, 256])
def test_stem_wgrad_production(n):
    be = backend_of("cuda")
    check_tiles(be, n, 224, "many")
    check_wgrad(be, "round", n, 224, 224)


# ================================================================ discrimination (CPU, no kernels)
# Plausible wrong kernels, a few lines of torch each.  The helpers above must reject every one at the test shapes; the
# tolerances of the older GPU tests (allclose 2e-2, max-relative 2e-2 / 1e-2, sums 1e-3) accept some of them.
CPU = torch.device("cpu")


def old_gemm_ok(y, ref):
    return torch.allclose(y.float(), ref.float(), rtol=2e-2, atol=2e-2)


def old_rel(a, b):
    return (a.float() - b.float()).abs().max().item() / max(b.float().abs().max().item(), 1e-6)


def rejects(fn, *a, **k):
    try:
        fn(*a, **k)
    except AssertionError:
        return True
    return False


def rz_bf16(t32):
    """fp32 → bf16 rounding toward zero (drop the low 16 bits)."""
    return (t32.float().contiguous().view(torch.int32) & -65536).view(torch.float32).to(BF16)


def test_discriminates_rz_rounding_and_early_bias_rounding():
    old_accepts = 0
    for M, N, K, act in GEMM_CASES:
        x, w, bias, relu = gemm_data("round", M, N, K, "both", CPU, M + N + K)
        ref, absdot = gemm_ref(x, w, bias, relu)
        premise_exact(ref, absdot, False)
        premise_rounding(ref)
        rz = rz_bf16(ref)                                                     # RZ instead of RNE in pack_bf16x2
        early = (x.double() @ w.double().t() + bias.to(BF16).double()).relu()   # bias rounded to bf16 before the add
        assert rejects(assert_exact, rz, ref), (M, N, K)
        assert rejects(assert_exact, early.to(BF16), ref), (M, N, K)
        old_accepts += old_gemm_ok(rz, ref) and old_gemm_ok(early.to(BF16), ref)
    assert old_accepts > 0


def test_discriminates_gemm_structure_bugs():
    nk = nb = 0
    for M, N, K, act in GEMM_CASES:
        x, w, bias, relu = gemm_data("small", M, N, K, "both", CPU, M * N + K)
        ref, _ = gemm_ref(x, w, bias, relu)
        acc = x.double() @ w.double().t()
        after = (acc.relu() + bias.double()).to(BF16)                      # bias added after the ReLU
        assert rejects(assert_exact, after, ref), (M, N, K)
        nb += 1
        if K > 64 and K % 64:
            kk = K // 64 * 64                                               # the last, partial K block dropped
            drop = (x[:, :kk].double() @ w[:, :kk].double().t() + bias.double()).relu().to(BF16)
            assert rejects(assert_exact, drop, ref), (M, N, K)
            nk += 1
    assert nk >= 4 and nb == len(GEMM_CASES)


def test_discriminates_reduced_precision_accumulator():
    """A bf16 (or fp16) accumulator passes on integer data but not the random-regime bound."""
    for M, N, K in [(127, 64, 264), (129, 72, 784), (8, 256, 3072)]:
        x, w, bias, relu = gemm_data("random", M, N, K, "none", CPU, K)
        ref, absdot = gemm_ref(x, w, bias, relu)
        assert_bounded(ref.float().to(BF16), ref, absdot, K)              # the correct result is accepted
        for acc_dt in (BF16, torch.float16):
            acc = torch.zeros(M, N, dtype=acc_dt)
            for k in range(K):
                acc = (acc.float() + x[:, k:k + 1].float() * w[:, k].float()).to(acc_dt)
            assert rejects(assert_bounded, acc.float().to(BF16), ref, absdot, K), (M, N, K, acc_dt)


def test_discriminates_right_border_padding_tap():
    """One padding tap at the right image border reads the last real column instead of zero."""
    for n, h, w, _ in STEM_EMU + [(2, 30, 64, "few")]:
        x, wt = stem_data("small", n, h, w, CPU, 11)
        ref, _ = conv_ref(x, wt)
        xp = F.pad(x.double(), (3, 3, 3, 3))
        xp[..., 3 + w] = xp[..., 2 + w]
        bad = F.conv2d(xp, wt.double(), stride=2).to(BF16)
        assert rejects(assert_exact, bad, ref), (n, h, w)


def test_discriminates_bn_sums_missing_row():
    """Σy loses one output pixel of one tile (a sum loop stopping one short).  Non-negative data: the loss is then tiny
    relative to the sums."""
    old_accepts = 0
    for n, h, w in [(1, 13, 16), (3, 7, 40), (2, 30, 64), (4, 64, 64)]:
        g = _gen(CPU, 12)
        x, wt = cl(uints((n, 3, h, w), 1, g, CPU)), uints((64, 3, 7, 7), 1, g, CPU)
        y = conv_ref(x, wt)[0].to(BF16)
        yd = y.double()
        good = torch.cat([yd.sum((0, 2, 3)), (yd * yd).sum((0, 2, 3))]).float()
        assert_sums(good, y, True, 0)
        yd_drop = yd.clone()
        yd_drop[-1, :, -1, -1] = 0
        bad = torch.cat([yd_drop.sum((0, 2, 3)), (yd_drop * yd_drop).sum((0, 2, 3))]).float()
        assert rejects(assert_sums, bad, y, True, 0), (n, h, w)
        old_accepts += bool((((bad - good).abs() / (good.abs() + 1.0)).max() < 1e-3))
    assert old_accepts > 0


def test_discriminates_dropped_wgrad_partial():
    """The weight gradient loses one CTA's partial (here: the last output-row tile).  Non-negative data: the loss is then
    small relative to the gradient."""
    old_accepts = 0
    for n, h, w in [(1, 13, 16), (3, 7, 40), (4, 64, 64), (16, 224, 32)]:
        g = _gen(CPU, 13)
        x, gy = cl(uints((n, 3, h, w), 1, g, CPU)), cl(uints((n, 64) + out_hw(h, w), 1, g, CPU))
        ref, gabs = wgrad_ref(x, gy)
        premise_exact(ref, gabs, False)
        assert_exact(ref.to(BF16), ref)
        g2 = gy.clone()
        g2[-1, :, -1, :] = 0
        bad = wgrad_ref(x, g2)[0].to(BF16)
        assert rejects(assert_exact, bad, ref), (n, h, w)
        old_accepts += old_rel(bad, ref) < 1e-2
    assert old_accepts > 0
