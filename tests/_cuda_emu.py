"""Run the REAL CUDA source of the parameter-server kernels (``csrc/kernels/ps_kernels.cu`` + the conversion helpers of
``common.cuh``) on the CPU.

Every CUDA thread of a CTA is a user-level fiber (``ucontext``) on ONE OS thread, scheduled round-robin and switched at barriers
(CTAs one after another): ``__syncthreads`` / warp barriers are generation counters, warp shuffles / ballots go through a per-warp
exchange buffer, atomics are plain read-modify-writes (nothing runs concurrently), shared memory = function statics, system-scope loads / stores / fences
= plain accesses (one process, one address space: "peer" arenas are just other buffers).  Only the PTX wrappers (``ld.relaxed.sys``,
``st.release.sys``, ``multimem.*``, ``%globaltimer``) are replaced by hand-written equivalents; everything else — encode (cast /
scale / radix-select top-k), the fused gather-decode-sum-SGD/Adam-publish kernel, the flag kernels — is compiled from the
repository's ``.cu`` text with g++.  ``multimem.st`` / ``multimem.ld_reduce`` (NVLS) act on registered multicast windows: a
multicast address is an offset applied to every rank's buffer (store = replicate; load-reduce = fp32 sum over the ranks, rounded
once to the wire type).

This is a numerics / indexing oracle that runs in every CPU round; it says nothing about timing or memory-model races (those are the
GPU tests' and ``protocol_model.py``'s job)."""
from __future__ import annotations

import ctypes
import os
import re
import shutil
import subprocess
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KDIR = os.path.join(ROOT, "pytorch_ps_mpi_b200", "csrc", "kernels")
CUDA_INC = "/usr/local/cuda/include"


def cut_function(src: str, header_regex: str) -> str:
    """The text of the first function whose header matches ``header_regex`` (from the match to its closing brace)."""
    m = re.search(header_regex, src)
    if m is None:
        raise KeyError(header_regex)
    depth, i = 0, src.index("{", m.start())
    while True:
        depth += src[i] == "{"
        depth -= src[i] == "}"
        i += 1
        if depth == 0:
            return src[m.start():i]


SHIM_HEAD = r'''
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>
#include <ucontext.h>
#include <time.h>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>
#include <algorithm>
#undef __device__
#undef __global__
#undef __forceinline__
#undef __shared__
#undef __launch_bounds__
#define __device__
#define __global__
#define __forceinline__ inline
#define __shared__ static
#define __launch_bounds__(...)
#define __grid_constant__
#define __restrict__
using std::min;
using std::max;
using std::isfinite;

struct EmuIdx { unsigned x; };
static EmuIdx threadIdx, blockIdx, gridDim, blockDim;     // one OS thread: the scheduler sets threadIdx at every switch

// ---- fibers: one per CUDA thread of the running CTA ----
struct EmuFiber { ucontext_t ctx; bool done; };
static EmuFiber emu_fib[1024];
static char* emu_stacks = nullptr;
static const size_t EMU_STACK = 96 * 1024;
static ucontext_t emu_sched_ctx;
static int emu_cur = 0, emu_live = 0, emu_warp_live[32];
static int emu_bar_count = 0, emu_bar_gen = 0, emu_wbar_count[32], emu_wbar_gen[32];
static void (*emu_body_call)(void*) = nullptr;
static void* emu_body_obj = nullptr;
static uint64_t emu_xchg[32][32];
static int emu_pred[1024];

static inline void emu_yield() { swapcontext(&emu_fib[emu_cur].ctx, &emu_sched_ctx); }
static void emu_trampoline() {
  emu_body_call(emu_body_obj);
  const int w = emu_cur >> 5;
  emu_fib[emu_cur].done = true;
  --emu_live;
  --emu_warp_live[w];
  // like the hardware, an exited thread no longer counts at a barrier its siblings are waiting in
  if (emu_live > 0 && emu_bar_count >= emu_live && emu_bar_count > 0) { emu_bar_count = 0; ++emu_bar_gen; }
  if (emu_warp_live[w] > 0 && emu_wbar_count[w] >= emu_warp_live[w] && emu_wbar_count[w] > 0) { emu_wbar_count[w] = 0; ++emu_wbar_gen[w]; }
  swapcontext(&emu_fib[emu_cur].ctx, &emu_sched_ctx);
}
static inline void __syncthreads() {
  const int g = emu_bar_gen;
  if (++emu_bar_count >= emu_live) { emu_bar_count = 0; ++emu_bar_gen; }
  else while (emu_bar_gen == g) emu_yield();
}
static inline void emu_warp_barrier() {
  const int w = threadIdx.x >> 5, g = emu_wbar_gen[w];
  if (++emu_wbar_count[w] >= emu_warp_live[w]) { emu_wbar_count[w] = 0; ++emu_wbar_gen[w]; }
  else while (emu_wbar_gen[w] == g) emu_yield();
}
static inline int __syncthreads_and(int p) {
  emu_pred[threadIdx.x] = p;
  __syncthreads();
  int r = 1;
  for (unsigned i = 0; i < blockDim.x; ++i) r &= emu_pred[i] != 0;
  __syncthreads();
  return r;
}
static inline void __syncwarp() { emu_warp_barrier(); }
template <class T> static inline T emu_exchange(T v, int src_lane) {
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  uint64_t bits = 0; memcpy(&bits, &v, sizeof(T));
  emu_xchg[w][l] = bits;
  emu_warp_barrier();
  T out = v;
  if (src_lane >= 0 && src_lane < 32) memcpy(&out, &emu_xchg[w][src_lane], sizeof(T));
  emu_warp_barrier();
  return out;
}
template <class T> static inline T __shfl_up_sync(unsigned, T v, int off) { const int l = threadIdx.x & 31; return emu_exchange(v, l >= off ? l - off : -1); }
template <class T> static inline T __shfl_xor_sync(unsigned, T v, int m) { return emu_exchange(v, (int)((threadIdx.x & 31) ^ m)); }
static inline unsigned __ballot_sync(unsigned, int p) {
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  emu_xchg[w][l] = p != 0;
  emu_warp_barrier();
  unsigned r = 0;
  const unsigned lanes = std::min(32u, blockDim.x - 32u * w);
  for (unsigned i = 0; i < lanes; ++i) r |= (unsigned)(emu_xchg[w][i] != 0) << i;
  emu_warp_barrier();
  return r;
}
static inline int __any_sync(unsigned m, int p) { return __ballot_sync(m, p) != 0; }
static inline int __popc(unsigned v) { return __builtin_popcount(v); }
static inline int __clz(unsigned v) { return v ? __builtin_clz(v) : 32; }
static inline void __threadfence_system() { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
static inline void __threadfence() { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
static inline void __nanosleep(unsigned) { emu_yield(); }
static inline unsigned long long emu_now_ns() {       // stands in for %globaltimer
  timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts);
  return (unsigned long long)ts.tv_sec * 1000000000ull + (unsigned long long)ts.tv_nsec + 1ull;
}
template <class T> static inline T atomicAdd(T* p, T v) { return __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
static inline float atomicAdd(float* p, float v) {
  uint32_t* q = reinterpret_cast<uint32_t*>(p); uint32_t o = __atomic_load_n(q, __ATOMIC_SEQ_CST), n;
  float f;
  do { memcpy(&f, &o, 4); f += v; memcpy(&n, &f, 4); } while (!__atomic_compare_exchange_n(q, &o, n, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST));
  memcpy(&f, &o, 4); return f;
}
template <class T> static inline T atomicMax(T* p, T v) { T o = __atomic_load_n(p, __ATOMIC_SEQ_CST); while (o < v && !__atomic_compare_exchange_n(p, &o, v, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST)) {} return o; }
template <class T> static inline T atomicMin(T* p, T v) { T o = __atomic_load_n(p, __ATOMIC_SEQ_CST); while (o > v && !__atomic_compare_exchange_n(p, &o, v, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST)) {} return o; }
template <class T> static inline T atomicOr(T* p, T v) { return __atomic_fetch_or(p, v, __ATOMIC_SEQ_CST); }
static inline unsigned __float_as_uint(float f) { unsigned u; memcpy(&u, &f, 4); return u; }
static inline float __uint_as_float(unsigned u) { float f; memcpy(&f, &u, 4); return f; }
static inline float __fdiv_rn(float a, float b) { return a / b; }
static inline float __fsqrt_rn(float a) { return sqrtf(a); }
static inline int __float2int_rn(float a) { return (int)nearbyintf(a); }

#include "common.cuh"      // constants, TileInfo, GroupHyper, wire_elem_bytes (host part of the real header)

namespace psb {
// ---- hand-written stand-ins for the PTX wrappers of common.cuh ----
static inline uint64_t ld_acquire_sys(const uint64_t* p) { return __atomic_load_n(p, __ATOMIC_ACQUIRE); }
static inline uint64_t ld_relaxed_sys_u64(const uint64_t* p) { return __atomic_load_n(p, __ATOMIC_RELAXED); }
static inline void st_release_sys(uint64_t* p, uint64_t v) { __atomic_store_n(p, v, __ATOMIC_RELEASE); }
static inline void st_relaxed_sys_f32(float* p, float v) { *p = v; }
static inline uint4 ld_sys_v4(const void* p) { uint4 v; memcpy(&v, p, 16); return v; }
static inline uint2 ld_sys_v2(const void* p) { uint2 v; memcpy(&v, p, 8); return v; }
static inline float ld_sys_f32(const float* p) { return *p; }
static inline uint4 ld_stream_v4(const void* p) { uint4 v; memcpy(&v, p, 16); return v; }
static inline void st_v4(void* p, uint4 v) { memcpy(p, &v, 16); }
static inline void st_sys_v4(void* p, uint4 v) { memcpy(p, &v, 16); }
// ---- multicast windows (NVLS): a multicast address is an offset into a window bound to every rank's buffer ----
struct EmuMcWindow { const uint8_t* mc; size_t nbytes; int n; uint8_t* base[16]; };
static EmuMcWindow emu_mc[8];
static int emu_mc_n = 0;
static inline const EmuMcWindow& emu_mc_find(const void* p, size_t* off) {
  const uint8_t* q = static_cast<const uint8_t*>(p);
  for (int i = 0; i < emu_mc_n; ++i)
    if (q >= emu_mc[i].mc && q + 16 <= emu_mc[i].mc + emu_mc[i].nbytes) { *off = q - emu_mc[i].mc; return emu_mc[i]; }
  fprintf(stderr, "multimem access outside every registered multicast window\n");
  abort();
}
static inline void multimem_st_v4(void* mc, uint4 v) {            // multimem.st: the switch replicates the store
  size_t off;
  const EmuMcWindow& w = emu_mc_find(mc, &off);
  for (int r = 0; r < w.n; ++r) memcpy(w.base[r] + off, &v, 16);
}
static inline uint4 multimem_ld_reduce_f32x4(const void* mc) {    // multimem.ld_reduce.add.f32: one load per rank, summed
  size_t off;
  const EmuMcWindow& w = emu_mc_find(mc, &off);
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int r = 0; r < w.n; ++r) { float t[4]; memcpy(t, w.base[r] + off, 16); for (int j = 0; j < 4; ++j) acc[j] += t[j]; }
  uint4 v; memcpy(&v, acc, 16); return v;
}
static inline uint4 emu_mc_reduce_16bit(const void* mc, bool bf) {   // .acc::f32: fp32 accumulation, ONE rounding to the wire type
  size_t off;
  const EmuMcWindow& w = emu_mc_find(mc, &off);
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int r = 0; r < w.n; ++r) {
    uint16_t t[8]; memcpy(t, w.base[r] + off, 16);
    for (int j = 0; j < 8; ++j) {
      if (bf) { uint32_t u = (uint32_t)t[j] << 16; float f; memcpy(&f, &u, 4); acc[j] += f; }
      else { __half h; memcpy(&h, &t[j], 2); acc[j] += __half2float(h); }
    }
  }
  uint16_t o[8];
  for (int j = 0; j < 8; ++j) {
    if (bf) { __nv_bfloat16 b = __float2bfloat16_rn(acc[j]); memcpy(&o[j], &b, 2); }
    else { __half h = __float2half_rn(acc[j]); memcpy(&o[j], &h, 2); }
  }
  uint4 v; memcpy(&v, o, 16); return v;
}
static inline uint4 multimem_ld_reduce_bf16x8(const void* mc) { return emu_mc_reduce_16bit(mc, true); }
static inline uint4 multimem_ld_reduce_f16x8(const void* mc) { return emu_mc_reduce_16bit(mc, false); }
'''

def real_spin(common: str) -> str:
    """The repository's bounded spin (``common.cuh::spin_until_ge``: time-out → error slot), reading the emulated clock."""
    return cut_function(common, r"__device__ __forceinline__ bool spin_until_ge\(").replace(
        'asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));', "now = emu_now_ns();")


CONVERSIONS = ["unpack_bf16x8", "unpack_f16x8", "unpack_fp8x8", "unpack_i8x8", "pack_bf16x2", "pack_f16x2_sat", "pack_f16x2",
               "pack_fp8x4", "pack_i8x4", "load8_local", "pack8"]

RUNNER = r'''
// ---- CTA runner: the threads of a CTA are fibers scheduled round-robin on this OS thread; CTAs run one after another ----
template <class F> static void emu_call_body(void* p) { (*static_cast<F*>(p))(); }
template <class F> static void emu_launch(int grid, int block, F body) {
  gridDim.x = grid; blockDim.x = block;
  if (emu_stacks == nullptr) emu_stacks = static_cast<char*>(malloc(EMU_STACK * 1024));
  emu_body_call = &emu_call_body<F>;
  emu_body_obj = &body;
  const int warps = (block + 31) / 32;
  for (int b = 0; b < grid; ++b) {
    blockIdx.x = b;
    emu_live = block; emu_bar_count = 0;
    for (int w = 0; w < warps; ++w) { emu_warp_live[w] = std::min(32, block - 32 * w); emu_wbar_count[w] = 0; }
    for (int t = 0; t < block; ++t) {
      getcontext(&emu_fib[t].ctx);
      emu_fib[t].ctx.uc_stack.ss_sp = emu_stacks + (size_t)t * EMU_STACK;
      emu_fib[t].ctx.uc_stack.ss_size = EMU_STACK;
      emu_fib[t].ctx.uc_link = nullptr;
      emu_fib[t].done = false;
      makecontext(&emu_fib[t].ctx, emu_trampoline, 0);
    }
    while (emu_live > 0)
      for (int t = 0; t < block; ++t)
        if (!emu_fib[t].done) { emu_cur = t; threadIdx.x = t; swapcontext(&emu_sched_ctx, &emu_fib[t].ctx); }
  }
}

'''

LAUNCH_RE = re.compile(r"(\w+(?:<[^<>;]*>)?)<<<([^;]*?),\s*([^,;]*?),\s*([^,;]*?),\s*s>>>\((.*?)\)(\s*;|\s*\n)", re.S)


def rewrite_launches(text: str):
    """``kernel<<<grid, block, smem, s>>>(args);`` → ``emu_launch(grid, block, [&] { kernel(args); });`` (returns text, count)."""
    return LAUNCH_RE.subn(lambda m: f"emu_launch({m.group(2)}, {m.group(3)}, [&] {{ {m.group(1)}({m.group(5)}); }}){m.group(6)}", text)


CUDA_RT_SHIM = r'''
static inline int emu_cudaGetDevice(int* d) { *d = 0; return 0; }
// the "GPU" has emu_sm_count SMs (148 = B200).  Tests shrink it so that the launchers' grid caps bind on small tensors and the
// kernels' grid-stride loops run more than one iteration per CTA — on hardware that is the normal case (ResNet-18: 14 336 pool rows
// on 2 368 CTAs).  Weak: one copy shared by every emulated translation unit of a library.
__attribute__((weak)) int emu_sm_count = 148;
extern "C" __attribute__((weak)) void emu_set_sm_count(int n) { emu_sm_count = n; }
static inline int emu_cudaDeviceGetAttribute(int* v, int, int) { *v = emu_sm_count; return 0; }
static inline int emu_cudaMemsetAsync(void* p, int v, size_t n, cudaStream_t) { memset(p, v, n); return 0; }
'''

DRIVER = r'''
extern "C" int emu_encode(int kind, int wire, int n, const void** src, const int* first_tile, const int* ntiles, const int* param,
                          const void* tiles, void* wire_arena, float* scales, uint32_t* amax, float* residual, int bpt, int cap,
                          double ratio, int grad_dt, uint64_t** sig_targets, int nsig, int sig_slot, uint64_t sig_value,
                          unsigned* sig_counter) {
  EncodeArgs a{};
  a.batch.n = n; a.batch.cum[0] = 0;
  for (int i = 0; i < n; ++i) { a.batch.src[i] = src[i]; a.batch.first_tile[i] = first_tile[i]; a.batch.param[i] = param[i]; a.batch.cum[i + 1] = a.batch.cum[i] + ntiles[i]; }
  a.tiles = reinterpret_cast<const TileInfo*>(tiles); a.wire = wire_arena; a.scales = scales; a.amax_bits = amax; a.residual = residual;
  a.bytes_per_tile = bpt; a.cap = cap; a.ratio = ratio; a.grad_dt = grad_dt;
  a.nsig = nsig; for (int i = 0; i < nsig; ++i) a.sig_targets[i] = sig_targets[i];
  a.sig_slot = sig_slot; a.sig_value = sig_value; a.sig_counter = sig_counter;
  // the REAL launchers (dispatch tables included): an unsupported (kind, wire) pair launches nothing and the caller's
  // comparison with the oracle fails
  if (kind == KIND_SCALED) psb_launch_absmax(nullptr, a);
  psb_launch_encode(nullptr, kind, wire, a);
  return 0;
}

// async-only arguments of the next emu_update call (consumed by it): version published, device-side selection, averaging
static uint64_t emu_x_version = 0; static const uint64_t* emu_x_select = nullptr; static int emu_x_avg = 0;
static double emu_x_timeout = 2.0;
extern "C" void emu_update_extra(uint64_t version, const uint64_t* select_out, int average_dynamic, double timeout_s) {
  emu_x_version = version; emu_x_select = select_out; emu_x_avg = average_dynamic; emu_x_timeout = timeout_s;
}
// multicast (NVLS) arguments of the next emu_update call + the window registry
static void* emu_x_param_mc = nullptr; static const void* emu_x_wire_mc = nullptr; static int emu_x_reduce = 0;
extern "C" void emu_update_mc(void* param_mc, const void* wire_mc, int reduce) {
  emu_x_param_mc = param_mc; emu_x_wire_mc = wire_mc; emu_x_reduce = reduce;
}
extern "C" int emu_mc_register(const void* mc, size_t nbytes, int n, void** bases) {
  if (psb::emu_mc_n >= 8 || n > 16) return -1;
  psb::EmuMcWindow& w = psb::emu_mc[psb::emu_mc_n];
  w.mc = static_cast<const uint8_t*>(mc); w.nbytes = nbytes; w.n = n;
  for (int r = 0; r < n; ++r) w.base[r] = static_cast<uint8_t*>(bases[r]);
  return psb::emu_mc_n++;
}
extern "C" void emu_mc_clear() { psb::emu_mc_n = 0; }
extern "C" int emu_update(int kind, int wire, int opt, int world, int rank, void** wire_p, float** scales_p, void** param_dst,
                          void* param_local, float* master, float* buf0, float* buf1, float* buf2, const void* tiles,
                          const uint8_t* active, const float* param_hyper, uint64_t* signal_local, uint64_t** signal_peer,
                          unsigned* done_counter, uint32_t* stats, const float* hyper /* ngroups x 11 */, int ngroups, int ntiles,
                          int bpt, int cap, int param_dt, int bcast, uint32_t contrib, uint32_t wait_mask, float inv_count,
                          uint64_t epoch, uint64_t wait_value, int tile_begin, int tile_end, int wait_grads, int signal_mode,
                          uint32_t ack_mask, int grid) {
  UpdateArgs a{};
  for (int r = 0; r < world; ++r) { a.wire[r] = wire_p[r]; a.scales[r] = scales_p[r]; a.param_dst[r] = param_dst[r]; a.signal_peer[r] = signal_peer[r]; }
  a.param_local = param_local; a.master = master; a.buf0 = buf0; a.buf1 = buf1; a.buf2 = buf2;
  a.tiles = reinterpret_cast<const TileInfo*>(tiles); a.active = active; a.param_hyper = reinterpret_cast<const float2*>(param_hyper);
  a.signal_local = signal_local; a.done_counter = done_counter; a.stats = stats;
  for (int g = 0; g < ngroups; ++g) {
    const float* h = hyper + 11 * g; GroupHyper& o = a.groups[g];
    o.lr = h[0]; o.weight_decay = h[1]; o.momentum = h[2]; o.dampening = h[3]; o.beta1 = h[4]; o.beta2 = h[5]; o.eps = h[6];
    o.step_size = h[7]; o.nesterov = (int)h[8]; o.amsgrad = (int)h[9]; o.first_step = (int)h[10]; o.pad = 0;
  }
  a.world = world; a.rank = rank; a.ntiles = ntiles; a.bytes_per_tile = bpt; a.cap = cap; a.param_dt = param_dt; a.bcast = bcast;
  a.reduce = emu_x_reduce; a.param_mc = emu_x_param_mc; a.wire_mc = emu_x_wire_mc;
  emu_x_reduce = REDUCE_P2P; emu_x_param_mc = nullptr; emu_x_wire_mc = nullptr;
  a.contrib_mask = contrib; a.wait_mask = wait_mask; a.inv_count = inv_count; a.epoch = epoch;
  a.wait_value = wait_value; a.tile_begin = tile_begin; a.tile_end = tile_end; a.wait_grads = wait_grads; a.signal_mode = signal_mode;
  a.ack_mask = ack_mask; a.ack_last = 1; a.timeout_ns = (unsigned long long)(emu_x_timeout * 1e9);
  a.version = emu_x_version; a.select_out = emu_x_select; a.average_dynamic = emu_x_avg;
  emu_x_version = 0; emu_x_select = nullptr; emu_x_avg = 0; emu_x_timeout = 2.0;
  psb_launch_update(nullptr, kind, wire, opt, a, grid);
  return 0;
}

extern "C" void emu_select(const uint64_t* signal_local, uint64_t* consumed, uint32_t cand_mask, int quota, uint64_t* out,
                           uint64_t version, uint64_t** begin_targets, int nbegin, double timeout_s) {
  psb_launch_select(nullptr, signal_local, consumed, cand_mask, quota, out, (unsigned long long)(timeout_s * 1e9), version,
                    begin_targets, nbegin);
}

extern "C" void emu_signal(uint64_t** targets, int n, int slot, uint64_t value, uint64_t* extra_base, int extra_slot,
                           uint64_t extra_value, uint64_t* version_local, int version_slot) {
  psb_launch_signal(nullptr, targets, n, slot, value, extra_base, extra_slot, extra_value, version_local, version_slot);
}

extern "C" void emu_wait(const uint64_t* signal_local, int slot0, uint32_t mask, uint64_t want, double timeout_s) {
  psb_launch_wait(nullptr, signal_local, slot0, mask, want, (unsigned long long)(timeout_s * 1e9));
}

extern "C" void emu_snapshot(const uint64_t* signal_local, const void* stage, void* shadow, void* params, size_t nbytes,
                             unsigned long long* scratch, int attempts) {
  psb_launch_snapshot(nullptr, signal_local, stage, shadow, params, nbytes, scratch, attempts, 148);
}
'''


_LIB = None


def kernel_source() -> str:
    """The emulated translation unit of ``ps_kernels.cu``: shim + conversions + the file's own text (kernels AND launchers)."""
    common = open(os.path.join(KDIR, "common.cuh")).read()
    ps = open(os.path.join(KDIR, "ps_kernels.cu")).read()
    conv = "\n".join(cut_function(common, r"(template <int FP8KIND>[^\n]*\n)?__device__ __forceinline__ [^\n]*\b" + name + r"\(")
                     for name in CONVERSIONS)
    conv += "\n" + real_spin(common)
    # ps_kernels.cu from its first kernel to the end: the anonymous namespace with the kernels AND the launchers behind it
    # (dispatch tables, grids), their <<< >>> launches rewritten to the fiber runner
    body = ps[ps.index('#include "kernels.h"') + len('#include "kernels.h"'):]
    body = body.replace('asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));', "now = emu_now_ns();")
    for fn in ("cudaGetDevice", "cudaDeviceGetAttribute"):
        body = body.replace(fn + "(", "emu_" + fn + "(")
    body, nlaunch = rewrite_launches(body)
    assert nlaunch >= 8 and "<<<" not in body, nlaunch
    kernels_h = open(os.path.join(KDIR, "kernels.h")).read()
    structs = kernels_h[kernels_h.index("#define PSB_ENCODE_MAX"): kernels_h.index("void psb_launch_absmax")]
    # the anonymous namespace's kernels stay private to the launchers, exactly as in the real translation unit
    return SHIM_HEAD + conv + "\n}  // namespace psb\n" + CUDA_RT_SHIM + RUNNER + structs + body + DRIVER


def _conversions() -> str:
    common = open(os.path.join(KDIR, "common.cuh")).read()
    return "\n".join(cut_function(common, r"(template <int FP8KIND>[^\n]*\n)?__device__ __forceinline__ [^\n]*\b" + name + r"\(")
                     for name in CONVERSIONS)


def _count_launch(define: bool) -> str:
    return "void psb_count_launch(int) {}\n" if define else "void psb_count_launch(int);\n"


def bn_source(define_count_launch: bool = True) -> str:
    """The emulated translation unit of ``bn_kernels.cu`` (kernels + launchers, dynamic shared memory as a static buffer)."""
    src = open(os.path.join(KDIR, "bn_kernels.cu")).read()
    body = src[src.index('#include "kernels.h"') + len('#include "kernels.h"'):]
    body = body.replace("extern __shared__ float smem[];", "float* smem = emu_dyn_smem;")
    for fn in ("cudaGetDevice", "cudaDeviceGetAttribute", "cudaMemsetAsync"):
        body = body.replace(fn + "(", "emu_" + fn + "(")
    body, n = rewrite_launches(body)
    assert n >= 8 and "<<<" not in body, n
    body = body.replace("namespace {\nusing namespace psb;", "namespace emu_bn {\nusing namespace psb;", 1).replace(
        "}  // namespace\n", "}  // namespace emu_bn\nusing namespace emu_bn;\n", 1)
    extra = "static float emu_dyn_smem[65536];\nstatic inline float rsqrtf(float v) { return 1.0f / sqrtf(v); }\n"
    return SHIM_HEAD + _conversions() + "\n}  // namespace psb\n" + extra + _count_launch(define_count_launch) + CUDA_RT_SHIM + \
        RUNNER + body


def pool_source(define_count_launch: bool = True) -> str:
    """``pool_kernels.cu`` (max-pool, input normalisers, stem im2col: kernels + launchers) plus the one plain-CUDA kernel of
    ``stem_kernels.cu`` (Σ of the weight-gradient partials; everything else there is tcgen05 / TMA)."""
    src = open(os.path.join(KDIR, "pool_kernels.cu")).read()
    body = src[src.index('#include "kernels.h"') + len('#include "kernels.h"'):]
    for fn in ("cudaGetDevice", "cudaDeviceGetAttribute"):
        body = body.replace(fn + "(", "emu_" + fn + "(")
    stem = open(os.path.join(KDIR, "stem_kernels.cu")).read()
    body += "\nnamespace { constexpr int SK = 176;\n" + cut_function(
        stem, r"__global__ void __launch_bounds__\(256\) psb_stem_wgrad_finalize_kernel\(") + "\n}\n" + cut_function(
        stem, r"void psb_stem_wgrad_finalize_launch\(")
    body, n = rewrite_launches(body)
    assert n == 8 and "<<<" not in body, n
    return SHIM_HEAD + _conversions() + "\n}  // namespace psb\n" + CUDA_RT_SHIM + RUNNER + _count_launch(define_count_launch) + body


_TMP_DIRS = []


def _scratch_dir(prefix: str) -> str:
    """A per-process build directory, removed at interpreter exit (the loaded library stays mapped)."""
    if not _TMP_DIRS:
        import atexit
        atexit.register(lambda: [shutil.rmtree(d, ignore_errors=True) for d in _TMP_DIRS])
    d = tempfile.mkdtemp(prefix=prefix)
    _TMP_DIRS.append(d)
    return d


def compile_shared(source: str, prefix: str):
    """g++ one emulated translation unit (+ its extern "C" driver) into a ctypes library."""
    d = _scratch_dir(prefix)
    open(os.path.join(d, "emu.cpp"), "w").write(source)
    p = subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-pthread", "-w", "-I", CUDA_INC, "-I", KDIR,
                        "-o", os.path.join(d, "emu.so"), os.path.join(d, "emu.cpp")], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True)
    if p.returncode != 0:
        raise RuntimeError("emulator build failed:\n" + p.stdout[-4000:])
    return ctypes.CDLL(os.path.join(d, "emu.so"))


def build():
    """Compile the emulator once per process; returns the ctypes library (or ``None`` without g++)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if shutil.which("g++") is None:
        return None
    d = _scratch_dir("psb_emu_")
    open(os.path.join(d, "emu.cpp"), "w").write(kernel_source())
    cmd = ["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-pthread", "-w", "-I", CUDA_INC, "-I", KDIR, "-o", os.path.join(d, "emu.so"),
           os.path.join(d, "emu.cpp")]
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if p.returncode != 0:
        raise RuntimeError("emulator build failed:\n" + p.stdout[-4000:])
    _LIB = ctypes.CDLL(os.path.join(d, "emu.so"))
    return _LIB


# ---------------------------------------------------------------------------------------------------------------------
# The REAL Python bindings (csrc/bindings.cpp: UpdatePlan with its window loop, encode batching, signal / wait / select /
# snapshot marshalling) linked against the emulated kernels: an importable stand-in for ``_psb200_cuda``.
# ---------------------------------------------------------------------------------------------------------------------
_EXT = None


def bindings_source() -> str:
    src = open(os.path.join(ROOT, "pytorch_ps_mpi_b200", "csrc", "bindings.cpp")).read()

    def drop(text, what):
        assert what in text, what
        return text.replace(what, "")

    for inc in ("#include <ATen/cuda/CUDAContext.h>\n", "#include <c10/cuda/CUDAGuard.h>\n", "#include <c10/cuda/CUDAStream.h>\n",
                '#include "symm_mem.h"\n'):
        src = drop(src, inc)
    # no CUDA runtime underneath: launches cannot fail, there is one "stream", 148 "SMs"
    src = src.replace('#include "kernels.h"\n', '#include "kernels.h"\n#define cudaGetLastError() cudaSuccess\n'
                      '#define cudaGetDevice(p) (*(p) = 0)\nextern int emu_sm_count;\n#define cudaDeviceGetAttribute(p, a, d) (*(p) = emu_sm_count)\n', 1)
    src = drop(src, "c10::cuda::getCurrentCUDAStream().stream()").replace("cudaStream_t cur_stream() { return ; }",
                                                                          "cudaStream_t cur_stream() { return nullptr; }")
    assert "cur_stream() { return nullptr; }" in src
    src = src.replace("at::kCUDA", "at::kCPU")
    src = drop(src, "!g.is_cuda() || ")                      # host tensors stand in for device tensors
    a = src.index("  py::class_<psb::SymmBlock")
    b = src.index(';', src.index('.def("ptr", &psb::SymmBlock::ptr)')) + 1
    return src[:a] + src[b:]                                 # the VMM runtime (driver API) is not part of the emulation


GEMM_STANDINS = r"""
// ---- the tensor-core kernels (tcgen05 / TMEM / TMA) are NOT emulated: reference math through ATen with the same contract ----
at::Tensor bcast_gemm(const at::Tensor& x, uint64_t w_ptr, int64_t N, int64_t K, c10::optional<at::Tensor> bias, bool relu,
                      uint64_t flag_ptr, uint64_t epoch, double timeout_s, int variant) {
  TORCH_CHECK(x.scalar_type() == at::kBFloat16 && x.dim() == 2 && x.size(1) == K, "x must be [M,K] bf16");
  if (flag_ptr) TORCH_CHECK(*reinterpret_cast<const volatile uint64_t*>(flag_ptr) >= epoch, "gate: PARAMS_READY not reached");
  auto w = at::from_blob(reinterpret_cast<void*>(w_ptr), {N, K}, x.options());
  auto y = at::matmul(x.to(at::kFloat), w.to(at::kFloat).t());
  if (bias.has_value() && bias->defined()) y = y + bias->to(at::kFloat);
  if (relu) y = at::relu(y);
  return y.to(at::kBFloat16);
}

std::vector<at::Tensor> stem_fwd(const at::Tensor& x, const at::Tensor& w2d, bool want_sums, uint64_t flag_ptr, uint64_t epoch,
                                 double timeout_s) {
  TORCH_CHECK(x.scalar_type() == at::kBFloat16 && x.dim() == 4 && x.size(1) == 3, "x must be [N,3,H,W] bf16");
  TORCH_CHECK(x.is_contiguous(at::MemoryFormat::ChannelsLast), "x must be channels_last contiguous");
  TORCH_CHECK(w2d.dim() == 2 && w2d.size(0) == 64 && w2d.size(1) == 176 && w2d.is_contiguous(), "w2d must be [64,176]");
  if (flag_ptr) TORCH_CHECK(*reinterpret_cast<const volatile uint64_t*>(flag_ptr) >= epoch, "gate: PARAMS_READY not reached");
  const int64_t N = x.size(0), H = x.size(2), W = x.size(3), OH = (H - 1) / 2 + 1, OW = (W - 1) / 2 + 1;
  TORCH_CHECK(W % 8 == 0 && W <= 256 && W >= 8, "fused stem: W must be a multiple of 8 and <= 256");
  auto a = im2col_stem(x);                                           // the REAL (emulated) patch-matrix kernel
  auto y32 = at::matmul(a.to(at::kFloat), w2d.to(at::kFloat).t());   // [M,64], fp32 accumulators
  auto y = y32.to(at::kBFloat16);
  // like the kernel's epilogue: the sums are taken over the bf16 values it stores, not over the fp32 accumulators
  auto yr = y.to(at::kFloat);
  at::Tensor sums = want_sums ? at::cat({yr.sum(0), (yr * yr).sum(0)}).contiguous() : at::Tensor();
  return {y.view({N, OH, OW, 64}).permute({0, 3, 1, 2}), sums};
}

at::Tensor stem_wgrad(const at::Tensor& x, const at::Tensor& gy) {
  check_nhwc(gy, "gy");
  auto a = im2col_stem(x);                                           // [M,176]
  auto g = gy.permute({0, 2, 3, 1}).reshape({-1, 64});               // NHWC rows
  return at::matmul(a.to(at::kFloat).t(), g.to(at::kFloat)).unsqueeze(0).contiguous();   // one "CTA" partial [1,176,64]
}
"""


def gemm_bindings_source() -> str:
    """``csrc/gemm_bindings.cpp`` for the emulated extension: the bindings of every plain-CUDA op are the repository's own text
    (BatchNorm forward / presummed / backward, max-pool, normalisers, im2col, wgrad finalize, ``bind_gemm``); the three
    tensor-core entry points are replaced by ATen reference math (``GEMM_STANDINS``)."""
    src = open(os.path.join(ROOT, "pytorch_ps_mpi_b200", "csrc", "gemm_bindings.cpp")).read()
    real = ["void check_nhwc", "std::vector<at::Tensor> bn_forward", "std::vector<at::Tensor> bn_backward",
            "std::vector<at::Tensor> maxpool_forward", "at::Tensor maxpool_backward", "at::Tensor normalize_pad8",
            "std::vector<at::Tensor> bn_forward_presummed", "at::Tensor stem_wgrad_finalize", "at::Tensor im2col_stem",
            "at::Tensor normalize_nhwc3"]
    parts = [cut_function(src, re.escape(h) + r"\(") for h in real]
    text = "\n\n".join(parts[:1] + [parts[8]] + parts[1:8] + parts[9:])          # im2col_stem before its users
    text = text.replace("c10::cuda::getCurrentCUDAStream().stream()", "nullptr").replace(".is_cuda()", ".defined()").replace(
        "->is_cuda()", "->defined()")
    head = ('#include <torch/extension.h>\n#include "kernels.h"\n#define cudaGetLastError() cudaSuccess\n'
            '#define cudaGetErrorString(e) "n/a"\nnamespace py = pybind11;\nint psb_bcast_gemm_smem_bytes() { return 0; }\nnamespace {\n')
    return head + text + GEMM_STANDINS + "\n}  // namespace\n" + cut_function(src, r"void bind_gemm\(py::module_& m\)") + "\n"


def build_extension():
    """Compile ``bindings.cpp`` (transformed as above) + the emulated kernels into ``_psb200_emu``; returns the imported module
    (or ``None`` without g++).  Cached in the temp directory by source hash: torch's headers take about a minute to compile."""
    global _EXT
    if _EXT is not None:
        return _EXT
    if shutil.which("g++") is None:
        return None
    import hashlib
    import importlib.machinery
    import importlib.util
    import sysconfig

    import pybind11
    import torch
    from torch.utils import cpp_extension as ce
    ksrc, bsrc = kernel_source(), bindings_source()
    extra = {"emu_bn": bn_source(False), "emu_pool": pool_source(False), "gemm_emu": gemm_bindings_source()}
    tag = hashlib.sha1((ksrc + bsrc + "".join(extra.values()) + torch.__version__).encode()).hexdigest()[:16]
    d = os.path.join(tempfile.gettempdir(), f"psb_emu_ext_{tag}")
    so = os.path.join(d, "_psb200_emu.so")
    if not os.path.exists(so):
        os.makedirs(d, exist_ok=True)
        open(os.path.join(d, "emu_kernels.cpp"), "w").write(ksrc)
        open(os.path.join(d, "bindings_emu.cpp"), "w").write(bsrc)
        abi = getattr(torch._C, "_GLIBCXX_USE_CXX11_ABI", True)
        inc = ["-I" + KDIR, "-I" + CUDA_INC, "-I" + sysconfig.get_paths()["include"], "-I" + pybind11.get_include()]
        inc += ["-I" + p for p in ce.include_paths()]
        jobs = [["g++", "-O1", "-std=c++17", "-fPIC", "-pthread", "-w", *inc, "-c", os.path.join(d, "emu_kernels.cpp"), "-o",
                 os.path.join(d, "emu_kernels.o")],
                ["g++", "-O1", "-std=c++17", "-fPIC", "-pthread", "-w", f"-D_GLIBCXX_USE_CXX11_ABI={int(abi)}",
                 "-DTORCH_EXTENSION_NAME=_psb200_emu", "-DTORCH_API_INCLUDE_EXTENSION_H", *inc, "-c",
                 os.path.join(d, "bindings_emu.cpp"), "-o", os.path.join(d, "bindings_emu.o")]]
        for name, text in extra.items():
            open(os.path.join(d, name + ".cpp"), "w").write(text)
            flags = [f"-D_GLIBCXX_USE_CXX11_ABI={int(abi)}", "-DTORCH_API_INCLUDE_EXTENSION_H"] if name == "gemm_emu" else []
            jobs.append(["g++", "-O1", "-std=c++17", "-fPIC", "-pthread", "-w", *flags, *inc, "-c", os.path.join(d, name + ".cpp"),
                         "-o", os.path.join(d, name + ".o")])
        procs = [subprocess.Popen(j, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for j in jobs]
        for pr in procs:
            out, _ = pr.communicate()
            if pr.returncode != 0:
                raise RuntimeError("emulated extension build failed:\n" + out[-4000:])
        libdirs = ce.library_paths()
        link = ["g++", "-shared", "-o", so + ".tmp", os.path.join(d, "bindings_emu.o"), os.path.join(d, "emu_kernels.o"),
                *[os.path.join(d, name + ".o") for name in extra],
                *["-L" + x for x in libdirs], *["-Wl,-rpath," + x for x in libdirs], "-lc10", "-ltorch_cpu", "-ltorch", "-ltorch_python",
                "-pthread"]
        p = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if p.returncode != 0:
            raise RuntimeError("emulated extension link failed:\n" + p.stdout[-4000:])
        os.replace(so + ".tmp", so)
    loader = importlib.machinery.ExtensionFileLoader("_psb200_emu", so)
    spec = importlib.util.spec_from_file_location("_psb200_emu", so, loader=loader)
    mod = importlib.util.module_from_spec(spec)
    loader.exec_module(mod)
    mod.emu = ctypes.CDLL(so)              # the emulator's own entry points (multicast windows) of the SAME library
    _EXT = mod
    return mod
