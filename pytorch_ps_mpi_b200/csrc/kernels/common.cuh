// Shared device helpers for the pytorch_ps_mpi_b200 sm_100a kernels.
//
// Layout contract (mirrors pytorch_ps_mpi_b200/codings.py and parallel/layout.py):
//   * every parameter occupies an integral number of PSB_TILE-element tiles of one flat arena,
//   * tile t of the wire arena starts at byte t * bytes_per_tile,
//   * thread `tid` of a 256-thread CTA owns elements [8*tid, 8*tid+8) of its tile, so thread
//     order == index order (the block-wise top-k relies on it).
#pragma once
#ifdef __CUDACC__
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>
#endif
#include <cuda_runtime.h>
#include <stdint.h>

#define PSB_TILE 2048
#define PSB_THREADS 256
#define PSB_EPT 8            // elements per thread
#define PSB_MAX_RANKS 16
#define PSB_MAX_GROUPS 16

// wire element types (codings.py WIRE_*)
enum : int { WIRE_F32 = 0, WIRE_BF16 = 1, WIRE_F16 = 2, WIRE_E4M3 = 3, WIRE_E5M2 = 4, WIRE_I8 = 5 };
// coding kinds (codings.py KIND_*)
enum : int { KIND_DENSE = 0, KIND_SCALED = 1, KIND_TOPK = 2, KIND_QSGD = 3 };
// parameter / gradient dtypes
enum : int { DT_F32 = 0, DT_BF16 = 1, DT_F16 = 2 };
// optimizers
enum : int { OPT_SGD = 0, OPT_ADAM = 1 };
// how the updated parameter tile is published
enum : int { BCAST_LOCAL = 0, BCAST_UNICAST = 1, BCAST_MULTICAST = 2 };
// how the gradient tiles are gathered
enum : int { REDUCE_P2P = 0, REDUCE_NVLS = 1 };

// signal-pad slots (uint64 each); pad is PSB_SIGNAL_SLOTS * 8 bytes at the start of the block
#define PSB_SIGNAL_SLOTS 512
#define SIG_GRAD_READY 0      // [0, 64): rank r's "my gradients for epoch e are in my arena"
#define SIG_PARAMS_READY 64   // PS → everyone: parameters of epoch e are published
#define SIG_CONSUMED 128      // [128, 192): rank r finished READING everyone's gradients (allgather mode)
#define SIG_ERROR 200         // non-zero → a spin timed out somewhere
#define SIG_VERSION 201       // async: parameter version published by the PS
#define SIG_STAGE_BEGIN 202   // async + consistent reads: version the PS STARTED publishing (sequence lock with SIG_VERSION)
#define SIG_SEEN_VERSION 203  // async worker, local: parameter version sampled when the previous gradient was posted
#define SIG_ACK 256           // [256, 320): async: PS consumed rank r's gradient of epoch e
#define SIG_GRAD_VERSION 320  // [320, 384): async: parameter version rank r's gradient was computed on

struct __align__(16) TileInfo {
  int32_t param;   // parameter index
  int32_t valid;   // real elements in this tile (<= PSB_TILE)
  int32_t group;   // param_group index (hyper-parameters)
  int32_t first;   // first tile of this parameter
};

struct GroupHyper {
  float lr, weight_decay, momentum, dampening;
  float beta1, beta2, eps, step_size;   // step_size = lr*sqrt(1-b2^t)/(1-b1^t) (ps.py:257-259)
  int32_t nesterov, amsgrad, first_step, pad;
};

#ifdef __CUDACC__
namespace psb {

__device__ __forceinline__ uint64_t ld_acquire_sys(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint64_t ld_relaxed_sys_u64(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(uint64_t* p, uint64_t v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys_f32(float* p, float v) {
  asm volatile("st.relaxed.sys.global.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

// 16-byte load that is coherent at system scope (peer memory over NVLink; never the stale-L1 path)
__device__ __forceinline__ uint4 ld_sys_v4(const void* p) {
  uint4 v;
  asm volatile("ld.relaxed.sys.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p)
               : "memory");
  return v;
}
__device__ __forceinline__ uint2 ld_sys_v2(const void* p) {
  uint2 v;
  asm volatile("ld.relaxed.sys.global.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float ld_sys_f32(const float* p) {
  float v;
  asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
  return v;
}
// streaming local 16-byte load / store (touch-once data: keep it out of L1)
__device__ __forceinline__ uint4 ld_stream_v4(const void* p) {
  uint4 v;
  asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p));
  return v;
}
__device__ __forceinline__ void st_v4(void* p, uint4 v) {
  asm volatile("st.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// peer store, system scope
__device__ __forceinline__ void st_sys_v4(void* p, uint4 v) {
  asm volatile("st.relaxed.sys.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}
// NVLS: one store, the switch replicates it into every GPU bound to the multicast object
__device__ __forceinline__ void multimem_st_v4(void* mc, uint4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(mc), "r"(v.x), "r"(v.y), "r"(v.z),
               "r"(v.w)
               : "memory");
}
// NVLS: the switch sums the same address across every bound GPU and returns one vector
__device__ __forceinline__ uint4 multimem_ld_reduce_f32x4(const void* mc) {
  uint4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(mc)
               : "memory");
  return v;
}
__device__ __forceinline__ uint4 multimem_ld_reduce_bf16x8(const void* mc) {
  uint4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.bf16x2 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(mc)
               : "memory");
  return v;
}
__device__ __forceinline__ uint4 multimem_ld_reduce_f16x8(const void* mc) {
  uint4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.f16x2 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(mc)
               : "memory");
  return v;
}

// Bounded spin: returns false (and raises the error slot) on time-out so a dead peer can never
// hang the GPU (every waiting kernel then exits and the host raises).
__device__ __forceinline__ bool spin_until_ge(const uint64_t* flag, uint64_t want, uint64_t* err_slot,
                                              unsigned long long timeout_ns) {
  unsigned long long t0 = 0;
  unsigned spins = 0;
  while (true) {
    if (ld_acquire_sys(flag) >= want) return true;
    if (ld_relaxed_sys_u64(err_slot) != 0) return false;
    if ((++spins & 63u) == 0) {
      unsigned long long now;
      asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      if (now - t0 > timeout_ns) {
        st_release_sys(err_slot, 1ull);
        return false;
      }
      __nanosleep(64);
    }
  }
}

// ---- element conversions ------------------------------------------------------------------
__device__ __forceinline__ void unpack_bf16x8(const uint4& v, float* f) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f[2 * i] = __uint_as_float(w[i] << 16);
    f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}
__device__ __forceinline__ void unpack_f16x8(const uint4& v, float* f) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __half2 h = *reinterpret_cast<const __half2*>(&w[i]);
    float2 t = __half22float2(h);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
template <int FP8KIND>  // WIRE_E4M3 or WIRE_E5M2
__device__ __forceinline__ void unpack_fp8x8(const uint2& v, float* f) {
  const uint32_t w[2] = {v.x, v.y};
#pragma unroll
  for (int i = 0; i < 2; ++i) {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      __nv_fp8x2_storage_t s = (__nv_fp8x2_storage_t)((w[i] >> (16 * j)) & 0xffffu);
      __half2_raw hr = __nv_cvt_fp8x2_to_halfraw2(s, FP8KIND == WIRE_E4M3 ? __NV_E4M3 : __NV_E5M2);
      float2 t = __half22float2(*reinterpret_cast<__half2*>(&hr));
      f[4 * i + 2 * j] = t.x;
      f[4 * i + 2 * j + 1] = t.y;
    }
  }
}
__device__ __forceinline__ void unpack_i8x8(const uint2& v, float* f) {
  const uint32_t w[2] = {v.x, v.y};
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) f[4 * i + j] = (float)(int8_t)((w[i] >> (8 * j)) & 0xffu);
}

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack_f16x2_sat(float a, float b) {
  a = fminf(fmaxf(a, -65504.f), 65504.f);
  b = fminf(fmaxf(b, -65504.f), 65504.f);
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack_f16x2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
template <int FP8KIND>
__device__ __forceinline__ uint32_t pack_fp8x4(float a, float b, float c, float d) {
  const __nv_fp8_interpretation_t k = FP8KIND == WIRE_E4M3 ? __NV_E4M3 : __NV_E5M2;
  uint32_t lo = __nv_cvt_float2_to_fp8x2(make_float2(a, b), __NV_SATFINITE, k);
  uint32_t hi = __nv_cvt_float2_to_fp8x2(make_float2(c, d), __NV_SATFINITE, k);
  return lo | (hi << 16);
}
__device__ __forceinline__ uint32_t pack_i8x4(float a, float b, float c, float d) {
  auto q = [](float x) -> uint32_t {
    int v = __float2int_rn(x);
    v = max(-127, min(127, v));
    return (uint32_t)(uint8_t)(int8_t)v;
  };
  return q(a) | (q(b) << 8) | (q(c) << 16) | (q(d) << 24);
}

// Load 8 consecutive elements of dtype DT (f32 / bf16 / f16) starting at element offset `e`.
__device__ __forceinline__ void load8_local(const void* base, int dt, size_t e, float* f) {
  if (dt == DT_F32) {
    const float* p = reinterpret_cast<const float*>(base) + e;
    uint4 a = ld_stream_v4(p), b = ld_stream_v4(p + 4);
    f[0] = __uint_as_float(a.x), f[1] = __uint_as_float(a.y), f[2] = __uint_as_float(a.z), f[3] = __uint_as_float(a.w);
    f[4] = __uint_as_float(b.x), f[5] = __uint_as_float(b.y), f[6] = __uint_as_float(b.z), f[7] = __uint_as_float(b.w);
  } else {
    uint4 a = ld_stream_v4(reinterpret_cast<const uint16_t*>(base) + e);
    if (dt == DT_BF16) unpack_bf16x8(a, f);
    else unpack_f16x8(a, f);
  }
}

// Encode 8 floats into dtype DT bits (for parameter publication). Returns the number of uint4 used.
__device__ __forceinline__ int pack8(int dt, const float* f, uint4* out) {
  if (dt == DT_F32) {
    out[0] = make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]), __float_as_uint(f[3]));
    out[1] = make_uint4(__float_as_uint(f[4]), __float_as_uint(f[5]), __float_as_uint(f[6]), __float_as_uint(f[7]));
    return 2;
  }
  if (dt == DT_BF16)
    out[0] = make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
  else
    out[0] = make_uint4(pack_f16x2(f[0], f[1]), pack_f16x2(f[2], f[3]), pack_f16x2(f[4], f[5]), pack_f16x2(f[6], f[7]));
  return 1;
}

}  // namespace psb
#endif  // __CUDACC__

namespace psb {
#ifndef __CUDACC__
#define PSB_HD
#else
#define PSB_HD __host__ __device__
#endif
PSB_HD constexpr int wire_elem_bytes(int wire) {
  return wire == WIRE_F32 ? 4 : (wire == WIRE_BF16 || wire == WIRE_F16) ? 2 : 1;
}
PSB_HD constexpr float wire_qmax(int wire) {
  return wire == WIRE_E4M3 ? 448.f : wire == WIRE_E5M2 ? 57344.f : wire == WIRE_I8 ? 127.f : 65504.f;
}

}  // namespace psb
