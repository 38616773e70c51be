// Parameter-server hot path for sm_100a: gradient encode, fused gather-reduce-decode-update-
// broadcast, and the epoch-flag signalling kernels.
//
// What these replace in the reference (citations into /root/reference):
//   * encode + to_np + pickle + blosc per parameter on a thread pool (ps.py:92-101,
//     mpi_comms.py:186-193)                         → psb_encode_kernel (one launch per bucket)
//   * Igatherv / Iallgatherv of host bytes (mpi_comms.py:88,162), H2D copies (mpi_comms.py:48-50),
//     decode (ps.py:165-167), sum(grads) (ps.py:176), the eager SGD/Adam ops (ps.py:197-261) and
//     the Ibcast of fresh parameters (mpi_comms.py:132)  → psb_update_kernel: ONE launch that
//     pulls every rank's wire tile over NVLink (P2P loads, or one multimem.ld_reduce through the
//     switch), decodes and sums in registers / shared memory in fixed rank order, applies the
//     optimizer to fp32 master state and publishes the new parameter tile to every GPU
//     (multimem.st through the switch, or unicast peer stores), then raises the epoch flag.
//   * MPI requests / req.Wait() (ps.py:146, mpi_comms.py:110,121)  → monotonically increasing epoch
//     flags in the symmetric signal pad (st.release.sys / ld.acquire.sys), bounded spins.
#include <algorithm>
#include <cstdlib>

#include "kernels.h"

namespace {
using namespace psb;

// ------------------------------------------------------------------------------------------
// small block-level helpers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t* warp_tot /*[8]*/, uint32_t* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    uint32_t n = __shfl_up_sync(0xffffffffu, incl, off);
    if (lane >= off) incl += n;
  }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  uint32_t base = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < PSB_THREADS / 32; ++w) {
    uint32_t t = warp_tot[w];
    if (w < warp) base += t;
    tot += t;
  }
  __syncthreads();   // warp_tot may be reused by the caller
  if (total) *total = tot;
  return base + incl - v;
}

__device__ __forceinline__ float block_max(float v, float* red /*[8]*/) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, off));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float m = red[0];
#pragma unroll
  for (int w = 1; w < PSB_THREADS / 32; ++w) m = fmaxf(m, red[w]);
  __syncthreads();
  return m;
}

// which batch entry / arena tile does this CTA work on
__device__ __forceinline__ void locate(const EncodeBatch& b, int cta, int& entry, int& tile) {
  int e = 0;
  while (e + 1 < b.n && b.cum[e + 1] <= cta) ++e;
  entry = e;
  tile = b.first_tile[e] + (cta - b.cum[e]);
}

__device__ __forceinline__ void load_grad8(const EncodeArgs& a, int entry, const TileInfo& ti, int tile, float* g) {
  const size_t off = (size_t)(tile - ti.first) * PSB_TILE + threadIdx.x * PSB_EPT;
  const int base = threadIdx.x * PSB_EPT;
  if (base < ti.valid) {
    load8_local(a.batch.src[entry], a.grad_dt, off, g);
#pragma unroll
    for (int j = 0; j < PSB_EPT; ++j)
      if (base + j >= ti.valid) g[j] = 0.f;
  } else {
#pragma unroll
    for (int j = 0; j < PSB_EPT; ++j) g[j] = 0.f;
  }
}

// A product rounded on its own, which the compiler may not fuse with a following add into an FMA: the QSGD tile norm is
// specified operation by operation (codings.qsgd_blockwise reproduces it).  Compiled as plain host C++, as the CPU
// emulator does, there is no FMA to fuse into.
#ifdef __CUDACC__
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
#else
inline float mul_rn(float a, float b) { return a * b; }
#endif

// Philox4x32-10 (Salmon et al., SC'11; Random123 constants).  The mul-hi is the top half of a 64-bit product so that the
// same text runs in the CPU emulator; codings.qsgd_uniform16 is the Python mirror.
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                              uint32_t* out) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    c0 = n0, c1 = (uint32_t)p1, c2 = n2, c3 = (uint32_t)p0;
    k0 += 0x9E3779B9u, k1 += 0xBB67AE85u;
  }
  out[0] = c0, out[1] = c1, out[2] = c2, out[3] = c3;
}

// ------------------------------------------------------------------------------------------
// abs-max pre-pass for Scale codings: one atomicMax per tile into amax_bits[param]
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(PSB_THREADS) psb_absmax_kernel(const __grid_constant__ EncodeArgs a) {
  __shared__ float red[PSB_THREADS / 32];
  int entry, tile;
  locate(a.batch, blockIdx.x, entry, tile);
  const TileInfo ti = a.tiles[tile];
  float g[PSB_EPT];
  load_grad8(a, entry, ti, tile, g);
  float m = 0.f;
#pragma unroll
  for (int j = 0; j < PSB_EPT; ++j) m = fmaxf(m, fabsf(g[j]));   // NaN-ignoring, like a finite-only max
  m = block_max(m, red);
  if (threadIdx.x == 0) atomicMax(a.amax_bits + ti.param, __float_as_uint(m));
}

// ------------------------------------------------------------------------------------------
// encode: gradient tile → wire tile (dense cast | abs-max scaled | block-wise top-k | block-wise QSGD)
// ------------------------------------------------------------------------------------------
template <int WIRE>
__device__ __forceinline__ void store_dense(void* wire_tile, const float* q) {
  const int tid = threadIdx.x;
  if constexpr (WIRE == WIRE_F32) {
    uint4* p = reinterpret_cast<uint4*>(reinterpret_cast<float*>(wire_tile) + tid * PSB_EPT);
    st_v4(p, make_uint4(__float_as_uint(q[0]), __float_as_uint(q[1]), __float_as_uint(q[2]), __float_as_uint(q[3])));
    st_v4(p + 1, make_uint4(__float_as_uint(q[4]), __float_as_uint(q[5]), __float_as_uint(q[6]), __float_as_uint(q[7])));
  } else if constexpr (WIRE == WIRE_BF16) {
    st_v4(reinterpret_cast<uint16_t*>(wire_tile) + tid * PSB_EPT,
          make_uint4(pack_bf16x2(q[0], q[1]), pack_bf16x2(q[2], q[3]), pack_bf16x2(q[4], q[5]), pack_bf16x2(q[6], q[7])));
  } else if constexpr (WIRE == WIRE_F16) {
    st_v4(reinterpret_cast<uint16_t*>(wire_tile) + tid * PSB_EPT,
          make_uint4(pack_f16x2_sat(q[0], q[1]), pack_f16x2_sat(q[2], q[3]), pack_f16x2_sat(q[4], q[5]),
                     pack_f16x2_sat(q[6], q[7])));
  } else if constexpr (WIRE == WIRE_E4M3 || WIRE == WIRE_E5M2) {
    uint2 v = make_uint2(pack_fp8x4<WIRE>(q[0], q[1], q[2], q[3]), pack_fp8x4<WIRE>(q[4], q[5], q[6], q[7]));
    *reinterpret_cast<uint2*>(reinterpret_cast<uint8_t*>(wire_tile) + tid * PSB_EPT) = v;
  } else {  // WIRE_I8
    uint2 v = make_uint2(pack_i8x4(q[0], q[1], q[2], q[3]), pack_i8x4(q[4], q[5], q[6], q[7]));
    *reinterpret_cast<uint2*>(reinterpret_cast<uint8_t*>(wire_tile) + tid * PSB_EPT) = v;
  }
}

template <int KIND, int WIRE>
__global__ void __launch_bounds__(PSB_THREADS) psb_encode_kernel(const __grid_constant__ EncodeArgs a) {
  int entry, tile;
  locate(a.batch, blockIdx.x, entry, tile);
  const TileInfo ti = a.tiles[tile];
  const int tid = threadIdx.x;
  uint8_t* wire_tile = reinterpret_cast<uint8_t*>(a.wire) + (size_t)tile * a.bytes_per_tile;
  float g[PSB_EPT];
  load_grad8(a, entry, ti, tile, g);

  if constexpr (KIND == KIND_DENSE) {
    store_dense<WIRE>(wire_tile, g);
  } else if constexpr (KIND == KIND_SCALED) {
    float amax = __uint_as_float(a.amax_bits[ti.param]);
    if (!(amax > 0.f) || !isfinite(amax)) amax = 1.f;
    const float inv = __fdiv_rn(amax, wire_qmax(WIRE));
    if (tile == ti.first && tid == 0) a.scales[ti.param] = inv;
    float q[PSB_EPT];
#pragma unroll
    for (int j = 0; j < PSB_EPT; ++j) q[j] = __fdiv_rn(g[j], inv);
    store_dense<WIRE>(wire_tile, q);
  } else if constexpr (KIND == KIND_QSGD) {
    // block-wise QSGD: q = sign(g) * stochastic_round(|g| * levels / ||tile||), scale = ||tile|| / levels in the slot trailer.
    // The sum of squares runs in a fixed order that codings.qsgd_blockwise reproduces bit for bit: each thread's 8 elements in
    // sequence, an xor butterfly over lanes (offsets 16..1), then the 8 warp sums in index order; the squares are not fused
    // into the sum (mul_rn).  The rest is adds, subtractions and products that have no FMA form.
    __shared__ float s_warp[PSB_THREADS / 32];
    float ss = 0.f;
#pragma unroll
    for (int j = 0; j < PSB_EPT; ++j) ss += mul_rn(g[j], g[j]);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
    if ((tid & 31) == 0) s_warp[tid >> 5] = ss;
    __syncthreads();
    float sum = s_warp[0];
#pragma unroll
    for (int w = 1; w < PSB_THREADS / 32; ++w) sum += s_warp[w];
    const float norm = __fsqrt_rn(sum);
    const float lv = (float)a.levels;
    const bool live = norm > 0.f && isfinite(norm);     // an all-zero or non-finite tile travels as q = 0, scale = 0
    float q[PSB_EPT];
    if (live) {
      // one Philox call per thread: counter = (arena element / 8, step, rank), key = seed → 8 uniforms of 16 bits
      const uint64_t grp = ((uint64_t)tile * PSB_TILE + tid * PSB_EPT) / PSB_EPT;
      uint32_t u[4];
      philox4x32_10((uint32_t)grp, (uint32_t)(grp >> 32), a.rng_step, (uint32_t)a.rank, (uint32_t)a.seed,
                    (uint32_t)(a.seed >> 32), u);
      const float r = __fdiv_rn(lv, norm);
#pragma unroll
      for (int j = 0; j < PSB_EPT; ++j) {
        const float x = fminf(fabsf(g[j]) * r, lv);   // rounding can land one ulp above `levels`: clamp
        const float l = floorf(x);
        const float u16 = (float)((u[j >> 1] >> (16 * (j & 1))) & 0xffffu);
        const float up = u16 < (x - l) * 65536.f ? 1.f : 0.f;
        q[j] = copysignf(l + up, g[j]);
      }
    } else {
#pragma unroll
      for (int j = 0; j < PSB_EPT; ++j) q[j] = 0.f;
    }
    store_dense<WIRE>(wire_tile, q);
    if (tid == 0)
      st_v4(wire_tile + PSB_TILE, make_uint4(__float_as_uint(live ? __fdiv_rn(norm, lv) : 0.f), 0u, 0u, 0u));
  } else {  // KIND_TOPK: block-wise magnitude top-k, ties → lower index, entries in index order
    __shared__ uint32_t hist[256];
    __shared__ uint32_t warp_tot[PSB_THREADS / 32];
    __shared__ uint32_t s_prefix, s_k;
    const size_t e0 = (size_t)tile * PSB_TILE + tid * PSB_EPT;
    if (a.residual) {
      const float4* r = reinterpret_cast<const float4*>(a.residual + e0);
      float4 r0 = r[0], r1 = r[1];
      g[0] += r0.x, g[1] += r0.y, g[2] += r0.z, g[3] += r0.w;
      g[4] += r1.x, g[5] += r1.y, g[6] += r1.z, g[7] += r1.w;
    }
    uint32_t key[PSB_EPT];
#pragma unroll
    for (int j = 0; j < PSB_EPT; ++j) key[j] = (tid * PSB_EPT + j < ti.valid) ? (__float_as_uint(g[j]) & 0x7fffffffu) : 0u;
    int k = (int)ceil((double)a.ratio * (double)ti.valid - 1e-9);
    k = max(1, min(ti.valid, k));
    uint32_t prefix = 0, mask = 0, kk = (uint32_t)k;
#pragma unroll 1
    for (int shift = 24; shift >= 0; shift -= 8) {
      hist[tid] = 0;
      __syncthreads();
#pragma unroll
      for (int j = 0; j < PSB_EPT; ++j)
        if ((key[j] & mask) == prefix) atomicAdd(&hist[(key[j] >> shift) & 0xffu], 1u);
      __syncthreads();
      if (tid < 32) {
        uint32_t c[8], sum = 0;
#pragma unroll
        for (int b = 0; b < 8; ++b) {
          c[b] = hist[255 - 8 * tid - b];
          sum += c[b];
        }
        uint32_t incl = sum;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
          uint32_t n = __shfl_up_sync(0xffffffffu, incl, off);
          if (tid >= off) incl += n;
        }
        const uint32_t excl = incl - sum;
        if (excl < kk && kk <= incl) {
          uint32_t run = excl;
#pragma unroll
          for (int b = 0; b < 8; ++b) {
            if (run + c[b] >= kk) {
              s_prefix = prefix | ((uint32_t)(255 - 8 * tid - b) << shift);
              s_k = kk - run;
              break;
            }
            run += c[b];
          }
        }
      }
      __syncthreads();
      prefix = s_prefix;
      kk = s_k;
      mask |= 0xffu << shift;
      __syncthreads();
    }
    const uint32_t T = prefix;   // k-th largest magnitude; take every key > T and the first kk keys == T
    uint32_t eqc = 0;
#pragma unroll
    for (int j = 0; j < PSB_EPT; ++j) eqc += (key[j] == T);
    uint32_t eq_before = block_excl_scan(eqc, warp_tot, nullptr);
    uint32_t selbits = 0, selc = 0;
#pragma unroll
    for (int j = 0; j < PSB_EPT; ++j) {
      bool s = key[j] > T;
      if (key[j] == T) {
        s = eq_before < kk;
        ++eq_before;
      }
      if (s) {
        selbits |= 1u << j;
        ++selc;
      }
    }
    uint32_t total = 0;
    uint32_t pos = block_excl_scan(selc, warp_tot, &total);
#pragma unroll
    for (int j = 0; j < PSB_EPT; ++j) {
      if (selbits >> j & 1u) {
        const uint32_t idx = tid * PSB_EPT + j;
        if constexpr (WIRE == WIRE_BF16) {
          __nv_bfloat16 hv = __float2bfloat16_rn(g[j]);
          const uint32_t bits = *reinterpret_cast<uint16_t*>(&hv);
          reinterpret_cast<uint32_t*>(wire_tile)[pos] = (idx << 16) | bits;
          g[j] -= __bfloat162float(hv);       // what stays behind as residual
        } else {
          reinterpret_cast<uint2*>(wire_tile)[pos] = make_uint2(idx, __float_as_uint(g[j]));
          g[j] = 0.f;
        }
        ++pos;
      }
    }
    for (uint32_t p = total + tid; p < (uint32_t)a.cap; p += PSB_THREADS) {   // pad: idx == PSB_TILE is "no entry"
      if constexpr (WIRE == WIRE_BF16) reinterpret_cast<uint32_t*>(wire_tile)[p] = (uint32_t)PSB_TILE << 16;
      else reinterpret_cast<uint2*>(wire_tile)[p] = make_uint2(PSB_TILE, 0u);
    }
    if (a.residual) {
      float4* r = reinterpret_cast<float4*>(a.residual + e0);
      r[0] = make_float4(g[0], g[1], g[2], g[3]);
      r[1] = make_float4(g[4], g[5], g[6], g[7]);
    }
  }

  // ---- fused flag raise (last encode launch of the step): the last CTA to finish publishes GRAD_READY ----
  if (a.nsig > 0) {
    __shared__ int s_last;
    __syncthreads();
    if (tid == 0) {
      __threadfence_system();                       // this CTA's wire tile is visible system-wide
      s_last = (atomicAdd(a.sig_counter, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (s_last) {
      if (tid == 0) *a.sig_counter = 0;
      __threadfence_system();
      if (tid < a.nsig && a.sig_targets[tid] != nullptr) st_release_sys(a.sig_targets[tid] + a.sig_slot, a.sig_value);
    }
  }
}

// ------------------------------------------------------------------------------------------
// the fused PS kernel
// ------------------------------------------------------------------------------------------
template <int WIRE>
__device__ __forceinline__ void issue_dense(const void* wire_base, size_t tile_byte_off, uint4& v0, uint4& v1) {
  const uint8_t* p = reinterpret_cast<const uint8_t*>(wire_base) + tile_byte_off +
                     (size_t)threadIdx.x * PSB_EPT * wire_elem_bytes(WIRE);
  if constexpr (WIRE == WIRE_F32) {
    v0 = ld_sys_v4(p);
    v1 = ld_sys_v4(p + 16);
  } else if constexpr (WIRE == WIRE_BF16 || WIRE == WIRE_F16) {
    v0 = ld_sys_v4(p);
  } else {
    uint2 t = ld_sys_v2(p);
    v0.x = t.x, v0.y = t.y;
  }
}

template <int WIRE>
__device__ __forceinline__ void decode_dense(const uint4& v0, const uint4& v1, float* f) {
  if constexpr (WIRE == WIRE_F32) {
    f[0] = __uint_as_float(v0.x), f[1] = __uint_as_float(v0.y), f[2] = __uint_as_float(v0.z), f[3] = __uint_as_float(v0.w);
    f[4] = __uint_as_float(v1.x), f[5] = __uint_as_float(v1.y), f[6] = __uint_as_float(v1.z), f[7] = __uint_as_float(v1.w);
  } else if constexpr (WIRE == WIRE_BF16) {
    unpack_bf16x8(v0, f);
  } else if constexpr (WIRE == WIRE_F16) {
    unpack_f16x8(v0, f);
  } else if constexpr (WIRE == WIRE_E4M3 || WIRE == WIRE_E5M2) {
    unpack_fp8x8<WIRE>(make_uint2(v0.x, v0.y), f);
  } else {
    unpack_i8x8(make_uint2(v0.x, v0.y), f);
  }
}

// Optimizer + publication for ONE tile whose summed gradient is already in `acc` (and whose state
// `w`, `b0`, `b1`, `b2` has been loaded): the epilogue shared by every gather flavour.
template <int OPT>
__device__ __forceinline__ void apply_and_publish(const UpdateArgs& a, const TileInfo& ti, size_t e0, float inv_count,
                                                  const float* acc, float* w, float* m, float* v, float* vm) {
  GroupHyper h = a.groups[ti.group];
  if (a.param_hyper != nullptr) {
    // parameters whose step count differs from their group's (a gradient that first arrived late, a layer that was frozen
    // for a while): the reference keeps state PER PARAMETER (/root/reference/ps.py:203-205,226-241), so the bias-corrected
    // Adam step size and SGD's first-step momentum rule come from a per-parameter table
    const float2 ph = a.param_hyper[ti.param];
    h.step_size = ph.x;
    h.first_step = ph.y != 0.f;
  }
  float g[PSB_EPT];
#pragma unroll
  for (int j = 0; j < PSB_EPT; ++j) g[j] = acc[j] * inv_count;
  if (h.weight_decay != 0.f) {
#pragma unroll
    for (int j = 0; j < PSB_EPT; ++j) g[j] = fmaf(h.weight_decay, w[j], g[j]);
  }
  if constexpr (OPT == OPT_SGD) {   // /root/reference/ps.py:197-214
    if (h.momentum != 0.f) {
#pragma unroll
      for (int j = 0; j < PSB_EPT; ++j) {
        m[j] = h.first_step ? g[j] : fmaf(h.momentum, m[j], (1.f - h.dampening) * g[j]);
        g[j] = h.nesterov ? fmaf(h.momentum, m[j], g[j]) : m[j];
      }
      float4* bp = reinterpret_cast<float4*>(a.buf0 + e0);
      bp[0] = make_float4(m[0], m[1], m[2], m[3]);
      bp[1] = make_float4(m[4], m[5], m[6], m[7]);
    }
#pragma unroll
    for (int j = 0; j < PSB_EPT; ++j) w[j] = fmaf(-h.lr, g[j], w[j]);
  } else {                          // /root/reference/ps.py:218-261
#pragma unroll
    for (int j = 0; j < PSB_EPT; ++j) {
      m[j] = fmaf(h.beta1, m[j], (1.f - h.beta1) * g[j]);
      v[j] = fmaf(h.beta2, v[j], (1.f - h.beta2) * g[j] * g[j]);
      float den_src = v[j];
      if (h.amsgrad) {
        vm[j] = fmaxf(vm[j], v[j]);
        den_src = vm[j];
      }
      const float denom = __fsqrt_rn(den_src) + h.eps;
      w[j] = fmaf(-h.step_size, __fdiv_rn(m[j], denom), w[j]);
    }
    float4* mp = reinterpret_cast<float4*>(a.buf0 + e0);
    mp[0] = make_float4(m[0], m[1], m[2], m[3]);
    mp[1] = make_float4(m[4], m[5], m[6], m[7]);
    float4* vp = reinterpret_cast<float4*>(a.buf1 + e0);
    vp[0] = make_float4(v[0], v[1], v[2], v[3]);
    vp[1] = make_float4(v[4], v[5], v[6], v[7]);
    if (h.amsgrad) {
      float4* xp = reinterpret_cast<float4*>(a.buf2 + e0);
      xp[0] = make_float4(vm[0], vm[1], vm[2], vm[3]);
      xp[1] = make_float4(vm[4], vm[5], vm[6], vm[7]);
    }
  }
  if (a.master != nullptr) {
    float4* wp = reinterpret_cast<float4*>(a.master + e0);
    wp[0] = make_float4(w[0], w[1], w[2], w[3]);
    wp[1] = make_float4(w[4], w[5], w[6], w[7]);
  }
  // publish the fresh parameter tile (the Ibcast of mpi_comms.py:132)
  uint4 out[2];
  const int nv = pack8(a.param_dt, w, out);
  const size_t pbytes = e0 * (a.param_dt == DT_F32 ? 4 : 2);
  if (a.bcast == BCAST_MULTICAST) {
    uint8_t* p = reinterpret_cast<uint8_t*>(a.param_mc) + pbytes;
    multimem_st_v4(p, out[0]);
    if (nv == 2) multimem_st_v4(p + 16, out[1]);
  } else if (a.bcast == BCAST_UNICAST) {
    for (int r = 0; r < a.world; ++r) {
      uint8_t* p = reinterpret_cast<uint8_t*>(a.param_dst[r]) + pbytes;
      st_sys_v4(p, out[0]);
      if (nv == 2) st_sys_v4(p + 16, out[1]);
    }
  } else {
    uint8_t* p = reinterpret_cast<uint8_t*>(a.param_local) + pbytes;
    st_v4(p, out[0]);
    if (nv == 2) st_v4(p + 16, out[1]);
  }
}

// Issue the (local, independent) optimizer-state loads for one tile: they fly while the peer loads do.
template <int OPT>
__device__ __forceinline__ void load_state(const UpdateArgs& a, const TileInfo& ti, size_t e0, float* w, float* m, float* v,
                                           float* vm) {
  if (a.master != nullptr) load8_local(a.master, DT_F32, e0, w);
  else load8_local(a.param_local, a.param_dt, e0, w);
  const GroupHyper& h = a.groups[ti.group];
  if constexpr (OPT == OPT_SGD) {
    if (h.momentum != 0.f) load8_local(a.buf0, DT_F32, e0, m);
  } else {
    load8_local(a.buf0, DT_F32, e0, m);
    load8_local(a.buf1, DT_F32, e0, v);
    if (h.amsgrad) load8_local(a.buf2, DT_F32, e0, vm);
  }
}

// One launch covers arena tiles [tile_begin, tile_end): the whole model, or ONE CHUNK of the per-bucket pipeline — the
// device analogue of the reference posting one non-blocking collective per parameter and consuming each as it completes
// (/root/reference/ps.py:140-148,159-162).  The engine launches chunk k's update while backward is still producing
// chunk k+1; GRAD_READY carries a monotone progress value ((epoch-1)*nchunks + chunk + 1), so one flag per rank serves
// every chunk.
//
// NVLS_U = tiles a thread keeps in flight on the multimem.ld_reduce path: one 16-byte switch reduction per tile is far too
// little to cover the NVLS round trip, so four are issued back to back before the first is consumed.
constexpr int NVLS_U = 4;

template <int KIND, int WIRE, int OPT>
__global__ void __launch_bounds__(PSB_THREADS, 3) psb_update_kernel(const __grid_constant__ UpdateArgs a) {
  __shared__ float s_acc[KIND == KIND_TOPK ? PSB_TILE : 1];
  __shared__ int s_flag;
  const int tid = threadIdx.x;
  uint64_t* err_slot = a.signal_local + SIG_ERROR;
  uint32_t contrib = a.contrib_mask, ack = a.ack_mask;
  float inv_count = a.inv_count;
  if (a.select_out != nullptr) {   // async: the contributor set was chosen on the device
    contrib = (uint32_t)a.select_out[0];
    ack = a.ack_last ? contrib : 0u;
    const uint32_t cnt = (uint32_t)a.select_out[1];
    if (cnt == 0) return;          // nothing to apply (all workers finished, or the select timed out)
    if (a.average_dynamic) inv_count = 1.f / (float)cnt;
  }

  // ---- 1. the req.Wait() of the reference: every contributor's progress flag ----
  // (the pipelined engine waits in a one-warp kernel queued just ahead of this one instead — a full update grid spinning
  //  on its peers would hold every SM's registers while this rank's backward still runs; then only the error slot is checked:
  //  a timed-out wait must not be followed by an update over stale tiles)
  if (a.wait_grads) {
    bool ok = true;
    if (tid < a.world && (contrib & a.wait_mask) >> tid & 1u)
      ok = spin_until_ge(a.signal_local + SIG_GRAD_READY + tid, a.wait_value, err_slot, a.timeout_ns);
    if (!__syncthreads_and(ok)) return;
  } else if (a.world > 1) {
    bool ok = true;
    if (tid == 0) ok = ld_relaxed_sys_u64(err_slot) == 0;
    if (!__syncthreads_and(ok)) return;
  }

  if constexpr (KIND == KIND_TOPK) {
    // ---- block-wise top-k: every rank's (index, value) entries are fetched with 16-byte peer loads, ALL ranks in
    // flight at once (2 vectors per thread per round), then scatter-added into a shared-memory tile rank by rank
    // (rank order = summation order, so the sum stays bit-reproducible) ----
    constexpr int ENT = (WIRE == WIRE_BF16) ? 4 : 2;     // entries per 16-byte vector
    constexpr int VPT = 2;                               // vectors per thread per round
    const int nv = a.bytes_per_tile >> 4;                // vectors per rank per tile
    const int total = a.world * nv;
    for (int tile = a.tile_begin + blockIdx.x; tile < a.tile_end; tile += gridDim.x) {
      const TileInfo ti = a.tiles[tile];
      if (a.active != nullptr && a.active[ti.param] == 0) continue;
      const size_t e0 = (size_t)tile * PSB_TILE + tid * PSB_EPT;
      const size_t tile_off = (size_t)tile * a.bytes_per_tile;
      float w[PSB_EPT], m[PSB_EPT], v[PSB_EPT], vm[PSB_EPT];
      load_state<OPT>(a, ti, e0, w, m, v, vm);           // local; flies while the peer loads do
      for (int j = tid; j < PSB_TILE; j += PSB_THREADS) s_acc[j] = 0.f;
      __syncthreads();
      for (int base = 0; base < total; base += VPT * PSB_THREADS) {
        uint4 q[VPT];
        int qr[VPT], qj[VPT];
#pragma unroll
        for (int k = 0; k < VPT; ++k) {
          const int vid = base + k * PSB_THREADS + tid;
          qr[k] = -1;
          qj[k] = 0;
          if (vid < total) {
            const int r = vid / nv;
            if (contrib >> r & 1u) {
              qr[k] = r;
              qj[k] = vid - r * nv;
              q[k] = ld_sys_v4(reinterpret_cast<const uint8_t*>(a.wire[r]) + tile_off + 16 * (size_t)qj[k]);
            }
          }
        }
        const int r_lo = base / nv, r_hi = (min(total, base + VPT * PSB_THREADS) - 1) / nv;
        for (int r = r_lo; r <= r_hi; ++r) {
#pragma unroll
          for (int k = 0; k < VPT; ++k) {
            if (qr[k] != r) continue;
            const uint32_t wd[4] = {q[k].x, q[k].y, q[k].z, q[k].w};
#pragma unroll
            for (int e = 0; e < ENT; ++e) {
              if (qj[k] * ENT + e >= a.cap) break;       // alignment padding behind the last entry
              uint32_t idx;
              float val;
              if constexpr (WIRE == WIRE_BF16) {
                idx = wd[e] >> 16;
                val = __uint_as_float(wd[e] << 16);
              } else {
                idx = wd[2 * e];
                val = __uint_as_float(wd[2 * e + 1]);
              }
              if (idx < PSB_TILE) s_acc[idx] += val;     // indices are unique within one rank's tile
            }
          }
          __syncthreads();
        }
      }
      float acc[PSB_EPT];
#pragma unroll
      for (int j = 0; j < PSB_EPT; ++j) acc[j] = s_acc[tid * PSB_EPT + j];
      __syncthreads();
      apply_and_publish<OPT>(a, ti, e0, inv_count, acc, w, m, v, vm);
    }
  } else {
    constexpr bool NVLS_OK = KIND == KIND_DENSE && (WIRE == WIRE_F32 || WIRE == WIRE_BF16 || WIRE == WIRE_F16);
    if (NVLS_OK && a.reduce == REDUCE_NVLS) {
      if constexpr (NVLS_OK) {
        // ---- the switch adds all ranks (multimem.ld_reduce): server ingress is 1x the vector, not (N-1)x ----
        for (int tile0 = a.tile_begin + blockIdx.x; tile0 < a.tile_end; tile0 += NVLS_U * gridDim.x) {
          uint4 v0[NVLS_U], v1[NVLS_U];
          TileInfo ti[NVLS_U];
          bool live[NVLS_U];
#pragma unroll
          for (int u = 0; u < NVLS_U; ++u) {
            const int tile = tile0 + u * gridDim.x;
            live[u] = tile < a.tile_end;
            if (live[u]) {
              ti[u] = a.tiles[tile];
              if (a.active != nullptr && a.active[ti[u].param] == 0) live[u] = false;
            }
            if (live[u]) {
              const uint8_t* p = reinterpret_cast<const uint8_t*>(a.wire_mc) + (size_t)tile * a.bytes_per_tile +
                                 (size_t)tid * PSB_EPT * wire_elem_bytes(WIRE);
              if constexpr (WIRE == WIRE_F32) {
                v0[u] = multimem_ld_reduce_f32x4(p);
                v1[u] = multimem_ld_reduce_f32x4(p + 16);
              } else if constexpr (WIRE == WIRE_BF16) {
                v0[u] = multimem_ld_reduce_bf16x8(p);
              } else {
                v0[u] = multimem_ld_reduce_f16x8(p);
              }
            }
          }
#pragma unroll
          for (int u = 0; u < NVLS_U; ++u) {
            if (!live[u]) continue;
            const size_t e0 = (size_t)(tile0 + u * gridDim.x) * PSB_TILE + tid * PSB_EPT;
            float acc[PSB_EPT], w[PSB_EPT], m[PSB_EPT], v[PSB_EPT], vm[PSB_EPT];
            load_state<OPT>(a, ti[u], e0, w, m, v, vm);
            decode_dense<WIRE>(v0[u], v1[u], acc);
            apply_and_publish<OPT>(a, ti[u], e0, inv_count, acc, w, m, v, vm);
          }
        }
      }
    } else {
      // ---- dense / scaled wires over P2P: up to CH ranks of 16-byte peer loads in flight per thread, local optimizer
      // state issued first (independent of the gather, so it overlaps the NVLink latency) ----
      constexpr int CH = 4;
      for (int tile = a.tile_begin + blockIdx.x; tile < a.tile_end; tile += gridDim.x) {
        const TileInfo ti = a.tiles[tile];
        if (a.active != nullptr && a.active[ti.param] == 0) continue;
        const size_t e0 = (size_t)tile * PSB_TILE + tid * PSB_EPT;
        float acc[PSB_EPT], w[PSB_EPT], m[PSB_EPT], v[PSB_EPT], vm[PSB_EPT];
#pragma unroll
        for (int j = 0; j < PSB_EPT; ++j) acc[j] = 0.f;
        load_state<OPT>(a, ti, e0, w, m, v, vm);
        for (int r0 = 0; r0 < a.world; r0 += CH) {
          uint4 v0[CH], v1[CH];
          float sc[CH];
#pragma unroll
          for (int c = 0; c < CH; ++c) {
            const int r = r0 + c;
            sc[c] = 1.f;
            if (r < a.world && (contrib >> r & 1u)) {
              issue_dense<WIRE>(a.wire[r], (size_t)tile * a.bytes_per_tile, v0[c], v1[c]);
              if constexpr (KIND == KIND_SCALED) sc[c] = ld_sys_f32(a.scales[r] + ti.param);
              if constexpr (KIND == KIND_QSGD)      // the tile's own scale, in the trailer of its wire slot
                sc[c] = ld_sys_f32(reinterpret_cast<const float*>(reinterpret_cast<const uint8_t*>(a.wire[r]) +
                                                                  (size_t)tile * a.bytes_per_tile + PSB_TILE));
            }
          }
#pragma unroll
          for (int c = 0; c < CH; ++c) {       // fixed rank order → deterministic fp32 sum
            const int r = r0 + c;
            if (r < a.world && (contrib >> r & 1u)) {
              float f[PSB_EPT];
              decode_dense<WIRE>(v0[c], v1[c], f);
#pragma unroll
              for (int j = 0; j < PSB_EPT; ++j) {
                if constexpr (KIND == KIND_SCALED || KIND == KIND_QSGD) acc[j] += f[j] * sc[c];
                else acc[j] += f[j];
              }
            }
          }
        }
        apply_and_publish<OPT>(a, ti, e0, inv_count, acc, w, m, v, vm);
      }
    }
  }

  // ---- completion: the last CTA raises the epoch flags ----
  // Launches that raise nothing (every pipeline chunk but the last; any launch at N = 1) skip the block: the system-scope
  // fence + completion atomic cost each CTA a round trip its warps wait out at the barrier (ncu: `barrier` was the top
  // stall of a 2-3-tile chunk launch).  Their stores are ordered before the last chunk's flag by the stream: a kernel's
  // writes — peer and multimem stores included — are complete when the kernel is.
  if (a.signal_mode == 0 && ack == 0u) return;
  __syncthreads();
  if (tid == 0) {
    __threadfence_system();
    const unsigned prev = atomicAdd(a.done_counter, 1u);
    s_flag = (prev == gridDim.x - 1);
  }
  __syncthreads();
  if (s_flag) {
    if (tid == 0) {
      *a.done_counter = 0;
      if (a.stats) atomicAdd(a.stats, 1u);
    }
    __threadfence_system();
    if (tid < a.world) {
      if (a.signal_mode == 1) {
        st_release_sys(a.signal_peer[tid] + SIG_VERSION, a.version);
        st_release_sys(a.signal_peer[tid] + SIG_PARAMS_READY, a.epoch);
      } else if (a.signal_mode == 2) {
        st_release_sys(a.signal_peer[tid] + SIG_CONSUMED + a.rank, a.epoch);
      }
      if (ack >> tid & 1u) {
        const uint64_t e = ld_relaxed_sys_u64(a.signal_local + SIG_GRAD_READY + tid);
        st_release_sys(a.signal_peer[tid] + SIG_ACK, e);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// flags
// ------------------------------------------------------------------------------------------
struct SignalArgs {
  uint64_t* targets[PSB_MAX_RANKS];
  int32_t n, slot;
  uint64_t value;
  uint64_t* extra_base;
  int32_t extra_slot;
  uint64_t extra_value;
  // async staleness accounting: when set, the kernel first posts "the parameter version this gradient was computed on"
  // (sampled into `version_local[SIG_SEEN_VERSION]` when the PREVIOUS gradient was posted, i.e. right before the forward
  // pass that produced this one started) into targets[t][version_slot], then re-samples the latest published version.
  uint64_t* version_local;
  int32_t version_slot;
};

__global__ void psb_signal_kernel(const __grid_constant__ SignalArgs a) {
  __threadfence_system();
  const int t = threadIdx.x;
  uint64_t seen = 0;
  if (a.version_local != nullptr) seen = ld_relaxed_sys_u64(a.version_local + SIG_SEEN_VERSION);
  if (t < a.n) {
    if (a.extra_base != nullptr && a.targets[t] != nullptr) st_release_sys(a.targets[t] + a.extra_slot, a.extra_value);
    if (a.version_local != nullptr && a.targets[t] != nullptr) st_release_sys(a.targets[t] + a.version_slot, seen);
    if (a.targets[t] != nullptr) st_release_sys(a.targets[t] + a.slot, a.value);
  }
  __syncwarp();      // every lane has read `seen` before lane 0 replaces it (several targets: one lane each)
  if (a.version_local != nullptr && t == 0)
    st_release_sys(a.version_local + SIG_SEEN_VERSION, ld_acquire_sys(a.version_local + SIG_VERSION));
}

__global__ void psb_wait_kernel(const uint64_t* signal_local, int slot0, uint32_t mask, uint64_t want,
                                unsigned long long timeout_ns) {
  const int t = threadIdx.x;
  if (mask >> t & 1u)
    spin_until_ge(signal_local + slot0 + t, want, const_cast<uint64_t*>(signal_local) + SIG_ERROR, timeout_ns);
}

// async PS: wait until `quota` candidate workers (ANY source, README.md:65-70) have a gradient newer
// than what was consumed.  Workers that posted the DONE epoch are reported in out[40] and never chosen.
// The whole server iteration is device-resident: this kernel also
//   * opens the consistent-read sequence lock (SIG_STAGE_BEGIN = version on every rank) iff something was selected,
//   * records the staleness of every selected gradient (updates applied since the parameters it was computed on):
//     out[44 + r] = (version - 1) - SIG_GRAD_VERSION[r],
// so the host never has to look at the result before queueing the update kernel and the next select.
#define PSB_DONE_EPOCH (1ull << 62)
struct SelectArgs {
  const uint64_t* signal_local;
  uint64_t* consumed;
  uint64_t* out;
  uint64_t* begin_targets[PSB_MAX_RANKS];   // every rank's signal pad (consistent=True) or all nullptr
  int32_t nbegin;
  uint32_t cand_mask;
  int32_t quota;
  uint64_t version;                          // the version the following update kernel will publish
  unsigned long long timeout_ns;
};

__global__ void psb_select_kernel(const __grid_constant__ SelectArgs a) {
  const uint64_t* signal_local = a.signal_local;
  uint64_t* consumed = a.consumed;
  uint64_t* out = a.out;
  const uint32_t cand_mask = a.cand_mask;
  const int quota = a.quota;
  const int t = threadIdx.x;   // one warp
  uint64_t* err = const_cast<uint64_t*>(signal_local) + SIG_ERROR;
  unsigned long long t0 = 0;
  uint32_t ready = 0, fin = 0;
  uint64_t e = 0;
  int need = 0;
  while (true) {
    const bool cand = cand_mask >> t & 1u;
    e = cand ? ld_acquire_sys(signal_local + SIG_GRAD_READY + t) : 0;
    const bool f = cand && e >= PSB_DONE_EPOCH;
    const bool r = cand && !f && e > consumed[t];
    ready = __ballot_sync(0xffffffffu, r);
    fin = __ballot_sync(0xffffffffu, f);
    need = min(quota, __popc(cand_mask & ~fin));
    if (need == 0 || __popc(ready) >= need) break;
    unsigned long long now;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));
    if (t0 == 0) t0 = now;
    bool bad = (now - t0 > a.timeout_ns) || ld_relaxed_sys_u64(err) != 0;
    if (__any_sync(0xffffffffu, bad)) {
      if (t == 0) {
        st_release_sys(err, 2ull);
        out[0] = 0;
        out[1] = 0;
        out[40] = fin;
      }
      return;
    }
    __nanosleep(200);
  }
  // rotating priority so no worker starves: start after the last served rank
  const int start = (int)(consumed[63] % 32);
  uint32_t chosen = 0;
  int cnt = 0;
  for (int i = 0; i < 32 && cnt < need; ++i) {
    const int r = (start + 1 + i) % 32;
    if (ready >> r & 1u) {
      chosen |= 1u << r;
      ++cnt;
    }
  }
  __syncwarp();
  if (chosen >> t & 1u) {
    consumed[t] = e;
    out[2 + t] = e;
    const uint64_t gv = ld_acquire_sys(signal_local + SIG_GRAD_VERSION + t);
    out[44 + t] = a.version - 1 >= gv ? a.version - 1 - gv : 0;
  }
  if (chosen != 0 && t < a.nbegin && a.begin_targets[t] != nullptr)
    st_release_sys(a.begin_targets[t] + SIG_STAGE_BEGIN, a.version);   // sequence lock: BEGIN(v) … stores … VERSION(v)
  if (t == 0) {
    if (chosen) consumed[63] = (uint64_t)(31 - __clz(chosen));
    out[0] = chosen;
    out[1] = (uint64_t)cnt;
    out[40] = fin;
    out[41] = a.version;
  }
}

// ------------------------------------------------------------------------------------------
// consistent reads (async, README.md:79-81 "a buffered broadcast"): device-side sequence-lock snapshot
// ------------------------------------------------------------------------------------------
// The server publishes version v into every rank's STAGING arena between SIG_STAGE_BEGIN = v and SIG_VERSION = v.
// A worker adopts whole versions only, with no host involvement:
//   psb_snapshot_fetch   every CTA: read BEGIN / VERSION; if they agree on a version newer than the adopted one, copy its
//                        slice staging → shadow and re-read BEGIN; any disagreement (publication in progress, torn copy,
//                        CTAs that saw different versions) vetoes.  The last CTA writes the verdict: status = v or 0.
//   psb_snapshot_commit  if status != 0: shadow → live parameter arena (purely local, the server never writes there), and the
//                        adopted version becomes v.  A vetoed attempt leaves the live parameters on the previous whole version.
struct SnapshotArgs {
  const uint64_t* signal_local;
  const uint4* stage;
  uint4* shadow;
  uint4* params;
  size_t nvec;                   // 16-byte vectors
  unsigned long long* scratch;   // [0] veto  [1] min version  [2] max version  [3] CTAs done  [4] status  [5] adopted version
};

__global__ void __launch_bounds__(256) psb_snapshot_fetch(const __grid_constant__ SnapshotArgs a) {
  __shared__ unsigned long long s_v;
  __shared__ int s_go;
  if (threadIdx.x == 0) {
    const uint64_t vb = ld_acquire_sys(a.signal_local + SIG_STAGE_BEGIN), ve = ld_acquire_sys(a.signal_local + SIG_VERSION);
    s_v = ve;
    s_go = (vb == ve) && (ve != a.scratch[5]) && (ve != 0);
  }
  __syncthreads();
  const unsigned long long v = s_v;
  bool veto = !s_go;
  if (s_go) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.nvec; i += (size_t)gridDim.x * blockDim.x)
      a.shadow[i] = ld_sys_v4(a.stage + i);       // coherent loads: the server's multimem.st / peer stores land here
    __syncthreads();
    if (threadIdx.x == 0) veto = ld_acquire_sys(a.signal_local + SIG_STAGE_BEGIN) != v;
  }
  if (threadIdx.x == 0) {
    if (veto) atomicOr(a.scratch + 0, 1ull);
    atomicMin(a.scratch + 1, v);
    atomicMax(a.scratch + 2, v);
    __threadfence();
    if (atomicAdd(a.scratch + 3, 1ull) == gridDim.x - 1) {
      __threadfence();
      const bool ok = a.scratch[0] == 0 && a.scratch[1] == a.scratch[2];
      a.scratch[4] = ok ? a.scratch[1] : 0ull;
      a.scratch[0] = 0, a.scratch[1] = ~0ull, a.scratch[2] = 0, a.scratch[3] = 0;
    }
  }
}

__global__ void __launch_bounds__(256) psb_snapshot_commit(const __grid_constant__ SnapshotArgs a) {
  const unsigned long long v = a.scratch[4];
  if (v == 0) return;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.nvec; i += (size_t)gridDim.x * blockDim.x)
    a.params[i] = a.shadow[i];
  if (blockIdx.x == 0 && threadIdx.x == 0) a.scratch[5] = v;     // stream-ordered: the next fetch reads it after this kernel
}

template <int KIND, int WIRE, int OPT>
void launch_update_t(cudaStream_t s, const UpdateArgs& a, int grid) {
  // (a variant with two P2P tiles in flight per thread and no state prefetch measured slower, 72.6 us vs 52.5 us on the
  //  ResNet-18 arena at N = 1, and was removed: profiles/psb_update_kernel_resnet18_n1_v2.ncu.txt)
  psb_update_kernel<KIND, WIRE, OPT><<<grid, PSB_THREADS, 0, s>>>(a);
}
template <int KIND, int WIRE>
void launch_update_o(cudaStream_t s, int opt, const UpdateArgs& a, int grid) {
  if (opt == OPT_SGD) launch_update_t<KIND, WIRE, OPT_SGD>(s, a, grid);
  else launch_update_t<KIND, WIRE, OPT_ADAM>(s, a, grid);
}

}  // namespace

// ------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------
#include <atomic>
static std::atomic<unsigned long long> g_psb_launches{0};
void psb_count_launch(int n) { g_psb_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }
unsigned long long psb_launch_count() { return g_psb_launches.load(std::memory_order_relaxed); }

void psb_launch_absmax(cudaStream_t s, const EncodeArgs& a) {
  const int ctas = a.batch.cum[a.batch.n];
  if (ctas > 0) {
    psb_absmax_kernel<<<ctas, PSB_THREADS, 0, s>>>(a);
    psb_count_launch(1);
  }
}

void psb_launch_encode(cudaStream_t s, int kind, int wire, const EncodeArgs& a) {
  const int ctas = a.batch.cum[a.batch.n];
  if (ctas <= 0) return;
  psb_count_launch(1);
#define ENC(K, W)                                            \
  if (kind == K && wire == W) {                              \
    psb_encode_kernel<K, W><<<ctas, PSB_THREADS, 0, s>>>(a); \
    return;                                                  \
  }
  ENC(KIND_DENSE, WIRE_F32) ENC(KIND_DENSE, WIRE_BF16) ENC(KIND_DENSE, WIRE_F16) ENC(KIND_DENSE, WIRE_E4M3)
  ENC(KIND_DENSE, WIRE_E5M2) ENC(KIND_SCALED, WIRE_I8) ENC(KIND_SCALED, WIRE_E4M3) ENC(KIND_SCALED, WIRE_E5M2)
  ENC(KIND_SCALED, WIRE_F16) ENC(KIND_TOPK, WIRE_F32) ENC(KIND_TOPK, WIRE_BF16) ENC(KIND_QSGD, WIRE_I8)
#undef ENC
}

void psb_launch_update(cudaStream_t s, int kind, int wire, int opt, const UpdateArgs& a, int grid) {
  psb_count_launch(1);
#define UPD(K, W)                                \
  if (kind == K && wire == W) {                  \
    launch_update_o<K, W>(s, opt, a, grid);      \
    return;                                      \
  }
  UPD(KIND_DENSE, WIRE_F32) UPD(KIND_DENSE, WIRE_BF16) UPD(KIND_DENSE, WIRE_F16) UPD(KIND_DENSE, WIRE_E4M3)
  UPD(KIND_DENSE, WIRE_E5M2) UPD(KIND_SCALED, WIRE_I8) UPD(KIND_SCALED, WIRE_E4M3) UPD(KIND_SCALED, WIRE_E5M2)
  UPD(KIND_SCALED, WIRE_F16) UPD(KIND_TOPK, WIRE_F32) UPD(KIND_TOPK, WIRE_BF16) UPD(KIND_QSGD, WIRE_I8)
#undef UPD
}

int psb_update_max_grid(int kind, int wire, int opt) {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  (void)kind, (void)wire, (void)opt;
  return sms * 3;   // __launch_bounds__(256, 3): all CTAs co-resident (the completion counter needs no more)
}

void psb_launch_signal(cudaStream_t s, uint64_t* const* targets, int ntargets, int slot, uint64_t value,
                       uint64_t* extra_slot_base, int extra_slot, uint64_t extra_value, uint64_t* version_local,
                       int version_slot) {
  SignalArgs a{};
  a.n = ntargets;
  for (int i = 0; i < ntargets && i < PSB_MAX_RANKS; ++i) a.targets[i] = targets[i];
  a.slot = slot;
  a.value = value;
  a.extra_base = extra_slot_base;
  a.extra_slot = extra_slot;
  a.extra_value = extra_value;
  a.version_local = version_local;
  a.version_slot = version_slot;
  psb_signal_kernel<<<1, 32, 0, s>>>(a);
  psb_count_launch(1);
}

void psb_launch_snapshot(cudaStream_t s, const uint64_t* signal_local, const void* stage, void* shadow, void* params, size_t nbytes,
                         unsigned long long* scratch, int attempts, int num_sms) {
  SnapshotArgs a{};
  a.signal_local = signal_local;
  a.stage = reinterpret_cast<const uint4*>(stage);
  a.shadow = reinterpret_cast<uint4*>(shadow);
  a.params = reinterpret_cast<uint4*>(params);
  a.nvec = nbytes / 16;
  a.scratch = scratch;
  const int grid = (int)std::max<size_t>(1, std::min<size_t>((size_t)num_sms * 4, (a.nvec + 255) / 256));
  for (int i = 0; i < attempts; ++i) {
    psb_snapshot_fetch<<<grid, 256, 0, s>>>(a);
    psb_snapshot_commit<<<grid, 256, 0, s>>>(a);
    psb_count_launch(2);
  }
}

void psb_launch_wait(cudaStream_t s, const uint64_t* signal_local, int slot0, uint32_t mask, uint64_t want,
                     unsigned long long timeout_ns) {
  psb_wait_kernel<<<1, 32, 0, s>>>(signal_local, slot0, mask, want, timeout_ns);
  psb_count_launch(1);
}

void psb_launch_select(cudaStream_t s, const uint64_t* signal_local, uint64_t* consumed, uint32_t cand_mask,
                       int quota, uint64_t* out, unsigned long long timeout_ns, uint64_t version,
                       uint64_t* const* begin_targets, int nbegin) {
  SelectArgs a{};
  a.signal_local = signal_local;
  a.consumed = consumed;
  a.out = out;
  a.cand_mask = cand_mask;
  a.quota = quota;
  a.version = version;
  a.timeout_ns = timeout_ns;
  a.nbegin = nbegin;
  for (int i = 0; i < nbegin && i < PSB_MAX_RANKS; ++i) a.begin_targets[i] = begin_targets[i];
  psb_select_kernel<<<1, 32, 0, s>>>(a);
  psb_count_launch(1);
}
