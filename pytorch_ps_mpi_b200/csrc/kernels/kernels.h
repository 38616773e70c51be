// Host-callable launchers of the sm_100a kernels (plain C++ types; no torch headers here).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"

#define PSB_ENCODE_MAX 64

// One launch encodes up to PSB_ENCODE_MAX gradient tensors (a "bucket" of hook firings).
struct EncodeBatch {
  const void* src[PSB_ENCODE_MAX];     // gradient tensors (contiguous, 16-byte aligned)
  int32_t first_tile[PSB_ENCODE_MAX];  // first arena tile of each
  int32_t cum[PSB_ENCODE_MAX + 1];     // prefix sum of tile counts
  int32_t param[PSB_ENCODE_MAX];       // parameter index of each
  int32_t n;
};

struct EncodeArgs {
  EncodeBatch batch;
  const TileInfo* tiles;
  void* wire;            // local wire arena
  float* scales;         // local per-parameter scale table (KIND_SCALED)
  uint32_t* amax_bits;   // per-parameter abs-max scratch (float bits, atomicMax)
  float* residual;       // error-feedback residual (flat fp32) or nullptr
  int32_t bytes_per_tile;
  int32_t cap;           // top-k entries per tile
  double ratio;
  int32_t grad_dt;
  // block-wise QSGD (KIND_QSGD): quantisation levels and the Philox key / counter words of this launch
  int32_t levels;
  uint64_t seed;
  uint32_t rng_step;
  int32_t rank;
  // optional fused flag raise: when this is the LAST encode launch of the step, its last CTA publishes
  // GRAD_READY itself (saves the separate psb_signal_kernel launch on the critical path)
  uint64_t* sig_targets[PSB_MAX_RANKS];
  int32_t nsig;
  int32_t sig_slot;
  uint64_t sig_value;
  unsigned int* sig_counter;   // zero before launch; left zero
};

struct UpdateArgs {
  const void* wire[PSB_MAX_RANKS];     // every rank's wire arena as mapped in THIS process
  const float* scales[PSB_MAX_RANKS];  // every rank's scale table
  void* param_dst[PSB_MAX_RANKS];      // every rank's parameter arena (unicast publication)
  void* param_mc;                      // multicast alias of the parameter arena (NVLS) or nullptr
  const void* wire_mc;                 // multicast alias of the wire arena (NVLS reduce) or nullptr
  void* param_local;                   // this rank's parameter arena
  float* master;                       // fp32 master weights (nullptr → parameters are the master)
  float* buf0;                         // momentum_buffer / exp_avg
  float* buf1;                         // exp_avg_sq
  float* buf2;                         // max_exp_avg_sq
  const TileInfo* tiles;
  const uint8_t* active;               // per-parameter "got a gradient this step" (nullptr = all)
  const float2* param_hyper;           // per-parameter {step_size, first_step} overriding the group's (nullptr = uniform)
  uint64_t* signal_local;
  uint64_t* signal_peer[PSB_MAX_RANKS];
  unsigned int* done_counter;          // zero before launch; the kernel leaves it zero
  uint32_t* stats;                     // [0]=tiles processed (debug / tests), may be nullptr
  GroupHyper groups[PSB_MAX_GROUPS];
  int32_t world, rank, ntiles, bytes_per_tile, cap;
  int32_t param_dt, bcast, reduce;
  uint32_t contrib_mask;               // ranks whose gradient is summed
  uint32_t wait_mask;                  // ranks whose GRAD_READY flag is awaited (the launching rank's own gradient is
                                       // ordered by the stream, so it is normally excluded)
  float inv_count;                     // 1 or 1/#contributors (average=True)
  uint64_t epoch;                      // value published to SIG_PARAMS_READY / SIG_CONSUMED when the LAST chunk is done
  uint64_t wait_value;                 // SIG_GRAD_READY progress value awaited: (epoch-1)*nchunks + chunk + 1 (the
                                       // reference's per-parameter req.Wait(), ps.py:159-162, at chunk granularity)
  int32_t tile_begin, tile_end;        // this launch covers arena tiles [tile_begin, tile_end) — one chunk of the
                                       // pipeline (or the whole arena)
  int32_t wait_grads;                  // spin on SIG_GRAD_READY of every contributor first
  int32_t signal_mode;                 // 0 none | 1 SIG_PARAMS_READY → all | 2 SIG_CONSUMED[rank] → all
  uint32_t ack_mask;                   // async: ranks to acknowledge (SIG_ACK) when done
  int32_t ack_last;                    // 1 on the last window of a launch sequence: the async contributors (chosen on the
                                       // device, select_out) are acknowledged only then
  uint64_t version;                    // async: value published to SIG_VERSION
  const uint64_t* select_out;          // async: device-side {mask, count, epochs…} from psb_select_kernel (or nullptr)
  int32_t average_dynamic;             // async: divide by the selected count
  unsigned long long timeout_ns;
};

void psb_launch_absmax(cudaStream_t s, const EncodeArgs& a);
void psb_launch_encode(cudaStream_t s, int kind, int wire, const EncodeArgs& a);
void psb_launch_update(cudaStream_t s, int kind, int wire, int opt, const UpdateArgs& a, int grid);
void psb_launch_signal(cudaStream_t s, uint64_t* const* targets, int ntargets, int slot, uint64_t value,
                       uint64_t* extra_slot_base, int extra_slot, uint64_t extra_value, uint64_t* version_local = nullptr,
                       int version_slot = 0);
void psb_launch_wait(cudaStream_t s, const uint64_t* signal_local, int slot0, uint32_t mask, uint64_t want,
                     unsigned long long timeout_ns);
// async PS: block until >= quota workers of `cand_mask` have SIG_GRAD_READY > consumed[r]; writes the
// chosen mask + their epochs to `out` (out[0]=mask, out[1]=count, out[2+r]=epoch of rank r)
// (out[40] = finished mask, out[41] = version, out[44+r] = staleness of rank r's gradient; opens the consistent-read sequence
//  lock on `begin_targets` when something was selected)
void psb_launch_select(cudaStream_t s, const uint64_t* signal_local, uint64_t* consumed, uint32_t cand_mask,
                       int quota, uint64_t* out, unsigned long long timeout_ns, uint64_t version = 0,
                       uint64_t* const* begin_targets = nullptr, int nbegin = 0);
// consistent reads: `attempts` x (fetch staging → shadow under the sequence lock, commit shadow → params); scratch = 6 x u64
// initialised to {0, ~0, 0, 0, 0, 0}; scratch[5] = the adopted version
void psb_launch_snapshot(cudaStream_t s, const uint64_t* signal_local, const void* stage, void* shadow, void* params, size_t nbytes,
                         unsigned long long* scratch, int attempts, int num_sms);
int psb_update_max_grid(int kind, int wire, int opt);

// bcast_gemm.cu — tcgen05 / TMEM / TMA GEMM whose weight tiles are gated on the PS broadcast epoch
struct BcastGemmArgs {
  const void* tmap_a;   // CUtensorMap* (host memory, passed as __grid_constant__ by value in launcher)
  const void* tmap_b;
  const void* tmap_c;
  const float* bias;    // nullable
  const uint64_t* ready_flag;   // nullable: SIG_PARAMS_READY slot to acquire before the first weight TMA
  uint64_t ready_epoch;
  int32_t M, N, K;
  int32_t relu;
  int32_t two_cta;      // 1 → cta_group::2 kernel (256x256 tiles per CTA pair; B box = 128 rows)
  const void* tmap_out; // 2-CTA only: CUtensorMap* of the [M,N] output (box 64 x 32, 128B swizzle) for the TMA-store
                        // epilogue; nullptr (or N % 8 != 0) → staged full-line stores
  unsigned long long timeout_ns;
};
void psb_launch_bcast_gemm(cudaStream_t s, const BcastGemmArgs& a, int num_sms);
// bcast_gemm2.cu — the cta_group::2 kernel; epi -1 = auto (TMA-store / staged epilogue), 0 / 1 / 3 = force (bench/gemm_variants.py)
void psb_launch_bcast_gemm2(cudaStream_t s, const BcastGemmArgs& a, int num_sms, int epi, const void* tmap_out);

// bn_kernels.cu — fused channels-last bf16 BatchNorm (+residual, +ReLU), forward and backward
void psb_bn_forward(cudaStream_t s, const void* x, const void* res, const void* gamma, const void* beta, void* y, float* sums,
                    float* mean, float* rstd, float* scale, float* shift, float* running_mean, float* running_var,
                    long long pixels, int C, float eps, float momentum, int relu, int training,
                    void* mask = nullptr /* [pixels * C/8] bytes: 1 bit per element, y > 0 (relu + training) */);
void psb_bn_forward_presummed(cudaStream_t s, const void* x, const void* res, const void* gamma, const void* beta, void* y,
                              const float* sums, float* mean, float* rstd, float* scale, float* shift, float* running_mean,
                              float* running_var, long long pixels, int C, float eps, float momentum, int relu,
                              void* mask = nullptr);
void psb_bn_backward(cudaStream_t s, const void* dy, const void* x, const void* y, const void* gamma, const float* mean,
                     const float* rstd, float* sums, float* coef, void* dx, void* dres, void* dgamma, void* dbeta,
                     long long pixels, int C, int relu, const void* mask = nullptr /* the forward's ReLU bit mask, replaces y */);

// pool_kernels.cu — channels-last bf16 3x3/s2/p1 max pooling
void psb_maxpool3x3s2_forward(cudaStream_t s, const void* x, void* y, void* arg, int N, int H, int W, int C);
void psb_maxpool3x3s2_backward(cudaStream_t s, const void* dy, const void* arg, void* dx, int N, int H, int W, int C);
void psb_normalize_pad8_launch(cudaStream_t s, const void* x, void* y, const float* mean, const float* inv_std, int N, long long HW);
void psb_im2col_stem_launch(cudaStream_t s, const void* x, void* a, int N, int H, int W);
void psb_normalize_nhwc3_launch(cudaStream_t s, const void* x, void* y, const float* mean, const float* inv_std, int N, long long HW);

// stem_kernels.cu — fused implicit-GEMM ResNet stem (7x7/s2, 3 → 64) with BN statistics in the epilogue
int psb_stem_fwd_smem_bytes();
void psb_stem_fwd_launch(cudaStream_t s, const void* tmap_w, const void* tmap_y, const void* x, float* sums, int N, int H, int W,
                         int num_sms, const uint64_t* ready_flag, uint64_t ready_epoch, unsigned long long timeout_ns);

int psb_stem_wgrad_grid(int N, int H, int num_sms);
void psb_stem_wgrad_finalize_launch(cudaStream_t s, const float* partial, int grid, void* out_bf16);
void psb_stem_wgrad_launch(cudaStream_t s, const void* tmap_g, const void* x, float* partial, int N, int H, int W, int num_sms);

// process-wide count of OUR kernel launches (every psb_* launcher adds to it; bench.py reports the delta)
void psb_count_launch(int n);
unsigned long long psb_launch_count();
