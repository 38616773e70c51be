// Python bindings of the CUDA extension (_psb200_cuda): symmetric memory, kernel launchers.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/extension.h>

#include <algorithm>
#include <cstring>
#include <memory>

#include "kernels.h"
#include "symm_mem.h"

namespace py = pybind11;

namespace {

void check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) throw std::runtime_error(std::string(what) + ": " + cudaGetErrorString(e));
}

cudaStream_t cur_stream() { return c10::cuda::getCurrentCUDAStream().stream(); }
// explicit raw stream handle (torch.cuda.Stream.cuda_stream) or 0 = torch's current stream: lets the engine launch on its
// side stream without the Python cost of switching the current stream
cudaStream_t pick_stream(uint64_t s) { return s ? reinterpret_cast<cudaStream_t>(s) : cur_stream(); }

int dt_code(at::ScalarType t) {
  switch (t) {
    case at::kFloat: return DT_F32;
    case at::kBFloat16: return DT_BF16;
    case at::kHalf: return DT_F16;
    default: throw std::runtime_error("unsupported dtype (need float32 / bfloat16 / float16)");
  }
}

// A tensor view over raw (VMM-mapped) device memory; `owner` keeps the mapping alive.
at::Tensor blob_tensor(uint64_t ptr, std::vector<int64_t> shape, at::ScalarType dtype, int device, py::object owner) {
  auto keep = std::make_shared<py::object>(std::move(owner));
  auto deleter = [keep](void*) mutable {
    py::gil_scoped_acquire g;
    keep.reset();
  };
  auto opts = at::TensorOptions().dtype(dtype).device(at::kCUDA, device);
  // target_device: a peer's block is mapped into THIS device's address space, but the pointer
  // attributes still name the owning GPU — tell ATen which device the view belongs to.
  return at::for_blob(reinterpret_cast<void*>(ptr), shape)
      .options(opts)
      .target_device(c10::Device(at::kCUDA, (c10::DeviceIndex)device))
      .deleter(deleter)
      .make_tensor();
}

// Static part of the fused PS launch (pointers never change after the arenas are built).
struct UpdatePlan {
  UpdateArgs a{};
  int kind = 0, wire = 0, opt = 0, grid = 0;
  int64_t window_bytes = 128ll << 20;

  void set_rank_ptrs(int r, uint64_t wire_p, uint64_t scales_p, uint64_t param_p, uint64_t signal_p) {
    if (r < 0 || r >= PSB_MAX_RANKS) throw std::runtime_error("rank out of range");
    a.wire[r] = reinterpret_cast<const void*>(wire_p);
    a.scales[r] = reinterpret_cast<const float*>(scales_p);
    a.param_dst[r] = reinterpret_cast<void*>(param_p);
    a.signal_peer[r] = reinterpret_cast<uint64_t*>(signal_p);
  }

  void launch(uint64_t epoch, const std::vector<std::vector<double>>& groups, uint32_t contrib_mask, double inv_count,
              int wait_grads, int signal_mode, uint32_t ack_mask, uint64_t version, uint64_t select_out,
              int average_dynamic, uint64_t active_ptr, double timeout_s, uint32_t wait_mask, uint64_t stream,
              int tile_begin, int tile_end, uint64_t wait_value, uint64_t param_hyper) {
    if (groups.size() > PSB_MAX_GROUPS) throw std::runtime_error("too many param groups for one launch");
    for (size_t i = 0; i < groups.size(); ++i) {
      const auto& g = groups[i];
      if (g.size() != 11) throw std::runtime_error("group hyper tuple must have 11 entries");
      GroupHyper& h = a.groups[i];
      h.lr = (float)g[0], h.weight_decay = (float)g[1], h.momentum = (float)g[2], h.dampening = (float)g[3];
      h.beta1 = (float)g[4], h.beta2 = (float)g[5], h.eps = (float)g[6], h.step_size = (float)g[7];
      h.nesterov = (int)g[8], h.amsgrad = (int)g[9], h.first_step = (int)g[10], h.pad = 0;
    }
    a.epoch = epoch;
    // one chunk of the pipeline (tile_end < 0: the whole arena, waiting for the plain epoch value)
    a.tile_begin = tile_end < 0 ? 0 : tile_begin;
    a.tile_end = tile_end < 0 ? a.ntiles : tile_end;
    if (a.tile_begin < 0 || a.tile_end > a.ntiles || a.tile_begin >= a.tile_end) throw std::runtime_error("bad tile range");
    a.wait_value = tile_end < 0 ? epoch : wait_value;
    a.contrib_mask = contrib_mask;
    a.wait_mask = wait_mask;
    a.inv_count = (float)inv_count;
    a.wait_grads = wait_grads;
    a.signal_mode = signal_mode;
    a.ack_mask = ack_mask;
    a.version = version;
    a.select_out = reinterpret_cast<const uint64_t*>(select_out);
    a.average_dynamic = average_dynamic;
    a.active = reinterpret_cast<const uint8_t*>(active_ptr);
    a.param_hyper = reinterpret_cast<const float2*>(param_hyper);
    a.timeout_ns = (unsigned long long)(timeout_s * 1e9);
    // Window the chunk: one launch touches at most `window_bytes` of every rank's wire arena.  A single kernel that walks
    // >= 1 GB of mapped peer memory on each of 8 ranks falls off a TLB cliff (194 GB/s, profiles/bw_sweep_n8.json);
    // back-to-back launches over <= 128 MB windows do not.  Only the first window waits for the flags (the rest is
    // stream-ordered behind it) and only the last one raises PARAMS_READY / CONSUMED / ACK.
    const int64_t per_tile = std::max<int64_t>(a.bytes_per_tile, 1);
    // (sparse wires have tiny tiles: also bound the window by the parameter bytes it publishes through peer / multicast memory)
    const int win = (int)std::max<int64_t>(1, std::min<int64_t>(window_bytes / per_tile, 4 * window_bytes / (PSB_TILE * 4)));
    const int lo = a.tile_begin, hi = a.tile_end;
    const int wait_grads_all = a.wait_grads, signal_all = a.signal_mode;
    const uint32_t ack_all = a.ack_mask;
    for (int b = lo; b < hi; b += win) {
      a.tile_begin = b;
      a.tile_end = std::min(hi, b + win);
      const bool first = b == lo, last = a.tile_end == hi;
      a.wait_grads = first ? wait_grads_all : 0;
      a.signal_mode = last ? signal_all : 0;
      a.ack_mask = last ? ack_all : 0;
      a.ack_last = last ? 1 : 0;
      psb_launch_update(pick_stream(stream), kind, wire, opt, a, std::min(grid, a.tile_end - a.tile_begin));
      check_launch("psb_update_kernel launch");
    }
    a.tile_begin = lo, a.tile_end = hi, a.wait_grads = wait_grads_all, a.signal_mode = signal_all, a.ack_mask = ack_all;
  }
};

void encode(int kind, int wire, const std::vector<at::Tensor>& grads, const std::vector<int>& first_tile,
            const std::vector<int>& ntiles, const std::vector<int>& param_idx, uint64_t tiles_ptr, uint64_t wire_ptr,
            uint64_t scales_ptr, uint64_t amax_ptr, uint64_t residual_ptr, int bytes_per_tile, int cap, double ratio,
            const std::vector<uint64_t>& sig_targets, int sig_slot, uint64_t sig_value, uint64_t sig_counter,
            uint64_t stream, int levels, uint64_t seed, uint32_t rng_step, int rank) {
  const size_t n = grads.size();
  if (first_tile.size() != n || ntiles.size() != n || param_idx.size() != n) throw std::runtime_error("encode: length mismatch");
  if (n == 0) return;
  cudaStream_t s = pick_stream(stream);
  EncodeArgs a{};
  a.tiles = reinterpret_cast<const TileInfo*>(tiles_ptr);
  a.wire = reinterpret_cast<void*>(wire_ptr);
  a.scales = reinterpret_cast<float*>(scales_ptr);
  a.amax_bits = reinterpret_cast<uint32_t*>(amax_ptr);
  a.residual = reinterpret_cast<float*>(residual_ptr);
  a.bytes_per_tile = bytes_per_tile;
  a.cap = cap;
  a.ratio = ratio;
  a.grad_dt = dt_code(grads[0].scalar_type());
  if (kind == KIND_QSGD) {
    if (levels < 1 || levels > 127) throw std::runtime_error("encode: QSGD levels must be in [1, 127] (int8 wire)");
    if (bytes_per_tile < PSB_TILE + 16) throw std::runtime_error("encode: a QSGD wire slot needs TILE + 16 bytes");
  }
  a.levels = levels;
  a.seed = seed;
  a.rng_step = rng_step;
  a.rank = rank;
  for (size_t base = 0; base < n; base += PSB_ENCODE_MAX) {
    const int m = (int)std::min<size_t>(PSB_ENCODE_MAX, n - base);
    a.batch.n = m;
    a.batch.cum[0] = 0;
    for (int i = 0; i < m; ++i) {
      const at::Tensor& g = grads[base + i];
      if (!g.is_cuda() || !g.is_non_overlapping_and_dense()) throw std::runtime_error("encode: gradients must be dense CUDA tensors");
      if (dt_code(g.scalar_type()) != a.grad_dt) throw std::runtime_error("encode: mixed gradient dtypes in one bucket");
      if (reinterpret_cast<uintptr_t>(g.data_ptr()) % 16 != 0) throw std::runtime_error("encode: gradient not 16-byte aligned");
      a.batch.src[i] = g.data_ptr();
      a.batch.first_tile[i] = first_tile[base + i];
      a.batch.param[i] = param_idx[base + i];
      a.batch.cum[i + 1] = a.batch.cum[i] + ntiles[base + i];
    }
    if (kind == KIND_SCALED) {
      psb_launch_absmax(s, a);
      check_launch("psb_absmax_kernel launch");
    }
    a.nsig = 0;
    if (!sig_targets.empty() && base + PSB_ENCODE_MAX >= n) {   // only the last launch of this call raises the flag
      if (sig_targets.size() > PSB_MAX_RANKS) throw std::runtime_error("encode: too many signal targets");
      a.nsig = (int)sig_targets.size();
      for (size_t i = 0; i < sig_targets.size(); ++i) a.sig_targets[i] = reinterpret_cast<uint64_t*>(sig_targets[i]);
      a.sig_slot = sig_slot;
      a.sig_value = sig_value;
      a.sig_counter = reinterpret_cast<unsigned int*>(sig_counter);
    }
    psb_launch_encode(s, kind, wire, a);
    check_launch("psb_encode_kernel launch");
  }
}

void signal(const std::vector<uint64_t>& targets, int slot, uint64_t value, int extra_slot, uint64_t extra_value,
            uint64_t stream, uint64_t version_local, int version_slot) {
  std::vector<uint64_t*> t;
  for (auto p : targets) t.push_back(reinterpret_cast<uint64_t*>(p));
  psb_launch_signal(pick_stream(stream), t.data(), (int)t.size(), slot, value,
                    extra_slot >= 0 ? reinterpret_cast<uint64_t*>(1) : nullptr, extra_slot < 0 ? 0 : extra_slot, extra_value,
                    reinterpret_cast<uint64_t*>(version_local), version_slot);
  check_launch("psb_signal_kernel launch");
}

void wait_flags(uint64_t signal_local, int slot0, uint32_t mask, uint64_t want, double timeout_s, uint64_t stream) {
  psb_launch_wait(pick_stream(stream), reinterpret_cast<const uint64_t*>(signal_local), slot0, mask, want,
                  (unsigned long long)(timeout_s * 1e9));
  check_launch("psb_wait_kernel launch");
}

void select_ready(uint64_t signal_local, uint64_t consumed, uint32_t cand_mask, int quota, uint64_t out, double timeout_s,
                  uint64_t version, const std::vector<uint64_t>& begin_targets, uint64_t stream) {
  std::vector<uint64_t*> bt;
  for (auto p : begin_targets) bt.push_back(reinterpret_cast<uint64_t*>(p));
  psb_launch_select(pick_stream(stream), reinterpret_cast<const uint64_t*>(signal_local), reinterpret_cast<uint64_t*>(consumed),
                    cand_mask, quota, reinterpret_cast<uint64_t*>(out), (unsigned long long)(timeout_s * 1e9), version,
                    bt.data(), (int)bt.size());
  check_launch("psb_select_kernel launch");
}

void snapshot(uint64_t signal_local, uint64_t stage, uint64_t shadow, uint64_t params, uint64_t nbytes, uint64_t scratch,
              int attempts, uint64_t stream) {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  psb_launch_snapshot(pick_stream(stream), reinterpret_cast<const uint64_t*>(signal_local), reinterpret_cast<const void*>(stage),
                      reinterpret_cast<void*>(shadow), reinterpret_cast<void*>(params), (size_t)nbytes,
                      reinterpret_cast<unsigned long long*>(scratch), attempts, sms);
  check_launch("psb_snapshot launch");
}

}  // namespace

void bind_gemm(py::module_& m);   // gemm_bindings.cpp

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "pytorch_ps_mpi_b200 CUDA runtime: VMM symmetric memory + sm_100a kernels";
  m.attr("TILE") = PSB_TILE;
  m.attr("SIGNAL_SLOTS") = PSB_SIGNAL_SLOTS;
  m.attr("SIG_GRAD_READY") = SIG_GRAD_READY;
  m.attr("SIG_PARAMS_READY") = SIG_PARAMS_READY;
  m.attr("SIG_CONSUMED") = SIG_CONSUMED;
  m.attr("SIG_ERROR") = SIG_ERROR;
  m.attr("SIG_VERSION") = SIG_VERSION;
  m.attr("SIG_ACK") = SIG_ACK;
  m.attr("SIG_GRAD_VERSION") = SIG_GRAD_VERSION;
  m.attr("MAX_RANKS") = PSB_MAX_RANKS;
  m.attr("MAX_GROUPS") = PSB_MAX_GROUPS;

  py::class_<psb::SymmBlock, std::shared_ptr<psb::SymmBlock>>(m, "SymmBlock")
      .def(py::init<int, int, int, size_t, const std::string&>(), py::arg("rank"), py::arg("world"), py::arg("device"),
           py::arg("bytes"), py::arg("sock_prefix"), py::call_guard<py::gil_scoped_release>())
      .def("map_peers", &psb::SymmBlock::map_peers, py::call_guard<py::gil_scoped_release>())
      .def("mc_supported", &psb::SymmBlock::mc_supported)
      .def("mc_create", &psb::SymmBlock::mc_create)
      .def("mc_import", &psb::SymmBlock::mc_import, py::call_guard<py::gil_scoped_release>())
      .def("mc_add_device", &psb::SymmBlock::mc_add_device)
      .def("mc_bind_and_map", &psb::SymmBlock::mc_bind_and_map)
      .def("stop_server", &psb::SymmBlock::stop_server, py::call_guard<py::gil_scoped_release>())
      .def_property_readonly("size", &psb::SymmBlock::size)
      .def_property_readonly("rank", &psb::SymmBlock::rank)
      .def_property_readonly("world", &psb::SymmBlock::world)
      .def_property_readonly("device", &psb::SymmBlock::device)
      .def_property_readonly("ptrs", &psb::SymmBlock::ptrs)
      .def_property_readonly("mc_ptr", &psb::SymmBlock::mc_ptr)
      .def_property_readonly("last_error", &psb::SymmBlock::last_error)
      .def("ptr", &psb::SymmBlock::ptr);

  m.def("blob_tensor",
        [](uint64_t ptr, int64_t nbytes, int device, py::object owner) {
          return blob_tensor(ptr, {nbytes}, at::kByte, device, std::move(owner));
        },
        "uint8 tensor view over raw device memory (owner is kept alive by the tensor); .view(dtype) it in Python");

  py::class_<UpdatePlan>(m, "UpdatePlan")
      .def(py::init<>())
      .def_readwrite("kind", &UpdatePlan::kind)
      .def_readwrite("wire", &UpdatePlan::wire)
      .def_readwrite("opt", &UpdatePlan::opt)
      .def_readwrite("grid", &UpdatePlan::grid)
      .def_readwrite("window_bytes", &UpdatePlan::window_bytes)
      .def("set_rank_ptrs", &UpdatePlan::set_rank_ptrs)
      .def("configure",
           [](UpdatePlan& p, int world, int rank, int ntiles, int bytes_per_tile, int cap, int param_dt, int bcast, int reduce,
              uint64_t param_mc, uint64_t wire_mc, uint64_t param_local, uint64_t master, uint64_t buf0, uint64_t buf1,
              uint64_t buf2, uint64_t tiles, uint64_t signal_local, uint64_t done_counter, uint64_t stats) {
             p.a.world = world, p.a.rank = rank, p.a.ntiles = ntiles, p.a.bytes_per_tile = bytes_per_tile, p.a.cap = cap;
             p.a.param_dt = param_dt, p.a.bcast = bcast, p.a.reduce = reduce;
             p.a.param_mc = reinterpret_cast<void*>(param_mc);
             p.a.wire_mc = reinterpret_cast<const void*>(wire_mc);
             p.a.param_local = reinterpret_cast<void*>(param_local);
             p.a.master = reinterpret_cast<float*>(master);
             p.a.buf0 = reinterpret_cast<float*>(buf0);
             p.a.buf1 = reinterpret_cast<float*>(buf1);
             p.a.buf2 = reinterpret_cast<float*>(buf2);
             p.a.tiles = reinterpret_cast<const TileInfo*>(tiles);
             p.a.signal_local = reinterpret_cast<uint64_t*>(signal_local);
             p.a.done_counter = reinterpret_cast<unsigned int*>(done_counter);
             p.a.stats = reinterpret_cast<uint32_t*>(stats);
           })
      .def("launch", &UpdatePlan::launch, py::arg("epoch"), py::arg("groups"), py::arg("contrib_mask"),
           py::arg("inv_count"), py::arg("wait_grads"), py::arg("signal_mode"), py::arg("ack_mask") = 0,
           py::arg("version") = 0, py::arg("select_out") = 0, py::arg("average_dynamic") = 0, py::arg("active_ptr") = 0,
           py::arg("timeout_s") = 30.0, py::arg("wait_mask") = 0xffffffffu, py::arg("stream") = 0,
           py::arg("tile_begin") = 0, py::arg("tile_end") = -1, py::arg("wait_value") = 0, py::arg("param_hyper") = 0);

  m.def("update_max_grid", &psb_update_max_grid);
  m.def("launch_count", []() { return (uint64_t)psb_launch_count(); }, "kernels of ours launched by this process so far");
  m.def("encode", &encode, py::arg("kind"), py::arg("wire"), py::arg("grads"), py::arg("first_tile"), py::arg("ntiles"),
        py::arg("param_idx"), py::arg("tiles_ptr"), py::arg("wire_ptr"), py::arg("scales_ptr"), py::arg("amax_ptr"),
        py::arg("residual_ptr"), py::arg("bytes_per_tile"), py::arg("cap"), py::arg("ratio"),
        py::arg("sig_targets") = std::vector<uint64_t>{}, py::arg("sig_slot") = 0, py::arg("sig_value") = 0,
        py::arg("sig_counter") = 0, py::arg("stream") = 0, py::arg("levels") = 0, py::arg("seed") = 0, py::arg("rng_step") = 0,
        py::arg("rank") = 0);
  m.def("signal", &signal, py::arg("targets"), py::arg("slot"), py::arg("value"), py::arg("extra_slot") = -1,
        py::arg("extra_value") = 0, py::arg("stream") = 0, py::arg("version_local") = 0, py::arg("version_slot") = 0);
  m.def("wait_flags", &wait_flags, py::arg("signal_local"), py::arg("slot0"), py::arg("mask"), py::arg("want"),
        py::arg("timeout_s"), py::arg("stream") = 0);
  m.def("select_ready", &select_ready, py::arg("signal_local"), py::arg("consumed"), py::arg("cand_mask"), py::arg("quota"),
        py::arg("out"), py::arg("timeout_s"), py::arg("version") = 0, py::arg("begin_targets") = std::vector<uint64_t>{},
        py::arg("stream") = 0);
  m.def("snapshot", &snapshot, py::arg("signal_local"), py::arg("stage"), py::arg("shadow"), py::arg("params"), py::arg("nbytes"),
        py::arg("scratch"), py::arg("attempts") = 2, py::arg("stream") = 0,
        "consistent reads: device-side sequence-lock snapshot staging → shadow → parameters (no host reads)");
  m.attr("SIG_STAGE_BEGIN") = SIG_STAGE_BEGIN;
  m.attr("SIG_SEEN_VERSION") = SIG_SEEN_VERSION;
  bind_gemm(m);
}
