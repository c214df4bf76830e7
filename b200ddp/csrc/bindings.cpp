// Python bindings.  The only translation unit that sees torch headers.  Which reference call site each op stands in for is
// documented on the Python side (b200ddp/ops/functional.py, parallel/peer.py, optim/sgd.py) and in docs/INVENTORY.md.
#include <torch/extension.h>
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>

#include "comm.h"
#include "comm_kernels.cuh"
#include "conv.h"
#include "gemm.h"
#include "ops.h"
#include "peer_mem.h"
#include "reducer.h"

namespace py = pybind11;
using namespace b200;

namespace {

DType dtype_of(const at::Tensor& t) {
  switch (t.scalar_type()) {
    case at::kFloat: return DType::F32;
    case at::kBFloat16: return DType::BF16;
    case at::kByte: return DType::U8;
    case at::kLong: return DType::I64;
    default: throw std::runtime_error("b200ddp: unsupported dtype " + std::string(c10::toString(t.scalar_type())));
  }
}

cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }

void check_cuda(const at::Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor");
  TORCH_CHECK(t.is_contiguous() || t.is_non_overlapping_and_dense(), name, " must be dense");
}

CommCtx make_ctx(PeerArena& a, size_t pad_off, double timeout_s) {
  CommCtx c;
  c.base = a.base();
  c.mc_base = a.mc_base();
  c.stride = a.stride();
  c.pad_off = pad_off;
  c.error_word = a.error_word_dev();
  c.timeout_ns = (unsigned long long)(timeout_s * 1e9);
  c.rank = a.rank();
  c.world = a.world();
  return c;
}

// Standalone fused allreduce of a list of tensors treated as one flat bucket (tests, sweeps,
// PeerCollectives.allreduce_).  Slots are padded to 8 elements, a flags tail is appended.
void allreduce_tensors(PeerArena& arena, const std::vector<at::Tensor>& tensors, const std::string& wire, int algo,
                       int blocks, size_t stage_off, size_t stage_bytes, double scale, int pad_set, double timeout_s,
                       c10::optional<at::Tensor> sq_partials) {
  TORCH_CHECK(!tensors.empty() && (int)tensors.size() <= kMaxBucketTensors, "allreduce_tensors: 1..", kMaxBucketTensors, " tensors");
  const DType in_dt = dtype_of(tensors[0]);
  const DType wire_dt = wire == "fp32" ? DType::F32 : DType::BF16;
  BucketTable tab;
  uint32_t off = 0;
  tab.count = (int)tensors.size();
  for (int k = 0; k < tab.count; ++k) {
    const at::Tensor& t = tensors[k];
    check_cuda(t, "tensor");
    TORCH_CHECK(dtype_of(t) == in_dt, "allreduce_tensors: mixed dtypes in one bucket");
    tab.t[k].ptr = t.data_ptr();
    tab.t[k].numel = (uint32_t)t.numel();
    tab.t[k].off = off;
    off += (uint32_t)((t.numel() + 7) / 8 * 8);
  }
  tab.data_elems = off;
  tab.total_elems = off + (uint32_t)((tab.count + 7) / 8 * 8);
  tab._pad = 0;
  TORCH_CHECK((size_t)tab.total_elems * dtype_size(wire_dt) <= stage_bytes, "allreduce_tensors: staging region too small");
  CommCtx ctx = make_ctx(arena, (size_t)pad_set * kPadSetBytes, timeout_s);
  if (algo == kAlgoAuto) algo = arena.has_multicast() ? kAlgoNvls : kAlgoTwoShot;
  float* sq = sq_partials.has_value() ? sq_partials->data_ptr<float>() : nullptr;
  launch_bucket_allreduce(ctx, tab, stage_off, in_dt, wire_dt, algo, blocks, nullptr, sq, nullptr, (float)scale,
                          /*scatter=*/true, cur_stream());
}

// Broadcast arbitrary tensors from `src`; chunked through the staging region.
int broadcast_tensors(PeerArena& arena, const std::vector<at::Tensor>& tensors, int src, size_t stage_off,
                      size_t stage_bytes, bool use_mc, int blocks, int pad_set, double timeout_s) {
  CommCtx ctx = make_ctx(arena, (size_t)pad_set * kPadSetBytes, timeout_s);
  int launches = 0;
  size_t i = 0;
  const size_t n = tensors.size();
  // a tensor larger than the staging region is sent in pieces
  size_t piece_off = 0;
  while (i < n) {
    BucketTable tab;
    tab.count = 0;
    uint32_t off = 0;
    while (i < n && tab.count < kMaxBucketTensors) {
      const at::Tensor& t = tensors[i];
      check_cuda(t, "tensor");
      const size_t nbytes = (size_t)t.numel() * t.element_size() - piece_off;
      const size_t room = stage_bytes - off;
      if (room < 16) break;
      size_t take = nbytes <= room ? nbytes : (room / 16) * 16;
      if (take == 0) break;
      tab.t[tab.count].ptr = static_cast<char*>(t.data_ptr()) + piece_off;
      tab.t[tab.count].numel = (uint32_t)take;
      tab.t[tab.count].off = off;
      ++tab.count;
      off += (uint32_t)((take + 15) / 16 * 16);
      if (take == nbytes) { ++i; piece_off = 0; } else { piece_off += take; break; }
    }
    if (tab.count == 0) throw std::runtime_error("broadcast_tensors: staging region too small");
    tab.data_elems = off;
    tab.total_elems = off;
    tab._pad = 0;
    launch_peer_broadcast(ctx, tab, stage_off, src, use_mc, blocks, cur_stream());
    ++launches;
  }
  return launches;
}

// ---- optimizer ---------------------------------------------------------------------------------
struct SgdPlan {
  std::vector<uintptr_t> params;
  std::vector<long long> numels, flat_offs;
  DType p_dtype, g_dtype;
  int total_blocks = 0;
  SgdPlan(std::vector<uintptr_t> p, std::vector<long long> n, std::vector<long long> fo, int pd, int gd)
      : params(std::move(p)), numels(std::move(n)), flat_offs(std::move(fo)), p_dtype((DType)pd), g_dtype((DType)gd) {
    for (auto v : numels) total_blocks += ceil_div(v, kOptChunk);
  }
  template <typename F>
  void for_each_table(const std::vector<uintptr_t>& grads, F&& fn) const {
    size_t i = 0;
    int block_base = 0;
    while (i < params.size()) {
      OptTable tab;
      tab.count = 0;
      tab.total_blocks = 0;
      while (i < params.size() && tab.count < kMaxOptTensors) {
        OptSlot& s = tab.t[tab.count++];
        s.p = reinterpret_cast<void*>(params[i]);
        s.g = reinterpret_cast<const void*>(grads[i]);
        s.flat_off = (unsigned long long)flat_offs[i];
        s.numel = (uint32_t)numels[i];
        s.blk0 = (uint32_t)tab.total_blocks;
        tab.total_blocks += ceil_div(numels[i], kOptChunk);
        ++i;
      }
      fn(tab, block_base);
      block_base += tab.total_blocks;
    }
  }
  int sqnorm(const std::vector<uintptr_t>& grads, uintptr_t partials, uintptr_t stream) const {
    TORCH_CHECK(grads.size() == params.size(), "SgdPlan: gradient list length mismatch");
    for_each_table(grads, [&](const OptTable& tab, int base) {
      launch_multi_sqnorm(tab, g_dtype, reinterpret_cast<float*>(partials) + base, reinterpret_cast<cudaStream_t>(stream));
    });
    return total_blocks;
  }
  void step(const std::vector<uintptr_t>& grads, uintptr_t lr, uintptr_t clip_coef, uintptr_t master, uintptr_t mom,
            uintptr_t step_count, double momentum, double dampening, double weight_decay, double grad_scale, bool nesterov,
            bool zero_grad, uintptr_t stream) const {
    TORCH_CHECK(grads.size() == params.size(), "SgdPlan: gradient list length mismatch");
    SgdHyper h;
    h.lr = reinterpret_cast<const float*>(lr);
    h.clip_coef = reinterpret_cast<const float*>(clip_coef);
    h.master = reinterpret_cast<float*>(master);
    h.momentum_buf = reinterpret_cast<float*>(mom);
    h.step_count = reinterpret_cast<const int*>(step_count);
    h.momentum = (float)momentum;
    h.dampening = (float)dampening;
    h.weight_decay = (float)weight_decay;
    h.grad_scale = (float)grad_scale;
    h.nesterov = nesterov ? 1 : 0;
    h.zero_grad = zero_grad ? 1 : 0;
    for_each_table(grads, [&](const OptTable& tab, int) {
      launch_multi_sgd(tab, p_dtype, g_dtype, h, reinterpret_cast<cudaStream_t>(stream));
    });
  }
};

// ---- fused BatchNorm: what the plain and the from-partials entry points share ------------------------------------------
template <typename T>
T* opt_ptr(const c10::optional<at::Tensor>& t) { return t.has_value() ? t->data_ptr<T>() : nullptr; }

// Checked input x [N, C, H, W] channels_last (+ residual) and the outputs: y, stats = [4, C] (save_mean, save_rstd, scale,
// shift) and, with relu, the [R, C/8] ReLU bitmask.
struct BnForwardIo {
  int R, C;
  const void* res;
  at::Tensor y, stats, mask;
};
BnForwardIo bn_forward_io(const char* op, const at::Tensor& x, const c10::optional<at::Tensor>& residual, const at::Tensor& gamma,
                          const at::Tensor& beta, bool relu) {
  check_cuda(x, "x");
  TORCH_CHECK(x.dim() == 4 && x.is_contiguous(at::MemoryFormat::ChannelsLast), op, ": x must be 4-D channels_last");
  TORCH_CHECK(gamma.scalar_type() == at::kFloat && beta.scalar_type() == at::kFloat, op, ": fp32 affine parameters");
  BnForwardIo io;
  io.C = (int)x.size(1);
  io.R = (int)(x.numel() / io.C);
  io.res = nullptr;
  if (residual.has_value()) {
    TORCH_CHECK(residual->sizes() == x.sizes() && residual->dtype() == x.dtype() && residual->is_contiguous(at::MemoryFormat::ChannelsLast),
                op, ": residual must match x (shape, dtype, channels_last)");
    io.res = residual->data_ptr();
  }
  io.y = at::empty_like(x);
  io.stats = at::empty({4, io.C}, x.options().dtype(at::kFloat));
  if (relu) io.mask = at::empty({(int64_t)io.R, (int64_t)(io.C / 8)}, x.options().dtype(at::kByte));
  return io;
}

// Checked ReLU bitmask and the outputs: dx, dres (when asked for) and dparams = [rows, C] (dgamma, dbeta, then per-entry rows).
struct BnBackwardIo {
  int R, C;
  const void* relu_mask;
  at::Tensor dx, dres, dparams;
};
BnBackwardIo bn_backward_io(const char* op, const at::Tensor& dy, const at::Tensor& x, const c10::optional<at::Tensor>& y, bool relu,
                            bool need_dres, int param_rows) {
  check_cuda(dy, "dy");
  TORCH_CHECK(!relu || (y.has_value() && y->scalar_type() == at::kByte), op, ": needs the ReLU bitmask written by bn_forward");
  BnBackwardIo io;
  io.C = (int)x.size(1);
  io.R = (int)(x.numel() / io.C);
  io.relu_mask = relu ? y->data_ptr() : nullptr;
  io.dx = at::empty_like(x);
  if (need_dres) io.dres = at::empty_like(x);
  io.dparams = at::empty({param_rows, io.C}, x.options().dtype(at::kFloat));
  return io;
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "b200ddp native extension (sm_100a)";
  m.attr("MAX_BUCKET_TENSORS") = kMaxBucketTensors;
  m.attr("MAX_COMM_BLOCKS") = kMaxCommBlocks;
  m.attr("SIGNAL_BYTES") = (long long)kSignalBytes;
  m.attr("ALGO_AUTO") = (int)kAlgoAuto;
  m.attr("ALGO_ONE_SHOT") = (int)kAlgoOneShot;
  m.attr("ALGO_TWO_SHOT") = (int)kAlgoTwoShot;
  m.attr("ALGO_NVLS") = (int)kAlgoNvls;
  m.attr("ALGO_NVLS_ONE_SHOT") = (int)kAlgoNvlsOneShot;

  m.def("launch_count", []() { return (long long)launch_counter().load(); });
  m.def("assign_by_size", &assign_by_size, py::arg("nbytes"), py::arg("keys"), py::arg("limits"), py::arg("max_tensors") = 0);

  py::class_<PeerArena>(m, "PeerArena")
      .def(py::init<int, int, int, size_t, const std::string&>())
      .def("bind_socket", &PeerArena::bind_socket)
      .def("exchange", &PeerArena::exchange, py::call_guard<py::gil_scoped_release>())
      .def("multicast_supported", &PeerArena::multicast_supported)
      .def("multicast_create", &PeerArena::multicast_create, py::call_guard<py::gil_scoped_release>())
      .def("multicast_add_device", &PeerArena::multicast_add_device)
      .def("multicast_bind", &PeerArena::multicast_bind)
      .def("disable_multicast", &PeerArena::disable_multicast)
      .def("has_multicast", &PeerArena::has_multicast)
      .def("alloc", &PeerArena::alloc, py::arg("nbytes"), py::arg("align") = 256)
      .def("used", &PeerArena::used)
      .def("rewind", &PeerArena::rewind)
      .def("bytes", &PeerArena::bytes)
      .def("rank", &PeerArena::rank)
      .def("world", &PeerArena::world)
      .def("local_ptr", [](PeerArena& a) { return (uintptr_t)a.local(); })
      .def("peer_ptr", [](PeerArena& a, int r) { return (uintptr_t)a.peer(r); })
      .def("mc_ptr", [](PeerArena& a) { return (uintptr_t)a.mc_base(); })
      .def("check_error", &PeerArena::check_error)
      .def("clear_error", &PeerArena::clear_error)
      .def("close", &PeerArena::close);

  m.def("allreduce_tensors", &allreduce_tensors, py::arg("arena"), py::arg("tensors"), py::arg("wire") = "bf16",
        py::arg("algo") = (int)kAlgoAuto, py::arg("blocks") = 32, py::arg("stage_off"), py::arg("stage_bytes"),
        py::arg("scale") = 1.0, py::arg("pad_set") = 1, py::arg("timeout_s") = 30.0, py::arg("sq_partials") = py::none());
  m.def("arena_tensor", [](PeerArena& a, size_t offset, int64_t numel, int dtype_code) {
    auto dt = dtype_code == 1 ? at::kBFloat16 : dtype_code == 2 ? at::kByte : at::kFloat;
    auto opts = at::TensorOptions().dtype(dt).device(at::kCUDA, a.device());
    return at::from_blob(a.local() + offset, {numel}, [](void*) {}, opts);
  });
  m.def("allreduce_symmetric", [](PeerArena& a, size_t buf_off, int64_t numel, int dtype_code, int algo, int blocks, double scale,
                                  int pad_set, double timeout_s) {
    CommCtx ctx = make_ctx(a, (size_t)pad_set * kPadSetBytes, timeout_s);
    if (algo == kAlgoAuto) algo = a.has_multicast() ? kAlgoNvls : kAlgoTwoShot;
    launch_symmetric_allreduce(ctx, buf_off, (size_t)numel, (DType)dtype_code, algo, blocks, (float)scale, cur_stream());
  });
  m.def("broadcast_tensors", &broadcast_tensors, py::arg("arena"), py::arg("tensors"), py::arg("src") = 0, py::arg("stage_off"),
        py::arg("stage_bytes"), py::arg("use_mc") = false, py::arg("blocks") = 32, py::arg("pad_set") = 1,
        py::arg("timeout_s") = 30.0);
  m.def("peer_pull", [](PeerArena& a, int peer, size_t src_off, at::Tensor dst, size_t bytes, int blocks) {
    launch_peer_pull(make_ctx(a, 0, 30.0), peer, src_off, dst.data_ptr(), bytes, blocks, cur_stream());
  });
  m.def("peer_push", [](PeerArena& a, int peer, size_t dst_off, at::Tensor src, size_t bytes, int blocks) {
    launch_peer_push(make_ctx(a, 0, 30.0), peer, dst_off, src.data_ptr(), bytes, blocks, cur_stream());
  });
  m.def("peer_barrier", [](PeerArena& a, int blocks, int pad_set, double timeout_s) {
    launch_peer_barrier(make_ctx(a, (size_t)pad_set * kPadSetBytes, timeout_s), blocks, cur_stream());
  }, py::arg("arena"), py::arg("blocks") = 1, py::arg("pad_set") = 1, py::arg("timeout_s") = 30.0);

  py::class_<BucketPlan>(m, "BucketPlan")
      .def(py::init<>())
      .def_readwrite("param_indices", &BucketPlan::param_indices)
      .def_readwrite("numels", &BucketPlan::numels)
      .def_readwrite("offsets", &BucketPlan::offsets)
      .def_readwrite("data_elems", &BucketPlan::data_elems)
      .def_readwrite("total_elems", &BucketPlan::total_elems)
      .def_readwrite("grad_dtype", &BucketPlan::grad_dtype)
      .def_readwrite("wire_dtype", &BucketPlan::wire_dtype)
      .def_readwrite("tail", &BucketPlan::tail);

  py::class_<Reducer>(m, "Reducer")
      .def(py::init([](PeerArena& arena, std::vector<BucketPlan> plans, int num_params, int algo,
                       int max_blocks, int tail_blocks, long long one_shot_max_bytes, bool as_view, bool find_unused, double extra_scale,
                       double timeout_s, int serial, int wide_blocks, long long tail_one_shot_max_bytes) {
             ReducerOptions o;
             o.algo = algo;
             o.max_blocks = max_blocks;
             o.tail_blocks = tail_blocks;
             o.one_shot_max_bytes = one_shot_max_bytes;
             o.as_view = as_view;
             o.find_unused = find_unused;
             o.extra_scale = (float)extra_scale;
             o.timeout_s = timeout_s;
             o.serial = serial;
             o.wide_blocks = wide_blocks;
             o.tail_one_shot_max_bytes = tail_one_shot_max_bytes;
             return std::make_unique<Reducer>(&arena, std::move(plans), num_params, o);
           }),
           py::keep_alive<1, 2>())
      .def("num_buckets", &Reducer::num_buckets)
      .def("bucket_blocks", &Reducer::bucket_blocks)
      .def("bucket_algo", &Reducer::bucket_algo)
      .def("set_flat_out", &Reducer::set_flat_out)
      .def("set_sq_partials", &Reducer::set_sq_partials)
      .def("reset", &Reducer::reset)
      .def("mark_ready", &Reducer::mark_ready)
      .def("finalize", &Reducer::finalize)
      .def("read_used_flags", &Reducer::read_used_flags)
      .def("synchronize", &Reducer::synchronize)
      .def("comm_stream", &Reducer::comm_stream)
      .def("runs_inline", &Reducer::runs_inline)
      .def("note_comm_stream_used", &Reducer::note_comm_stream_used)
      .def("set_eager_inline", &Reducer::set_eager_inline)
      .def("error_code", &Reducer::error_code)
      .def_readonly("launches", &Reducer::launches)
      .def_readonly("bytes_on_wire", &Reducer::bytes_on_wire)
      .def_readonly("iterations", &Reducer::iterations)
      .def_readonly("ready_order", &Reducer::ready_order);

  py::class_<SgdPlan>(m, "SgdPlan")
      .def(py::init<std::vector<uintptr_t>, std::vector<long long>, std::vector<long long>, int, int>())
      .def_readonly("total_blocks", &SgdPlan::total_blocks)
      .def("sqnorm", &SgdPlan::sqnorm)
      .def("step", &SgdPlan::step);
  m.def("clip_coef", [](at::Tensor partials, int n, double max_norm, double grad_scale, at::Tensor coef, at::Tensor norm) {
    launch_clip_coef(partials.data_ptr<float>(), n, (float)max_norm, (float)grad_scale, coef.data_ptr<float>(),
                     norm.data_ptr<float>(), cur_stream());
  });

  // ---- losses -----------------------------------------------------------------------------------
  m.def("mse_fwd_bwd", [](at::Tensor out, at::Tensor target, double gscale) {
    check_cuda(out, "out"); check_cuda(target, "target");
    TORCH_CHECK(out.is_contiguous() && target.is_contiguous() && out.sizes() == target.sizes() && out.dtype() == target.dtype(),
                "mse_fwd_bwd: out/target must be contiguous with equal shape and dtype");
    c10::cuda::CUDAGuard guard(out.device());
    const size_t n = (size_t)out.numel();
    const int blocks = mse_blocks(n);
    at::Tensor loss = at::empty({}, out.options().dtype(at::kFloat));
    at::Tensor dout = at::empty_like(out);
    at::Tensor scratch = at::zeros({blocks + 1}, out.options().dtype(at::kFloat));
    launch_mse_fwd_bwd(out.data_ptr(), target.data_ptr(), dtype_of(out), n, (float)gscale, loss.data_ptr<float>(), dout.data_ptr(),
                       scratch.data_ptr<float>(), blocks, cur_stream());
    return std::make_tuple(loss, dout);
  });
  m.def("xent_fwd_bwd", [](at::Tensor logits, at::Tensor targets, long long ignore_index, double gscale) {
    check_cuda(logits, "logits"); check_cuda(targets, "targets");
    TORCH_CHECK(logits.dim() == 2 && logits.is_contiguous() && targets.is_contiguous() && targets.scalar_type() == at::kLong &&
                targets.numel() == logits.size(0), "xent_fwd_bwd: logits [rows, cols] contiguous, targets int64 [rows]");
    c10::cuda::CUDAGuard guard(logits.device());
    const int rows = (int)logits.size(0), cols = (int)logits.size(1);
    at::Tensor loss = at::empty({}, logits.options().dtype(at::kFloat));
    at::Tensor row_loss = at::empty({rows + 1}, logits.options().dtype(at::kFloat));
    at::Tensor dlogits = at::empty_like(logits);
    launch_xent_fwd_bwd(logits.data_ptr(), targets.data_ptr<int64_t>() ? (const long long*)targets.data_ptr<int64_t>() : nullptr,
                        dtype_of(logits), rows, cols, ignore_index, (float)gscale, row_loss.data_ptr<float>(), loss.data_ptr<float>(),
                        dlogits.data_ptr(), cur_stream());
    return std::make_tuple(loss, dlogits);
  });

  m.def("gelu_fwd", [](at::Tensor pre) {
    check_cuda(pre, "pre");
    TORCH_CHECK(pre.is_contiguous(), "gelu_fwd: contiguous input");
    c10::cuda::CUDAGuard guard(pre.device());
    at::Tensor out = at::empty_like(pre);
    launch_gelu(pre.data_ptr(), nullptr, out.data_ptr(), dtype_of(pre), (size_t)pre.numel(), false, cur_stream());
    return out;
  });
  m.def("gelu_bwd", [](at::Tensor dy, at::Tensor pre) {
    check_cuda(pre, "pre");
    TORCH_CHECK(pre.is_contiguous() && dy.is_contiguous() && dy.dtype() == pre.dtype() && dy.numel() == pre.numel(), "gelu_bwd: matching contiguous tensors");
    c10::cuda::CUDAGuard guard(pre.device());
    at::Tensor out = at::empty_like(pre);
    launch_gelu(pre.data_ptr(), dy.data_ptr(), out.data_ptr(), dtype_of(pre), (size_t)pre.numel(), true, cur_stream());
    return out;
  });

  // ---- layer norm -------------------------------------------------------------------------------
  m.def("layernorm_fwd", [](at::Tensor x, at::Tensor gamma, at::Tensor beta, double eps) {
    check_cuda(x, "x");
    TORCH_CHECK(x.is_contiguous() && gamma.is_contiguous() && beta.is_contiguous(), "layernorm_fwd: contiguous inputs");
    TORCH_CHECK(gamma.dtype() == x.dtype() && beta.dtype() == x.dtype(), "layernorm_fwd: gamma/beta dtype must match x");
    c10::cuda::CUDAGuard guard(x.device());
    const int cols = (int)x.size(-1);
    const int rows = (int)(x.numel() / cols);
    at::Tensor y = at::empty_like(x);
    at::Tensor mean = at::empty({rows}, x.options().dtype(at::kFloat));
    at::Tensor rstd = at::empty({rows}, x.options().dtype(at::kFloat));
    launch_layernorm_fwd(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), dtype_of(x), rows, cols, (float)eps, y.data_ptr(),
                         mean.data_ptr<float>(), rstd.data_ptr<float>(), cur_stream());
    return std::make_tuple(y, mean, rstd);
  });
  m.def("layernorm_bwd", [](at::Tensor dy, at::Tensor x, at::Tensor gamma, at::Tensor mean, at::Tensor rstd) {
    check_cuda(dy, "dy");
    TORCH_CHECK(dy.is_contiguous() && x.is_contiguous(), "layernorm_bwd: contiguous inputs");
    c10::cuda::CUDAGuard guard(x.device());
    const int cols = (int)x.size(-1);
    const int rows = (int)(x.numel() / cols);
    const int parts = layernorm_partial_rows(rows);
    at::Tensor dx = at::empty_like(x);
    at::Tensor dgp = at::empty({parts, cols}, x.options().dtype(at::kFloat));
    at::Tensor dbp = at::empty({parts, cols}, x.options().dtype(at::kFloat));
    at::Tensor dgamma = at::empty_like(gamma);
    at::Tensor dbeta = at::empty_like(gamma);
    launch_layernorm_bwd(dy.data_ptr(), x.data_ptr(), gamma.data_ptr(), mean.data_ptr<float>(), rstd.data_ptr<float>(), dtype_of(x),
                         rows, cols, dx.data_ptr(), dgp.data_ptr<float>(), dbp.data_ptr<float>(), parts, dgamma.data_ptr(),
                         dbeta.data_ptr(), cur_stream());
    return std::make_tuple(dx, dgamma, dbeta);
  });

  // ---- linears ----------------------------------------------------------------------------------
  m.def("small_linear_fwd", [](at::Tensor x, at::Tensor w, c10::optional<at::Tensor> b, bool relu) {
    check_cuda(x, "x");
    TORCH_CHECK(x.scalar_type() == at::kFloat && w.scalar_type() == at::kFloat && x.is_contiguous() && w.is_contiguous(),
                "small_linear_fwd: fp32 contiguous");
    c10::cuda::CUDAGuard guard(x.device());
    const int K = (int)x.size(-1), N = (int)w.size(0);
    const int M = (int)(x.numel() / K);
    auto sizes = x.sizes().vec();
    sizes.back() = N;
    at::Tensor y = at::empty(sizes, x.options());
    launch_small_linear_fwd(x.data_ptr<float>(), w.data_ptr<float>(), b.has_value() ? b->data_ptr<float>() : nullptr,
                            y.data_ptr<float>(), M, N, K, relu ? 1 : 0, cur_stream());
    return y;
  });
  m.def("small_linear_bwd", [](at::Tensor dy, at::Tensor x, at::Tensor w, at::Tensor y, bool relu, bool need_dx, bool has_bias) {
    check_cuda(dy, "dy");
    c10::cuda::CUDAGuard guard(x.device());
    const int K = (int)x.size(-1), N = (int)w.size(0);
    const int M = (int)(x.numel() / K);
    at::Tensor dyc = dy.contiguous();
    at::Tensor dx = need_dx ? at::empty_like(x) : at::Tensor();
    at::Tensor dw = at::empty_like(w);
    at::Tensor db = has_bias ? at::empty({N}, w.options()) : at::Tensor();
    launch_small_linear_bwd(dyc.data_ptr<float>(), x.data_ptr<float>(), w.data_ptr<float>(), y.data_ptr<float>(),
                            need_dx ? dx.data_ptr<float>() : nullptr, dw.data_ptr<float>(), has_bias ? db.data_ptr<float>() : nullptr,
                            M, N, K, relu ? 1 : 0, 0, cur_stream());
    return std::make_tuple(dx, dw, db);
  });

  // tcgen05 GEMM: D[M,N] = act(A[M,K] @ B[N,K]^T + bias) ; all bf16 row-major, fp32 accumulate in TMEM
  m.def("gemm_nt", [](at::Tensor a, at::Tensor b, c10::optional<at::Tensor> bias, int epilogue, c10::optional<at::Tensor> out) {
    check_cuda(a, "a"); check_cuda(b, "b");
    TORCH_CHECK(a.scalar_type() == at::kBFloat16 && b.scalar_type() == at::kBFloat16, "gemm_nt: bf16 operands");
    TORCH_CHECK(a.dim() == 2 && b.dim() == 2 && a.size(1) == b.size(1) && a.is_contiguous() && b.is_contiguous(),
                "gemm_nt: A [M,K], B [N,K], both K-major contiguous");
    c10::cuda::CUDAGuard guard(a.device());
    const int M = (int)a.size(0), K = (int)a.size(1), N = (int)b.size(0);
    at::Tensor d = out.has_value() ? *out : at::empty({M, N}, a.options());
    TORCH_CHECK(d.is_contiguous() && d.size(0) == M && d.size(1) == N, "gemm_nt: bad output");
    const void* bias_ptr = nullptr;
    if (bias.has_value()) {
      TORCH_CHECK(bias->scalar_type() == at::kBFloat16 && bias->numel() == N, "gemm_nt: bias bf16 [N]");
      bias_ptr = bias->data_ptr();
    }
    launch_gemm_nt_bf16(a.data_ptr(), b.data_ptr(), d.data_ptr(), bias_ptr, M, N, K, epilogue, dtype_of(d), cur_stream());
    return d;
  }, py::arg("a"), py::arg("b"), py::arg("bias") = py::none(), py::arg("epilogue") = 0, py::arg("out") = py::none());
  // general form: a_mn=false -> a is [M,K]; true -> a is stored [K,M].  b_mn=false -> b is [N,K]; true -> stored [K,N].
  m.def("gemm", [](at::Tensor a, at::Tensor b, c10::optional<at::Tensor> bias, bool a_mn, bool b_mn, int epilogue, bool out_fp32,
                   c10::optional<at::Tensor> out) {
    check_cuda(a, "a"); check_cuda(b, "b");
    TORCH_CHECK(a.scalar_type() == at::kBFloat16 && b.scalar_type() == at::kBFloat16, "gemm: bf16 operands");
    TORCH_CHECK(a.dim() == 2 && b.dim() == 2 && a.is_contiguous() && b.is_contiguous(), "gemm: 2-D contiguous operands");
    c10::cuda::CUDAGuard guard(a.device());
    const int M = (int)(a_mn ? a.size(1) : a.size(0)), K = (int)(a_mn ? a.size(0) : a.size(1));
    const int N = (int)(b_mn ? b.size(1) : b.size(0)), Kb = (int)(b_mn ? b.size(0) : b.size(1));
    TORCH_CHECK(K == Kb, "gemm: reduction dims differ (", K, " vs ", Kb, ")");
    bool accumulate = false;
    at::Tensor d;
    if (out.has_value()) { d = *out; accumulate = d.scalar_type() == at::kFloat && out_fp32; }
    else d = at::empty({M, N}, a.options().dtype(out_fp32 ? at::kFloat : at::kBFloat16));
    TORCH_CHECK(d.is_contiguous() && d.size(0) == M && d.size(1) == N, "gemm: bad output");
    const void* bias_ptr = nullptr;
    if (bias.has_value()) {
      TORCH_CHECK(bias->scalar_type() == at::kBFloat16 && bias->numel() == N, "gemm: bias bf16 [N]");
      bias_ptr = bias->data_ptr();
    }
    launch_gemm_bf16(a.data_ptr(), b.data_ptr(), d.data_ptr(), bias_ptr, M, N, K, a_mn, b_mn, epilogue, dtype_of(d), accumulate,
                     cur_stream());
    return d;
  }, py::arg("a"), py::arg("b"), py::arg("bias") = py::none(), py::arg("a_mn") = false, py::arg("b_mn") = false,
     py::arg("epilogue") = 0, py::arg("out_fp32") = false, py::arg("out") = py::none());
  // forward GEMM (a [M,K], b [N,K]) that also returns per-32-row partial column statistics of its output: [2][ceil(M/32)][N]
  m.def("gemm_stats", [](at::Tensor a, at::Tensor b) {
    check_cuda(a, "a"); check_cuda(b, "b");
    TORCH_CHECK(a.scalar_type() == at::kBFloat16 && b.scalar_type() == at::kBFloat16, "gemm_stats: bf16 operands");
    TORCH_CHECK(a.dim() == 2 && b.dim() == 2 && a.is_contiguous() && b.is_contiguous() && a.size(1) == b.size(1), "gemm_stats: [M,K] x [N,K]");
    c10::cuda::CUDAGuard guard(a.device());
    const int M = (int)a.size(0), K = (int)a.size(1), N = (int)b.size(0);
    at::Tensor d = at::empty({M, N}, a.options());
    at::Tensor stats = at::empty({2, (M + 31) / 32, N}, a.options().dtype(at::kFloat));
    launch_gemm_bf16(a.data_ptr(), b.data_ptr(), d.data_ptr(), nullptr, M, N, K, false, false, 0, DType::BF16, false, cur_stream(),
                     stats.data_ptr<float>());
    return std::make_tuple(d, stats);
  });
  m.def("gemm_supported", &gemm_shape_supported);
  m.def("set_gemm_cta_mode", &set_gemm_cta_mode);
  m.def("set_gemm_group_m", &set_gemm_group_m);
  m.def("set_gemm_tma_store", &set_gemm_tma_store);
  m.def("gemm_tile_order", [](int num_m, int num_n, int group_m) {
    // host mirror of the device rasterisation: tile id -> (m block, n block)
    std::vector<std::pair<int, int>> out((size_t)num_m * num_n);
    for (int t = 0; t < num_m * num_n; ++t) gemm_tile_coords(t, num_m, num_n, group_m, &out[t].first, &out[t].second);
    return out;
  });

  // ---- convolutions on tcgen05 (conv_tcgen05.cu / conv_wgrad_tcgen05.cu): channels_last bf16, stride 1, 1x1 or 3x3 ------
  m.def("conv_fprop", [](at::Tensor x, at::Tensor w, int stride, int pad, int mode, int block_n, int base_offset, bool stats,
                         c10::optional<at::Tensor> debug, int kc) {
    check_cuda(x, "x"); check_cuda(w, "w");
    TORCH_CHECK(x.scalar_type() == at::kBFloat16 && w.scalar_type() == at::kBFloat16, "conv_fprop: bf16 tensors");
    TORCH_CHECK(x.dim() == 4 && x.is_contiguous(at::MemoryFormat::ChannelsLast), "conv_fprop: x must be 4-D channels_last");
    TORCH_CHECK(w.dim() == 4 && w.size(1) == x.size(1) && w.is_contiguous(at::MemoryFormat::ChannelsLast), "conv_fprop: filter must be [K, C, R, S] channels_last");
    const int R = (int)w.size(2), S = (int)w.size(3);
    TORCH_CHECK(stride == 1 && R == S && pad == (R - 1) / 2, "conv_fprop: stride 1, 'same' padding");
    c10::cuda::CUDAGuard guard(x.device());
    const int N = (int)x.size(0), C = (int)x.size(1), H = (int)x.size(2), W = (int)x.size(3), K = (int)w.size(0);
    at::Tensor y = at::empty({N, K, H, W}, x.options().memory_format(at::MemoryFormat::ChannelsLast));
    ConvLaunchCfg cfg; cfg.mode = mode; cfg.block_n = block_n; cfg.set_base_offset = base_offset; cfg.kc = kc;
    if (debug.has_value()) { TORCH_CHECK(debug->scalar_type() == at::kLong && debug->numel() >= 16 && debug->is_cuda(), "debug: int64[16] cuda"); cfg.debug_counters = debug->data_ptr(); }
    at::Tensor st;
    float* stp = nullptr;
    if (stats) {
      const int groups = conv_stat_groups(N, H, W, C, K, R, S, cfg);
      TORCH_CHECK(groups > 0, "conv_fprop: no tile plan");
      st = at::empty({2, groups, K}, x.options().dtype(at::kFloat));
      stp = st.data_ptr<float>();
    }
    launch_conv_tap_gemm(x.data_ptr(), w.data_ptr(), y.data_ptr(), N, H, W, C, K, R, S, false, cfg, stp, cur_stream());
    return std::make_tuple(y, st);
  }, py::arg("x"), py::arg("w"), py::arg("stride") = 1, py::arg("pad") = 0, py::arg("mode") = -1, py::arg("block_n") = 0,
     py::arg("base_offset") = 0, py::arg("stats") = false, py::arg("debug") = py::none(), py::arg("kc") = 0);
  // optional epilogue fusion: addend [N,C,H,W] is added to dx; (bn_x, bn_mask, bn_stats) make the epilogue also emit the partial
  // sums of the BatchNorm backward that consumes dx (returned as the second tensor, [2, G, C]; empty otherwise)
  m.def("conv_dgrad", [](at::Tensor dy, at::Tensor w, int stride, int pad, int mode, int block_n, int base_offset, int kc,
                         c10::optional<at::Tensor> addend, c10::optional<at::Tensor> bn_x, c10::optional<at::Tensor> bn_mask,
                         c10::optional<at::Tensor> bn_stats) {
    check_cuda(dy, "dy"); check_cuda(w, "w");
    TORCH_CHECK(dy.scalar_type() == at::kBFloat16 && w.scalar_type() == at::kBFloat16, "conv_dgrad: bf16 tensors");
    TORCH_CHECK(dy.dim() == 4 && dy.is_contiguous(at::MemoryFormat::ChannelsLast), "conv_dgrad: dy must be 4-D channels_last");
    TORCH_CHECK(w.dim() == 4 && w.size(0) == dy.size(1) && w.is_contiguous(at::MemoryFormat::ChannelsLast), "conv_dgrad: filter must be [K, C, R, S] channels_last");
    const int R = (int)w.size(2), S = (int)w.size(3);
    TORCH_CHECK(stride == 1 && R == S && pad == (R - 1) / 2, "conv_dgrad: stride 1, 'same' padding");
    c10::cuda::CUDAGuard guard(dy.device());
    const int N = (int)dy.size(0), K = (int)dy.size(1), H = (int)dy.size(2), W = (int)dy.size(3), C = (int)w.size(1);
    at::Tensor dx = at::empty({N, C, H, W}, dy.options().memory_format(at::MemoryFormat::ChannelsLast));
    ConvLaunchCfg cfg; cfg.mode = mode; cfg.block_n = block_n; cfg.set_base_offset = base_offset; cfg.kc = kc;
    ConvBwdFusion fuse;
    bool any = false;
    at::Tensor part;
    float* pp = nullptr;
    if (addend.has_value()) {
      TORCH_CHECK(addend->sizes() == dx.sizes() && addend->scalar_type() == at::kBFloat16 && addend->is_contiguous(at::MemoryFormat::ChannelsLast),
                  "conv_dgrad: addend must match dx (bf16, channels_last)");
      fuse.addend = addend->data_ptr(); any = true;
    }
    if (bn_x.has_value()) {
      TORCH_CHECK(bn_stats.has_value() && bn_stats->scalar_type() == at::kFloat && bn_stats->dim() == 2 && bn_stats->size(1) == C && bn_stats->size(0) >= 2,
                  "conv_dgrad: bn_stats must be fp32 [>=2, C] (rows: mean, rstd)");
      TORCH_CHECK(bn_x->sizes() == dx.sizes() && bn_x->scalar_type() == at::kBFloat16 && bn_x->is_contiguous(at::MemoryFormat::ChannelsLast),
                  "conv_dgrad: bn_x must match dx (bf16, channels_last)");
      fuse.bn_x = bn_x->data_ptr();
      if (bn_mask.has_value()) {
        TORCH_CHECK(bn_mask->scalar_type() == at::kByte && bn_mask->numel() == (int64_t)N * H * W * (C / 8), "conv_dgrad: bn_mask must be uint8 [N*H*W, C/8]");
        fuse.bn_mask = bn_mask->data_ptr();
      }
      fuse.bn_mean = bn_stats->data_ptr<float>();
      fuse.bn_rstd = bn_stats->data_ptr<float>() + C;
      // the statistics workspace of the data gradient has one row per CTA of an n-tile over the Cin columns
      const int groups = conv_stat_groups(N, H, W, K, C, R, S, cfg);
      TORCH_CHECK(groups > 0, "conv_dgrad: no tile plan");
      part = at::empty({2, groups, C}, dy.options().dtype(at::kFloat));
      pp = part.data_ptr<float>();
      any = true;
    }
    launch_conv_tap_gemm(dy.data_ptr(), w.data_ptr(), dx.data_ptr(), N, H, W, C, K, R, S, true, cfg, pp, cur_stream(), any ? &fuse : nullptr);
    return std::make_tuple(dx, part);
  }, py::arg("dy"), py::arg("w"), py::arg("stride") = 1, py::arg("pad") = 0, py::arg("mode") = -1, py::arg("block_n") = 0,
     py::arg("base_offset") = 0, py::arg("kc") = 0, py::arg("addend") = py::none(), py::arg("bn_x") = py::none(),
     py::arg("bn_mask") = py::none(), py::arg("bn_stats") = py::none());
  m.def("conv_wgrad", [](at::Tensor dy, at::Tensor x, int ksize, int stride, int pad, int split, int tile_m, int tile_n) {
    check_cuda(dy, "dy"); check_cuda(x, "x");
    TORCH_CHECK(dy.scalar_type() == at::kBFloat16 && x.scalar_type() == at::kBFloat16, "conv_wgrad: bf16 tensors");
    TORCH_CHECK(dy.dim() == 4 && dy.is_contiguous(at::MemoryFormat::ChannelsLast) && x.dim() == 4 && x.is_contiguous(at::MemoryFormat::ChannelsLast),
                "conv_wgrad: channels_last 4-D tensors");
    TORCH_CHECK(stride == 1 && pad == (ksize - 1) / 2 && dy.size(0) == x.size(0) && dy.size(2) == x.size(2) && dy.size(3) == x.size(3),
                "conv_wgrad: stride 1, 'same' padding");
    c10::cuda::CUDAGuard guard(dy.device());
    const int N = (int)x.size(0), C = (int)x.size(1), H = (int)x.size(2), W = (int)x.size(3), K = (int)dy.size(1);
    WgradCfg cfg; cfg.split = split; cfg.tile_m = tile_m; cfg.tile_n = tile_n;
    const size_t ws = conv_wgrad_workspace_floats(N, H, W, C, K, ksize, ksize, cfg);
    TORCH_CHECK(ws > 0, "conv_wgrad: unsupported geometry / tiling");
    at::Tensor work = at::empty({(int64_t)ws}, x.options().dtype(at::kFloat));
    at::Tensor dw = at::empty({K, C, ksize, ksize}, x.options().memory_format(at::MemoryFormat::ChannelsLast));
    launch_conv_wgrad(dy.data_ptr(), x.data_ptr(), dw.data_ptr(), N, H, W, C, K, ksize, ksize, cfg, work.data_ptr<float>(), cur_stream());
    return dw;
  }, py::arg("dy"), py::arg("x"), py::arg("ksize"), py::arg("stride") = 1, py::arg("pad") = 0, py::arg("split") = 0,
     py::arg("tile_m") = 0, py::arg("tile_n") = 0);
  // strided 7x7 stem (3 -> 64 channels, stride 2, padding 3) on the tcgen05 tap-GEMM through an overlapping-window tensor map
  m.def("stem_conv_supported", [](int H, int W) { StemGeom g; return stem_geom(H, W, &g); });
  m.def("stem_pack_input", [](at::Tensor x) {
    check_cuda(x, "x");
    TORCH_CHECK(x.scalar_type() == at::kBFloat16 && x.dim() == 4 && x.size(1) == 3 && x.is_contiguous(at::MemoryFormat::ChannelsLast),
                "stem_pack_input: x must be bf16 [N,3,H,W] channels_last");
    c10::cuda::CUDAGuard guard(x.device());
    const int N = (int)x.size(0), H = (int)x.size(2), W = (int)x.size(3);
    StemGeom g;
    TORCH_CHECK(stem_geom(H, W, &g), "stem_pack_input: unsupported image size ", H, "x", W);
    at::Tensor xp = at::empty({N, g.Hp2, g.Wp, 8}, x.options());
    launch_stem_pack_input(x.data_ptr(), xp.data_ptr(), N, H, W, cur_stream());
    return xp;
  });
  m.def("stem_pack_weight", [](at::Tensor w) {
    check_cuda(w, "w");
    TORCH_CHECK(w.scalar_type() == at::kBFloat16 && w.dim() == 4 && w.size(0) == 64 && w.size(1) == 3 && w.size(2) == 7 && w.size(3) == 7 &&
                w.is_contiguous(at::MemoryFormat::ChannelsLast), "stem_pack_weight: w must be bf16 [64,3,7,7] channels_last");
    c10::cuda::CUDAGuard guard(w.device());
    at::Tensor w2 = at::empty({w.size(0), (int64_t)kStemK}, w.options().memory_format(at::MemoryFormat::Contiguous));
    launch_stem_pack_weight(w.data_ptr(), w2.data_ptr(), (int)w.size(0), cur_stream());
    return w2;
  });
  m.def("stem_conv_fprop_packed", [](at::Tensor xp, at::Tensor w2, int H, int W, bool stats, bool resident, bool debug) {
    check_cuda(xp, "xp"); check_cuda(w2, "w2");
    c10::cuda::CUDAGuard guard(xp.device());
    StemGeom g;
    const int N = (int)xp.size(0), K = (int)w2.size(0);
    TORCH_CHECK(stem_geom(H, W, &g) && xp.dim() == 4 && xp.size(1) == g.Hp2 && xp.size(2) == g.Wp && xp.size(3) == 8 && xp.is_contiguous() &&
                w2.dim() == 2 && w2.size(1) == kStemK && w2.is_contiguous() && xp.scalar_type() == at::kBFloat16 && w2.scalar_type() == at::kBFloat16,
                "stem_conv_fprop_packed: operands do not match the packed layout");
    at::Tensor y = at::empty({N, K, g.Ho, g.Wo}, xp.options().memory_format(at::MemoryFormat::ChannelsLast));
    at::Tensor part, dbg;
    float* sp = nullptr;
    if (stats) { part = at::empty({2, stem_stat_groups(N, H, W), K}, xp.options().dtype(at::kFloat)); sp = part.data_ptr<float>(); }
    if (debug) dbg = at::zeros({16}, xp.options().dtype(at::kLong));
    launch_stem_conv_fprop(xp.data_ptr(), w2.data_ptr(), y.data_ptr(), N, H, W, K, sp, resident, debug ? dbg.data_ptr() : nullptr, cur_stream());
    return std::make_tuple(y, part, dbg);
  }, py::arg("xp"), py::arg("w2"), py::arg("H"), py::arg("W"), py::arg("stats") = false, py::arg("resident") = true, py::arg("debug") = false);
  m.def("stem_conv_fprop", [](at::Tensor x, at::Tensor w, bool stats, bool resident) {
    check_cuda(x, "x"); check_cuda(w, "w");
    TORCH_CHECK(x.scalar_type() == at::kBFloat16 && w.scalar_type() == at::kBFloat16, "stem_conv_fprop: bf16 tensors");
    TORCH_CHECK(x.dim() == 4 && x.size(1) == 3 && x.is_contiguous(at::MemoryFormat::ChannelsLast), "stem_conv_fprop: x must be [N,3,H,W] channels_last");
    TORCH_CHECK(w.dim() == 4 && w.size(0) == 64 && w.size(1) == 3 && w.size(2) == 7 && w.size(3) == 7 && w.is_contiguous(at::MemoryFormat::ChannelsLast),
                "stem_conv_fprop: w must be [64,3,7,7] channels_last");
    c10::cuda::CUDAGuard guard(x.device());
    const int N = (int)x.size(0), H = (int)x.size(2), W = (int)x.size(3), K = (int)w.size(0);
    StemGeom g;
    TORCH_CHECK(stem_geom(H, W, &g), "stem_conv_fprop: unsupported image size ", H, "x", W);
    at::Tensor xp = at::empty({N, g.Hp2, g.Wp, 8}, x.options().memory_format(at::MemoryFormat::Contiguous));
    at::Tensor w2 = at::empty({K, (int64_t)kStemK}, x.options().memory_format(at::MemoryFormat::Contiguous));
    at::Tensor y = at::empty({N, K, g.Ho, g.Wo}, x.options().memory_format(at::MemoryFormat::ChannelsLast));
    at::Tensor part;
    float* sp = nullptr;
    if (stats) { part = at::empty({2, stem_stat_groups(N, H, W), K}, x.options().dtype(at::kFloat).memory_format(at::MemoryFormat::Contiguous)); sp = part.data_ptr<float>(); }
    cudaStream_t st = cur_stream();
    launch_stem_pack_input(x.data_ptr(), xp.data_ptr(), N, H, W, st);
    launch_stem_pack_weight(w.data_ptr(), w2.data_ptr(), K, st);
    launch_stem_conv_fprop(xp.data_ptr(), w2.data_ptr(), y.data_ptr(), N, H, W, K, sp, resident, nullptr, st);
    return std::make_tuple(y, part, xp);
  }, py::arg("x"), py::arg("w"), py::arg("stats") = false, py::arg("resident") = true);
  m.def("stem_conv_wgrad", [](at::Tensor dy, at::Tensor xp, int H, int W, int variant, bool unpack) {
    check_cuda(dy, "dy"); check_cuda(xp, "xp");
    TORCH_CHECK(dy.scalar_type() == at::kBFloat16 && xp.scalar_type() == at::kBFloat16, "stem_conv_wgrad: bf16 tensors");
    TORCH_CHECK(dy.dim() == 4 && dy.is_contiguous(at::MemoryFormat::ChannelsLast) && xp.is_contiguous(), "stem_conv_wgrad: dy channels_last, xp packed");
    TORCH_CHECK(variant == 0 || variant == 1, "stem_conv_wgrad: variant 0 (dedicated kernel) or 1 (generic kernel)");
    c10::cuda::CUDAGuard guard(dy.device());
    const int N = (int)dy.size(0), K = (int)dy.size(1);
    StemGeom g;
    TORCH_CHECK(stem_geom(H, W, &g) && dy.size(2) == g.Ho && dy.size(3) == g.Wo && xp.dim() == 4 && xp.size(0) == N && xp.size(1) == g.Hp2 &&
                xp.size(2) == g.Wp && xp.size(3) == 8, "stem_conv_wgrad: geometry mismatch");
    const size_t ws = stem_wgrad_workspace_floats(N, H, W, K, variant);
    TORCH_CHECK(ws > 0, "stem_conv_wgrad: unsupported geometry");
    auto plain = dy.options().memory_format(at::MemoryFormat::Contiguous);
    at::Tensor work = at::empty({(int64_t)ws}, plain.dtype(at::kFloat));
    at::Tensor dw2 = variant == 0 ? at::empty({(int64_t)kStemK, K}, plain) : at::empty({K, (int64_t)kStemK}, plain);
    cudaStream_t st = cur_stream();
    launch_stem_conv_wgrad(dy.data_ptr(), xp.data_ptr(), dw2.data_ptr(), N, H, W, K, variant, work.data_ptr<float>(), st);
    if (!unpack) return dw2;
    at::Tensor dw = at::empty({K, 3, 7, 7}, dy.options().memory_format(at::MemoryFormat::ChannelsLast));
    launch_stem_unpack_wgrad(dw2.data_ptr(), dw.data_ptr(), K, variant == 0, st);
    return dw;
  }, py::arg("dy"), py::arg("xp"), py::arg("H"), py::arg("W"), py::arg("variant") = 0, py::arg("unpack") = true);
  m.def("conv_tile_plan", [](int N, int H, int W, int R, int S, int mode) {
    ConvTilePlan pl;
    const bool ok = conv_tile_plan(N, H, W, R, S, mode, &pl);
    return std::make_tuple(ok, pl.mode, pl.BH, pl.BI, pl.num_m_tiles, pl.dense_rows, pl.acc_rows, pl.a_rows);
  });

  // ---- fused BatchNorm ---------------------------------------------------------------------------
  m.def("bn_workspace", [](int R, int C) {
    size_t pf = 0, cn = 0;
    bn_workspace_sizes(R, C, &pf, &cn);
    return std::make_tuple((long long)pf, (long long)cn);
  });
  m.def("bn_forward", [](at::Tensor x, c10::optional<at::Tensor> residual, at::Tensor gamma, at::Tensor beta,
                         c10::optional<at::Tensor> running_mean, c10::optional<at::Tensor> running_var,
                         c10::optional<at::Tensor> num_batches, double eps, double momentum, bool relu, at::Tensor partial,
                         at::Tensor counters) {
    BnForwardIo io = bn_forward_io("bn_forward", x, residual, gamma, beta, relu);
    c10::cuda::CUDAGuard guard(x.device());
    float* st = io.stats.data_ptr<float>();
    launch_bn_forward(x.data_ptr(), io.res, io.y.data_ptr(), relu ? io.mask.data_ptr<uint8_t>() : nullptr, dtype_of(x), io.R, io.C,
                      gamma.data_ptr<float>(), beta.data_ptr<float>(), opt_ptr<float>(running_mean), opt_ptr<float>(running_var),
                      (long long*)opt_ptr<int64_t>(num_batches), st, st + io.C, st + 2 * io.C, st + 3 * io.C, partial.data_ptr<float>(),
                      (unsigned int*)counters.data_ptr<int>(), (float)eps, (float)momentum, relu, cur_stream());
    return std::make_tuple(io.y, io.stats, io.mask);
  });
  m.def("bn_forward_partials", [](at::Tensor x, c10::optional<at::Tensor> residual, at::Tensor gamma, at::Tensor beta,
                                  c10::optional<at::Tensor> running_mean, c10::optional<at::Tensor> running_var,
                                  c10::optional<at::Tensor> num_batches, double eps, double momentum, bool relu, at::Tensor partial) {
    BnForwardIo io = bn_forward_io("bn_forward_partials", x, residual, gamma, beta, relu);
    check_cuda(partial, "partial");
    TORCH_CHECK(partial.scalar_type() == at::kFloat && partial.dim() == 3 && partial.size(0) == 2 && partial.size(2) == io.C &&
                partial.is_contiguous(), "bn_forward_partials: partial statistics must be fp32 [2, groups, C]");
    c10::cuda::CUDAGuard guard(x.device());
    float* st = io.stats.data_ptr<float>();
    launch_bn_forward_from_partials(x.data_ptr(), io.res, io.y.data_ptr(), relu ? io.mask.data_ptr<uint8_t>() : nullptr, dtype_of(x), io.R,
                                    io.C, gamma.data_ptr<float>(), beta.data_ptr<float>(), opt_ptr<float>(running_mean),
                                    opt_ptr<float>(running_var), (long long*)opt_ptr<int64_t>(num_batches), st, st + io.C,
                                    partial.data_ptr<float>(), (int)partial.size(1), (float)eps, (float)momentum, relu, cur_stream());
    return std::make_tuple(io.y, io.stats, io.mask);
  });
  m.def("bn_backward_partials", [](at::Tensor dy, at::Tensor x, c10::optional<at::Tensor> y, at::Tensor gamma, at::Tensor stats, bool relu,
                                   bool need_dres, at::Tensor partial) {
    BnBackwardIo io = bn_backward_io("bn_backward_partials", dy, x, y, relu, need_dres, 2);   // dparams rows: dgamma, dbeta
    check_cuda(partial, "partial");
    TORCH_CHECK(partial.scalar_type() == at::kFloat && partial.dim() == 3 && partial.size(0) == 2 && partial.size(2) == io.C && partial.is_contiguous(),
                "bn_backward_partials: partial sums must be fp32 [2, groups, C]");
    TORCH_CHECK(dy.is_contiguous(at::MemoryFormat::ChannelsLast) && dy.sizes() == x.sizes() && dy.dtype() == x.dtype(),
                "bn_backward_partials: dy must match x");
    c10::cuda::CUDAGuard guard(x.device());
    float* dp = io.dparams.data_ptr<float>();
    const float* st = stats.data_ptr<float>();
    launch_bn_backward_from_partials(dy.data_ptr(), x.data_ptr(), io.relu_mask, io.dx.data_ptr(), need_dres ? io.dres.data_ptr() : nullptr,
                                     dtype_of(x), io.R, io.C, gamma.data_ptr<float>(), st, st + io.C, dp, dp + io.C,
                                     partial.data_ptr<float>(), (int)partial.size(1), relu, cur_stream());
    return std::make_tuple(io.dx, io.dres, io.dparams);
  });
  m.def("bn_backward", [](at::Tensor dy, at::Tensor x, c10::optional<at::Tensor> y, at::Tensor gamma, at::Tensor stats, bool relu,
                          bool need_dres, at::Tensor partial, at::Tensor counters) {
    BnBackwardIo io = bn_backward_io("bn_backward", dy, x, y, relu, need_dres, 4);   // dparams rows: dgamma, dbeta, coef1, coef2
    c10::cuda::CUDAGuard guard(x.device());
    at::Tensor dyc = dy.is_contiguous(at::MemoryFormat::ChannelsLast) ? dy : dy.contiguous(at::MemoryFormat::ChannelsLast);
    float* dp = io.dparams.data_ptr<float>();
    const float* st = stats.data_ptr<float>();
    launch_bn_backward(dyc.data_ptr(), x.data_ptr(), io.relu_mask, io.dx.data_ptr(), need_dres ? io.dres.data_ptr() : nullptr, dtype_of(x),
                       io.R, io.C, gamma.data_ptr<float>(), st, st + io.C, dp, dp + io.C, dp + 2 * io.C, partial.data_ptr<float>(),
                       (unsigned int*)counters.data_ptr<int>(), relu, cur_stream());
    return std::make_tuple(io.dx, io.dres, io.dparams);
  });

  // ---- max pooling ------------------------------------------------------------------------------
  m.def("maxpool3x3s2_fwd", [](at::Tensor x) {
    check_cuda(x, "x");
    TORCH_CHECK(x.dim() == 4 && x.is_contiguous(at::MemoryFormat::ChannelsLast), "maxpool3x3s2_fwd: 4-D channels_last input");
    c10::cuda::CUDAGuard guard(x.device());
    const int N = (int)x.size(0), C = (int)x.size(1), H = (int)x.size(2), W = (int)x.size(3);
    const int OH = (H + 2 - 3) / 2 + 1, OW = (W + 2 - 3) / 2 + 1;
    at::Tensor y = at::empty({N, C, OH, OW}, x.options().memory_format(at::MemoryFormat::ChannelsLast));
    at::Tensor idx = at::empty({N, C, OH, OW}, x.options().dtype(at::kByte).memory_format(at::MemoryFormat::ChannelsLast));
    launch_maxpool3x3s2_fwd(x.data_ptr(), y.data_ptr(), idx.data_ptr<uint8_t>(), dtype_of(x), N, H, W, C, cur_stream());
    return std::make_tuple(y, idx);
  });
  m.def("maxpool3x3s2_bwd", [](at::Tensor dy, at::Tensor idx, int64_t H, int64_t W) {
    check_cuda(dy, "dy");
    c10::cuda::CUDAGuard guard(dy.device());
    at::Tensor dyc = dy.is_contiguous(at::MemoryFormat::ChannelsLast) ? dy : dy.contiguous(at::MemoryFormat::ChannelsLast);
    const int N = (int)dy.size(0), C = (int)dy.size(1);
    at::Tensor dx = at::empty({N, C, H, W}, dy.options().memory_format(at::MemoryFormat::ChannelsLast));
    launch_maxpool3x3s2_bwd(dyc.data_ptr(), idx.data_ptr<uint8_t>(), dx.data_ptr(), dtype_of(dy), N, (int)H, (int)W, C, cur_stream());
    return dx;
  });

  // ---- input pipeline ---------------------------------------------------------------------------
  m.def("normalize_to_channels_last", [](at::Tensor src, at::Tensor dst, at::Tensor mean, at::Tensor inv_std, double in_scale) {
    check_cuda(src, "src"); check_cuda(dst, "dst");
    TORCH_CHECK(src.dim() == 4 && src.is_contiguous(), "normalize_to_channels_last: src NCHW contiguous");
    // dst may carry extra (zero-filled) channels: [N, C_out >= C, H, W]
    TORCH_CHECK(dst.dim() == 4 && dst.is_contiguous(at::MemoryFormat::ChannelsLast) && dst.size(0) == src.size(0) &&
                dst.size(1) >= src.size(1) && dst.size(2) == src.size(2) && dst.size(3) == src.size(3),
                "normalize_to_channels_last: dst must be channels_last [N, C_out >= C, H, W]");
    TORCH_CHECK(mean.numel() >= src.size(1) && inv_std.numel() >= src.size(1), "normalize_to_channels_last: mean/inv_std per source channel");
    c10::cuda::CUDAGuard guard(src.device());
    launch_normalize_to_channels_last(src.data_ptr(), dtype_of(src), dst.data_ptr(), dtype_of(dst), (int)src.size(0), (int)src.size(1),
                                      (int)dst.size(1), (int)src.size(2), (int)src.size(3), mean.data_ptr<float>(), inv_std.data_ptr<float>(),
                                      (float)in_scale, cur_stream());
  });
}
