// The autograd node of the distillation step as a compiled torch extension (host C++ only).
//
// `FeatureDistillation.distill` (mirror of mafed/methods/distillation.py:105-122) used to reach the C ABI through
// ctypes and a Python `torch.autograd.Function`: pointer tables, workspace and gradient allocation, stream lookup,
// launch and the backward fix-up cost ~300 us of interpreter time per step -- more than the kernels of every
// workload below ~0.3 ms of HBM traffic.  This file does the same work in C++: one call per step from Python, a
// `torch::autograd::Node` for the backward.  It contains no kernel and no arithmetic; it binds the C ABI of
// libmafed_distill.so (include/mafed_distill.h) at run time (`bind(path)`, dlopen of the same file the ctypes
// binding loads) and fails loudly when that library is missing.
#include <torch/extension.h>

#include <ATen/cuda/CUDAEvent.h>
#include <c10/cuda/CUDACachingAllocator.h>
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <dlfcn.h>
#include <torch/csrc/autograd/function.h>
#include <torch/csrc/autograd/functions/utils.h>
#include <torch/csrc/autograd/saved_variable.h>

#include <cstring>
#include <memory>
#include <string>
#include <tuple>
#include <vector>

#include "mafed_distill.h"

namespace {

using torch::autograd::Node;
using torch::autograd::SavedVariable;
using torch::autograd::variable_list;

// ---------------------------------------------------------------- the C ABI, bound at run time
struct Api {
  decltype(&mafed_distill_abi_version) abi_version = nullptr;
  decltype(&mafed_distill_error_string) error_string = nullptr;
  decltype(&mafed_distill_ws_bytes) ws_bytes = nullptr;
  decltype(&mafed_distill_step) step = nullptr;
  decltype(&mafed_distill_fwd_step) fwd_step = nullptr;
  decltype(&mafed_distill_bwd) bwd = nullptr;
  decltype(&mafed_distill_modality_masks) modality_masks = nullptr;
  decltype(&mafed_distill_prefetch_counts) prefetch_counts = nullptr;
  bool bound = false;
};
Api g_api;

template <typename F>
void load_symbol(void* lib, const char* name, F& fn) {
  fn = reinterpret_cast<F>(dlsym(lib, name));
  TORCH_CHECK(fn != nullptr, "libmafed_distill.so does not export ", name, ": rebuild it (python -m mafed_b200.build)");
}

void bind(const std::string& path) {
  void* lib = dlopen(path.c_str(), RTLD_NOW | RTLD_GLOBAL);
  TORCH_CHECK(lib != nullptr, "cannot load ", path, " (", dlerror(),
              "): build it with `python -m mafed_b200.build` -- the distillation path has no CPU / eager fallback");
  Api a;
  load_symbol(lib, "mafed_distill_abi_version", a.abi_version);
  load_symbol(lib, "mafed_distill_error_string", a.error_string);
  load_symbol(lib, "mafed_distill_ws_bytes", a.ws_bytes);
  load_symbol(lib, "mafed_distill_step", a.step);
  load_symbol(lib, "mafed_distill_fwd_step", a.fwd_step);
  load_symbol(lib, "mafed_distill_bwd", a.bwd);
  load_symbol(lib, "mafed_distill_modality_masks", a.modality_masks);
  load_symbol(lib, "mafed_distill_prefetch_counts", a.prefetch_counts);
  TORCH_CHECK(a.abi_version() == MAFED_ABI_VERSION, "libmafed_distill.so ABI version ", a.abi_version(),
              " != ", MAFED_ABI_VERSION, "; rebuild");
  a.bound = true;
  g_api = a;
}

const Api& api() {
  TORCH_CHECK(g_api.bound, "mafed_torch_node: bind(<path of libmafed_distill.so>) has not been called");
  return g_api;
}

void check_rc(int rc, const char* what) {
  TORCH_CHECK(rc == 0, what, " failed: ", api().error_string(rc), " (code ", rc, ")");
}

// ---------------------------------------------------------------- plan: the host tables of one configuration
struct Plan {
  mafed_weights_t w;
  int n_layers = 0;
  int loss_kind = MAFED_LOSS_MSE;
  bool cls = false;
  int n_vis = 256;
  double grad_multiplier = 1.0;   // e.g. world_size to undo DDP's gradient averaging
  bool single_pass = true;
  double assumed_grad_out = 1.0;  // upstream gradient the one-pass step bakes in

  Plan(int modality_kind, double distill_coeff, const std::vector<double>& layer_coeffs,
       const c10::optional<std::vector<double>>& lang_weights, int loss_kind_, bool cls_, int n_vis_,
       double grad_multiplier_, bool single_pass_, double assumed_grad_out_)
      : n_layers((int)layer_coeffs.size()), loss_kind(loss_kind_), cls(cls_), n_vis(n_vis_),
        grad_multiplier(grad_multiplier_), single_pass(single_pass_), assumed_grad_out(assumed_grad_out_) {
    TORCH_CHECK(n_layers >= 1 && n_layers <= MAFED_MAX_LAYERS, "1..", MAFED_MAX_LAYERS, " layers per call");
    std::memset(&w, 0, sizeof(w));
    w.modality_kind = modality_kind;
    w.distill_coeff = (float)distill_coeff;
    for (int i = 0; i < n_layers; ++i) w.layer_coeff[i] = (float)layer_coeffs[i];
    if (lang_weights.has_value()) {
      TORCH_CHECK((int)lang_weights->size() == n_layers, "lang_weights / layer_coeffs length mismatch");
      for (int i = 0; i < n_layers; ++i) w.lang_weight[i] = (float)(*lang_weights)[i];
    }
  }
  float fixed() const { return (float)(assumed_grad_out * grad_multiplier); }
};

// Token counts sent ahead of the step (mafed_distill_prefetch_counts).  The 1-CTA launch runs on a side stream,
// ordered behind whatever produced the mask, so it never sits between two kernels of the compute stream; the step
// that consumes the ticket makes its stream wait for `done` (long since recorded) before it launches.
struct CountsTicket {
  at::Tensor tensor;          // int64[4] on the device: {exchange epoch, bits(n_text), bits(n_vis rows), 0}
  at::Tensor mask;            // the mask the counts were taken from (kept alive until the ticket goes)
  at::cuda::CUDAEvent done;   // recorded on the side stream behind the launch
  void wait() {
    const auto dev = tensor.device();
    done.block(c10::cuda::getCurrentCUDAStream(dev.index()));
  }
};

c10::cuda::CUDAStream side_stream(c10::DeviceIndex dev) {
  static std::vector<c10::optional<c10::cuda::CUDAStream>> streams(64);
  auto& s = streams.at((size_t)dev);
  if (!s.has_value()) s = c10::cuda::getStreamFromPool(/*isHighPriority=*/true, dev);
  return *s;
}

int dtype_code(at::ScalarType t) {
  switch (t) {
    case at::kFloat: return MAFED_F32;
    case at::kBFloat16: return MAFED_BF16;
    case at::kHalf: return MAFED_F16;
    default: TORCH_CHECK_TYPE(false, "unsupported hidden-state dtype ", t, " (float32, bfloat16, float16)");
  }
}

// One [B, T, D] view per needed layer of ONE allocation (the caching allocator is paid once, not L times).
// Built without the dispatcher: the views share `buf`'s storage.
std::vector<at::Tensor> layer_views(const at::Tensor& buf, int64_t n) {
  std::vector<at::Tensor> out;
  out.reserve(n);
  const auto sizes = buf.sizes().slice(1);
  const auto strides = buf.strides().slice(1);
  const int64_t step = buf.stride(0);
  for (int64_t j = 0; j < n; ++j) {
    auto impl = c10::make_intrusive<c10::TensorImpl>(c10::TensorImpl::VIEW, c10::Storage(buf.storage()), buf.key_set(),
                                                     buf.dtype());
    impl->set_storage_offset(buf.storage_offset() + j * step);
    impl->set_sizes_and_strides(sizes, strides);
    out.emplace_back(std::move(impl));
  }
  return out;
}

// ---------------------------------------------------------------- the backward node
struct DistillBackward : public Node {
  std::shared_ptr<Plan> plan;
  mafed_shape_t shape;
  mafed_tuning_t tuning;           // a copy: the caller's knobs may be gone by the time backward runs
  bool has_tuning = false;
  std::vector<SavedVariable> students, teachers;   // version-checked on unpack: an in-place edit between forward
  SavedVariable mask;                               // and backward would silently change what the kernels read
  bool has_mask = false;
  at::Tensor scratch;              // workspace + scale table [+ sums]
  const float* bwd_scale = nullptr;
  at::Tensor grad_buf;             // one-pass step: the gradients, already written
  std::vector<bool> needs;
  float* seen = nullptr;           // pinned host word that receives the upstream gradient (kept alive by `seen_owner`)
  at::Tensor seen_owner;
  bool released = false;

  std::string name() const override { return "MafedDistillBackward"; }

  void release_variables() override {
    for (auto& s : students) s.reset_data();
    for (auto& t : teachers) t.reset_data();
    if (has_mask) mask.reset_data();
    scratch.reset();
    grad_buf.reset();
    released = true;
  }

  variable_list apply(variable_list&& grads_in) override {
    const size_t n = needs.size();
    variable_list out(n);
    if (grads_in.empty() || !grads_in[0].defined()) return out;
    TORCH_CHECK(!released, "Trying to backward through the distillation step a second time (its saved tensors have "
                           "been freed); pass retain_graph=True to the first backward");
    const Api& a = api();
    auto self = shared_from_this();
    std::vector<at::Tensor> s(n), t(n);
    const void* s_ptrs[MAFED_MAX_LAYERS];
    const void* t_ptrs[MAFED_MAX_LAYERS];
    void* g_ptrs[MAFED_MAX_LAYERS];
    for (size_t i = 0; i < n; ++i) {
      s[i] = students[i].unpack(self);
      t[i] = teachers[i].unpack(self);
      s_ptrs[i] = s[i].data_ptr();
      t_ptrs[i] = t[i].data_ptr();
    }
    at::Tensor m;
    if (has_mask) m = mask.unpack(self);
    const auto device = s[0].device();
    c10::cuda::CUDAGuard guard(device);
    const cudaStream_t stream = c10::cuda::getCurrentCUDAStream(device.index()).stream();
    at::AutoDispatchBelowADInplaceOrView below;
    at::Tensor g = grads_in[0];
    if (g.scalar_type() != at::kFloat || g.device() != device) g = g.to(device, at::kFloat);
    if (!g.is_contiguous()) g = g.contiguous();
    shape.tuning = has_tuning ? &tuning : nullptr;

    int64_t n_need = 0;
    for (bool b : needs) n_need += b ? 1 : 0;
    const bool gate = grad_buf.defined();   // one-pass step: gradients exist, fix them up only if g differs
    at::Tensor buf = grad_buf;
    if (!gate) {
      std::vector<int64_t> sz = {n_need, shape.B, shape.T, shape.D};
      buf = plan->cls ? at::zeros(sz, s[0].options()) : at::empty(sz, s[0].options());
    }
    auto views = layer_views(buf, n_need);
    for (size_t i = 0, j = 0; i < n; ++i) {
      g_ptrs[i] = needs[i] ? views[j].data_ptr() : nullptr;
      if (needs[i]) out[i] = std::move(views[j++]);
    }
    const float fixed = plan->fixed();
    check_rc(a.bwd(&shape, s_ptrs, t_ptrs, g_ptrs, has_mask ? m.data_ptr<int64_t>() : nullptr, bwd_scale,
                   g.data_ptr<float>(), (float)plan->grad_multiplier, gate ? &fixed : nullptr, gate ? seen : nullptr,
                   stream),
             "mafed_distill_bwd");
    grad_buf.reset();   // handed to autograd: a second backward (retain_graph) recomputes into a fresh buffer
    return out;
  }
};

// ---------------------------------------------------------------- forward
// students / teachers: the selected [B, T, D] hidden states (same shape and device; one dtype, or fp32 students with
// bf16 / fp16 teachers -- other mixes are up-cast to fp32).  attn_mask: int64 [B, T - n_vis]
// (ignored in cls mode).  masks_out: None, an int64 [2, B, T] tensor, or True to have one allocated here; it receives
// (lang_masks, image_masks).  comm: a mafed_comm_t* (0: single rank).  ticket: optional int64[4] from
// prefetch_counts.  seen: optional pinned float[1].
// Returns (total, aux, masks): the 0-dim fp32 loss with the node attached, the [3L] layer / (text, vision) losses,
// and the [2, B, T] mask tensor (None if not requested).
std::tuple<at::Tensor, at::Tensor, c10::optional<at::Tensor>> distill(
    const std::shared_ptr<Plan>& plan, std::vector<at::Tensor> students, std::vector<at::Tensor> teachers,
    const c10::optional<at::Tensor>& attn_mask, const py::object& masks_out, int64_t comm,
    const std::shared_ptr<CountsTicket>& ticket, const c10::optional<at::Tensor>& seen, int64_t tuning_addr) {
  const Api& a = api();
  const int L = plan->n_layers;
  TORCH_CHECK((int)students.size() == L && (int)teachers.size() == L, "students / teachers / plan length mismatch");
  {
    // One dtype everywhere, or fp32 students with teachers of one half-precision dtype: the kernels read the tensors
    // as they are (a teacher pair, MAFED_DTYPE_PAIR).  Any other mix -- layers of different dtypes, a student narrower
    // than its teacher -- is up-cast to fp32 on both sides, which is what the reference's autocast region does to
    // the inputs of its loss functions (distillation.py:90,244); the casts are ordinary autograd ops.
    const at::ScalarType s_type = students[0].scalar_type(), t_type = teachers[0].scalar_type();
    bool uniform = true;
    for (int i = 0; i < L && uniform; ++i)
      uniform = students[i].scalar_type() == s_type && teachers[i].scalar_type() == t_type;
    const bool native = uniform && (s_type == t_type || (s_type == at::kFloat && (t_type == at::kBFloat16 ||
                                                                                  t_type == at::kHalf)));
    if (!native)
      for (int i = 0; i < L; ++i) {
        students[i] = students[i].to(at::kFloat);
        teachers[i] = teachers[i].to(at::kFloat);
      }
  }
  const at::Tensor& s0 = students[0];
  TORCH_CHECK(s0.is_cuda(), "hidden_states is on ", s0.device(),
              ": the distillation path runs only as sm_100a CUDA kernels (there is no CPU fallback)");
  TORCH_CHECK_VALUE(s0.dim() == 3, "hidden states must be [B, T, D]");
  const int code = dtype_code(s0.scalar_type());
  const int t_code = dtype_code(teachers[0].scalar_type());
  const auto device = s0.device();
  const bool grad_mode = at::GradMode::is_enabled();
  std::vector<bool> needs(L, false);
  bool any_need = false;
  for (int i = 0; i < L; ++i) {
    at::Tensor& s = students[i];
    at::Tensor& t = teachers[i];
    TORCH_CHECK_VALUE(s.sizes() == s0.sizes() && t.sizes() == s0.sizes(),
                      "all selected hidden states must share one [B, T, D] shape");
    TORCH_CHECK_VALUE(s.scalar_type() == s0.scalar_type() && t.scalar_type() == teachers[0].scalar_type() &&
                          s.device() == device && t.device() == device,
                      "student / teacher dtype or device mismatch");
    needs[i] = grad_mode && s.requires_grad();
    any_need = any_need || needs[i];
  }
  // collect the graph edges before the tensors are replaced by contiguous copies
  torch::autograd::edge_list edges;
  if (any_need) edges = torch::autograd::collect_next_edges(students);

  at::AutoDispatchBelowADInplaceOrView below;
  for (int i = 0; i < L; ++i) {
    if (!students[i].is_contiguous()) students[i] = students[i].contiguous();
    if (!teachers[i].is_contiguous()) teachers[i] = teachers[i].contiguous();
  }
  const int64_t B = s0.size(0), T = s0.size(1), D = s0.size(2);
  mafed_shape_t shape;
  std::memset(&shape, 0, sizeof(shape));
  shape.n_layers = L;
  shape.B = (int32_t)B;
  shape.T = (int32_t)T;
  shape.n_vis = plan->cls ? (int32_t)std::min<int64_t>(plan->n_vis, T) : plan->n_vis;
  shape.D = (int32_t)D;
  shape.dtype = t_code == code ? code : MAFED_DTYPE_PAIR(code, t_code);
  shape.loss_kind = plan->loss_kind;
  shape.cls = plan->cls ? 1 : 0;
  shape.tuning = reinterpret_cast<const mafed_tuning_t*>(tuning_addr);

  at::Tensor mask;
  if (!plan->cls) {
    TORCH_CHECK_VALUE(attn_mask.has_value() && attn_mask->defined(), "attention_mask is required");
    mask = *attn_mask;
    TORCH_CHECK(mask.is_cuda(), "attention_mask is on ", mask.device(),
                ": the distillation path runs only as sm_100a CUDA kernels (there is no CPU fallback)");
    if (mask.scalar_type() != at::kLong) mask = mask.to(at::kLong);
    TORCH_CHECK_VALUE(mask.dim() == 2 && mask.size(0) == B && mask.size(1) == T - plan->n_vis, "attention_mask shape ",
                      mask.sizes(), " != (B, T - n_vis) = (", B, ", ", T - plan->n_vis, ")");
    if (!mask.is_contiguous()) mask = mask.contiguous();
  }

  c10::cuda::CUDAGuard guard(device);
  const cudaStream_t stream = c10::cuda::getCurrentCUDAStream(device.index()).stream();
  const size_t ws_bytes = (a.ws_bytes(L) + 255) & ~(size_t)255;
  const size_t scale_bytes = ((size_t)8 * L + 255) & ~(size_t)255;
  const bool sharded = comm != 0;
  const size_t sums_bytes = sharded ? (size_t)8 * (2 * L + 2) : 0;
  const auto byte_opts = at::TensorOptions().dtype(at::kByte).device(device);
  at::Tensor scratch = at::empty({(int64_t)(ws_bytes + scale_bytes + sums_bytes)}, byte_opts);
  at::Tensor out = at::empty({1 + 3 * (int64_t)L}, at::TensorOptions().dtype(at::kFloat).device(device));
  char* base = reinterpret_cast<char*>(scratch.data_ptr());
  float* bwd_scale = reinterpret_cast<float*>(base + ws_bytes);
  double* sums = sharded ? reinterpret_cast<double*>(base + ws_bytes + scale_bytes) : nullptr;

  const void* s_ptrs[MAFED_MAX_LAYERS];
  const void* t_ptrs[MAFED_MAX_LAYERS];
  void* g_ptrs[MAFED_MAX_LAYERS];
  for (int i = 0; i < L; ++i) {
    s_ptrs[i] = students[i].data_ptr();
    t_ptrs[i] = teachers[i].data_ptr();
    g_ptrs[i] = nullptr;
  }
  int64_t* lang = nullptr;
  int64_t* image = nullptr;
  c10::optional<at::Tensor> masks;
  if (!masks_out.is_none() && !plan->cls) {
    if (py::isinstance<py::bool_>(masks_out)) {
      if (masks_out.cast<bool>()) masks = at::empty({2, B, T}, at::TensorOptions().dtype(at::kLong).device(device));
    } else {
      masks = masks_out.cast<at::Tensor>();
    }
    if (masks.has_value()) {
      const at::Tensor& mo = *masks;
      TORCH_CHECK_VALUE(mo.is_cuda() && mo.scalar_type() == at::kLong && mo.is_contiguous() && mo.dim() == 3 &&
                            mo.size(0) == 2 && mo.size(1) == B && mo.size(2) == T,
                        "masks_out must be a contiguous int64 [2, B, T] CUDA tensor");
      lang = mo.data_ptr<int64_t>();
      image = lang + B * T;
    }
  }
  const int64_t* mask_ptr = mask.defined() ? mask.data_ptr<int64_t>() : nullptr;
  const int64_t* ticket_ptr = nullptr;
  if (ticket != nullptr) {
    ticket->wait();     // this stream behind the prefetch launch (a no-op wait: it finished a forward pass ago)
    ticket_ptr = ticket->tensor.data_ptr<int64_t>();
  }

  at::Tensor grad_buf;
  if (plan->single_pass && any_need) {
    int64_t n_need = 0;
    for (bool b : needs) n_need += b ? 1 : 0;
    std::vector<int64_t> sz = {n_need, B, T, D};
    // cls: only row 0 of each sample is written by the kernel
    grad_buf = plan->cls ? at::zeros(sz, s0.options().requires_grad(false)) : at::empty(sz, s0.options().requires_grad(false));
    char* g0 = reinterpret_cast<char*>(grad_buf.data_ptr());
    const size_t layer_bytes = (size_t)B * T * D * grad_buf.element_size();
    for (int i = 0, j = 0; i < L; ++i)
      if (needs[i]) g_ptrs[i] = g0 + (size_t)(j++) * layer_bytes;
    check_rc(a.step(&shape, s_ptrs, t_ptrs, g_ptrs, mask_ptr, &plan->w, plan->fixed(), base, out.data_ptr<float>(),
                    bwd_scale, sums, lang, image, reinterpret_cast<mafed_comm_t*>(comm), ticket_ptr, stream),
             "mafed_distill_step");
  } else {
    check_rc(a.fwd_step(&shape, s_ptrs, t_ptrs, mask_ptr, &plan->w, base, out.data_ptr<float>(), bwd_scale, sums,
                        reinterpret_cast<mafed_comm_t*>(comm), stream),
             "mafed_distill_fwd_step");
    if (lang != nullptr) check_rc(a.modality_masks(&shape, mask_ptr, lang, image, stream), "mafed_distill_modality_masks");
  }

  at::Tensor total = out.select(0, 0);
  at::Tensor aux = out.narrow(0, 1, 3 * (int64_t)L);
  if (any_need) {
    auto node = std::shared_ptr<DistillBackward>(new DistillBackward(), torch::autograd::deleteNode);
    node->set_next_edges(std::move(edges));
    node->plan = plan;
    node->shape = shape;
    if (shape.tuning != nullptr) {
      node->tuning = *shape.tuning;
      node->has_tuning = true;
    }
    node->shape.tuning = nullptr;
    node->students.reserve(L);
    node->teachers.reserve(L);
    for (int i = 0; i < L; ++i) {
      node->students.emplace_back(students[i], false);
      node->teachers.emplace_back(teachers[i], false);
    }
    if (mask.defined()) {
      node->mask = SavedVariable(mask, false);
      node->has_mask = true;
    }
    node->scratch = scratch;
    node->bwd_scale = bwd_scale;
    node->grad_buf = grad_buf;
    node->needs = needs;
    if (seen.has_value() && seen->defined()) {
      // must be device-accessible host memory (a pinned tensor): the gate kernel stores into it
      TORCH_CHECK_VALUE(seen->scalar_type() == at::kFloat && seen->device().is_cpu(), "seen must be a pinned float32 tensor");
      node->seen_owner = *seen;
      node->seen = seen->data_ptr<float>();
    }
    torch::autograd::set_history(total, node);
  }
  return std::make_tuple(std::move(total), std::move(aux), std::move(masks));
}

// Token counts ahead of the step (mafed_distill_prefetch_counts): launches on the side stream, returns the ticket.
std::shared_ptr<CountsTicket> prefetch_counts(const at::Tensor& attn_mask, int64_t n_vis, int64_t comm, int64_t tuning_addr) {
  const Api& a = api();
  TORCH_CHECK(attn_mask.is_cuda() && attn_mask.scalar_type() == at::kLong && attn_mask.is_contiguous() && attn_mask.dim() == 2,
              "prefetch_counts: attention_mask must be a contiguous int64 [B, txt] CUDA tensor");
  const auto device = attn_mask.device();
  c10::cuda::CUDAGuard guard(device);
  const auto current = c10::cuda::getCurrentCUDAStream(device.index());
  const auto side = side_stream(device.index());
  mafed_shape_t shape;
  std::memset(&shape, 0, sizeof(shape));
  shape.n_layers = 1;
  shape.B = (int32_t)attn_mask.size(0);
  shape.T = (int32_t)(n_vis + attn_mask.size(1));
  shape.n_vis = (int32_t)n_vis;
  shape.D = 1;
  shape.dtype = MAFED_F32;
  shape.tuning = reinterpret_cast<const mafed_tuning_t*>(tuning_addr);
  auto ticket = std::make_shared<CountsTicket>();
  ticket->tensor = at::empty({4}, at::TensorOptions().dtype(at::kLong).device(device));
  ticket->mask = attn_mask;
  // both allocations belong to the compute stream; tell the allocator that the side stream touches them too
  c10::cuda::CUDACachingAllocator::recordStream(ticket->tensor.storage().data_ptr(), side);
  c10::cuda::CUDACachingAllocator::recordStream(attn_mask.storage().data_ptr(), side);
  at::cuda::CUDAEvent ready;
  ready.record(current);        // behind the producer of the mask
  ready.block(side);
  check_rc(a.prefetch_counts(&shape, attn_mask.data_ptr<int64_t>(), reinterpret_cast<mafed_comm_t*>(comm),
                             ticket->tensor.data_ptr<int64_t>(), side.stream()),
           "mafed_distill_prefetch_counts");
  ticket->done.record(side);
  return ticket;
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "mafed_b200: compiled autograd node over the C ABI of libmafed_distill.so";
  m.def("bind", &bind, "dlopen libmafed_distill.so and resolve the C ABI");
  m.def("is_bound", [] { return g_api.bound; });
  py::class_<Plan, std::shared_ptr<Plan>>(m, "Plan")
      .def(py::init<int, double, const std::vector<double>&, const c10::optional<std::vector<double>>&, int, bool, int,
                    double, bool, double>(),
           py::arg("modality_kind"), py::arg("distill_coeff"), py::arg("layer_coeffs"), py::arg("lang_weights"),
           py::arg("loss_kind"), py::arg("cls"), py::arg("n_vis"), py::arg("grad_multiplier"), py::arg("single_pass"),
           py::arg("assumed_grad_out"))
      .def_readonly("n_layers", &Plan::n_layers)
      .def_readwrite("single_pass", &Plan::single_pass)
      .def_readwrite("assumed_grad_out", &Plan::assumed_grad_out)
      .def_readwrite("grad_multiplier", &Plan::grad_multiplier);
  py::class_<CountsTicket, std::shared_ptr<CountsTicket>>(m, "CountsTicket")
      .def_readonly("tensor", &CountsTicket::tensor)
      .def("wait", &CountsTicket::wait, "make the current stream wait for the prefetch launch")
      .def("data_ptr", [](CountsTicket& t) { return (uint64_t)(uintptr_t)t.tensor.data_ptr(); });
  m.def("distill", &distill, py::arg("plan"), py::arg("students"), py::arg("teachers"), py::arg("attn_mask"),
        py::arg("masks_out"), py::arg("comm"), py::arg("ticket"), py::arg("seen"), py::arg("tuning"));
  m.def("prefetch_counts", &prefetch_counts, py::arg("attn_mask"), py::arg("n_vis"), py::arg("comm"), py::arg("tuning"));
}
