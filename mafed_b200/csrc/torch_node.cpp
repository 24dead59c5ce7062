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

#include "mafed_cached_step.h"
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

// The step that reads the teacher straight from the teacher cache (include/mafed_cached_step.h): a library of its
// own, bound on first use (`bind_cached(path)`, mafed_b200.node.load_cached).
struct CachedApi {
  decltype(&mafed_cached_step_abi_version) abi_version = nullptr;
  decltype(&mafed_cached_step_error_string) error_string = nullptr;
  decltype(&mafed_cached_step_supported) supported = nullptr;
  decltype(&mafed_cached_step) step = nullptr;
  decltype(&mafed_cached_step_bwd) bwd = nullptr;
  bool bound = false;
};
CachedApi g_cached;

template <typename F>
void load_cached_symbol(void* lib, const char* name, F& fn) {
  fn = reinterpret_cast<F>(dlsym(lib, name));
  TORCH_CHECK(fn != nullptr, "libmafed_cached_step.so does not export ", name, ": rebuild it (python -m mafed_b200.build)");
}

void bind_cached(const std::string& path) {
  void* lib = dlopen(path.c_str(), RTLD_NOW | RTLD_LOCAL);
  TORCH_CHECK(lib != nullptr, "cannot load ", path, " (", dlerror(),
              "): build it with `python -m mafed_b200.build` -- the cached step has no eager fallback");
  CachedApi a;
  load_cached_symbol(lib, "mafed_cached_step_abi_version", a.abi_version);
  load_cached_symbol(lib, "mafed_cached_step_error_string", a.error_string);
  load_cached_symbol(lib, "mafed_cached_step_supported", a.supported);
  load_cached_symbol(lib, "mafed_cached_step", a.step);
  load_cached_symbol(lib, "mafed_cached_step_bwd", a.bwd);
  TORCH_CHECK(a.abi_version() == MAFED_CACHED_ABI_VERSION, "libmafed_cached_step.so ABI version ", a.abi_version(),
              " != ", MAFED_CACHED_ABI_VERSION, "; rebuild");
  a.bound = true;
  g_cached = a;
}

const CachedApi& cached_api() {
  TORCH_CHECK(g_cached.bound, "mafed_torch_node: bind_cached(<path of libmafed_cached_step.so>) has not been called");
  return g_cached;
}

// A step whose teacher rows come from the teacher cache: the teacher table holds the [M, T_c, D] cache tensors and
// sample b reads memory sample idx[b].
struct CacheRef {
  std::vector<int64_t> idx;
  int64_t M = 0;
  int32_t T_c = 0;
};

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

// ---------------------------------------------------------------- shared by the node and the torch.library ops
// Pointer tables of one launch.
struct Tables {
  const void* s[MAFED_MAX_LAYERS];
  const void* t[MAFED_MAX_LAYERS];
  void* g[MAFED_MAX_LAYERS];
};

void fill_tables(const std::vector<at::Tensor>& students, const std::vector<at::Tensor>& teachers, Tables& tb) {
  for (size_t i = 0; i < students.size(); ++i) {
    tb.s[i] = students[i].data_ptr();
    tb.t[i] = teachers[i].data_ptr();
    tb.g[i] = nullptr;
  }
}

// Gradient pointers into one [n_need, B, T, D] buffer: layer i gets the next slice if it needs a gradient.
void fill_grad_ptrs(const at::Tensor& buf, const std::vector<bool>& needs, Tables& tb) {
  char* g0 = reinterpret_cast<char*>(buf.data_ptr());
  const size_t layer_bytes = buf.size(0) == 0 ? 0 : (size_t)(buf.numel() / buf.size(0)) * buf.element_size();
  for (size_t i = 0, j = 0; i < needs.size(); ++i) tb.g[i] = needs[i] ? g0 + (j++) * layer_bytes : nullptr;
}

int64_t count_needs(const std::vector<bool>& needs) {
  int64_t n = 0;
  for (bool b : needs) n += b ? 1 : 0;
  return n;
}

// The gradient buffer of the needed layers; cls: only row 0 of each sample is written by the kernels.
at::Tensor alloc_grads(int64_t n_need, const at::Tensor& s0, bool cls) {
  std::vector<int64_t> sz = {n_need, s0.size(0), s0.size(1), s0.size(2)};
  const auto opts = s0.options().requires_grad(false);
  return cls ? at::zeros(sz, opts) : at::empty(sz, opts);
}

mafed_shape_t make_shape(const at::Tensor& s0, const at::Tensor& t0, int L, int loss_kind, bool cls, int n_vis,
                         int64_t tuning_addr) {
  const int code = dtype_code(s0.scalar_type());
  const int t_code = dtype_code(t0.scalar_type());
  const int64_t T = s0.size(1);
  mafed_shape_t shape;
  std::memset(&shape, 0, sizeof(shape));
  shape.n_layers = L;
  shape.B = (int32_t)s0.size(0);
  shape.T = (int32_t)T;
  shape.n_vis = cls ? (int32_t)std::min<int64_t>(n_vis, T) : n_vis;
  shape.D = (int32_t)s0.size(2);
  shape.dtype = t_code == code ? code : MAFED_DTYPE_PAIR(code, t_code);
  shape.loss_kind = loss_kind;
  shape.cls = cls ? 1 : 0;
  shape.tuning = reinterpret_cast<const mafed_tuning_t*>(tuning_addr);
  return shape;
}

// int64 [B, T - n_vis] contiguous attention mask on the device (undefined in cls mode, where it is not read).
at::Tensor prepare_mask(const c10::optional<at::Tensor>& attn_mask, bool cls, int n_vis, int64_t B, int64_t T) {
  at::Tensor mask;
  if (cls) return mask;
  TORCH_CHECK_VALUE(attn_mask.has_value() && attn_mask->defined(), "attention_mask is required");
  mask = *attn_mask;
  TORCH_CHECK(mask.is_cuda(), "attention_mask is on ", mask.device(),
              ": the distillation path runs only as sm_100a CUDA kernels (there is no CPU fallback)");
  if (mask.scalar_type() != at::kLong) mask = mask.to(at::kLong);
  TORCH_CHECK_VALUE(mask.dim() == 2 && mask.size(0) == B && mask.size(1) == T - n_vis, "attention_mask shape ",
                    mask.sizes(), " != (B, T - n_vis) = (", B, ", ", T - n_vis, ")");
  if (!mask.is_contiguous()) mask = mask.contiguous();
  return mask;
}

// One scratch allocation: the partial-sum workspace, then [the scale table,] then [the sharded fp64 sums].
struct Scratch {
  at::Tensor buf;
  char* ws = nullptr;
  float* bwd_scale = nullptr;
  double* sums = nullptr;
};

Scratch alloc_scratch(int L, c10::Device device, bool with_scale, bool sharded) {
  const size_t ws_bytes = (api().ws_bytes(L) + 255) & ~(size_t)255;
  const size_t scale_bytes = with_scale ? ((size_t)8 * L + 255) & ~(size_t)255 : 0;
  const size_t sums_bytes = sharded ? (size_t)8 * (2 * L + 2) : 0;
  Scratch sc;
  sc.buf = at::empty({(int64_t)(ws_bytes + scale_bytes + sums_bytes)},
                     at::TensorOptions().dtype(at::kByte).device(device));
  sc.ws = reinterpret_cast<char*>(sc.buf.data_ptr());
  if (with_scale) sc.bwd_scale = reinterpret_cast<float*>(sc.ws + ws_bytes);
  if (sharded) sc.sums = reinterpret_cast<double*>(sc.ws + ws_bytes + scale_bytes);
  return sc;
}

at::Tensor alloc_out(int L, c10::Device device) {
  return at::empty({1 + 3 * (int64_t)L}, at::TensorOptions().dtype(at::kFloat).device(device));
}

void launch_step(const mafed_shape_t& shape, const Tables& tb, const at::Tensor& mask, const mafed_weights_t& w,
                 float fixed, const Scratch& sc, float* out, float* bwd_scale, int64_t* lang, int64_t* image,
                 int64_t comm, const int64_t* ticket, cudaStream_t stream) {
  check_rc(api().step(&shape, tb.s, tb.t, tb.g, mask.defined() ? mask.data_ptr<int64_t>() : nullptr, &w, fixed, sc.ws,
                      out, bwd_scale, sc.sums, lang, image, reinterpret_cast<mafed_comm_t*>(comm), ticket, stream),
           "mafed_distill_step");
}

void launch_fwd_step(const mafed_shape_t& shape, const Tables& tb, const at::Tensor& mask, const mafed_weights_t& w,
                     const Scratch& sc, float* out, float* bwd_scale, int64_t* lang, int64_t* image, int64_t comm,
                     cudaStream_t stream) {
  const int64_t* mask_ptr = mask.defined() ? mask.data_ptr<int64_t>() : nullptr;
  check_rc(api().fwd_step(&shape, tb.s, tb.t, mask_ptr, &w, sc.ws, out, bwd_scale, sc.sums,
                          reinterpret_cast<mafed_comm_t*>(comm), stream),
           "mafed_distill_fwd_step");
  if (lang != nullptr) check_rc(api().modality_masks(&shape, mask_ptr, lang, image, stream), "mafed_distill_modality_masks");
}

// The gate (skip != nullptr) or the full backward into the pointers of `tb.g`.  g: the device fp32 upstream gradient.
void launch_bwd(const mafed_shape_t& shape, const Tables& tb, const at::Tensor& mask, const float* bwd_scale,
                const at::Tensor& g, float grad_out_scale, const float* skip, float* seen, cudaStream_t stream) {
  check_rc(api().bwd(&shape, tb.s, tb.t, tb.g, mask.defined() ? mask.data_ptr<int64_t>() : nullptr, bwd_scale,
                     g.data_ptr<float>(), grad_out_scale, skip, seen, stream),
           "mafed_distill_bwd");
}

void launch_cached_step(const mafed_shape_t& shape, const Tables& tb, const CacheRef& c, const at::Tensor& mask,
                        const mafed_weights_t& w, float fixed, const Scratch& sc, float* out, float* bwd_scale,
                        int64_t* lang, int64_t* image, cudaStream_t stream) {
  const CachedApi& a = cached_api();
  const int rc = a.step(&shape, tb.s, tb.t, c.M, c.T_c, c.idx.data(), tb.g, mask.defined() ? mask.data_ptr<int64_t>() : nullptr,
                        &w, fixed, sc.ws, out, bwd_scale, sc.sums, lang, image, stream);
  TORCH_CHECK(rc == 0, "mafed_cached_step failed: ", a.error_string(rc), " (code ", rc, ")");
}

void launch_cached_bwd(const mafed_shape_t& shape, const Tables& tb, const CacheRef& c, const at::Tensor& mask,
                       const float* bwd_scale, const at::Tensor& g, float grad_out_scale, const float* skip, float* seen,
                       cudaStream_t stream) {
  const CachedApi& a = cached_api();
  const int rc = a.bwd(&shape, tb.s, tb.t, c.M, c.T_c, c.idx.data(), tb.g, mask.defined() ? mask.data_ptr<int64_t>() : nullptr,
                       bwd_scale, g.data_ptr<float>(), grad_out_scale, skip, seen, stream);
  TORCH_CHECK(rc == 0, "mafed_cached_step_bwd failed: ", a.error_string(rc), " (code ", rc, ")");
}

// The upstream gradient as the kernels read it: fp32, contiguous, on `device`.
at::Tensor upstream(at::Tensor g, c10::Device device) {
  if (g.scalar_type() != at::kFloat || g.device() != device) g = g.to(device, at::kFloat);
  if (!g.is_contiguous()) g = g.contiguous();
  return g;
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
  std::shared_ptr<CacheRef> cache;  // a step read from the teacher cache: `teachers` are the cache tensors

  std::string name() const override { return cache ? "MafedCachedDistillBackward" : "MafedDistillBackward"; }

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
    auto self = shared_from_this();
    std::vector<at::Tensor> s(n), t(n);
    for (size_t i = 0; i < n; ++i) {
      s[i] = students[i].unpack(self);
      t[i] = teachers[i].unpack(self);
    }
    Tables tb;
    fill_tables(s, t, tb);
    at::Tensor m;
    if (has_mask) m = mask.unpack(self);
    const auto device = s[0].device();
    c10::cuda::CUDAGuard guard(device);
    const cudaStream_t stream = c10::cuda::getCurrentCUDAStream(device.index()).stream();
    at::AutoDispatchBelowADInplaceOrView below;
    const at::Tensor g = upstream(grads_in[0], device);
    shape.tuning = has_tuning ? &tuning : nullptr;

    const int64_t n_need = count_needs(needs);
    const bool gate = grad_buf.defined();   // one-pass step: gradients exist, fix them up only if g differs
    const at::Tensor buf = gate ? grad_buf : alloc_grads(n_need, s[0], plan->cls);
    fill_grad_ptrs(buf, needs, tb);
    auto views = layer_views(buf, n_need);
    for (size_t i = 0, j = 0; i < n; ++i)
      if (needs[i]) out[i] = std::move(views[j++]);
    const float fixed = plan->fixed();
    if (cache)   // the full-grid fix-up (libmafed_cached_step.so starts nothing from the device)
      launch_cached_bwd(shape, tb, *cache, m, bwd_scale, g, (float)plan->grad_multiplier, gate ? &fixed : nullptr,
                        gate ? seen : nullptr, stream);
    else
      launch_bwd(shape, tb, m, bwd_scale, g, (float)plan->grad_multiplier, gate ? &fixed : nullptr,
                 gate ? seen : nullptr, stream);
    grad_buf.reset();   // handed to autograd: a second backward (retain_graph) recomputes into a fresh buffer
    return out;
  }
};

// ---------------------------------------------------------------- forward
// students / teachers: the selected [B, T, D] hidden states (same shape and device; one dtype, or fp32 students with
// bf16 / fp16 teachers -- other mixes, the refused pairs, are up-cast to fp32).  attn_mask: int64 [B, T - n_vis]
// (ignored in cls mode).  masks_out: None, an int64 [2, B, T] tensor, or True to have one allocated here; it receives
// (lang_masks, image_masks).  comm: a mafed_comm_t* (0: single rank).  ticket: optional int64[4] from
// prefetch_counts.  seen: optional pinned float[1].
// Returns (total, aux, masks): the 0-dim fp32 loss with the node attached, the [3L] layer / (text, vision) losses,
// and the [2, B, T] mask tensor (None if not requested).
// cache: a one-pass step whose teachers are the [M, T_c, D] tensors of the teacher cache (distill_cached).
std::tuple<at::Tensor, at::Tensor, c10::optional<at::Tensor>> distill_impl(
    const std::shared_ptr<Plan>& plan, std::vector<at::Tensor> students, std::vector<at::Tensor> teachers,
    const c10::optional<at::Tensor>& attn_mask, const py::object& masks_out, int64_t comm,
    const std::shared_ptr<CountsTicket>& ticket, const c10::optional<at::Tensor>& seen, int64_t tuning_addr,
    const std::shared_ptr<CacheRef>& cache) {
  const int L = plan->n_layers;
  TORCH_CHECK((int)students.size() == L && (int)teachers.size() == L, "students / teachers / plan length mismatch");
  if (!cache) {
    // One dtype everywhere, or fp32 students with teachers of one half-precision dtype: the kernels read the tensors
    // as they are (a teacher pair, MAFED_DTYPE_PAIR).  distill_loss gives each dtype group of a step its own call, so
    // any other mix arriving here is the one group of pairs the kernels refuse (a student narrower than its teacher,
    // bf16 against fp16).  It is up-cast to fp32 on both sides, which is what the reference's autocast region does to
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
  const auto device = s0.device();
  const bool grad_mode = at::GradMode::is_enabled();
  std::vector<bool> needs(L, false);
  bool any_need = false;
  for (int i = 0; i < L; ++i) {
    at::Tensor& s = students[i];
    at::Tensor& t = teachers[i];
    if (cache) {
      TORCH_CHECK_VALUE(s.sizes() == s0.sizes() && t.dim() == 3 && t.size(0) == cache->M && t.size(1) == cache->T_c &&
                            t.size(2) == s0.size(2) && t.is_contiguous(),
                        "the teacher cache must hold one contiguous [M, T_c, D] tensor per selected layer");
    } else {
      TORCH_CHECK_VALUE(s.sizes() == s0.sizes() && t.sizes() == s0.sizes(),
                        "all selected hidden states must share one [B, T, D] shape");
    }
    TORCH_CHECK_VALUE(s.scalar_type() == s0.scalar_type() && t.scalar_type() == teachers[0].scalar_type() &&
                          s.device() == device && t.device() == device,
                      "student / teacher dtype or device mismatch");
    needs[i] = grad_mode && s.requires_grad();
    any_need = any_need || needs[i];
  }
  TORCH_CHECK(!cache || (plan->single_pass && any_need && comm == 0 && ticket == nullptr && !plan->cls),
              "distill_cached runs the one-pass step of one rank with gradients (single_pass, no CLS)");
  // collect the graph edges before the tensors are replaced by contiguous copies
  torch::autograd::edge_list edges;
  if (any_need) edges = torch::autograd::collect_next_edges(students);

  at::AutoDispatchBelowADInplaceOrView below;
  for (int i = 0; i < L; ++i) {
    if (!students[i].is_contiguous()) students[i] = students[i].contiguous();
    if (!teachers[i].is_contiguous()) teachers[i] = teachers[i].contiguous();
  }
  const int64_t B = s0.size(0), T = s0.size(1);
  const mafed_shape_t shape = make_shape(s0, teachers[0], L, plan->loss_kind, plan->cls, plan->n_vis, tuning_addr);
  const at::Tensor mask = prepare_mask(attn_mask, plan->cls, plan->n_vis, B, T);

  c10::cuda::CUDAGuard guard(device);
  const cudaStream_t stream = c10::cuda::getCurrentCUDAStream(device.index()).stream();
  const Scratch sc = alloc_scratch(L, device, /*with_scale=*/true, /*sharded=*/comm != 0);
  const at::Tensor scratch = sc.buf;
  float* bwd_scale = sc.bwd_scale;
  at::Tensor out = alloc_out(L, device);
  Tables tb;
  fill_tables(students, teachers, tb);
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
  const int64_t* ticket_ptr = nullptr;
  if (ticket != nullptr) {
    ticket->wait();     // this stream behind the prefetch launch (a no-op wait: it finished a forward pass ago)
    ticket_ptr = ticket->tensor.data_ptr<int64_t>();
  }

  at::Tensor grad_buf;
  if (plan->single_pass && any_need) {
    grad_buf = alloc_grads(count_needs(needs), s0, plan->cls);
    fill_grad_ptrs(grad_buf, needs, tb);
    if (cache)
      launch_cached_step(shape, tb, *cache, mask, plan->w, plan->fixed(), sc, out.data_ptr<float>(), bwd_scale, lang,
                         image, stream);
    else
      launch_step(shape, tb, mask, plan->w, plan->fixed(), sc, out.data_ptr<float>(), bwd_scale, lang, image, comm,
                  ticket_ptr, stream);
  } else {
    launch_fwd_step(shape, tb, mask, plan->w, sc, out.data_ptr<float>(), bwd_scale, lang, image, comm, stream);
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
    node->cache = cache;
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

std::tuple<at::Tensor, at::Tensor, c10::optional<at::Tensor>> distill(
    const std::shared_ptr<Plan>& plan, std::vector<at::Tensor> students, std::vector<at::Tensor> teachers,
    const c10::optional<at::Tensor>& attn_mask, const py::object& masks_out, int64_t comm,
    const std::shared_ptr<CountsTicket>& ticket, const c10::optional<at::Tensor>& seen, int64_t tuning_addr) {
  return distill_impl(plan, std::move(students), std::move(teachers), attn_mask, masks_out, comm, ticket, seen,
                      tuning_addr, nullptr);
}

// The one-pass step of one rank with the teacher rows read straight from the teacher cache: `cache` holds one
// contiguous [M, T_c, D] tensor per selected layer, `idx` the B memory indices of the batch (each in [0, M)).  Same
// result and node as `distill` on the gathered teachers; the node keeps the cache tensors (version-checked) and runs the
// library's full-grid fix-up as its backward.  The caller asks `cached_supported` first.
std::tuple<at::Tensor, at::Tensor, c10::optional<at::Tensor>> distill_cached(
    const std::shared_ptr<Plan>& plan, std::vector<at::Tensor> students, std::vector<at::Tensor> cache,
    std::vector<int64_t> idx, int64_t T_c, const c10::optional<at::Tensor>& attn_mask, const py::object& masks_out,
    const c10::optional<at::Tensor>& seen, int64_t tuning_addr) {
  cached_api();
  TORCH_CHECK_VALUE(!cache.empty() && cache[0].dim() == 3, "the teacher cache must hold [M, T_c, D] tensors");
  TORCH_CHECK_VALUE(!students.empty() && students[0].dim() == 3 && (int64_t)idx.size() == students[0].size(0),
                    "one memory index per sample of the batch");
  auto ref = std::make_shared<CacheRef>();
  ref->idx = std::move(idx);
  ref->M = cache[0].size(0);
  ref->T_c = (int32_t)T_c;
  return distill_impl(plan, std::move(students), std::move(cache), attn_mask, masks_out, 0, nullptr, seen, tuning_addr,
                      ref);
}

// Does libmafed_cached_step.so take this step (mafed_cached_step_supported)?  False for dtype mixes it has no kernel
// for; the caller then gathers the teacher rows and runs `distill`.
bool cached_supported(const std::shared_ptr<Plan>& plan, const std::vector<at::Tensor>& students,
                      const std::vector<at::Tensor>& cache, int64_t T_c, int64_t tuning_addr) {
  const CachedApi& a = cached_api();
  const int L = plan->n_layers;
  if ((int)students.size() != L || (int)cache.size() != L || plan->cls) return false;
  const at::Tensor& s0 = students[0];
  const at::Tensor& c0 = cache[0];
  if (s0.dim() != 3 || c0.dim() != 3 || !s0.is_cuda()) return false;
  const auto st = s0.scalar_type(), ct = c0.scalar_type();
  const bool native = st == ct || (st == at::kFloat && (ct == at::kBFloat16 || ct == at::kHalf));
  if (!native || (st != at::kFloat && st != at::kBFloat16 && st != at::kHalf)) return false;
  Tables tb;
  for (int i = 0; i < L; ++i) {
    const at::Tensor& s = students[i];
    const at::Tensor& c = cache[i];
    if (s.sizes() != s0.sizes() || s.scalar_type() != st || !s.is_contiguous() || s.device() != s0.device() ||
        c.sizes() != c0.sizes() || c.scalar_type() != ct || !c.is_contiguous() || c.device() != s0.device() ||
        c.size(2) != s0.size(2) || c.size(1) != T_c)
      return false;
    tb.s[i] = s.data_ptr();
    tb.t[i] = c.data_ptr();
  }
  const mafed_shape_t shape = make_shape(s0, c0, L, plan->loss_kind, false, plan->n_vis, tuning_addr);
  return a.supported(&shape, tb.s, tb.t, c0.size(0), (int32_t)T_c) == 1;
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

// ---------------------------------------------------------------- the step as torch.library ops
// `mafed::step`, `mafed::fwd_step` and `mafed::bwd` are the three C-ABI calls of a step as dispatcher ops, so that
// torch.compile can trace a step into the caller's graph (the pybind `distill` above builds its own autograd node,
// which Dynamo cannot trace).  Their fake implementations and the autograd formula live in mafed_b200/ops.py.  The
// plan arrives as plain values; the workspace is scratch from the caching allocator, as in `distill`.  The ops take
// one dtype everywhere, or fp32 students with bf16 / fp16 teachers: the caller splits a step into dtype groups and
// up-casts a group of refused pairs.

struct OpInputs {
  std::vector<at::Tensor> students, teachers;
  at::Tensor mask;
  mafed_shape_t shape;
  Tables tb;
};

OpInputs op_inputs(const at::TensorList students, const at::TensorList teachers, const c10::optional<at::Tensor>& mask,
                   int64_t loss_kind, bool cls, int64_t n_vis, int64_t tuning) {
  const int64_t L = (int64_t)students.size();
  TORCH_CHECK(L >= 1 && L <= MAFED_MAX_LAYERS, "1..", MAFED_MAX_LAYERS, " layers per call");
  TORCH_CHECK((int64_t)teachers.size() == L, "students / teachers length mismatch");
  OpInputs in;
  const at::Tensor& s0 = students[0];
  const at::Tensor& t0 = teachers[0];
  TORCH_CHECK_VALUE(s0.dim() == 3, "hidden states must be [B, T, D]");
  const bool native = s0.scalar_type() == t0.scalar_type() ||
                      (s0.scalar_type() == at::kFloat && (t0.scalar_type() == at::kBFloat16 || t0.scalar_type() == at::kHalf));
  TORCH_CHECK_TYPE(native, "student / teacher dtypes ", s0.scalar_type(), " / ", t0.scalar_type(),
                   ": one dtype, or float32 students with bfloat16 or float16 teachers");
  for (int64_t i = 0; i < L; ++i) {
    TORCH_CHECK_VALUE(students[i].sizes() == s0.sizes() && teachers[i].sizes() == s0.sizes(),
                      "all selected hidden states must share one [B, T, D] shape");
    TORCH_CHECK_VALUE(students[i].scalar_type() == s0.scalar_type() && teachers[i].scalar_type() == t0.scalar_type() &&
                          students[i].device() == s0.device() && teachers[i].device() == s0.device(),
                      "student / teacher dtype or device mismatch");
    in.students.push_back(students[i].contiguous());
    in.teachers.push_back(teachers[i].contiguous());
  }
  in.shape = make_shape(s0, t0, (int)L, (int)loss_kind, cls, (int)n_vis, tuning);
  in.mask = prepare_mask(mask, cls, (int)n_vis, s0.size(0), s0.size(1));
  fill_tables(in.students, in.teachers, in.tb);
  return in;
}

mafed_weights_t op_weights(int64_t L, at::ArrayRef<double> layer_coeffs, const c10::optional<at::ArrayRef<double>>& lang_weights,
                           int64_t modality_kind, double distill_coeff) {
  TORCH_CHECK((int64_t)layer_coeffs.size() == L, "layer_coeffs / students length mismatch");
  c10::optional<std::vector<double>> lw;
  if (lang_weights.has_value()) lw = lang_weights->vec();
  return Plan((int)modality_kind, distill_coeff, layer_coeffs.vec(), lw, MAFED_LOSS_MSE, false, 0, 1.0, true, 1.0).w;
}

std::vector<bool> op_needs(c10::List<bool> needs, int64_t L) {
  TORCH_CHECK((int64_t)needs.size() == L, "needs / students length mismatch");
  std::vector<bool> v(needs.begin(), needs.end());
  return v;
}

at::Tensor op_masks(bool want, bool cls, const at::Tensor& s0) {
  const auto opts = at::TensorOptions().dtype(at::kLong).device(s0.device());
  return want && !cls ? at::empty({2, s0.size(0), s0.size(1)}, opts) : at::empty({0}, opts);
}

// -> (out [1 + 3L]: total, then aux; grads [n_need, B, T, D]; bwd_scale [2L]; masks [2, B, T] or [0])
std::tuple<at::Tensor, at::Tensor, at::Tensor, at::Tensor> op_step(
    at::TensorList students, at::TensorList teachers, const c10::optional<at::Tensor>& mask,
    at::ArrayRef<double> layer_coeffs, c10::optional<at::ArrayRef<double>> lang_weights, int64_t modality_kind,
    double distill_coeff, int64_t loss_kind, bool cls, int64_t n_vis, double assumed_grad_out, double grad_multiplier,
    c10::List<bool> needs, int64_t comm, bool want_masks, int64_t tuning) {
  const int64_t L = (int64_t)students.size();
  OpInputs in = op_inputs(students, teachers, mask, loss_kind, cls, n_vis, tuning);
  const mafed_weights_t w = op_weights(L, layer_coeffs, lang_weights, modality_kind, distill_coeff);
  const std::vector<bool> nd = op_needs(needs, L);
  const at::Tensor& s0 = in.students[0];
  const auto device = s0.device();
  c10::cuda::CUDAGuard guard(device);
  const cudaStream_t stream = c10::cuda::getCurrentCUDAStream(device.index()).stream();
  const Scratch sc = alloc_scratch((int)L, device, /*with_scale=*/false, /*sharded=*/comm != 0);
  at::Tensor out = alloc_out((int)L, device);
  at::Tensor bwd_scale = at::empty({2 * L}, at::TensorOptions().dtype(at::kFloat).device(device));
  at::Tensor grads = alloc_grads(count_needs(nd), s0, cls);
  at::Tensor masks = op_masks(want_masks, cls, s0);
  int64_t* lang = masks.numel() ? masks.data_ptr<int64_t>() : nullptr;
  fill_grad_ptrs(grads, nd, in.tb);
  launch_step(in.shape, in.tb, in.mask, w, (float)(assumed_grad_out * grad_multiplier), sc, out.data_ptr<float>(),
              bwd_scale.data_ptr<float>(), lang, lang ? lang + s0.size(0) * s0.size(1) : nullptr, comm, nullptr, stream);
  return std::make_tuple(out, grads, bwd_scale, masks);
}

// -> (out [1 + 3L]: total, then aux; bwd_scale [2L]; masks [2, B, T] or [0])
std::tuple<at::Tensor, at::Tensor, at::Tensor> op_fwd_step(
    at::TensorList students, at::TensorList teachers, const c10::optional<at::Tensor>& mask,
    at::ArrayRef<double> layer_coeffs, c10::optional<at::ArrayRef<double>> lang_weights, int64_t modality_kind,
    double distill_coeff, int64_t loss_kind, bool cls, int64_t n_vis, double grad_multiplier, c10::List<bool> needs,
    int64_t comm, bool want_masks, int64_t tuning) {
  // grad_multiplier and needs are read by the autograd formula (its backward), not by the launch
  const int64_t L = (int64_t)students.size();
  op_needs(needs, L);
  OpInputs in = op_inputs(students, teachers, mask, loss_kind, cls, n_vis, tuning);
  const mafed_weights_t w = op_weights(L, layer_coeffs, lang_weights, modality_kind, distill_coeff);
  const at::Tensor& s0 = in.students[0];
  const auto device = s0.device();
  c10::cuda::CUDAGuard guard(device);
  const cudaStream_t stream = c10::cuda::getCurrentCUDAStream(device.index()).stream();
  const Scratch sc = alloc_scratch((int)L, device, /*with_scale=*/false, /*sharded=*/comm != 0);
  at::Tensor out = alloc_out((int)L, device);
  at::Tensor bwd_scale = at::empty({2 * L}, at::TensorOptions().dtype(at::kFloat).device(device));
  at::Tensor masks = op_masks(want_masks, cls, s0);
  int64_t* lang = masks.numel() ? masks.data_ptr<int64_t>() : nullptr;
  launch_fwd_step(in.shape, in.tb, in.mask, w, sc, out.data_ptr<float>(), bwd_scale.data_ptr<float>(), lang,
                  lang ? lang + s0.size(0) * s0.size(1) : nullptr, comm, stream);
  return std::make_tuple(out, bwd_scale, masks);
}

// The backward into `grads` ([n_need, B, T, D], mutated).  With `skip_if_equals` it is the one-pass step's 1-CTA gate:
// nothing happens when grad_out * grad_out_scale equals it, otherwise the exact backward overwrites `grads`.
void op_bwd(at::TensorList students, at::TensorList teachers, const c10::optional<at::Tensor>& mask,
            const at::Tensor& grads, const at::Tensor& bwd_scale, const at::Tensor& grad_out, double grad_out_scale,
            c10::optional<double> skip_if_equals, c10::List<bool> needs, int64_t loss_kind, bool cls, int64_t n_vis,
            int64_t tuning) {
  const int64_t L = (int64_t)students.size();
  OpInputs in = op_inputs(students, teachers, mask, loss_kind, cls, n_vis, tuning);
  const std::vector<bool> nd = op_needs(needs, L);
  const at::Tensor& s0 = in.students[0];
  TORCH_CHECK_VALUE(grads.is_contiguous() && grads.scalar_type() == s0.scalar_type() && grads.dim() == 4 &&
                        grads.size(0) == count_needs(nd) && grads.sizes().slice(1) == s0.sizes(),
                    "grads must be a contiguous [n_need, B, T, D] tensor of the student dtype");
  TORCH_CHECK_VALUE(bwd_scale.is_contiguous() && bwd_scale.scalar_type() == at::kFloat && bwd_scale.numel() == 2 * L,
                    "bwd_scale must be a contiguous float32 [2L] tensor");
  const auto device = s0.device();
  c10::cuda::CUDAGuard guard(device);
  const cudaStream_t stream = c10::cuda::getCurrentCUDAStream(device.index()).stream();
  const at::Tensor g = upstream(grad_out, device);
  fill_grad_ptrs(grads, nd, in.tb);
  const float skip = skip_if_equals.has_value() ? (float)*skip_if_equals : 0.f;
  launch_bwd(in.shape, in.tb, in.mask, bwd_scale.data_ptr<float>(), g, (float)grad_out_scale,
             skip_if_equals.has_value() ? &skip : nullptr, nullptr, stream);
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
  m.def("bind_cached", &bind_cached, "dlopen libmafed_cached_step.so and resolve its C ABI");
  m.def("cached_bound", [] { return g_cached.bound; });
  m.def("distill_cached", &distill_cached, py::arg("plan"), py::arg("students"), py::arg("cache"), py::arg("idx"),
        py::arg("T_c"), py::arg("attn_mask"), py::arg("masks_out"), py::arg("seen"), py::arg("tuning"));
  m.def("cached_supported", &cached_supported, py::arg("plan"), py::arg("students"), py::arg("cache"), py::arg("T_c"),
        py::arg("tuning"));
  m.def("prefetch_counts", &prefetch_counts, py::arg("attn_mask"), py::arg("n_vis"), py::arg("comm"), py::arg("tuning"));
}

TORCH_LIBRARY(mafed, m) {
  m.def("step(Tensor[] students, Tensor[] teachers, Tensor? mask, float[] layer_coeffs, float[]? lang_weights, "
        "int modality_kind, float distill_coeff, int loss_kind, bool cls, int n_vis, float assumed_grad_out, "
        "float grad_multiplier, bool[] needs, int comm, bool want_masks, int tuning) -> (Tensor, Tensor, Tensor, Tensor)");
  m.def("fwd_step(Tensor[] students, Tensor[] teachers, Tensor? mask, float[] layer_coeffs, float[]? lang_weights, "
        "int modality_kind, float distill_coeff, int loss_kind, bool cls, int n_vis, float grad_multiplier, bool[] needs, "
        "int comm, bool want_masks, int tuning) -> (Tensor, Tensor, Tensor)");
  m.def("bwd(Tensor[] students, Tensor[] teachers, Tensor? mask, Tensor(a!) grads, Tensor bwd_scale, Tensor grad_out, "
        "float grad_out_scale, float? skip_if_equals, bool[] needs, int loss_kind, bool cls, int n_vis, int tuning) -> ()");
}

TORCH_LIBRARY_IMPL(mafed, CUDA, m) {
  m.impl("step", &op_step);
  m.impl("fwd_step", &op_fwd_step);
  m.impl("bwd", &op_bwd);
}
