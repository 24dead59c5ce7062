// The one-pass step of a replay batch with its teacher rows read straight from the per-task teacher cache
// (include/mafed_cached_step.h).  The kernels are the TMA-ring step and backward of libmafed_distill.so
// (distill_tma.cuh) with the CacheTeacher addressing: the producer warp copies each sample's teacher rows out of the
// [M, T_c, D] cache instead of a gathered [B, T, D] tensor; ring, stage layout and consumers are the same, so the
// results are those of the gather followed by the ordinary step.
//
// A library of its own, so that libmafed_distill.so keeps its export list.  It launches every kernel with a plain
// stream launch (no programmatic-dependent-launch attribute): libmafed_distill.so remembers the streams its gate went
// to and launches its next kernel there fully serialised, but it cannot see this library's launches, and a persistent
// grid launched as a programmatic dependent right behind a gate could hold the SMs a backward started by that gate
// needs.  For the same reason the backward is the full-grid fix-up, which starts nothing from the device.
#include <atomic>
#include <cstring>

#include "distill_common.cuh"
#include "distill_dispatch.cuh"
#include "distill_epilogue.cuh"
#include "distill_tma.cuh"
#include "mafed_cached_step.h"

namespace mafed {
namespace {

static_assert(kCacheMaxSamples == MAFED_CACHED_MAX_SAMPLES, "index table capacity");

// Arrival counters of the in-kernel tail, as in distill_abi.cu (this library's own pool): zero whenever no kernel uses
// one, taken round-robin; launches recorded into a CUDA graph draw from the other half.
constexpr unsigned kDoneSlots = 256;
__device__ unsigned int g_cached_tail_done[kDoneSlots];
std::atomic<unsigned> g_tail_next{0};
std::atomic<unsigned> g_tail_next_captured{0};

unsigned int* next_tail_counter(cudaStream_t st) {
  static unsigned int* base[kMaxDevices] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return nullptr;
  if (base[dev] == nullptr) {
    void* p = nullptr;
    if (cudaGetSymbolAddress(&p, g_cached_tail_done) != cudaSuccess) return nullptr;
    base[dev] = reinterpret_cast<unsigned int*>(p);
  }
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) return nullptr;
  constexpr unsigned half = kDoneSlots / 2;
  if (cap == cudaStreamCaptureStatusActive) return base[dev] + half + (g_tail_next_captured.fetch_add(1) % half);
  return base[dev] + (g_tail_next.fetch_add(1) % half);
}

// What mafed_cached_step_supported checks, as a pure function of the arguments.  It is the TMA-ring eligibility of
// the step on gathered tensors (vector_path + tma_geometry in distill_dispatch.cuh) plus the cache's own alignment; the
// shared-memory budget of tma_geometry always admits a ring of rows <= 32 KB on sm_100 (227 KB per block).
bool supported(const mafed_shape_t* sh, const void* const* student_ptrs, const void* const* cache_ptrs, int64_t M,
               int32_t T_c) {
  if (check_shape(sh) != 0 || sh->cls || !student_ptrs || !cache_ptrs) return false;
  if (sh->B > kCacheMaxSamples || M < 1 || M > INT32_MAX || T_c < sh->T) return false;
  if ((long long)sh->B * sh->T > INT32_MAX) return false;
  if (tune(*sh, MAFED_TUNE_NO_TAIL) || chosen_variant(*sh) != 2) return false;
  const long long row_bytes = (long long)sh->D * (long long)student_size(*sh);
  if (row_bytes % 16 != 0 || row_bytes > 32768) return false;
  if (mixed_pair(*sh) && sh->D % 8 != 0) return false;
  for (int l = 0; l < sh->n_layers; ++l)
    if (!student_ptrs[l] || !cache_ptrs[l] || !aligned_to(student_ptrs[l], 16) || !aligned_to(cache_ptrs[l], 16))
      return false;
  return true;
}

// Argument checks shared by the step and its backward, then the kernel parameters: PathParams as the ordinary step
// fills them (the teacher table holds the cache pointers) and the index table.  Everything that can be checked
// without a device is checked first.
int fill_cached(const mafed_shape_t* sh, const void* const* student_ptrs, const void* const* cache_ptrs, int64_t M,
                int32_t T_c, const int64_t* idx, void* const* grad_ptrs, const int64_t* attn_mask, PathParams& p,
                CacheTeacher& c) {
  int rc = check_shape(sh);
  if (rc) return rc;
  if (!student_ptrs || !cache_ptrs || !idx || !grad_ptrs || (needs_mask(*sh) && !attn_mask)) return MAFED_E_ARG;
  if (sh->cls || sh->B > kCacheMaxSamples || M < 1 || M > INT32_MAX || T_c < sh->T) return MAFED_E_ARG;
  for (int b = 0; b < sh->B; ++b)
    if (idx[b] < 0 || idx[b] >= M) return MAFED_E_ARG;
  if (!supported(sh, student_ptrs, cache_ptrs, M, T_c)) return MAFED_E_ARG;
  rc = fill_params(sh, student_ptrs, cache_ptrs, grad_ptrs, attn_mask, p);
  if (rc) return rc;
  p.n_chunks = (int)((size_t)sh->D * student_size(*sh) / 16);
  memset(&c, 0, sizeof(c));
  for (int b = 0; b < sh->B; ++b) c.idx[b] = (int32_t)idx[b];
  c.T_c = T_c;
  c.shift = (long long)T_c - sh->T;
  return 0;
}

template <typename T, int LOSS, int MODE, typename TT>
int launch(const PathParams& p, const TmaGeom& geo, const CacheTeacher& c, cudaStream_t st) {
  auto kernel = &k_bwd_tma_cached<T, LOSS, MODE, TT>;
  static bool attr_set[kMaxDevices] = {};
  const DeviceInfo& dv = device_info();
  if (!dv.ok) return MAFED_E_NODEVICE;
  if (!attr_set[dv.index]) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dv.smem_optin - 16 * 1024);
    if (e != cudaSuccess) return (int)e;
    attr_set[dv.index] = true;
  }
  const long long total = ((p.n_rows + geo.rows - 1) / geo.rows) * p.n_layers;
  const unsigned grid = (unsigned)clamp_grid((long long)dv.sm_count, total);   // one persistent CTA per SM
  kernel<<<grid, kTmaConsumerThreads + 32, (size_t)geo.stages * geo.stage_bytes, st>>>(p, geo, c);
  return (int)cudaPeekAtLastError();
}

template <int MODE, typename T, typename TT>
int launch_loss(const mafed_shape_t& sh, const PathParams& p, const TmaGeom& geo, const CacheTeacher& c, cudaStream_t st) {
  if (sh.loss_kind == MAFED_LOSS_MSE) return launch<T, MAFED_LOSS_MSE, MODE, TT>(p, geo, c, st);
  return launch<T, MAFED_LOSS_COSINE, MODE, TT>(p, geo, c, st);
}

// The ring of the pass (the ordinary step's geometry for the same shape), then the kernel of the dtype pair.
template <int MODE>
int run(const mafed_shape_t& sh, const PathParams& p, const CacheTeacher& c, cudaStream_t st) {
  TmaGeom geo;
  if (!tma_geometry(sh, p, MODE == kFused ? kPassFused : kPassBwd, geo, sh.loss_kind)) return MAFED_E_ARG;
  if (mixed_pair(sh)) {
    if (teacher_dtype(sh) == MAFED_BF16) return launch_loss<MODE, float, __nv_bfloat16>(sh, p, geo, c, st);
    return launch_loss<MODE, float, __half>(sh, p, geo, c, st);
  }
  switch (student_dtype(sh)) {
    case MAFED_F32: return launch_loss<MODE, float, float>(sh, p, geo, c, st);
    case MAFED_BF16: return launch_loss<MODE, __nv_bfloat16, __nv_bfloat16>(sh, p, geo, c, st);
    default: return launch_loss<MODE, __half, __half>(sh, p, geo, c, st);
  }
}

}  // namespace
}  // namespace mafed

using namespace mafed;

extern "C" {

int mafed_cached_step_abi_version(void) { return MAFED_CACHED_ABI_VERSION; }

const char* mafed_cached_step_error_string(int code) {
  switch (code) {
    case 0: return "ok";
    case MAFED_E_ARG:
      return "invalid argument (null pointer, a memory index outside [0, M), T > T_c, T < n_vis, more than 2048 "
             "samples, or a step mafed_cached_step_supported refuses)";
    case MAFED_E_DTYPE: return "unsupported dtype or loss kind";
    case MAFED_E_ALIGN: return "pointer not aligned to its element size";
    case MAFED_E_NODEVICE: return "no usable CUDA device";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
  }
}

int mafed_cached_step_supported(const mafed_shape_t* shape, const void* const* student_ptrs,
                                const void* const* cache_ptrs, int64_t M, int32_t T_c) {
  return supported(shape, student_ptrs, cache_ptrs, M, T_c) ? 1 : 0;
}

int mafed_cached_step(const mafed_shape_t* shape, const void* const* student_ptrs, const void* const* cache_ptrs,
                      int64_t M, int32_t T_c, const int64_t* idx, void* const* grad_ptrs, const int64_t* attn_mask,
                      const mafed_weights_t* weights, float assumed_grad_out, void* ws, float* out, float* bwd_scale,
                      double* sums, int64_t* lang_mask, int64_t* image_mask, void* stream) {
  if (!weights || !out || !bwd_scale || !ws) return MAFED_E_ARG;
  if ((lang_mask == nullptr) != (image_mask == nullptr)) return MAFED_E_ARG;
  PathParams p;
  CacheTeacher c;
  int rc = fill_cached(shape, student_ptrs, cache_ptrs, M, T_c, idx, grad_ptrs, attn_mask, p, c);
  const cudaStream_t st = (cudaStream_t)stream;
  unsigned int* done = rc ? nullptr : next_tail_counter(st);
  if (!rc && done == nullptr) rc = (int)cudaErrorInvalidValue;
  if (!rc) {
    // as fused_impl in distill_abi.cu for a single rank whose step folds the losses into the kernel's last CTA
    p.bwd_scale = bwd_scale;
    p.fixed_gout = assumed_grad_out;
    p.ws = reinterpret_cast<float*>(ws);
    p.tail_done = done;
    p.tail_flags = kEpiReduce | kEpiLosses;
    p.tail_out = out;
    p.tail_sums = sums;
    p.lang_mask_out = lang_mask;
    p.image_mask_out = image_mask;
    p.loss_kind = shape->loss_kind;
    p.n_mask = mask_entries(*shape);
    p.n_vis_rows = vis_rows(*shape);
    p.w = *weights;
    if (mask_entries(*shape) <= 16384) {
      // every CTA derives the scale table from the mask itself while its first tiles are in flight
      p.inline_scale = 1;
      p.bwd_scale_out = bwd_scale;
    } else {
      // a large mask: one prologue launch leaves the counts in the ws header for the tail and writes the scale table
      double* counts = reinterpret_cast<double*>(p.ws + kWsCountsAt);
      p.tail_counts_in = counts;
      EpiParams e;
      memset(&e, 0, sizeof(e));
      e.a.mask = attn_mask;
      e.a.counts_out = counts;
      e.a.bwd_scale = bwd_scale;
      e.a.n_mask = mask_entries(*shape);
      e.a.n_vis_rows = vis_rows(*shape);
      e.a.n_layers = shape->n_layers;
      e.a.D = shape->D;
      e.a.loss_kind = shape->loss_kind;
      e.a.flags = MAFED_STAGE_COUNTS | MAFED_STAGE_SCALE;
      e.w = *weights;
      k_epilogue<<<1, kEpiThreads, 0, st>>>(e);
      rc = (int)cudaPeekAtLastError();
    }
    if (!rc) rc = run<kFused>(*shape, p, c, st);
  }
  return rc;
}

int mafed_cached_step_bwd(const mafed_shape_t* shape, const void* const* student_ptrs, const void* const* cache_ptrs,
                          int64_t M, int32_t T_c, const int64_t* idx, void* const* grad_ptrs, const int64_t* attn_mask,
                          const float* bwd_scale, const float* grad_out, float grad_out_scale,
                          const float* skip_if_equals, float* grad_out_seen, void* stream) {
  if (!bwd_scale) return MAFED_E_ARG;
  PathParams p;
  CacheTeacher c;
  int rc = fill_cached(shape, student_ptrs, cache_ptrs, M, T_c, idx, grad_ptrs, attn_mask, p, c);
  if (!rc) {
    p.bwd_scale = bwd_scale;
    p.grad_out = grad_out;
    p.gout_scale = grad_out_scale;
    if (skip_if_equals != nullptr) {   // the fix-up: a full grid whose CTAs return at once when there is nothing to fix
      p.skip_if_gout_equals = 1;
      p.fixed_gout = *skip_if_equals;
    }
    c.gout_seen = grad_out_seen;
    rc = run<kBackward>(*shape, p, c, (cudaStream_t)stream);
  }
  return rc;
}

}  // extern "C"
