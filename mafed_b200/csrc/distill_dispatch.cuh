// Host-side choice of kernel family and launch geometry for one streaming pass, shared by the two
// translation units of the library: distill_abi.cu (every ordinary launch) and distill_gate.cu (the gated
// backward, compiled as relocatable device code because its 1-CTA gate launches the backward from the device).
// The pass is a template parameter so that a unit instantiates only the kernels it launches, and the way a
// kernel is started is a `Launcher` policy: HostLaunch enqueues it on the stream, GateLaunch (distill_gate.cu)
// enqueues a gate that starts it from the device only when it has work to do.
//
// Nothing here is process-global: overrides arrive per call (mafed_shape_t::tuning) and the caches of
// occupancy / opt-in shared memory are per kernel and per device.
#pragma once
#include <cstring>

#include "distill_common.cuh"
#include "distill_ldg.cuh"
#include "distill_tma.cuh"

namespace MAFED_NS {

enum Pass { kPassFwd = 0, kPassBwd = 1, kPassFused = 2 };
constexpr int kMaxDevices = 64;

// key: MAFED_TUNE_* (include/mafed_distill.h)
inline int tune(const mafed_shape_t& sh, int key) { return sh.tuning != nullptr ? sh.tuning->v[key] : 0; }

// Launch with programmatic dependent launch enabled: the kernel may start its prologue while its
// predecessor in the stream is finishing; all kernels here call griddepcontrol.wait before touching
// global memory, so stream-order semantics are unchanged.
template <typename... KArgs, typename... Args>
void launch_pdl(void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t st, bool pdl,
                Args... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// The ordinary launcher: the kernel goes onto the stream.
struct HostLaunch {
  cudaStream_t st;
  bool pdl;
  template <typename Kernel, typename... Args>
  void run(unsigned grid, unsigned block, size_t smem, const Args&... args) const {
    launch_pdl(Kernel::host(), grid, block, smem, st, pdl, args...);
  }
};

struct DeviceInfo {
  int index = -1;
  int sm_count = 0;
  int smem_optin = 0;
  bool ok = false;
};

inline const DeviceInfo& device_info() {
  static DeviceInfo info[kMaxDevices];
  static DeviceInfo none;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return none;
  DeviceInfo& d = info[dev];
  if (!d.ok) {
    cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&d.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    d.index = dev;
    d.ok = d.sm_count > 0;
  }
  return d;
}

inline int check_shape(const mafed_shape_t* sh) {
  if (sh == nullptr) return MAFED_E_ARG;
  if (sh->n_layers < 1 || sh->n_layers > kMaxLayers) return MAFED_E_ARG;
  if (sh->B < 1 || sh->T < 1 || sh->D < 1 || sh->n_vis < 0 || sh->n_vis > sh->T) return MAFED_E_ARG;
  if (sh->dtype < MAFED_F32 || sh->dtype > MAFED_F16) return MAFED_E_DTYPE;
  if (sh->loss_kind != MAFED_LOSS_MSE && sh->loss_kind != MAFED_LOSS_COSINE) return MAFED_E_DTYPE;
  return 0;
}

inline size_t elem_size(int dtype) { return dtype == MAFED_F32 ? 4 : 2; }

// Fill the geometry part of PathParams.  CLS mode (distillation.py:251-257) is the same path over
// B rows (position 0 of every sample), all of them "visual", T*D elements apart.
inline void fill_geometry(const mafed_shape_t& sh, PathParams& p) {
  p.n_layers = sh.n_layers;
  p.D = sh.D;
  if (sh.cls) {
    p.n_rows = sh.B;
    p.row_stride = (long long)sh.T * sh.D;
    p.T = 1;
    p.n_vis = 1;
    p.txt = 0;
  } else {
    p.n_rows = (long long)sh.B * sh.T;
    p.row_stride = sh.D;
    p.T = sh.T;
    p.n_vis = sh.n_vis;
    p.txt = sh.T - sh.n_vis;
  }
}

inline bool aligned_to(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }
inline bool needs_mask(const mafed_shape_t& sh) { return !sh.cls && sh.T > sh.n_vis; }
inline long long mask_entries(const mafed_shape_t& sh) {
  return needs_mask(sh) ? (long long)sh.B * (sh.T - sh.n_vis) : 0;
}
inline double vis_rows(const mafed_shape_t& sh) { return sh.cls ? (double)sh.B : (double)sh.B * (double)sh.n_vis; }

// Common argument checks + pointer-table copy for the three streaming passes.
inline int fill_params(const mafed_shape_t* shape, const void* const* student_ptrs, const void* const* teacher_ptrs,
                       void* const* grad_ptrs, const int64_t* attn_mask, PathParams& p) {
  int rc = check_shape(shape);
  if (rc) return rc;
  if (!student_ptrs || !teacher_ptrs || (needs_mask(*shape) && !attn_mask)) return MAFED_E_ARG;
  if (!device_info().ok) return MAFED_E_NODEVICE;
  memset(&p, 0, sizeof(p));
  fill_geometry(*shape, p);
  p.gout_scale = 1.f;
  const size_t es = elem_size(shape->dtype);
  for (int l = 0; l < shape->n_layers; ++l) {
    if (!student_ptrs[l] || !teacher_ptrs[l]) return MAFED_E_ARG;
    if (!aligned_to(student_ptrs[l], es) || !aligned_to(teacher_ptrs[l], es)) return MAFED_E_ALIGN;
    p.s[l] = student_ptrs[l];
    p.t[l] = teacher_ptrs[l];
    if (grad_ptrs) {
      if (!aligned_to(grad_ptrs[l], es)) return MAFED_E_ALIGN;
      p.g[l] = grad_ptrs[l];
    }
  }
  p.mask = attn_mask;
  return 0;
}

// ---------------------------------------------------------------- launch helpers
template <typename K>
int blocks_per_sm(K kernel, int threads, size_t dyn_smem) {
  int n = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, threads, dyn_smem) != cudaSuccess) n = 1;
  return n < 1 ? 1 : n;
}

inline long long clamp_grid(long long grid, long long total) {
  if (grid > total) grid = total;
  if (grid > kMaxPartials) grid = kMaxPartials;
  return grid < 1 ? 1 : grid;
}

// A kernel as a TYPE: `host()` is its entry point for an ordinary launch; `tail_launch` (relocatable-device-code
// unit only) starts it from the device into the tail-launch stream of the running grid, i.e. stream-ordered right
// behind it.  (A kernel passed as a non-type template argument does not survive as the target of a device-side
// launch with nvcc 12.9 -- tools/probes/cdp_probe3.cu -- so the kernel is always named in the tag.)
#ifdef MAFED_DEVICE_LAUNCH
#define MAFED_TAIL_LAUNCH(...)                                                                                  \
  template <typename... A>                                                                                      \
  static __device__ __forceinline__ void tail_launch(unsigned grid, unsigned block, unsigned smem, const A&... a) { \
    __VA_ARGS__<<<grid, block, smem, cudaStreamTailLaunch>>>(a...);                                             \
  }
#else
#define MAFED_TAIL_LAUNCH(...)
#endif

template <typename T, int CPL, int RPI, int LOSS, int PASS>
struct LdgKernel;
template <typename T, int CPL, int RPI, int LOSS>
struct LdgKernel<T, CPL, RPI, LOSS, kPassFwd> {
  static auto host() { return &k_fwd_ldg<T, CPL, RPI, LOSS>; }
};
template <typename T, int CPL, int RPI, int LOSS>
struct LdgKernel<T, CPL, RPI, LOSS, kPassBwd> {
  static auto host() { return &k_bwd_ldg<T, CPL, RPI, LOSS, kBackward>; }
  MAFED_TAIL_LAUNCH(k_bwd_ldg<T, CPL, RPI, LOSS, kBackward>)
};
template <typename T, int CPL, int RPI, int LOSS>
struct LdgKernel<T, CPL, RPI, LOSS, kPassFused> {
  static auto host() { return &k_bwd_ldg<T, CPL, RPI, LOSS, kFused>; }
};

template <typename T, int LOSS, int PASS>
struct TmaKernel;
template <typename T, int LOSS>
struct TmaKernel<T, LOSS, kPassFwd> {
  static auto host() { return &k_fwd_tma<T, LOSS>; }
};
template <typename T, int LOSS>
struct TmaKernel<T, LOSS, kPassBwd> {
  static auto host() { return &k_bwd_tma<T, LOSS, kBackward>; }
  MAFED_TAIL_LAUNCH(k_bwd_tma<T, LOSS, kBackward>)
};
template <typename T, int LOSS>
struct TmaKernel<T, LOSS, kPassFused> {
  static auto host() { return &k_bwd_tma<T, LOSS, kFused>; }
};

template <typename T, int LOSS>
struct GenericFwdKernel {
  static auto host() { return &k_fwd_generic<T, LOSS>; }
};
template <typename T, int LOSS>
struct GenericBwdKernel {
  static auto host() { return &k_bwd_generic<T, LOSS>; }
  MAFED_TAIL_LAUNCH(k_bwd_generic<T, LOSS>)
};

template <typename T, int CPL, int RPI, int LOSS, int PASS, typename Launcher>
int launch_ldg(const PathParams& p, const Launcher& go) {
  static_assert(LOSS != kLossL2Norm || PASS == kPassFwd, "the token-norm reduction has no backward");
  using Kernel = LdgKernel<T, CPL, RPI, LOSS, PASS>;
  static int occ[kMaxDevices] = {};   // per kernel and per device
  const DeviceInfo& dv = device_info();
  if (occ[dv.index] == 0) occ[dv.index] = blocks_per_sm(Kernel::host(), kLdgThreads, 0);
  const long long rows_per_iter = (long long)kLdgWarps * RPI;
  const long long total = ((p.n_rows + rows_per_iter - 1) / rows_per_iter) * p.n_layers;
  const unsigned grid = (unsigned)clamp_grid((long long)dv.sm_count * occ[dv.index], total);
  go.template run<Kernel>(grid, kLdgThreads, 0, p);
  return (int)cudaPeekAtLastError();
}

template <typename T, int LOSS, int PASS, typename Launcher>
int dispatch_ldg(const PathParams& p, const Launcher& go) {
  const int cpl = (p.n_chunks + 31) / 32;
  // rows per warp per iteration: more independent loads in flight for short rows; the cosine gradient keeps the row
  // statistics and two coefficients per row as well, so it takes half as many rows at a time (with 4 / 2 it spilled
  // 150-250 bytes per thread under the 128-register cap)
  constexpr bool kHeavy = LOSS == MAFED_LOSS_COSINE && PASS != kPassFwd;
  if (cpl <= 1) return launch_ldg<T, 1, kHeavy ? 2 : 4, LOSS, PASS>(p, go);
  if (cpl <= 2) return launch_ldg<T, 2, kHeavy ? 2 : 4, LOSS, PASS>(p, go);
  if (cpl <= 3) return launch_ldg<T, 3, kHeavy ? 1 : 2, LOSS, PASS>(p, go);
  if (cpl <= 4) return launch_ldg<T, 4, kHeavy ? 1 : 2, LOSS, PASS>(p, go);
  if (cpl <= 6) return launch_ldg<T, 6, 1, LOSS, PASS>(p, go);
  return launch_ldg<T, 8, 1, LOSS, PASS>(p, go);  // multi-pass for rows longer than 4 KB
}

// Any D / any alignment: element-wise kernels.  The fused pass is simply forward then backward.
template <typename T, int LOSS, int PASS, typename Launcher>
int launch_generic(const mafed_shape_t& sh, const PathParams& p, const Launcher& go) {
  const DeviceInfo& dv = device_info();
  const long long total = ((p.n_rows + kLdgWarps - 1) / kLdgWarps) * p.n_layers;
  const unsigned grid = (unsigned)clamp_grid((long long)dv.sm_count * 4, total);
  if constexpr (PASS == kPassFwd || PASS == kPassFused) go.template run<GenericFwdKernel<T, LOSS>>(grid, kLdgThreads, 0, p);
  if constexpr (LOSS != kLossL2Norm && (PASS == kPassBwd || PASS == kPassFused))
    go.template run<GenericBwdKernel<T, LOSS>>(grid, kLdgThreads, 0, p, PASS == kPassFused ? 1 : 0);
  return (int)cudaPeekAtLastError();
}

inline bool tma_geometry(const mafed_shape_t& sh, const PathParams& p, int pass, TmaGeom& geo, int loss) {
  const DeviceInfo& dv = device_info();
  const long long row_bytes = (long long)p.n_chunks * 16;
  if (row_bytes > 32768) return false;
  const long long budget = (long long)dv.smem_optin - 16 * 1024;  // static smem + slack
  // Measured on B200 (profiles/r02l_geometry_sweep.txt: one-pass step, 13 shapes x 13 rings; r02q_geometry_sweep_
  // {fwd,bwd}.txt: the two passes; all after the producer stopped paying 64-bit divisions and the mask round trip
  // per tile).  What the memory system is sensitive to is the number of bytes in flight per SM:
  //  * forward pass (reads only): 2 stages x 96 KB -- best or within 2 % for every shape; ragged long text +13 %
  //    and cosine +5 % over 2 x 72 KB.
  //  * passes that also write the gradient (backward, one-pass step): 3 stages x 32 KB (96 KB in flight) is the best
  //    or within 2.5 % of it for every shape of 256 visual + ~32 text rows (base / 410M / 1B, bf16 and fp32, 16..256
  //    samples), 5-12 % ahead of 2 x 64 KB; 64 KB in flight is latency-bound (+20 %), 128 KB and more queue up in
  //    the memory system (+5-13 %).
  //  * the cosine gradient needs two sweeps over a row with a warp reduction in between, so a stage drains more
  //    slowly: 4 stages x 32 KB keep more rows in different phases at once.
  //  * text-heavy batches (more than a quarter of the rows behind the attention mask, where ragged masks make
  //    whole tiles zero-fill only) keep the coarse ring, 2 x 64-72 KB: fewer, larger tiles amortise the per-tile
  //    cost of the padded ones (3 x 32 KB is 4-16 % behind there).
  const bool text_heavy = (long long)(sh.T - sh.n_vis) * 4 > (long long)sh.T;
  const bool wide = pass == kPassFwd;
  const bool cosine_fine = !wide && loss == MAFED_LOSS_COSINE;
  const bool fused_fine = !wide && !cosine_fine && !text_heavy;
  const long long stage_target = wide ? 96 * 1024 : ((cosine_fine || fused_fine) ? 32 * 1024 : 72 * 1024);
  int rows = (int)(stage_target / (2 * row_bytes));
  if (rows >= 8 && !wide && !cosine_fine && !fused_fine) rows &= ~7;
  if (rows > kTmaMaxRows) rows = kTmaMaxRows;
  if (rows < 1) rows = 1;
  if (2 * rows * row_bytes > budget) rows = (int)(budget / (2 * row_bytes));
  if (rows < 1) return false;
  geo.rows = rows;
  geo.stage_bytes = (int)(2 * rows * row_bytes);
  int stages = cosine_fine ? 4 : (fused_fine ? 3 : ((wide || 2 * geo.stage_bytes >= 96 * 1024) ? 2 : 3));
  if (stages > kTmaMaxStages) stages = kTmaMaxStages;
  while (stages > 1 && (long long)stages * geo.stage_bytes > budget) --stages;
  geo.stages = stages;
  // Refill pacing (profiles/r02n_pace_sweep.txt).  The coarse ring of a text-heavy one-pass step, every row live:
  // 0.96 ms refilled at once, 0.90 ms with ~0.5 us between a free slot and its refill (in-flight bytes per SM are
  // what the memory system is sensitive to); with a ragged mask the same pause costs 4 %, so the producer drops it
  // at the first padded row it meets.
  geo.pace = pass != kPassFwd && !fused_fine && !cosine_fine;
  return true;
}

template <typename T, int LOSS, int PASS, typename Launcher>
int launch_tma(const PathParams& p, const TmaGeom& geo, const Launcher& go) {
  static_assert(LOSS != kLossL2Norm || PASS == kPassFwd, "the token-norm reduction has no backward");
  using Kernel = TmaKernel<T, LOSS, PASS>;
  // the opt-in shared-memory size is a per-device function attribute: remember it per kernel and device
  static bool attr_set[kMaxDevices] = {};
  const DeviceInfo& dv = device_info();
  const size_t dyn = (size_t)geo.stages * geo.stage_bytes;
  if (!attr_set[dv.index]) {
    cudaError_t e = cudaFuncSetAttribute(Kernel::host(), cudaFuncAttributeMaxDynamicSharedMemorySize, dv.smem_optin - 16 * 1024);
    if (e != cudaSuccess) return (int)e;
    attr_set[dv.index] = true;
  }
  const long long total = ((p.n_rows + geo.rows - 1) / geo.rows) * p.n_layers;
  const unsigned grid = (unsigned)clamp_grid((long long)dv.sm_count, total);   // one persistent CTA per SM
  go.template run<Kernel>(grid, kTmaConsumerThreads + 32, dyn, p, geo);   // + the producer warp
  return (int)cudaPeekAtLastError();
}

inline bool vector_path(const mafed_shape_t& sh, const PathParams& p, int pass) {
  // vector kernels: rows are whole, 16-byte aligned chunks
  const size_t es = elem_size(sh.dtype);
  bool ok = ((size_t)sh.D * es) % 16 == 0 && ((size_t)p.row_stride * es) % 16 == 0;
  for (int l = 0; l < sh.n_layers && ok; ++l)
    ok = aligned_to(p.s[l], 16) && aligned_to(p.t[l], 16) && (pass == kPassFwd || aligned_to(p.g[l], 16));
  return ok;
}

inline int chosen_variant(const mafed_shape_t& sh) {
  const int variant = tune(sh, MAFED_TUNE_VARIANT_ALL);
  return variant == 0 ? 2 : variant;   // 1 ldg, 2 tma (default)
}

template <typename T, int LOSS, int PASS, typename Launcher>
int dispatch_typed(const mafed_shape_t& sh, PathParams& p, bool vector_ok, const Launcher& go) {
  if (!vector_ok) return launch_generic<T, LOSS, PASS>(sh, p, go);
  if (chosen_variant(sh) == 2) {
    TmaGeom geo;
    if (tma_geometry(sh, p, PASS, geo, LOSS)) return launch_tma<T, LOSS, PASS>(p, geo, go);
  }
  return dispatch_ldg<T, LOSS, PASS>(p, go);
}

template <typename T, int PASS, typename Launcher>
int dispatch_loss(const mafed_shape_t& sh, PathParams& p, int loss, bool vector_ok, const Launcher& go) {
  if (loss == MAFED_LOSS_MSE) return dispatch_typed<T, MAFED_LOSS_MSE, PASS>(sh, p, vector_ok, go);
  if constexpr (PASS == kPassFwd) {
    if (loss == kLossL2Norm) return dispatch_typed<T, kLossL2Norm, PASS>(sh, p, vector_ok, go);
  }
  return dispatch_typed<T, MAFED_LOSS_COSINE, PASS>(sh, p, vector_ok, go);
}

template <int PASS, typename Launcher>
int dispatch(const mafed_shape_t& sh, PathParams& p, const Launcher& go, int loss_override = -1) {
  const bool vector_ok = vector_path(sh, p, PASS);
  p.n_chunks = vector_ok ? (int)((size_t)sh.D * elem_size(sh.dtype) / 16) : 0;
  const int loss = loss_override >= 0 ? loss_override : sh.loss_kind;
  switch (sh.dtype) {
    case MAFED_F32: return dispatch_loss<float, PASS>(sh, p, loss, vector_ok, go);
    case MAFED_BF16: return dispatch_loss<__nv_bfloat16, PASS>(sh, p, loss, vector_ok, go);
    default: return dispatch_loss<__half, PASS>(sh, p, loss, vector_ok, go);
  }
}

// Will `dispatch` take the TMA-ring kernels for this call?  (Same decision, made ahead of the launch.)
inline bool uses_tma(const mafed_shape_t& sh, const PathParams& p, int pass) {
  if (!vector_path(sh, p, pass) || chosen_variant(sh) != 2) return false;
  PathParams q = p;
  q.n_chunks = (int)((size_t)sh.D * elem_size(sh.dtype) / 16);
  TmaGeom geo;
  return tma_geometry(sh, q, pass, geo, MAFED_LOSS_MSE);   // eligibility does not depend on the loss kind
}

}  // namespace MAFED_NS
