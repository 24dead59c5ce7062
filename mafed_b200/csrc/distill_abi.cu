// C ABI (include/mafed_distill.h) over the sm_100a kernels.  No torch types, no allocation, no host
// synchronisation: every entry point validates its arguments, picks a launch geometry and enqueues
// kernels on the caller's stream.
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "distill_common.cuh"
#include "distill_dispatch.cuh"
#include "distill_epilogue.cuh"
#include "distill_gate.h"
#include "distill_host.cuh"
#include "distill_ldg.cuh"
#include "distill_tma.cuh"

namespace mafed {
namespace {

// May this launch be a programmatic dependent of its predecessor in `stream`?  Not right behind a gate
// (distill_gate.cu: the gate may have started a backward from the device that needs the SMs first).
bool pdl_allowed(void* stream) { return !mafed_gate::consume_gate_mark(stream); }

HostLaunch host_launch(void* stream) { return HostLaunch{(cudaStream_t)stream, pdl_allowed(stream)}; }

// Arrival counters of the in-kernel tail (distill_tma.cuh).  A counter is zero whenever no kernel is using it
// (the last CTA resets it), so launches take them round-robin: two kernels can only share one if 128 tailed
// launches are in flight at once on one device, and each of them is a persistent whole-GPU kernel.  Launches
// recorded into a CUDA graph keep their counter for every replay, so they draw from a separate half of the
// pool: an eager launch on another stream can never land on the counter of a graph that is replaying.
constexpr unsigned kDoneSlots = 256;
__device__ unsigned int g_tail_done[kDoneSlots];
std::atomic<unsigned> g_tail_next{0};
std::atomic<unsigned> g_tail_next_captured{0};

unsigned int* next_tail_counter(cudaStream_t st) {
  static unsigned int* base[kMaxDevices] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return nullptr;
  if (base[dev] == nullptr) {
    void* p = nullptr;
    if (cudaGetSymbolAddress(&p, g_tail_done) != cudaSuccess) return nullptr;
    base[dev] = reinterpret_cast<unsigned int*>(p);
  }
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) return nullptr;
  constexpr unsigned half = kDoneSlots / 2;
  if (cap == cudaStreamCaptureStatusActive) return base[dev] + half + (g_tail_next_captured.fetch_add(1) % half);
  return base[dev] + (g_tail_next.fetch_add(1) % half);
}

}  // namespace
}  // namespace mafed

// Host handle of the peer-memory communicator (see distill_comm.cuh).
struct mafed_comm {
  int world = 0;
  int rank = 0;
  void* local = nullptr;
  void* peers[mafed::kCommMaxRanks] = {};
  long long timeout_cycles = 0;
  double cycles_per_second = 1.9e9;
  bool loopback = false;
  int* status_host = nullptr;   // mapped pinned host word: the kernels write it on a timeout, the host just reads it
  int* status_dev = nullptr;    // its device address
};

namespace mafed {
namespace {

CommDev comm_dev(const mafed_comm* c) {
  CommDev d;
  memset(&d, 0, sizeof(d));
  if (c == nullptr || c->world <= 1) return d;
  d.world = c->world;
  d.rank = c->rank;
  d.timeout_cycles = c->timeout_cycles;
  for (int r = 0; r < c->world; ++r) d.ll[r] = reinterpret_cast<unsigned long long*>(c->peers[r]);
  char* tail = reinterpret_cast<char*>(c->local) + kCommTailAt;
  d.epoch = reinterpret_cast<unsigned long long*>(tail);
  d.epoch_counts = reinterpret_cast<unsigned long long*>(tail + 8);
  d.status = c->status_dev;
  d.trace = reinterpret_cast<unsigned long long*>(tail + 32);
  return d;
}

int launch_scalar_stage(const mafed_shape_t& sh, const mafed_weights_t* w, int flags, const int64_t* mask,
                        const void* ws, double* sums, float* out, float* bwd_scale, cudaStream_t st,
                        const mafed_comm* comm = nullptr, int comm_what = 0, double* counts_out = nullptr,
                        const double* counts_in = nullptr) {
  EpiParams e;
  memset(&e, 0, sizeof(e));
  e.comm = comm_dev(comm);
  if (e.comm.world > 1) {
    const int L2 = 2 * sh.n_layers;
    if (comm_what == (MAFED_COMM_SUMS | MAFED_COMM_COUNTS)) { e.a.comm_first = 0; e.a.comm_count = L2 + 2; }
    else if (comm_what == MAFED_COMM_SUMS) { e.a.comm_first = 0; e.a.comm_count = L2; }
    else if (comm_what == MAFED_COMM_COUNTS) { e.a.comm_first = L2; e.a.comm_count = 2; }
  }
  e.a.ws = reinterpret_cast<const float*>(ws);
  e.a.mask = mask;
  e.a.sums = sums;
  e.a.counts_out = counts_out;
  e.a.counts_in = counts_in;
  e.a.out = out;
  e.a.bwd_scale = bwd_scale;
  e.a.n_mask = mask_entries(sh);
  e.a.n_vis_rows = vis_rows(sh);
  e.a.n_layers = sh.n_layers;
  e.a.D = sh.D;
  e.a.loss_kind = sh.loss_kind;
  e.a.flags = flags;
  if (w != nullptr) e.w = *w;
  launch_pdl(k_epilogue, 1, kEpiThreads, 0, st, pdl_allowed(st), e);
  return (int)cudaPeekAtLastError();
}

// What mafed_distill_step wants produced besides the gradients; with it the fused kernel may run the loss
// algebra (and the modality masks) itself.
struct StepTail {
  float* out;
  double* sums;
  int64_t* lang_mask;
  int64_t* image_mask;
};

int fused_impl(const mafed_shape_t* shape, const void* const* student_ptrs, const void* const* teacher_ptrs,
               void* const* grad_ptrs, const int64_t* attn_mask, const mafed_weights_t* weights, float* bwd_scale,
               float assumed_grad_out, void* ws, mafed_comm* comm, const int64_t* counts_ticket, void* stream,
               const StepTail* tail, bool* folded) {
  if (!grad_ptrs || !bwd_scale || !ws) return MAFED_E_ARG;
  if (comm != nullptr && comm->world > 1 && (!weights || comm->world > kCommMaxRanks)) return MAFED_E_ARG;
  PathParams p;
  int rc = fill_params(shape, student_ptrs, teacher_ptrs, grad_ptrs, attn_mask, p);
  if (rc) return rc;
  p.bwd_scale = bwd_scale;
  p.fixed_gout = assumed_grad_out;
  p.ws = reinterpret_cast<float*>(ws);
  const bool sharded = comm != nullptr && comm->world > 1;
  const bool tma = uses_tma(*shape, p, kPassFused);
  const bool want_tail = tail != nullptr && weights != nullptr && tma && !tune(*shape, MAFED_TUNE_NO_TAIL);
  // with a ticket nobody sums the mask inside the streaming kernel, so the mask size does not matter
  const bool want_inline = weights != nullptr && tma && (counts_ticket != nullptr || mask_entries(*shape) <= 16384);
  // The arrival counter: needed for the tail and, in a sharded step without a ticket, for the in-kernel counts
  // exchange (the last CTA advances the device-side epoch).
  unsigned int* done = nullptr;
  if (want_tail || (want_inline && sharded && counts_ticket == nullptr)) done = next_tail_counter((cudaStream_t)stream);
  p.tail_done = done;
  if (done != nullptr && want_tail) {
    // the last CTA of the TMA kernel reduces the partials and forms the losses (and exchanges the sums with the
    // peers); all CTAs write the modality masks: no epilogue or mask launch
    p.tail_flags = kEpiReduce | kEpiLosses;
    p.tail_out = tail->out;
    p.tail_sums = tail->sums;
    p.lang_mask_out = tail->lang_mask;
    p.image_mask_out = tail->image_mask;
    p.tail_comm = sharded ? 1 : 0;
    if (folded != nullptr) *folded = true;
  }
  if (weights != nullptr) {
    p.loss_kind = shape->loss_kind;
    p.n_mask = mask_entries(*shape);
    p.n_vis_rows = vis_rows(*shape);
    p.w = *weights;
    if (sharded) p.comm = comm_dev(comm);
    // the scale table is this call's business.  Small masks: every CTA of the TMA kernel derives it itself while
    // its first tiles are in flight (the whole step is ONE launch; in a sharded step the counts exchange rides
    // inside the kernel); otherwise one prologue launch, which leaves the counts in the ws header for the tail.
    if (want_inline && (!sharded || done != nullptr || counts_ticket != nullptr)) {
      p.inline_scale = 1;
      p.bwd_scale_out = bwd_scale;
      p.comm_counts = sharded ? 1 : 0;
      p.counts_ticket = reinterpret_cast<const long long*>(counts_ticket);
    } else {
      double* counts = reinterpret_cast<double*>(p.ws + kWsCountsAt);
      p.tail_counts_in = counts;
      rc = launch_scalar_stage(*shape, weights, MAFED_STAGE_COUNTS | MAFED_STAGE_SCALE, attn_mask, nullptr, nullptr,
                               nullptr, bwd_scale, (cudaStream_t)stream, comm, MAFED_COMM_COUNTS, counts);
      if (rc) return rc;
    }
  }
  return dispatch<kPassFused>(*shape, p, host_launch(stream));
}

}  // namespace
}  // namespace mafed

using namespace mafed;

extern "C" {

int mafed_distill_abi_version(void) { return MAFED_ABI_VERSION; }

const char* mafed_distill_error_string(int code) {
  switch (code) {
    case 0: return "ok";
    case MAFED_E_ARG: return "invalid argument (null pointer, non-positive size or too many layers)";
    case MAFED_E_DTYPE: return "unsupported dtype or loss kind";
    case MAFED_E_ALIGN: return "pointer not aligned to its element size";
    case MAFED_E_NODEVICE: return "no usable CUDA device";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
  }
}

size_t mafed_distill_ws_bytes(int n_layers) {
  if (n_layers < 1) n_layers = 1;
  if (n_layers > kMaxLayers) n_layers = kMaxLayers;
  return sizeof(float) * ((size_t)kWsHeaderFloats + (size_t)kMaxPartials * n_layers * 2);
}

int mafed_distill_sums_len(int n_layers) { return 2 * n_layers + 2; }
int mafed_distill_out_len(int n_layers) { return 1 + 3 * n_layers; }

int mafed_distill_fwd(const mafed_shape_t* shape, const void* const* student_ptrs, const void* const* teacher_ptrs,
                      const int64_t* attn_mask, void* ws, void* stream) {
  PathParams p;
  int rc = fill_params(shape, student_ptrs, teacher_ptrs, nullptr, attn_mask, p);
  if (rc) return rc;
  if (!ws) return MAFED_E_ARG;
  p.ws = reinterpret_cast<float*>(ws);
  return dispatch<kPassFwd>(*shape, p, host_launch(stream));
}

int mafed_distill_token_norm_sums(const mafed_shape_t* shape, const void* const* tensor_ptrs, const int64_t* attn_mask,
                                  void* ws, void* stream) {
  PathParams p;
  int rc = fill_params(shape, tensor_ptrs, tensor_ptrs, nullptr, attn_mask, p);
  if (rc) return rc;
  if (!ws) return MAFED_E_ARG;
  p.ws = reinterpret_cast<float*>(ws);
  p.single_input = 1;
  return dispatch<kPassFwd>(*shape, p, host_launch(stream), kLossL2Norm);
}

int mafed_distill_scalar_stage(const mafed_shape_t* shape, const mafed_weights_t* weights, int flags,
                               const int64_t* attn_mask, const void* ws, double* sums, float* out, float* bwd_scale,
                               mafed_comm_t* comm, int comm_what, void* stream) {
  int rc = check_shape(shape);
  if (rc) return rc;
  if ((flags & MAFED_STAGE_REDUCE) && !ws) return MAFED_E_ARG;
  if ((flags & MAFED_STAGE_COUNTS) && needs_mask(*shape) && !attn_mask) return MAFED_E_ARG;
  if ((flags & (MAFED_STAGE_LOSSES | MAFED_STAGE_SCALE)) && !weights) return MAFED_E_ARG;
  if ((flags & MAFED_STAGE_LOSSES) && !out) return MAFED_E_ARG;
  if ((flags & MAFED_STAGE_SCALE) && !bwd_scale) return MAFED_E_ARG;
  const bool reads_sums = ((flags & MAFED_STAGE_LOSSES) && !(flags & MAFED_STAGE_REDUCE)) ||
                          ((flags & (MAFED_STAGE_LOSSES | MAFED_STAGE_SCALE)) && !(flags & MAFED_STAGE_COUNTS));
  const bool only_writes = (flags & (MAFED_STAGE_LOSSES | MAFED_STAGE_SCALE)) == 0;
  const bool sharded = comm != nullptr && comm->world > 1;
  // a sharded sequence always carries the sums vector between its stages
  if ((reads_sums || only_writes || sharded) && !sums) return MAFED_E_ARG;
  if (sharded && (comm->world > kCommMaxRanks || comm_what < 0 || comm_what > 3)) return MAFED_E_ARG;
  return launch_scalar_stage(*shape, weights, flags, attn_mask, ws, sums, out, bwd_scale, (cudaStream_t)stream,
                             sharded ? comm : nullptr, comm_what);
}

int mafed_comm_handle_bytes(void) { return (int)sizeof(cudaIpcMemHandle_t); }

int mafed_comm_create(int world, int rank, void* ipc_handle_out, mafed_comm_t** out) {
  if (world < 1 || world > kCommMaxRanks || rank < 0 || rank >= world || !ipc_handle_out || !out) return MAFED_E_ARG;
  mafed_comm* c = new mafed_comm();
  c->world = world;
  c->rank = rank;
  cudaError_t e = cudaMalloc(&c->local, kCommMailboxBytes);
  if (e == cudaSuccess) e = cudaMemset(c->local, 0, kCommMailboxBytes);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  cudaIpcMemHandle_t h;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, c->local);
  if (e == cudaSuccess) e = cudaHostAlloc(reinterpret_cast<void**>(&c->status_host), sizeof(int), cudaHostAllocMapped);
  if (e == cudaSuccess) {
    *c->status_host = 0;
    e = cudaHostGetDevicePointer(reinterpret_cast<void**>(&c->status_dev), c->status_host, 0);
  }
  if (e != cudaSuccess) {
    if (c->status_host) cudaFreeHost(c->status_host);
    if (c->local) cudaFree(c->local);
    delete c;
    return (int)e;
  }
  memcpy(ipc_handle_out, &h, sizeof(h));
  c->peers[rank] = c->local;
  int dev = 0, khz = 0;
  if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, dev) == cudaSuccess && khz > 0)
    c->cycles_per_second = 1e3 * (double)khz;
  double seconds = kCommDefaultTimeoutS;
  if (const char* env = getenv("MAFED_B200_COMM_TIMEOUT_S")) {
    const double v = atof(env);
    if (v > 0.0) seconds = v;
  }
  c->timeout_cycles = (long long)(seconds * c->cycles_per_second);
  *out = c;
  return 0;
}

int mafed_comm_set_timeout(mafed_comm_t* c, double seconds) {
  if (!c || !(seconds > 0.0)) return MAFED_E_ARG;
  c->timeout_cycles = (long long)(seconds * c->cycles_per_second);
  return 0;
}

int mafed_comm_connect(mafed_comm_t* c, const void* all_handles) {
  if (!c) return MAFED_E_ARG;
  if (!all_handles) {
    // diagnostic loop-back: every "peer" is this rank's own mailbox.  Rank r only ever fills slot r, so the other
    // ranks' slots stay empty and every exchange runs into the spin bound -- the way to test that bound on one GPU.
    for (int r = 0; r < c->world; ++r) c->peers[r] = c->local;
    c->loopback = true;
    return 0;
  }
  const char* hs = reinterpret_cast<const char*>(all_handles);
  for (int r = 0; r < c->world; ++r) {
    if (r == c->rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, hs + (size_t)r * sizeof(h), sizeof(h));
    cudaError_t e = cudaIpcOpenMemHandle(&c->peers[r], h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return (int)e;
  }
  return 0;
}

int mafed_comm_status(mafed_comm_t* c, int* status_out) {
  if (!c || !status_out) return MAFED_E_ARG;
  // the word lives in mapped pinned host memory: a plain read, no synchronisation.  It shows every timeout of the
  // kernels that have finished; a caller that needs the verdict for a particular step synchronises its stream first.
  *status_out = *const_cast<volatile int*>(c->status_host);
  return 0;
}

int mafed_comm_trace(mafed_comm_t* c, unsigned long long* out4) {
  if (!c || !out4) return MAFED_E_ARG;
  const char* tail = reinterpret_cast<const char*>(c->local) + kCommTailAt;
  return (int)cudaMemcpy(out4, tail + 32, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
}

int mafed_comm_trace_async(mafed_comm_t* c, unsigned long long* out4, void* stream) {
  if (!c || !out4) return MAFED_E_ARG;
  const char* tail = reinterpret_cast<const char*>(c->local) + kCommTailAt;
  return (int)cudaMemcpyAsync(out4, tail + 32, 4 * sizeof(unsigned long long), cudaMemcpyDefault,
                              static_cast<cudaStream_t>(stream));
}

int mafed_comm_destroy(mafed_comm_t* c) {
  if (!c) return 0;
  for (int r = 0; r < c->world; ++r)
    if (!c->loopback && r != c->rank && c->peers[r]) cudaIpcCloseMemHandle(c->peers[r]);
  if (c->local) cudaFree(c->local);
  if (c->status_host) cudaFreeHost(c->status_host);
  delete c;
  return 0;
}

int mafed_distill_prefetch_counts(const mafed_shape_t* shape, const int64_t* attn_mask, mafed_comm_t* comm,
                                  int64_t* ticket, void* stream) {
  int rc = check_shape(shape);
  if (rc) return rc;
  if (!ticket || (needs_mask(*shape) && !attn_mask)) return MAFED_E_ARG;
  if (comm != nullptr && comm->world > kCommMaxRanks) return MAFED_E_ARG;
  PrefetchParams pp;
  memset(&pp, 0, sizeof(pp));
  pp.mask = attn_mask;
  pp.n_mask = mask_entries(*shape);
  pp.n_vis_rows = vis_rows(*shape);
  pp.ticket = reinterpret_cast<long long*>(ticket);
  pp.comm = comm_dev(comm);
  launch_pdl(k_prefetch_counts, 1, kEpiThreads, 0, (cudaStream_t)stream, pdl_allowed(stream), pp);
  return (int)cudaPeekAtLastError();
}

int mafed_distill_bwd(const mafed_shape_t* shape, const void* const* student_ptrs, const void* const* teacher_ptrs,
                      void* const* grad_ptrs, const int64_t* attn_mask, const float* bwd_scale, const float* grad_out,
                      float grad_out_scale, const float* skip_if_equals, float* grad_out_seen, void* stream) {
  if (!grad_ptrs || !bwd_scale) return MAFED_E_ARG;
  int rc = check_shape(shape);
  if (rc) return rc;
  if (skip_if_equals != nullptr && !tune(*shape, MAFED_TUNE_NO_GATE)) {
    // the one-pass step's gate: a 1-CTA launch that starts the backward from the device only if it is needed
    // (distill_gate.cu, the relocatable-device-code unit of the library)
    return mafed_gate::gated_backward(shape, student_ptrs, teacher_ptrs, grad_ptrs, attn_mask, bwd_scale, grad_out,
                                      grad_out_scale, *skip_if_equals, grad_out_seen, stream);
  }
  PathParams p;
  rc = fill_params(shape, student_ptrs, teacher_ptrs, grad_ptrs, attn_mask, p);
  if (rc) return rc;
  p.bwd_scale = bwd_scale;
  p.grad_out = grad_out;
  p.gout_scale = grad_out_scale;
  if (skip_if_equals != nullptr) {   // MAFED_TUNE_NO_GATE: the round-1 form, a full grid whose CTAs return at once
    p.skip_if_gout_equals = 1;
    p.fixed_gout = *skip_if_equals;
  }
  return dispatch<kPassBwd>(*shape, p, host_launch(stream));
}

int mafed_distill_fused(const mafed_shape_t* shape, const void* const* student_ptrs, const void* const* teacher_ptrs,
                        void* const* grad_ptrs, const int64_t* attn_mask, const mafed_weights_t* weights, float* bwd_scale,
                        float assumed_grad_out, void* ws, mafed_comm_t* comm, void* stream) {
  return fused_impl(shape, student_ptrs, teacher_ptrs, grad_ptrs, attn_mask, weights, bwd_scale, assumed_grad_out, ws,
                    comm, nullptr, stream, nullptr, nullptr);
}

int mafed_distill_step(const mafed_shape_t* shape, const void* const* student_ptrs, const void* const* teacher_ptrs,
                       void* const* grad_ptrs, const int64_t* attn_mask, const mafed_weights_t* weights,
                       float assumed_grad_out, void* ws, float* out, float* bwd_scale, double* sums,
                       int64_t* lang_mask, int64_t* image_mask, mafed_comm_t* comm, const int64_t* counts_ticket,
                       void* stream) {
  if (!weights || !out) return MAFED_E_ARG;
  if ((lang_mask == nullptr) != (image_mask == nullptr)) return MAFED_E_ARG;
  const bool sharded = comm != nullptr && comm->world > 1;
  if (sharded && !sums) return MAFED_E_ARG;
  int rc = check_shape(shape);
  if (rc) return rc;
  if (lang_mask != nullptr && shape->cls) return MAFED_E_ARG;
  StepTail tail = {out, sums, lang_mask, image_mask};
  bool folded = false;
  rc = fused_impl(shape, student_ptrs, teacher_ptrs, grad_ptrs, attn_mask, weights, bwd_scale, assumed_grad_out, ws,
                  comm, counts_ticket, stream, &tail, &folded);
  if (rc || folded) return rc;
  // not a single-launch shape (rows > 32 KB, unaligned tensors, a mask of more than 16 Ki entries): same step as
  // separate launches
  if (lang_mask != nullptr) {
    rc = mafed_distill_modality_masks(shape, attn_mask, lang_mask, image_mask, stream);
    if (rc) return rc;
  }
  const int flags = MAFED_STAGE_REDUCE | MAFED_STAGE_COUNTS | MAFED_STAGE_LOSSES;
  return launch_scalar_stage(*shape, weights, flags, attn_mask, ws, sums, out, nullptr, (cudaStream_t)stream,
                             sharded ? comm : nullptr, MAFED_COMM_SUMS | MAFED_COMM_COUNTS);
}

int mafed_distill_fwd_step(const mafed_shape_t* shape, const void* const* student_ptrs,
                           const void* const* teacher_ptrs, const int64_t* attn_mask, const mafed_weights_t* weights,
                           void* ws, float* out, float* bwd_scale, double* sums, mafed_comm_t* comm, void* stream) {
  if (!weights || !out || !ws) return MAFED_E_ARG;
  const bool sharded = comm != nullptr && comm->world > 1;
  if (sharded && (!sums || comm->world > kCommMaxRanks)) return MAFED_E_ARG;
  PathParams p;
  int rc = fill_params(shape, student_ptrs, teacher_ptrs, nullptr, attn_mask, p);
  if (rc) return rc;
  p.ws = reinterpret_cast<float*>(ws);
  const int flags = MAFED_STAGE_REDUCE | MAFED_STAGE_COUNTS | MAFED_STAGE_LOSSES | (bwd_scale ? MAFED_STAGE_SCALE : 0);
  unsigned int* done = nullptr;
  if (!tune(*shape, MAFED_TUNE_NO_TAIL) && uses_tma(*shape, p, kPassFwd)) done = next_tail_counter((cudaStream_t)stream);
  if (done != nullptr) {
    p.tail_flags = flags;
    p.tail_done = done;
    p.tail_out = out;
    p.tail_sums = sums;
    p.tail_bwd_scale = bwd_scale;
    p.loss_kind = shape->loss_kind;
    p.n_mask = mask_entries(*shape);
    p.n_vis_rows = vis_rows(*shape);
    p.w = *weights;
    if (sharded) {   // sums + counts exchange inside the tail
      p.comm = comm_dev(comm);
      p.tail_comm = 1;
    }
    return dispatch<kPassFwd>(*shape, p, host_launch(stream));
  }
  rc = dispatch<kPassFwd>(*shape, p, host_launch(stream));
  if (rc) return rc;
  return launch_scalar_stage(*shape, weights, flags, attn_mask, ws, sums, out, bwd_scale, (cudaStream_t)stream,
                             sharded ? comm : nullptr, MAFED_COMM_SUMS | MAFED_COMM_COUNTS);
}

int mafed_distill_modality_masks(const mafed_shape_t* shape, const int64_t* attn_mask, int64_t* lang_mask,
                                 int64_t* image_mask, void* stream) {
  int rc = check_shape(shape);
  if (rc) return rc;
  if (!lang_mask || !image_mask || (needs_mask(*shape) && !attn_mask)) return MAFED_E_ARG;
  const long long n = (long long)shape->B * shape->T;
  const unsigned grid = (unsigned)clamp_grid((n + 255) / 256, 1 << 20);
  launch_pdl(k_modality_masks, grid > 1184 ? 1184u : grid, 256, 0, (cudaStream_t)stream, pdl_allowed(stream),
             attn_mask, lang_mask, image_mask, n, (int)shape->T, (int)shape->n_vis);
  return (int)cudaPeekAtLastError();
}

// ---------------------------------------------------------------- host-buffer step
size_t mafed_host_step_device_bytes(const mafed_shape_t* shape) {
  if (check_shape(shape)) return 0;
  const size_t layer = (size_t)shape->B * shape->T * shape->D * elem_size(shape->dtype);
  const size_t mask = needs_mask(*shape) ? (size_t)shape->B * (shape->T - shape->n_vis) * sizeof(int64_t) : 0;
  return 3 * layer * shape->n_layers + mask + (size_t)shape->n_layers * (mafed_distill_ws_bytes(1) + 128) + 4096;
}

int mafed_host_step_create(const mafed_shape_t* shape, mafed_host_step_t** out) {
  int rc = check_shape(shape);
  if (rc) return rc;
  if (!out || shape->cls) return MAFED_E_ARG;
  if (!device_info().ok) return MAFED_E_NODEVICE;
  mafed_host_step* h = new mafed_host_step();
  h->shape = *shape;
  const int L = shape->n_layers;
  h->layer_bytes = (((size_t)shape->B * shape->T * shape->D * elem_size(shape->dtype)) + 255) & ~(size_t)255;
  h->mask_bytes = ((needs_mask(*shape) ? (size_t)shape->B * (shape->T - shape->n_vis) * sizeof(int64_t) : 0) + 255) & ~(size_t)255;
  h->ws_bytes = (mafed_distill_ws_bytes(1) + 255) & ~(size_t)255;
  const size_t total = 3 * h->layer_bytes * L + h->mask_bytes + (size_t)L * h->ws_bytes + (size_t)L * 6 * sizeof(float) +
                       (size_t)L * 4 * sizeof(double) + 4 * sizeof(int64_t) + 1024;
  cudaError_t e = cudaMalloc(&h->d_pool, total);
  if (e == cudaSuccess) e = cudaMallocHost(&h->h_out, sizeof(float) * 4 * L);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->s_run, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    mafed_host_step_destroy(h);
    return (int)e;
  }
  char* p = h->d_pool;
  for (int l = 0; l < L; ++l) { h->d_s.push_back(p); p += h->layer_bytes; }
  for (int l = 0; l < L; ++l) { h->d_t.push_back(p); p += h->layer_bytes; }
  for (int l = 0; l < L; ++l) { h->d_g.push_back(p); p += h->layer_bytes; }
  h->d_mask = reinterpret_cast<int64_t*>(p); p += h->mask_bytes;
  h->d_ws = p; p += (size_t)L * h->ws_bytes;
  h->d_sums = reinterpret_cast<double*>(p); p += sizeof(double) * 4 * L;      // per layer [2 sums + 2 counts]
  h->d_ticket = reinterpret_cast<int64_t*>(p); p += sizeof(int64_t) * 4;
  h->d_out = reinterpret_cast<float*>(p); p += sizeof(float) * 4 * L;
  h->d_scale = reinterpret_cast<float*>(p);
  h->ev_in.resize(L);
  h->ev_run.resize(L);
  for (int l = 0; l < L; ++l) {
    cudaEventCreateWithFlags(&h->ev_in[l], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&h->ev_run[l], cudaEventDisableTiming);
  }
  cudaEventCreateWithFlags(&h->ev_mask, cudaEventDisableTiming);
  *out = h;
  return 0;
}

int mafed_host_step_run(mafed_host_step_t* h, const mafed_weights_t* weights, const void* const* h_student,
                        const void* const* h_teacher, void* const* h_grad, const int64_t* h_mask, float grad_out,
                        float* h_out, mafed_comm_t* comm) {
  if (!h || !weights || !h_student || !h_teacher || !h_grad || !h_out) return MAFED_E_ARG;
  const bool sharded = comm != nullptr && comm->world > 1;
  const mafed_shape_t& sh = h->shape;
  const int L = sh.n_layers;
  if (needs_mask(sh) && !h_mask) return MAFED_E_ARG;
  const size_t layer = (size_t)sh.B * sh.T * sh.D * elem_size(sh.dtype);
  const size_t mask = needs_mask(sh) ? (size_t)sh.B * (sh.T - sh.n_vis) * sizeof(int64_t) : 0;
  cudaError_t e = cudaSuccess;
  if (mask) e = cudaMemcpyAsync(h->d_mask, h_mask, mask, cudaMemcpyHostToDevice, h->s_in);
  if (sharded && e == cudaSuccess) {
    // batch-sharded: this rank's token counts leave for the peers as soon as the mask is on the device, while the
    // first layer's activations are still crossing PCIe; every layer's step then reads the same ticket
    e = cudaEventRecord(h->ev_mask, h->s_in);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(h->s_run, h->ev_mask, 0);
    if (e != cudaSuccess) return (int)e;
    int rc = mafed_distill_prefetch_counts(&sh, h->d_mask, comm, h->d_ticket, h->s_run);
    if (rc) return rc;
  }
  for (int l = 0; l < L && e == cudaSuccess; ++l) {
    e = cudaMemcpyAsync(h->d_s[l], h_student[l], layer, cudaMemcpyHostToDevice, h->s_in);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h->d_t[l], h_teacher[l], layer, cudaMemcpyHostToDevice, h->s_in);
    if (e == cudaSuccess) e = cudaEventRecord(h->ev_in[l], h->s_in);
  }
  if (e != cudaSuccess) return (int)e;
  mafed_shape_t one = sh;
  one.n_layers = 1;
  for (int l = 0; l < L; ++l) {
    mafed_weights_t w;
    memset(&w, 0, sizeof(w));
    w.modality_kind = weights->modality_kind;
    w.distill_coeff = weights->distill_coeff;
    w.layer_coeff[0] = weights->layer_coeff[l];
    w.lang_weight[0] = weights->lang_weight[l];
    cudaStreamWaitEvent(h->s_run, h->ev_in[l], 0);
    const void* sp[1] = {h->d_s[l]};
    const void* tp[1] = {h->d_t[l]};
    void* gp[1] = {h->d_g[l]};
    char* ws = h->d_ws + (size_t)l * h->ws_bytes;
    int rc = mafed_distill_step(&one, sp, tp, gp, h->d_mask, &w, grad_out, ws, h->d_out + 4 * l, h->d_scale + 2 * l,
                                sharded ? h->d_sums + 4 * l : nullptr, nullptr, nullptr, sharded ? comm : nullptr,
                                sharded ? h->d_ticket : nullptr, h->s_run);
    if (rc) return rc;
    cudaEventRecord(h->ev_run[l], h->s_run);
    cudaStreamWaitEvent(h->s_out, h->ev_run[l], 0);
    e = cudaMemcpyAsync(h_grad[l], h->d_g[l], layer, cudaMemcpyDeviceToHost, h->s_out);
    if (e != cudaSuccess) return (int)e;
  }
  e = cudaMemcpyAsync(h->h_out, h->d_out, sizeof(float) * 4 * L, cudaMemcpyDeviceToHost, h->s_out);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->s_out);
  if (e != cudaSuccess) return (int)e;
  // out[1+3L] layout of the device path: total, layer losses, (text, vision) losses
  double total = 0.0;
  for (int l = 0; l < L; ++l) {
    total += (double)h->h_out[4 * l];
    h_out[1 + l] = h->h_out[4 * l + 1];
    h_out[1 + L + 2 * l] = h->h_out[4 * l + 2];
    h_out[1 + L + 2 * l + 1] = h->h_out[4 * l + 3];
  }
  h_out[0] = (float)total;
  return 0;
}

int mafed_host_step_destroy(mafed_host_step_t* h) {
  if (!h) return 0;
  for (cudaEvent_t ev : h->ev_in) cudaEventDestroy(ev);
  for (cudaEvent_t ev : h->ev_run) cudaEventDestroy(ev);
  if (h->ev_mask) cudaEventDestroy(h->ev_mask);
  if (h->s_in) cudaStreamDestroy(h->s_in);
  if (h->s_run) cudaStreamDestroy(h->s_run);
  if (h->s_out) cudaStreamDestroy(h->s_out);
  if (h->h_out) cudaFreeHost(h->h_out);
  if (h->d_pool) cudaFree(h->d_pool);
  delete h;
  return 0;
}

int mafed_host_register(void* ptr, size_t bytes) { return (int)cudaHostRegister(ptr, bytes, cudaHostRegisterDefault); }
int mafed_host_unregister(void* ptr) { return (int)cudaHostUnregister(ptr); }

}  // extern "C"
