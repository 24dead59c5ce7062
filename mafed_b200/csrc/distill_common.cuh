// Shared device helpers for the MAFED distillation kernels (sm_100a).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "mafed_distill.h"

// The kernels live in `mafed`; the relocatable-device-code unit that holds the gated backward (distill_gate.cu)
// compiles the same headers into `mafed_gate`, so that the two units never share a kernel symbol.
#ifndef MAFED_NS
#define MAFED_NS mafed
#endif

namespace MAFED_NS {

constexpr int kMaxLayers = MAFED_MAX_LAYERS;
// Third "loss": per-token L2 norm of a single tensor (no teacher), for the gradient-norm modality
// importances of distillation_loss_weights.py:91-146.  Forward kernels only.
constexpr int kLossL2Norm = 2;
constexpr float kCosEps = 1e-12f;  // EPSILON of ATen's cosine_embedding_loss
constexpr int kMaxPartials = 2048;  // upper bound on CTAs writing partial sums
// ws header: [0] = number of partial blocks (int); [2..5] = two doubles, the (global) token counts a prologue
// launch leaves for the in-kernel tail of the streaming kernel that follows it
constexpr int kWsHeaderFloats = 8;
constexpr int kWsCountsAt = 2;

// Peer-memory communicator as the kernels see it (see distill_comm.cuh).
constexpr int kCommMaxRanks = 16;
constexpr int kCommSlots = 2 * kMaxLayers + 2;  // one full `sums` vector
constexpr double kCommDefaultTimeoutS = 60.0;  // spin bound of an exchange (MAFED_B200_COMM_TIMEOUT_S / mafed_comm_set_timeout)

struct CommDev {
  unsigned long long* ll[kCommMaxRanks];    // mailbox of every rank (peer-mapped; [rank] is local), see distill_comm.cuh
  unsigned long long* epoch;                // local: collectives issued so far
  unsigned long long* epoch_counts;         // local: count prefetches issued so far
  int* status;                              // 0 ok, 1 timeout; mapped pinned HOST memory (the host reads it without a sync)
  unsigned long long* trace;                // local: SM-cycle totals [counts exchange, publish, wait for peers, calls]
  long long timeout_cycles;                 // spin bound of one wait, in SM cycles
  int world;                                // 0 = no communicator (single rank)
  int rank;
};

// Kernel-parameter block shared by forward and backward kernels (passed by value, < 4 KB).
struct PathParams {
  const void* s[kMaxLayers];
  const void* t[kMaxLayers];
  void* g[kMaxLayers];           // backward only
  const int64_t* mask;           // [B, txt] int64 (unused in cls mode)
  float* ws;                     // forward: partial sums
  const float* bwd_scale;        // backward: [L][2]
  const float* grad_out;         // backward: device scalar or nullptr
  long long n_rows;              // rows per layer (B*T, or B in cls mode)
  long long row_stride;          // elements between consecutive rows
  int n_layers;
  int T;                         // positions per sample as seen by the modality rule
  int n_vis;
  int txt;                       // T - n_vis
  int D;
  int n_chunks;                  // 16-byte chunks per row (vector kernels)
  float fixed_gout;              // fused pass: upstream gradient assumed at forward time (host value)
  float gout_scale;              // backward: host factor on *grad_out (e.g. world_size to undo DDP's averaging)
  int skip_if_gout_equals;       // backward fix-up: return at once when *grad_out == fixed_gout
  int single_input;              // 1: only `s` is read (token-norm sums); the teacher table is ignored
  // one-pass step with the prologue folded in: every CTA derives the scale table from the mask itself
  int inline_scale;              // 1: compute counts + scale in the kernel (weights below), else read bwd_scale
  int loss_kind;
  long long n_mask;              // B * txt
  double n_vis_rows;             // B * n_vis
  float* bwd_scale_out;          // CTA 0 publishes the table for the later backward fix-up
  mafed_weights_t w;
  // batch-sharded one-pass step: the token counts are exchanged inside this kernel (comm.world > 1).  Every CTA
  // reads the device-side epoch counter at its start; only the LAST CTA to finish (tail) advances it, so all
  // CTAs of a launch agree on the epoch and the sequence stays CUDA-graph replayable.
  int comm_counts;               // 1: exchange the counts in this kernel (epoch = device-side counter + 1)
  const long long* counts_ticket;  // counts sent ahead of the step (k_prefetch_counts): {epoch, bits(n_text), bits(n_vis rows)}
  CommDev comm;
  // In-kernel tail (TMA kernels): the last CTA to finish runs the scalar stage on the partial sums, so the step
  // needs no epilogue launch.  Needs w / loss_kind / n_mask / n_vis_rows above (and comm for a sharded step).
  int tail_flags;                // 0: no tail; else EpiFlags of the stage to run
  const double* tail_counts_in;  // [2] counts from a prologue launch (fused pass without the in-kernel scale table)
  int tail_comm;                 // 1: allreduce the sums (+ counts when computed in the tail) over the peer mailboxes
  unsigned int* tail_done;       // arrival counter: zero on entry, reset by the last CTA
  double* tail_sums;             // optional [2L + 2] copy of the (global) sums and counts
  float* tail_out;               // [1 + 3L] losses
  float* tail_bwd_scale;         // [2L] scale table (two-pass forward)
  // one-pass step: the two [B, T] int64 modality masks of distillation.py:134-144, written by the same kernel
  int64_t* lang_mask_out;
  int64_t* image_mask_out;
};

// What a "backward-shaped" kernel does: kBackward writes gradients only; kFused also accumulates
// the loss sums in the same pass over student and teacher (3*D*e bytes per token*layer instead of 5).
enum PassMode { kBackward = 1, kFused = 2 };

// ---------------------------------------------------------------- element packing (16-byte vectors)
template <typename T> struct Pack;

template <> struct Pack<float> {
  static constexpr int kPer16 = 4;
  __device__ __forceinline__ static void unpack(const uint4& v, float (&f)[4]) {
    f[0] = __uint_as_float(v.x); f[1] = __uint_as_float(v.y);
    f[2] = __uint_as_float(v.z); f[3] = __uint_as_float(v.w);
  }
  __device__ __forceinline__ static uint4 pack(const float (&f)[4]) {
    return make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]), __float_as_uint(f[3]));
  }
  __device__ __forceinline__ static float load1(const void* p, long long i) { return ((const float*)p)[i]; }
  __device__ __forceinline__ static void store1(void* p, long long i, float v) { ((float*)p)[i] = v; }
  // one 32-bit word at a time (keeps few values live: the register-resident row forms)
  static constexpr int kPerWord = 1;
  __device__ __forceinline__ static void unpack_word(uint32_t w, float (&f)[1]) { f[0] = __uint_as_float(w); }
  __device__ __forceinline__ static uint32_t pack_word(const float (&f)[1]) { return __float_as_uint(f[0]); }
};

template <> struct Pack<__nv_bfloat16> {
  static constexpr int kPer16 = 8;
  __device__ __forceinline__ static void unpack(const uint4& v, float (&f)[8]) {
    // bf16 -> fp32 is exact: the 16 payload bits become the high half of the fp32 word
    f[0] = __uint_as_float(v.x << 16); f[1] = __uint_as_float(v.x & 0xffff0000u);
    f[2] = __uint_as_float(v.y << 16); f[3] = __uint_as_float(v.y & 0xffff0000u);
    f[4] = __uint_as_float(v.z << 16); f[5] = __uint_as_float(v.z & 0xffff0000u);
    f[6] = __uint_as_float(v.w << 16); f[7] = __uint_as_float(v.w & 0xffff0000u);
  }
  __device__ __forceinline__ static uint32_t pack2(float lo, float hi) {
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);  // round-to-nearest-even, once
    return *reinterpret_cast<uint32_t*>(&h);
  }
  __device__ __forceinline__ static uint4 pack(const float (&f)[8]) {
    return make_uint4(pack2(f[0], f[1]), pack2(f[2], f[3]), pack2(f[4], f[5]), pack2(f[6], f[7]));
  }
  static constexpr int kPerWord = 2;
  __device__ __forceinline__ static void unpack_word(uint32_t w, float (&f)[2]) {
    f[0] = __uint_as_float(w << 16);
    f[1] = __uint_as_float(w & 0xffff0000u);
  }
  __device__ __forceinline__ static uint32_t pack_word(const float (&f)[2]) { return pack2(f[0], f[1]); }
  __device__ __forceinline__ static float load1(const void* p, long long i) {
    return __bfloat162float(((const __nv_bfloat16*)p)[i]);
  }
  __device__ __forceinline__ static void store1(void* p, long long i, float v) {
    ((__nv_bfloat16*)p)[i] = __float2bfloat16_rn(v);
  }
};

template <> struct Pack<__half> {
  static constexpr int kPer16 = 8;
  __device__ __forceinline__ static void up2(uint32_t w, float& a, float& b) {
    float2 r = __half22float2(*reinterpret_cast<const __half2*>(&w));
    a = r.x; b = r.y;
  }
  __device__ __forceinline__ static void unpack(const uint4& v, float (&f)[8]) {
    up2(v.x, f[0], f[1]); up2(v.y, f[2], f[3]); up2(v.z, f[4], f[5]); up2(v.w, f[6], f[7]);
  }
  __device__ __forceinline__ static uint32_t pack2(float lo, float hi) {
    __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
  }
  __device__ __forceinline__ static uint4 pack(const float (&f)[8]) {
    return make_uint4(pack2(f[0], f[1]), pack2(f[2], f[3]), pack2(f[4], f[5]), pack2(f[6], f[7]));
  }
  static constexpr int kPerWord = 2;
  __device__ __forceinline__ static void unpack_word(uint32_t w, float (&f)[2]) { up2(w, f[0], f[1]); }
  __device__ __forceinline__ static uint32_t pack_word(const float (&f)[2]) { return pack2(f[0], f[1]); }
  __device__ __forceinline__ static float load1(const void* p, long long i) {
    return __half2float(((const __half*)p)[i]);
  }
  __device__ __forceinline__ static void store1(void* p, long long i, float v) {
    ((__half*)p)[i] = __float2half_rn(v);
  }
};

// ---------------------------------------------------------------- global memory access
// Streaming 128-bit load: read-only path, do not allocate in L1 (every byte is used exactly once).
__device__ __forceinline__ uint4 ldg_stream(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_128(void* p, const uint4& v) {
  asm volatile("st.global.v4.u32 [%0], {%1, %2, %3, %4};"
               :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// ---------------------------------------------------------------- programmatic dependent launch
// Every kernel of the path is launched with programmaticStreamSerialization: it may become resident
// while its predecessor in the stream is still running (hiding launch latency and prologue work) and
// blocks in pdl_wait() -- before its first global-memory access -- until the predecessor has completed
// and flushed.  pdl_launch_dependents() lets the successor do the same with respect to this kernel.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---------------------------------------------------------------- reductions
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------- modality rule
// distillation.py:134-144: t < n_vis -> visual token, weight 1; else text token weighted by the
// attention mask value.  Returns the weight; sets `modality` (0 = text, 1 = vision).
__device__ __forceinline__ float row_weight(const PathParams& p, long long row, int& modality) {
  const long long b = row / p.T;
  const int t = (int)(row - b * p.T);
  if (t < p.n_vis) { modality = 1; return 1.f; }
  modality = 0;
  return (float)__ldg(p.mask + b * p.txt + (t - p.n_vis));
}

// Modality weights of layer l (distillation_loss_weights.py:71-79,148-174) as (w_text, w_vision).
__device__ __forceinline__ void modality_weights(const mafed_weights_t& w, int l, double n_text, double n_vis,
                                                 double& wt, double& wv) {
  if (w.modality_kind == MAFED_MODW_EQUAL) {
    wt = (double)(float)(n_text / (n_text + n_vis));
    wv = (double)(float)(n_vis / (n_text + n_vis));
  } else if (w.modality_kind == MAFED_MODW_TABLE) {
    wt = (double)w.lang_weight[l];
    wv = (double)(float)(1.0 - wt);
  } else if (w.modality_kind == MAFED_MODW_TEXT_ONLY) {
    wt = 1.0;
    wv = 0.0;
  } else {  // CLS: vision slot only
    wt = 0.0;
    wv = 1.0;
  }
}

// Backward scale of layer l: c_l * coeff * w_m * k / n_m with k = 2/D (mse) or 1 (cosine).
__device__ __forceinline__ void backward_scales(const mafed_weights_t& w, int l, double n_text, double n_vis,
                                                int loss_kind, int D, float& s_text, float& s_vis) {
  double wt, wv;
  modality_weights(w, l, n_text, n_vis, wt, wv);
  const double c = (double)w.layer_coeff[l] * (double)w.distill_coeff;
  const double g = (loss_kind == MAFED_LOSS_MSE) ? 2.0 / (double)D : 1.0;
  s_text = (w.modality_kind == MAFED_MODW_CLS) ? 0.f : (float)(c * wt * g / n_text);
  s_vis = (w.modality_kind == MAFED_MODW_TEXT_ONLY) ? 0.f : (float)(c * wv * g / n_vis);
}

// Per-element math.  mse: sum (h-p)^2.  cosine: dot, |h|^2, |p|^2.
template <int LOSS, int NE>
__device__ __forceinline__ void accumulate(const float (&a)[NE], const float (&b)[NE], float& x, float& y, float& z) {
#pragma unroll
  for (int i = 0; i < NE; ++i) {
    if (LOSS == MAFED_LOSS_MSE) {
      const float d = a[i] - b[i];
      x = fmaf(d, d, x);
    } else if (LOSS == kLossL2Norm) {
      x = fmaf(a[i], a[i], x);
    } else {
      x = fmaf(a[i], b[i], x);
      y = fmaf(a[i], a[i], y);
      z = fmaf(b[i], b[i], z);
    }
  }
}

// Per-row loss value from the warp-reduced statistics.
template <int LOSS>
__device__ __forceinline__ float row_value(float x, float y, float z) {
  if (LOSS == MAFED_LOSS_MSE) return x;  // division by D happens once, in the epilogue
  if (LOSS == kLossL2Norm) return sqrtf(x);
  const float den = sqrtf((y + kCosEps) * (z + kCosEps));
  return 1.f - x / den;
}

// Per-CTA accumulation of [layer][modality] partial sums.  One slot per warp (no atomics: the
// result is bit-reproducible for a fixed launch geometry), combined in fixed order at kernel end.
template <int WARPS>
struct CtaSums {
  float v[WARPS][kMaxLayers][2];
};

template <int WARPS>
__device__ __forceinline__ void cta_sums_zero(CtaSums<WARPS>& s, int n_layers) {
  for (int i = threadIdx.x; i < WARPS * kMaxLayers * 2; i += blockDim.x) (&s.v[0][0][0])[i] = 0.f;
}

template <int WARPS>
__device__ __forceinline__ void cta_sums_flush(CtaSums<WARPS>& s, int warp, int lane, int layer, float text, float vis) {
  text = warp_sum(text);
  vis = warp_sum(vis);
  if (lane == 0 && layer >= 0) {
    s.v[warp][layer][0] += text;
    s.v[warp][layer][1] += vis;
  }
}

// ws layout: [0..3] header (int n_partials), then [block][layer][2].
template <int WARPS>
__device__ __forceinline__ void cta_sums_store(const CtaSums<WARPS>& s, float* ws, int n_layers, int first_thread,
                                               int n_threads) {
  if (blockIdx.x == 0 && (int)threadIdx.x == first_thread) reinterpret_cast<int*>(ws)[0] = gridDim.x;
  float* dst = ws + kWsHeaderFloats + (size_t)blockIdx.x * n_layers * 2;
  for (int i = (int)threadIdx.x - first_thread; i < n_layers * 2; i += n_threads) {
    const int l = i >> 1, m = i & 1;
    float acc = 0.f;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) acc += s.v[w][l][m];
    dst[i] = acc;
  }
}

}  // namespace MAFED_NS
