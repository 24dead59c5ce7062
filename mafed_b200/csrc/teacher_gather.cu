// Teacher hidden states of a replay step gathered from the per-task cache (include/mafed_teacher_gather.h).
//
// One launch covers every layer and sample of the step (up to 64 layers and 2048 samples; more take more launches).
// Each (layer, sample) output region is T rows of D elements, made of two contiguous runs of the cache: the n_vis
// visual rows at the sample's start and the T - n_vis text rows at its end (the text block is right-aligned in the
// cache, which pads it on the left).  The regions are cut into chunks of kThreads * kUnroll copy units; a persistent
// grid walks the chunks, each thread keeping kUnroll independent loads in flight before its stores.  The copy unit is
// 16 bytes when D * e and every pointer allow it, else the widest of 8 / 4 / 2 bytes that does (the element-wise path
// for odd row sizes).  The layer pointer tables and the sample indices travel in the kernel parameters, read through
// __grid_constant__ so that a dynamic index does not copy them to local memory.
#include <cuda_runtime.h>
#include <stdint.h>

#include "mafed_teacher_gather.h"

namespace {

constexpr int kLayers = 64;
constexpr int kSamples = 2048;
constexpr int kThreads = 256;
constexpr int kUnroll = 4;
constexpr int kBlocksPerSM = 8;     // 8 x 256 threads: a full SM, 128 KB of loads in flight on it

struct GatherParams {
  char* out[kLayers];
  const char* cache[kLayers];
  int32_t idx[kSamples];            // -1: index out of range (NaN rows)
  int B;
  int64_t vis_units;                // visual rows of a sample, in copy units
  int64_t region_units;             // T rows (one output region)
  int64_t shift_units;              // (T_c - T) rows: where a sample's text block starts in the cache, past n_vis
  int64_t sample_units;             // T_c rows (cache stride of a sample)
  int64_t chunks;                   // chunks per region
  int64_t n_work;                   // n_layers * B * chunks
  uint64_t nan8;                    // 8 bytes of the element type's NaN
};

template <typename V> __device__ __forceinline__ V nan_unit(uint64_t p);
template <> __device__ __forceinline__ uint4 nan_unit<uint4>(uint64_t p) {
  return make_uint4(uint32_t(p), uint32_t(p >> 32), uint32_t(p), uint32_t(p >> 32));
}
template <> __device__ __forceinline__ uint2 nan_unit<uint2>(uint64_t p) { return make_uint2(uint32_t(p), uint32_t(p >> 32)); }
template <> __device__ __forceinline__ unsigned int nan_unit<unsigned int>(uint64_t p) { return uint32_t(p); }
template <> __device__ __forceinline__ unsigned short nan_unit<unsigned short>(uint64_t p) { return uint16_t(p); }

template <typename V>
__global__ void __launch_bounds__(kThreads) mafed_teacher_gather_kernel(const __grid_constant__ GatherParams p) {
  constexpr int64_t kChunk = int64_t(kThreads) * kUnroll;
  for (int64_t w = blockIdx.x; w < p.n_work; w += gridDim.x) {
    const int64_t region = w / p.chunks;
    const int64_t begin = (w - region * p.chunks) * kChunk;
    const int64_t end = min(begin + kChunk, p.region_units);
    const int l = int(region / p.B);
    const int b = int(region - int64_t(l) * p.B);
    V* dst = reinterpret_cast<V*>(p.out[l]) + int64_t(b) * p.region_units;
    const int s = p.idx[b];
    if (s < 0) {
      const V nan = nan_unit<V>(p.nan8);
      for (int64_t u = begin + threadIdx.x; u < end; u += kThreads) dst[u] = nan;
      continue;
    }
    const V* src = reinterpret_cast<const V*>(p.cache[l]) + int64_t(s) * p.sample_units;
    V v[kUnroll];
#pragma unroll
    for (int k = 0; k < kUnroll; ++k) {
      const int64_t u = begin + threadIdx.x + int64_t(k) * kThreads;
      if (u < end) v[k] = __ldcs(src + (u < p.vis_units ? u : u + p.shift_units));   // the cache is read once a step
    }
#pragma unroll
    for (int k = 0; k < kUnroll; ++k) {
      const int64_t u = begin + threadIdx.x + int64_t(k) * kThreads;
      if (u < end) dst[u] = v[k];                  // default policy: the step reads these next, some from L2
    }
  }
}

int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return -1;
  if (dev < 0 || dev >= 64) return -1;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) return -1;
    cached[dev] = n;
  }
  return cached[dev];
}

template <typename V>
int launch(GatherParams& p, int64_t row_bytes, int T, int T_c, int n_vis, int n_layers, cudaStream_t stream, int sms) {
  const int64_t row = row_bytes / int64_t(sizeof(V));
  p.vis_units = int64_t(n_vis) * row;
  p.region_units = int64_t(T) * row;
  p.shift_units = int64_t(T_c - T) * row;
  p.sample_units = int64_t(T_c) * row;
  p.chunks = (p.region_units + int64_t(kThreads) * kUnroll - 1) / (int64_t(kThreads) * kUnroll);
  p.n_work = int64_t(n_layers) * p.B * p.chunks;
  const int64_t cap = int64_t(sms) * kBlocksPerSM;
  const unsigned grid = unsigned(p.n_work < cap ? p.n_work : cap);
  mafed_teacher_gather_kernel<V><<<grid, kThreads, 0, stream>>>(p);
  return cudaGetLastError() == cudaSuccess ? MAFED_GATHER_OK : MAFED_GATHER_ECUDA;
}

}  // namespace

extern "C" int mafed_teacher_gather_abi_version(void) { return MAFED_GATHER_ABI_VERSION; }

extern "C" const char* mafed_teacher_gather_error_string(int code) {
  switch (code) {
    case MAFED_GATHER_OK: return "ok";
    case MAFED_GATHER_EINVAL:
      return "invalid argument (needs n_layers >= 1, 1 <= B, 1 <= M <= 2^31 - 1, 0 <= n_vis <= T <= T_c, D >= 1, "
             "dtype 0/1/2, non-NULL tables and pointers aligned to the element size)";
    case MAFED_GATHER_ECUDA: return "CUDA error (device query or kernel launch)";
    default: return "unknown error code";
  }
}

extern "C" int mafed_teacher_gather(void* const* out, const void* const* cache, const int64_t* idx, int n_layers,
                                    int B, int64_t M, int T, int T_c, int n_vis, int D, int dtype, void* stream) {
  if (!out || !cache || !idx || n_layers < 1 || B < 1 || M < 1 || M > INT32_MAX || n_vis < 0 || T < n_vis ||
      T > T_c || T < 1 || D < 1 || dtype < MAFED_GATHER_F32 || dtype > MAFED_GATHER_F16)
    return MAFED_GATHER_EINVAL;
  const int64_t e = dtype == MAFED_GATHER_F32 ? 4 : 2;
  const uint64_t nan1 = dtype == MAFED_GATHER_F32 ? 0x7FC00000ull : dtype == MAFED_GATHER_BF16 ? 0x7FC0ull : 0x7E00ull;
  const int64_t row_bytes = int64_t(D) * e;
  // the widest copy unit that the row size and every pointer allow
  uintptr_t align = uintptr_t(row_bytes);
  for (int l = 0; l < n_layers; ++l) {
    if (!out[l] || !cache[l]) return MAFED_GATHER_EINVAL;
    align |= reinterpret_cast<uintptr_t>(out[l]) | reinterpret_cast<uintptr_t>(cache[l]);
  }
  if (align % uintptr_t(e)) return MAFED_GATHER_EINVAL;
  const int width = align % 16 == 0 ? 16 : align % 8 == 0 ? 8 : align % 4 == 0 ? 4 : 2;
  const int sms = sm_count();
  if (sms < 0) return MAFED_GATHER_ECUDA;

  GatherParams p;
  p.nan8 = e == 4 ? (nan1 | nan1 << 32) : (nan1 | nan1 << 16 | nan1 << 32 | nan1 << 48);
  const int64_t region_bytes = int64_t(T) * row_bytes;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (int l0 = 0; l0 < n_layers; l0 += kLayers) {
    const int nl = n_layers - l0 < kLayers ? n_layers - l0 : kLayers;
    for (int b0 = 0; b0 < B; b0 += kSamples) {
      p.B = B - b0 < kSamples ? B - b0 : kSamples;
      for (int l = 0; l < nl; ++l) {
        p.out[l] = static_cast<char*>(out[l0 + l]) + int64_t(b0) * region_bytes;
        p.cache[l] = static_cast<const char*>(cache[l0 + l]);
      }
      for (int b = 0; b < p.B; ++b) {
        const int64_t s = idx[b0 + b];
        p.idx[b] = s >= 0 && s < M ? int32_t(s) : -1;
      }
      int rc;
      switch (width) {
        case 16: rc = launch<uint4>(p, row_bytes, T, T_c, n_vis, nl, st, sms); break;
        case 8: rc = launch<uint2>(p, row_bytes, T, T_c, n_vis, nl, st, sms); break;
        case 4: rc = launch<unsigned int>(p, row_bytes, T, T_c, n_vis, nl, st, sms); break;
        default: rc = launch<unsigned short>(p, row_bytes, T, T_c, n_vis, nl, st, sms); break;
      }
      if (rc != MAFED_GATHER_OK) return rc;
    }
  }
  return MAFED_GATHER_OK;
}
