// Teacher hidden states of a replay step gathered from the per-task cache (include/mafed_teacher_gather.h).
//
// One launch covers every layer and sample of the step (up to 64 layers and 2048 samples; more take more launches).
// Each (layer, sample) output region is T rows of D elements, made of two contiguous runs of the cache: the n_vis
// visual rows at the sample's start and the T - n_vis text rows at its end (the text block is right-aligned in the
// cache, which pads it on the left).  The regions are cut into chunks of kThreads * kUnroll copy units; a persistent
// grid walks the chunks, each thread keeping kUnroll independent loads in flight before its stores.  The copy unit is
// 16 bytes when D * e and every pointer allow it, else the widest of 8 / 4 / 2 bytes that does (the element-wise path
// for odd row sizes).  The layer tables and the samples' (rank, slot) travel in the kernel parameters, read through
// __grid_constant__ so that a dynamic index does not copy them to local memory.
//
// A sample's rows start at base[rank] + off[layer] + slot * T_c * D * e.  The sharded cache (one buffer per rank of a
// box, mapped into every peer through CUDA IPC) gives each rank's base and the layer offsets shared by every shard; the
// one-rank gather is the same kernel with base[0] = 0 and the layer pointers as offsets.  Peer rows arrive over NVLink
// through the kernel's own loads.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include "mafed_teacher_gather.h"

namespace {

constexpr int kLayers = 64;
constexpr int kSamples = 2048;
constexpr int kRanks = 16;          // the communicator's limit (one NVLink box)
constexpr int kThreads = 256;
constexpr int kUnroll = 4;
constexpr int kBlocksPerSM = 8;     // 8 x 256 threads: a full SM, 128 KB of loads in flight on it

struct GatherParams {
  char* out[kLayers];
  uint64_t base[kRanks];            // address of each rank's shard (0 on the one-rank path)
  uint64_t off[kLayers];            // byte offset of each layer from a rank's base (the layer pointer on that path)
  int32_t idx[kSamples];            // slot in its rank's shard; -1: out of range (NaN rows)
  uint8_t rank[kSamples];           // the rank whose shard holds the sample
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
    const V* src = reinterpret_cast<const V*>(p.base[p.rank[b]] + p.off[l]) + int64_t(s) * p.sample_units;
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

// The checks and launches shared by both entry points.  Layer l's rows sit at base[r] + off(l), where off(l) is
// cache[l] (one rank, base[0] = 0) or layer_off[l] (a sharded cache); sample b is slot slot[b] of rank src_rank[b]
// (rank 0 when src_rank is NULL), and a slot outside [0, slots) or a rank outside [0, n_ranks) gives NaN rows.
int gather(void* const* out, const uint64_t* base, int n_ranks, const void* const* cache, const int64_t* layer_off,
           const int32_t* src_rank, const int64_t* slot, int n_layers, int B, int64_t slots, int T, int T_c, int n_vis,
           int D, int dtype, cudaStream_t st) {
  const int64_t e = dtype == MAFED_GATHER_F32 ? 4 : 2;
  const uint64_t nan1 = dtype == MAFED_GATHER_F32 ? 0x7FC00000ull : dtype == MAFED_GATHER_BF16 ? 0x7FC0ull : 0x7E00ull;
  const int64_t row_bytes = int64_t(D) * e;
  // the widest copy unit that the row size and every pointer allow
  uintptr_t align = uintptr_t(row_bytes);
  for (int r = 0; r < n_ranks; ++r) align |= uintptr_t(base[r]);
  for (int l = 0; l < n_layers; ++l) {
    if (!out[l] || (cache ? !cache[l] : layer_off[l] < 0)) return MAFED_GATHER_EINVAL;
    align |= reinterpret_cast<uintptr_t>(out[l]) |
             (cache ? reinterpret_cast<uintptr_t>(cache[l]) : uintptr_t(layer_off[l]));
  }
  if (align % uintptr_t(e)) return MAFED_GATHER_EINVAL;
  const int width = align % 16 == 0 ? 16 : align % 8 == 0 ? 8 : align % 4 == 0 ? 4 : 2;
  const int sms = sm_count();
  if (sms < 0) return MAFED_GATHER_ECUDA;

  GatherParams p;
  p.nan8 = e == 4 ? (nan1 | nan1 << 32) : (nan1 | nan1 << 16 | nan1 << 32 | nan1 << 48);
  for (int r = 0; r < n_ranks; ++r) p.base[r] = base[r];
  const int64_t region_bytes = int64_t(T) * row_bytes;
  for (int l0 = 0; l0 < n_layers; l0 += kLayers) {
    const int nl = n_layers - l0 < kLayers ? n_layers - l0 : kLayers;
    for (int b0 = 0; b0 < B; b0 += kSamples) {
      p.B = B - b0 < kSamples ? B - b0 : kSamples;
      for (int l = 0; l < nl; ++l) {
        p.out[l] = static_cast<char*>(out[l0 + l]) + int64_t(b0) * region_bytes;
        p.off[l] = cache ? uint64_t(reinterpret_cast<uintptr_t>(cache[l0 + l])) : uint64_t(layer_off[l0 + l]);
      }
      for (int b = 0; b < p.B; ++b) {
        const int64_t s = slot[b0 + b];
        const int r = src_rank ? src_rank[b0 + b] : 0;
        const bool in = s >= 0 && s < slots && r >= 0 && r < n_ranks;
        p.idx[b] = in ? int32_t(s) : -1;
        p.rank[b] = in ? uint8_t(r) : 0;
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

bool bad_sizes(int n_layers, int B, int64_t M, int T, int T_c, int n_vis, int D, int dtype) {
  return n_layers < 1 || B < 1 || M < 1 || M > INT32_MAX || n_vis < 0 || T < n_vis || T > T_c || T < 1 || D < 1 ||
         dtype < MAFED_GATHER_F32 || dtype > MAFED_GATHER_F16;
}

}  // namespace

struct mafed_teacher_shard {
  int world = 0, rank = 0;
  bool connected = false;
  void* local = nullptr;
  void* peers[kRanks] = {};     // peers[rank] is `local`; the others are IPC mappings of the peers' shards
};

extern "C" int mafed_teacher_gather_abi_version(void) { return MAFED_GATHER_ABI_VERSION; }

extern "C" const char* mafed_teacher_gather_error_string(int code) {
  switch (code) {
    case MAFED_GATHER_OK: return "ok";
    case MAFED_GATHER_EINVAL:
      return "invalid argument (needs n_layers >= 1, 1 <= B, 1 <= M <= 2^31 - 1, 0 <= n_vis <= T <= T_c, D >= 1, "
             "dtype 0/1/2, non-NULL tables and pointers aligned to the element size)";
    case MAFED_GATHER_ECUDA: return "CUDA error (device query or kernel launch)";
    case MAFED_GATHER_ESHARD: return "CUDA error allocating, exporting or mapping a teacher-cache shard";
    default: return "unknown error code";
  }
}

extern "C" int mafed_teacher_gather(void* const* out, const void* const* cache, const int64_t* idx, int n_layers,
                                    int B, int64_t M, int T, int T_c, int n_vis, int D, int dtype, void* stream) {
  if (!out || !cache || !idx || bad_sizes(n_layers, B, M, T, T_c, n_vis, D, dtype)) return MAFED_GATHER_EINVAL;
  const uint64_t zero = 0;
  return gather(out, &zero, 1, cache, nullptr, nullptr, idx, n_layers, B, M, T, T_c, n_vis, D, dtype,
                static_cast<cudaStream_t>(stream));
}

extern "C" int mafed_teacher_gather_sharded(void* const* out, const void* const* bases, int n_ranks,
                                            const int64_t* layer_off, const int32_t* src_rank, const int64_t* slot,
                                            int n_layers, int B, int64_t slots, int T, int T_c, int n_vis, int D,
                                            int dtype, void* stream) {
  if (!out || !bases || !layer_off || !src_rank || !slot || n_ranks < 1 || n_ranks > kRanks ||
      bad_sizes(n_layers, B, slots, T, T_c, n_vis, D, dtype))
    return MAFED_GATHER_EINVAL;
  uint64_t base[kRanks];
  for (int r = 0; r < n_ranks; ++r) {
    if (!bases[r]) return MAFED_GATHER_EINVAL;
    base[r] = uint64_t(reinterpret_cast<uintptr_t>(bases[r]));
  }
  return gather(out, base, n_ranks, nullptr, layer_off, src_rank, slot, n_layers, B, slots, T, T_c, n_vis, D, dtype,
                static_cast<cudaStream_t>(stream));
}

extern "C" int mafed_teacher_shard_handle_bytes(void) { return int(sizeof(cudaIpcMemHandle_t)); }

extern "C" int mafed_teacher_shard_create(int world, int rank, int64_t bytes, void* ipc_handle_out,
                                          mafed_teacher_shard_t** out) {
  if (world < 1 || world > kRanks || rank < 0 || rank >= world || bytes < 1 || !ipc_handle_out || !out)
    return MAFED_GATHER_EINVAL;
  mafed_teacher_shard* s = new mafed_teacher_shard();
  s->world = world;
  s->rank = rank;
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaMalloc(&s->local, size_t(bytes));
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, s->local);
  if (e != cudaSuccess) {
    cudaGetLastError();         // leave no error behind for the next launch check
    if (s->local) cudaFree(s->local);
    delete s;
    return MAFED_GATHER_ESHARD;
  }
  memcpy(ipc_handle_out, &h, sizeof(h));
  s->peers[rank] = s->local;
  *out = s;
  return MAFED_GATHER_OK;
}

extern "C" int mafed_teacher_shard_connect(mafed_teacher_shard_t* s, const void* all_handles) {
  if (!s || !all_handles || s->connected) return MAFED_GATHER_EINVAL;
  const char* hs = static_cast<const char*>(all_handles);
  for (int r = 0; r < s->world; ++r) {
    if (r == s->rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, hs + size_t(r) * sizeof(h), sizeof(h));
    if (cudaIpcOpenMemHandle(&s->peers[r], h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
      cudaGetLastError();
      s->peers[r] = nullptr;
      return MAFED_GATHER_ESHARD;
    }
  }
  s->connected = true;
  return MAFED_GATHER_OK;
}

extern "C" int mafed_teacher_shard_base(const mafed_teacher_shard_t* s, int rank, void** base_out) {
  if (!s || rank < 0 || rank >= s->world || !base_out || !s->peers[rank]) return MAFED_GATHER_EINVAL;
  *base_out = s->peers[rank];
  return MAFED_GATHER_OK;
}

extern "C" int mafed_teacher_shard_destroy(mafed_teacher_shard_t* s) {
  if (!s) return MAFED_GATHER_OK;
  for (int r = 0; r < s->world; ++r)
    if (r != s->rank && s->peers[r]) cudaIpcCloseMemHandle(s->peers[r]);
  if (s->local) cudaFree(s->local);
  delete s;
  return MAFED_GATHER_OK;
}
