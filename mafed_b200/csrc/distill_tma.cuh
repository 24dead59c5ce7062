// TMA-staged kernels: one producer warp streams row tiles global -> shared with bulk async copies
// (cp.async.bulk + mbarrier complete_tx; SASS: UBLKCP) through a multi-stage ring; consumer warps
// read the staged rows with conflict-free 128-bit shared loads.  One persistent CTA per SM; the ring
// keeps up to ~190 KB per SM in flight without spending registers on it.
#pragma once
#include <type_traits>

#include "distill_comm.cuh"
#include "distill_common.cuh"
#include "distill_epilogue.cuh"

namespace MAFED_NS {

constexpr int kTmaMaxStages = 8;
constexpr int kTmaMaxRows = 32;  // rows per stage (one per producer lane)
// 16 consumer warps: two stages are drained concurrently when a stage holds <= 8 rows (+2.6 % on the 1B shape over
// 8 warps, neutral elsewhere; profiles/r01_call4_sweep_extra.json)
constexpr int kTmaConsumerWarps = 16;
constexpr int kTmaConsumerThreads = kTmaConsumerWarps * 32;
constexpr unsigned kTmaPaceNs = 500;  // refill pause of a paced ring (see tma_geometry)

struct TmaGeom {
  int stages;
  int rows;         // rows per stage
  int stage_bytes;  // rows * (student row bytes + teacher row bytes)
  int pace;         // 1: the producer pauses kTmaPaceNs between a slot becoming free and its refill, as long as this
                    // CTA has met no padded row (the batch looks dense)
};

struct TmaStageMeta {
  float w[kTmaMaxRows];
  int mod[kTmaMaxRows];
  int layer;
  int n_rows;
  long long row0;
};

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  } while (!ok);
}
// 1-D bulk async copy global -> shared, completion signalled on an mbarrier (bytes % 16 == 0).
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ uint4 lds_128(uint32_t addr) {
  uint4 r;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
  return r;
}
__device__ __forceinline__ uint2 lds_64(uint32_t addr) {
  uint2 r;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(r.x), "=r"(r.y) : "r"(addr));
  return r;
}
// the teacher's share of a staged chunk (TeacherChunk::Vec): LDS.128, or LDS.64 for a half-precision teacher
template <typename V> __device__ __forceinline__ V lds_vec(uint32_t addr);
template <> __device__ __forceinline__ uint4 lds_vec<uint4>(uint32_t addr) { return lds_128(addr); }
template <> __device__ __forceinline__ uint2 lds_vec<uint2>(uint32_t addr) { return lds_64(addr); }
__device__ __forceinline__ void named_bar_sync(int id, int n_threads) {
  asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(n_threads) : "memory");
}

// ---------------------------------------------------------------- teacher-row addressing
// Where the producer finds the teacher row of row (b, t) of layer l.
//  * DenseTeacher: the [B, T, D] tensors of an ordinary step, t[l] + row * t_row_pitch.
//  * CacheTeacher: the per-task teacher cache (include/mafed_cached_step.h), one contiguous [M, T_c, D] tensor per
//    layer at t[l]; sample b is memory sample idx[b], its visual rows t < n_vis at the start of the sample's T_c rows
//    and its text rows right-aligned at their end -- the mapping of the teacher-cache gather, so that the step reads
//    the rows a gathered tensor would hold.  The table travels in the kernel parameters (__grid_constant__).
struct DenseTeacher {
  static constexpr bool kCache = false;
};

constexpr int kCacheMaxSamples = 2048;
struct CacheTeacher {
  static constexpr bool kCache = true;
  int32_t idx[kCacheMaxSamples];   // memory index of each sample, in [0, M)
  long long T_c;                   // cache rows of one sample
  long long shift;                 // T_c - T: offset of the text rows past n_vis
  float* gout_seen;                // backward fix-up: receives the upstream gradient it saw (optional)
};

// ---------------------------------------------------------------- producer
// All 32 lanes of the producer warp run this; lane r owns row r of every stage.  The backward walks its tiles
// last-to-first, so that it starts on the rows the forward left in L2.  A stage holds its rows' student bytes, then
// their teacher bytes (TT: the teacher's element type; its rows are row_bytes >> TeacherChunk::kShift long).
template <typename T, typename TT, typename TA = DenseTeacher>
__device__ __forceinline__ void tma_producer(const PathParams& p, const TmaGeom& geo, unsigned char* data,
                                             uint64_t* full, uint64_t* empty, TmaStageMeta* meta, int lane,
                                             bool for_backward, const TA& ta = TA()) {
  const long long tiles_per_layer = (p.n_rows + geo.rows - 1) / geo.rows;
  const long long total = tiles_per_layer * p.n_layers;
  const uint32_t row_bytes = (uint32_t)p.n_chunks * 16u;
  const uint32_t t_row_bytes = row_bytes >> TeacherChunk<T, TT>::kShift;
  const long long row_pitch = p.row_stride * (long long)sizeof(T);
  const long long t_row_pitch = p.row_stride * (long long)sizeof(TT);
  const bool contiguous = row_pitch == (long long)row_bytes;
  int stage = 0;
  uint32_t phase = 0;
  // The row weights of a tile come from the attention mask (an L2 round trip).  They are fetched one tile ahead, so
  // that the trip overlaps the wait for a free slot: a run of padded tiles (long, half-empty text) is otherwise paced
  // by this warp's load latency instead of by the zero-fill's bandwidth.
  // trow: the lane's teacher row in the cache (CacheTeacher only)
  struct Tile { int l, n_rows, m; long long row0; float w; long long trow; };
  // (layer, tile in layer) of this CTA's tiles advance by gridDim.x per step: kept incrementally, no 64-bit division
  // on the per-tile path; the row -> (sample, position) split is a 32-bit division whenever the row count allows it
  // (always for the cache, whose host side admits at most 2^31 - 1 rows)
  const bool rows32 = TA::kCache || p.n_rows <= 0x7fffffffLL;
  int f_l = (int)((long long)blockIdx.x / tiles_per_layer);
  long long f_til = (long long)blockIdx.x - (long long)f_l * tiles_per_layer;
  auto fetch = [&]() {
    Tile x;
    x.l = for_backward ? (p.n_layers - 1 - f_l) : f_l;
    x.row0 = (for_backward ? (tiles_per_layer - 1 - f_til) : f_til) * geo.rows;
    x.n_rows = (int)min((long long)geo.rows, p.n_rows - x.row0);
    x.m = 1;
    x.w = 0.f;
    if constexpr (TA::kCache) x.trow = 0;
    if (lane < x.n_rows) {
      if (rows32) {
        const unsigned row = (unsigned)x.row0 + (unsigned)lane;
        const unsigned bb = row / (unsigned)p.T;
        const int t = (int)(row - bb * (unsigned)p.T);
        if (t < p.n_vis) x.w = 1.f;
        else { x.m = 0; x.w = (float)__ldg(p.mask + (long long)bb * p.txt + (t - p.n_vis)); }
        if constexpr (TA::kCache) x.trow = (long long)ta.idx[bb] * ta.T_c + t + (t < p.n_vis ? 0 : ta.shift);
      } else {
        x.w = row_weight(p, x.row0 + lane, x.m);
      }
    }
    if (for_backward && p.g[x.l] == nullptr) x.w = 0.f;
    f_til += gridDim.x;
    while (f_til >= tiles_per_layer) { f_til -= tiles_per_layer; ++f_l; }
    return x;
  };
  Tile next = {};
  bool seen_padded = false;
  if ((long long)blockIdx.x < total) next = fetch();
  for (long long t0 = blockIdx.x; t0 < total; t0 += gridDim.x) {
    const Tile cur = next;
    if (t0 + gridDim.x < total) next = fetch();
    const int l = cur.l, n_rows = cur.n_rows, m = cur.m;
    const long long row0 = cur.row0;
    const float w = cur.w;
    mbar_wait(smem_u32(&empty[stage]), phase ^ 1u);  // slot free (first lap passes immediately)
    // Pacing (see tma_geometry): with every row live the step is bound by DRAM, and a coarse ring refilled at once
    // queues more in the memory system than it can use; with padded rows about, the CTAs holding more live rows are
    // the critical path and must not be held back.
    if (lane < n_rows && w == 0.f) seen_padded = true;
    seen_padded = __any_sync(0xffffffffu, seen_padded);
    if (geo.pace && !seen_padded) __nanosleep(kTmaPaceNs);

    const unsigned valid = __ballot_sync(0xffffffffu, w != 0.f);
    TmaStageMeta& mt = meta[stage];
    mt.w[lane] = w;
    mt.mod[lane] = m;
    if (lane == 0) { mt.layer = l; mt.n_rows = n_rows; mt.row0 = row0; }
    __syncwarp();
    const uint32_t bar = smem_u32(&full[stage]);
    const bool both = !p.single_input;
    if (lane == 0) {
      const uint32_t live_bytes = std::is_same<T, TT>::value ? (both ? 2u : 1u) * row_bytes
                                                             : row_bytes + (both ? t_row_bytes : 0u);
      mbar_arrive_expect_tx(bar, (uint32_t)__popc(valid) * live_bytes);
    }
    __syncwarp();
    const uint32_t s_dst = smem_u32(data + (size_t)stage * geo.stage_bytes);
    const uint32_t t_dst = s_dst + (uint32_t)geo.rows * row_bytes;
    const char* sb = reinterpret_cast<const char*>(p.s[l]) + row0 * row_pitch;
    const char* tb = reinterpret_cast<const char*>(p.t[l]) + row0 * t_row_pitch;
    const unsigned all = (n_rows >= 32) ? 0xffffffffu : ((1u << n_rows) - 1u);
    if constexpr (TA::kCache) {
      // the lane's teacher row in the cache (a sample's rows are two runs there: visual prefix, text block)
      const char* tr = reinterpret_cast<const char*>(p.t[l]) + cur.trow * (long long)t_row_bytes;
      if (contiguous && valid == all) {
        if (lane == 0) bulk_g2s(s_dst, sb, (uint32_t)n_rows * row_bytes, bar);
        // one bulk copy per contiguous run of teacher rows: a lane starts a run unless its row follows the previous
        // lane's in memory (same bytes in flight as a single copy: expect_tx is unchanged)
        const unsigned long long a = reinterpret_cast<unsigned long long>(tr);
        const unsigned long long prev = __shfl_up_sync(0xffffffffu, a, 1);
        const bool start = lane < n_rows && (lane == 0 || a != prev + t_row_bytes);
        const unsigned starts = __ballot_sync(0xffffffffu, start);
        if (start && both) {
          const unsigned later = starts & (0xfffffffeu << lane);   // the runs that start after this lane
          const int end = later ? __ffs(later) - 1 : n_rows;
          bulk_g2s(t_dst + (uint32_t)lane * t_row_bytes, tr, (uint32_t)(end - lane) * t_row_bytes, bar);
        }
      } else if (w != 0.f) {
        bulk_g2s(s_dst + (uint32_t)lane * row_bytes, sb + (long long)lane * row_pitch, row_bytes, bar);
        if (both) bulk_g2s(t_dst + (uint32_t)lane * t_row_bytes, tr, t_row_bytes, bar);
      }
    } else {
      if (contiguous && valid == all) {
        // whole tile live: one bulk copy per tensor
        if (lane == 0) bulk_g2s(s_dst, sb, (uint32_t)n_rows * row_bytes, bar);
        if (lane == 1 && both) bulk_g2s(t_dst, tb, (uint32_t)n_rows * t_row_bytes, bar);
      } else if (w != 0.f) {
        // ragged tile: only live rows are fetched (padded text rows cost no bandwidth)
        bulk_g2s(s_dst + (uint32_t)lane * row_bytes, sb + (long long)lane * row_pitch, row_bytes, bar);
        if (both) bulk_g2s(t_dst + (uint32_t)lane * t_row_bytes, tb + (long long)lane * t_row_pitch, t_row_bytes, bar);
      }
    }
    if (++stage == geo.stages) { stage = 0; phase ^= 1u; }
  }
}

struct TmaSmem {
  uint64_t full[kTmaMaxStages];
  uint64_t empty[kTmaMaxStages];
  TmaStageMeta meta[kTmaMaxStages];
};

__device__ __forceinline__ void tma_prologue(TmaSmem& sm, const TmaGeom& geo) {
  if (threadIdx.x == 0) {
    for (int i = 0; i < geo.stages; ++i) {
      mbar_init(smem_u32(&sm.full[i]), 1);      // producer's arrive.expect_tx
      mbar_init(smem_u32(&sm.empty[i]), kTmaConsumerWarps);   // one arrive per consumer warp
    }
    mbar_fence_init();
  }
  __syncthreads();
  // everything above overlapped the predecessor kernel's tail; from here on we touch global memory
  pdl_launch_dependents();
  pdl_wait();
}

// ---------------------------------------------------------------- in-kernel tail
// Called by the NT consumer threads of every CTA after its partial sums are in `ws`: the CTA that arrives
// last at the counter reduces all partials in fixed order and runs the scalar stage (losses, scale table,
// peer exchange) -- what a separate single-CTA epilogue launch would do.  The order of the reduction does
// not depend on which CTA is last, so results stay bit-reproducible.
template <int NT>
__device__ __forceinline__ void tma_tail(const PathParams& p, const double* counts_in,
                                         unsigned long long counts_epoch = 0ull) {
  __shared__ int s_last;
  __shared__ EpiSmem s_epi;
  __threadfence();  // this thread's partial-sum stores are visible device-wide before the arrival below
  named_bar_sync(1, NT);
  if (threadIdx.x == 0) {
    __threadfence();  // release: the CTA's stores (ordered before this point by the barrier) precede the arrival
    s_last = atomicAdd(p.tail_done, 1u) == gridDim.x - 1u;
    __threadfence();  // acquire: the other CTAs' stores are visible after the last arrival is observed
  }
  named_bar_sync(1, NT);
  if (!s_last) return;
  __threadfence();
  if (threadIdx.x == 0) *p.tail_done = 0u;  // every other CTA has arrived: leave the counter clean for its next user
  if (!p.tail_flags) {
    // no scalar stage here; after an in-kernel counts exchange the epoch counter still has to move on
    if (counts_epoch != 0ull && threadIdx.x == 0) *p.comm.epoch = counts_epoch;
    return;
  }
  EpiArgs a;
  a.ws = p.ws;
  a.mask = p.mask;
  a.sums = p.tail_sums;
  a.counts_out = nullptr;
  a.counts_in = counts_in;
  a.out = p.tail_out;
  a.bwd_scale = p.tail_bwd_scale;
  a.n_mask = p.n_mask;
  a.n_vis_rows = p.n_vis_rows;
  a.n_part = (int)gridDim.x;
  a.n_layers = p.n_layers;
  a.D = p.D;
  a.loss_kind = p.loss_kind;
  a.flags = p.tail_flags;
  a.comm_first = 0;
  a.comm_count = p.tail_comm ? (2 * p.n_layers + ((p.tail_flags & kEpiCounts) ? 2 : 0)) : 0;
  // after an in-kernel counts exchange at epoch e the sums exchange is e + 1 (and the counter becomes e + 1);
  // otherwise the next value of the counter
  a.comm_epoch = counts_epoch != 0ull ? counts_epoch + 1ull : 0ull;
  if (counts_epoch != 0ull && a.comm_count == 0 && threadIdx.x == 0) *p.comm.epoch = counts_epoch;
  scalar_stage<NT>(a, p.comm, p.w, s_epi, (int)threadIdx.x, SyncNamed<NT>());
}

// ---------------------------------------------------------------- forward
template <typename T, int LOSS, typename TT = T>
__global__ void __launch_bounds__(kTmaConsumerThreads + 32, 1)
k_fwd_tma(const __grid_constant__ PathParams p, const __grid_constant__ TmaGeom geo) {
  constexpr int NE = Pack<T>::kPer16;
  using Tch = TeacherChunk<T, TT>;
  using TV = typename Tch::Vec;
  extern __shared__ __align__(128) unsigned char dyn_smem[];
  __shared__ TmaSmem sm;
  __shared__ CtaSums<kTmaConsumerWarps> sums;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  cta_sums_zero(sums, p.n_layers);
  tma_prologue(sm, geo);

  if (warp == kTmaConsumerWarps) {
    tma_producer<T, TT>(p, geo, dyn_smem, sm.full, sm.empty, sm.meta, lane, false);
    return;
  }
  const long long tiles_per_layer = (p.n_rows + geo.rows - 1) / geo.rows;
  const long long total = tiles_per_layer * p.n_layers;
  const uint32_t row_bytes = (uint32_t)p.n_chunks * 16u;
  const uint32_t t_row_bytes = row_bytes >> Tch::kShift;
  float acc_text = 0.f, acc_vis = 0.f;
  int cur = -1, stage = 0;
  uint32_t phase = 0;
  long long it = 0;
  for (long long t0 = blockIdx.x; t0 < total; t0 += gridDim.x, ++it) {
    mbar_wait(smem_u32(&sm.full[stage]), phase);
    const TmaStageMeta& mt = sm.meta[stage];
    const int l = mt.layer;
    if (l != cur) {
      cta_sums_flush(sums, warp, lane, cur, acc_text, acc_vis);
      acc_text = acc_vis = 0.f;
      cur = l;
    }
    const uint32_t s_base = smem_u32(dyn_smem + (size_t)stage * geo.stage_bytes);
    const uint32_t t_base = s_base + (uint32_t)geo.rows * row_bytes;
    // rotate the row->warp map with the iteration so short tiles still use every warp over time
    const int first =
        (int)((warp + kTmaConsumerWarps - (int)((it * geo.rows) % kTmaConsumerWarps)) % kTmaConsumerWarps);
    for (int r = first; r < mt.n_rows; r += kTmaConsumerWarps) {
      const float w = mt.w[r];
      if (w == 0.f) continue;
      const uint32_t sa = s_base + (uint32_t)r * row_bytes, ta = t_base + (uint32_t)r * t_row_bytes;
      float x = 0.f, y = 0.f, z = 0.f;
      int c = lane;
      for (; c + 96 < p.n_chunks; c += 128) {
        uint4 sv[4];
        TV tv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          sv[u] = lds_128(sa + (uint32_t)(c + 32 * u) * 16u);
          if constexpr (LOSS == kLossL2Norm) tv[u] = sv[u];
          else tv[u] = lds_vec<TV>(ta + (uint32_t)(c + 32 * u) * (uint32_t)Tch::kBytes);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          float a[NE], b[NE];
          Pack<T>::unpack(sv[u], a);
          Tch::unpack(tv[u], b);
          accumulate<LOSS, NE>(a, b, x, y, z);
        }
      }
      for (; c < p.n_chunks; c += 32) {
        float a[NE], b[NE];
        const uint4 sv1 = lds_128(sa + (uint32_t)c * 16u);
        Pack<T>::unpack(sv1, a);
        if constexpr (LOSS == kLossL2Norm) Tch::unpack(sv1, b);
        else Tch::unpack(lds_vec<TV>(ta + (uint32_t)c * (uint32_t)Tch::kBytes), b);
        accumulate<LOSS, NE>(a, b, x, y, z);
      }
      float val;
      if (LOSS == MAFED_LOSS_MSE) {
        val = x;
      } else {
        x = warp_sum(x); y = warp_sum(y); z = warp_sum(z);
        val = (lane == 0) ? row_value<LOSS>(x, y, z) : 0.f;
      }
      if (mt.mod[r] == 0) acc_text = fmaf(w, val, acc_text);
      else acc_vis = fmaf(w, val, acc_vis);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(smem_u32(&sm.empty[stage]));
    if (++stage == geo.stages) { stage = 0; phase ^= 1u; }
  }
  cta_sums_flush(sums, warp, lane, cur, acc_text, acc_vis);
  named_bar_sync(1, kTmaConsumerThreads);
  cta_sums_store(sums, p.ws, p.n_layers, 0, kTmaConsumerThreads);
  if (p.tail_done != nullptr) tma_tail<kTmaConsumerThreads>(p, nullptr);
}

// ---------------------------------------------------------------- backward
template <int LOSS, int NE>
__device__ __forceinline__ void grad_elems_tma(const float (&a)[NE], const float (&b)[NE], float scale, float ch,
                                               float cp, float (&o)[NE]) {
#pragma unroll
  for (int i = 0; i < NE; ++i) {
    if (LOSS == MAFED_LOSS_MSE) o[i] = scale * (a[i] - b[i]);
    else o[i] = fmaf(ch, a[i], -cp * b[i]);
  }
}

// Cosine gradient of one SHORT row of exactly 32 * CPL chunks with compile-time trip counts: the shared-memory loads
// of a batch are issued back to back, there is no loop control, and the row scalars cost one reciprocal instead of
// three divisions.  KEEP: the lane's share of the row pair stays in registers between the statistics and the gradient
// (no second sweep over shared memory) -- affordable up to CPL = 3 in the 16-warp build (96 registers per thread);
// otherwise the row is swept twice in batches of two chunks.  At 1.5-2 KB rows the generic two-sweep loop further
// down is bound by instruction issue (61 % of the issue slots at 4 warps per scheduler,
// profiles/r02a_ncu_fused_C2_cosine_raw.csv), not by HBM.  Returns the row's loss value 1 - cos (all lanes hold it).
template <typename T>
__device__ __forceinline__ void cosine_stats_chunk(const uint4& sv, const uint4& tv, float& x, float& y, float& z) {
  constexpr int NW = Pack<T>::kPerWord;
  // word by word, so that only a handful of unpacked values is live at any time
  const uint32_t sw[4] = {sv.x, sv.y, sv.z, sv.w}, tw[4] = {tv.x, tv.y, tv.z, tv.w};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    float a[NW], b[NW];
    Pack<T>::unpack_word(sw[k], a);
    Pack<T>::unpack_word(tw[k], b);
    accumulate<MAFED_LOSS_COSINE, NW>(a, b, x, y, z);
  }
}

template <typename T>
__device__ __forceinline__ uint4 cosine_grad_chunk(const uint4& sv, const uint4& tv, float ch, float cp) {
  constexpr int NW = Pack<T>::kPerWord;
  const uint32_t sw[4] = {sv.x, sv.y, sv.z, sv.w}, tw[4] = {tv.x, tv.y, tv.z, tv.w};
  uint32_t ow[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    float a[NW], b[NW], o[NW];
    Pack<T>::unpack_word(sw[k], a);
    Pack<T>::unpack_word(tw[k], b);
#pragma unroll
    for (int i = 0; i < NW; ++i) o[i] = fmaf(ch, a[i], -cp * b[i]);
    ow[k] = Pack<T>::pack_word(o);
  }
  return make_uint4(ow[0], ow[1], ow[2], ow[3]);
}

template <typename T, int CPL, bool KEEP>
__device__ __forceinline__ float cosine_row_unrolled(uint32_t sa, uint32_t ta, int lane, float w, char* grow) {
  constexpr int NB = KEEP ? CPL : 2;          // chunks per batch of loads
  static_assert(CPL % NB == 0, "batches of two chunks");
  uint4 sv[NB], tv[NB];
  float x = 0.f, y = 0.f, z = 0.f;
#pragma unroll
  for (int u0 = 0; u0 < CPL; u0 += NB) {
#pragma unroll
    for (int u = 0; u < NB; ++u) {
      sv[u] = lds_128(sa + (uint32_t)(lane + 32 * (u0 + u)) * 16u);
      tv[u] = lds_128(ta + (uint32_t)(lane + 32 * (u0 + u)) * 16u);
    }
#pragma unroll
    for (int u = 0; u < NB; ++u) cosine_stats_chunk<T>(sv[u], tv[u], x, y, z);
  }
  x = warp_sum(x); y = warp_sum(y); z = warp_sum(z);
  // cos = x / den, den = sqrt((|h|^2 + eps)(|p|^2 + eps));  d(1 - cos)/dh = (cos / (|h|^2 + eps)) h - p / den
  const float aa = y + kCosEps, den = sqrtf(aa * (z + kCosEps));
  const float r = __frcp_rn(den * aa);          // one correctly rounded reciprocal serves both quotients
  const float inv_den = r * aa, cosv = x * inv_den;
  const float ch = w * cosv * (r * den), cp = w * inv_den;
  if (grow != nullptr) {
#pragma unroll
    for (int u0 = 0; u0 < CPL; u0 += NB) {
      if (!KEEP) {
#pragma unroll
        for (int u = 0; u < NB; ++u) {
          sv[u] = lds_128(sa + (uint32_t)(lane + 32 * (u0 + u)) * 16u);
          tv[u] = lds_128(ta + (uint32_t)(lane + 32 * (u0 + u)) * 16u);
        }
      }
#pragma unroll
      for (int u = 0; u < NB; ++u)
        stg_128(grow + (lane + 32 * (u0 + u)) * 16, cosine_grad_chunk<T>(sv[u], tv[u], ch, cp));
    }
  }
  return 1.f - cosv;
}

// MODE = kBackward: gradients only.  MODE = kFused: the consumers also accumulate the forward's loss
// sums from the rows they already hold in shared memory (one pass over student and teacher per step).
// TA: the teacher-row addressing (k_bwd_tma: DenseTeacher; k_bwd_tma_cached: CacheTeacher); only the producer
// reads it, so the consumers' arithmetic is the same for both.
template <typename T, int LOSS, int MODE, typename TT, typename TA>
__device__ __forceinline__ void bwd_tma_body(const PathParams& p, const TmaGeom& geo, const TA& ta) {
  constexpr int NE = Pack<T>::kPer16;
  constexpr bool FUSED = MODE == kFused;
  // a half-precision teacher under an fp32 student: no unrolled short-row cosine forms (general two-sweep loop)
  constexpr bool kSameType = std::is_same<T, TT>::value;
  using Tch = TeacherChunk<T, TT>;
  using TV = typename Tch::Vec;
  extern __shared__ __align__(128) unsigned char dyn_smem[];
  __shared__ TmaSmem sm;
  __shared__ CtaSums<FUSED ? kTmaConsumerWarps : 1> sums;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (FUSED) cta_sums_zero(sums, p.n_layers);
  tma_prologue(sm, geo);
  float gout;
  if (FUSED) {
    gout = p.fixed_gout;
  } else {
    gout = (p.grad_out ? __ldg(p.grad_out) : 1.f) * p.gout_scale;
    if constexpr (TA::kCache) {
      if (ta.gout_seen != nullptr && blockIdx.x == 0 && threadIdx.x == 0) *ta.gout_seen = gout;
    }
    if (p.skip_if_gout_equals && gout == p.fixed_gout) return;  // fix-up launch with nothing to fix
  }
  if (warp == kTmaConsumerWarps) {
    tma_producer<T, TT, TA>(p, geo, dyn_smem, sm.full, sm.empty, sm.meta, lane, !FUSED, ta);
    return;
  }
  // Scale table in shared memory.  One-pass step with the prologue folded in: while the producer's first
  // tiles are in flight, the consumer warps count the valid text tokens themselves (the mask is a few KB,
  // L2-resident) and derive the table; CTA 0 publishes it for the later backward fix-up.
  __shared__ float s_scale[2 * kMaxLayers];
  __shared__ double s_counts[2];  // (global) token counts, kept for the tail
  unsigned long long counts_epoch = 0ull;
  if (FUSED && p.lang_mask_out != nullptr) {
    // the masks the reference leaves in `batch` (distillation.py:134-144): a few hundred KB spread over all CTAs
    const long long n = p.n_rows;
    for (long long i = (long long)blockIdx.x * kTmaConsumerThreads + threadIdx.x; i < n;
         i += (long long)gridDim.x * kTmaConsumerThreads) {
      const long long b = i / p.T;
      const int t = (int)(i - b * p.T);
      const bool vis = t < p.n_vis;
      p.lang_mask_out[i] = vis ? 0 : p.mask[b * p.txt + (t - p.n_vis)];
      p.image_mask_out[i] = vis ? 1 : 0;
    }
  }
  if (FUSED && p.inline_scale) {
    __shared__ long long s_cnt[kTmaConsumerWarps];
    __shared__ double s_peer[kCommMaxRanks][2];
    const CommDev& c = p.comm;
    const bool sharded = c.world > 1 && p.comm_counts;
    double n_text, n_vis_rows;
    if (p.counts_ticket != nullptr) {
      // The counts were computed -- and, across batch shards, sent to every peer -- when the batch was drawn
      // (k_prefetch_counts), long before this kernel: nothing to sum, and the poll below finds every peer's words
      // already in the own mailbox (local L2).  The prefetch has its own epoch counter and slot generations, so the
      // sums exchange in the tail simply takes the next value of the main counter (counts_epoch stays 0).
      if (sharded) {
        const unsigned long long e = (unsigned long long)__ldcg(p.counts_ticket);
        const long long t_x0 = clock64();
        if ((int)threadIdx.x < 2 * c.world) {
          const int r = threadIdx.x >> 1, k = threadIdx.x & 1;
          s_peer[r][k] = ll_wait(ll_count_slot(c.ll[c.rank], (int)(e % kCommCountSlots), r, k), ll_tag(e), c.status,
                                 c.timeout_cycles);
        }
        named_bar_sync(1, kTmaConsumerThreads);
        if (blockIdx.x == 0 && threadIdx.x == 0) c.trace[0] += (unsigned long long)(clock64() - t_x0);
        n_text = 0.0;
        n_vis_rows = 0.0;
        for (int r = 0; r < c.world; ++r) {
          n_text += s_peer[r][0];
          n_vis_rows += s_peer[r][1];
        }
      } else {
        n_text = __longlong_as_double(__ldcg(p.counts_ticket + 1));
        n_vis_rows = __longlong_as_double(__ldcg(p.counts_ticket + 2));
      }
    } else {
      long long cnt = 0;
      for (long long i = threadIdx.x; i < p.n_mask; i += kTmaConsumerThreads) cnt += p.mask[i];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
      if (lane == 0) s_cnt[warp] = cnt;
      named_bar_sync(1, kTmaConsumerThreads);
      long long n_text_local = 0;
#pragma unroll
      for (int i = 0; i < kTmaConsumerWarps; ++i) n_text_local += s_cnt[i];
      n_text = (double)n_text_local;
      n_vis_rows = p.n_vis_rows;
      if (sharded) {
        // Batch-sharded step: the two token counts are exchanged right here.  CTA 0 fires this rank's counts into
        // every rank's mailbox as self-validating words (distill_comm.cuh: no fence, no flag); every CTA then polls
        // its OWN rank's mailbox (local L2) for all peers and sums in rank order.  The one-way NVLink trip hides
        // behind the first tiles.
        const long long t_x0 = clock64();
        // nobody writes the counter before the last CTA's tail: every CTA of this launch reads the same value
        const unsigned long long e = __ldcg(c.epoch) + 1ull;
        counts_epoch = e;
        const int par = (int)(e & 1ull);
        const uint32_t tag = ll_tag(e);
        if (blockIdx.x == 0) {
          if ((int)threadIdx.x < 2 * c.world) {
            const int peer = threadIdx.x >> 1, k = threadIdx.x & 1;
            ll_store(ll_slot(c.ll[peer], par, c.rank, k), k == 0 ? n_text : n_vis_rows, tag);
          }
        }
        if ((int)threadIdx.x < 2 * c.world) {
          const int r = threadIdx.x >> 1, k = threadIdx.x & 1;
          s_peer[r][k] = ll_wait(ll_slot(c.ll[c.rank], par, r, k), tag, c.status, c.timeout_cycles);
        }
        named_bar_sync(1, kTmaConsumerThreads);
        if (blockIdx.x == 0 && threadIdx.x == 0) c.trace[0] += (unsigned long long)(clock64() - t_x0);
        n_text = 0.0;
        n_vis_rows = 0.0;
        for (int r = 0; r < c.world; ++r) {
          n_text += s_peer[r][0];
          n_vis_rows += s_peer[r][1];
        }
      }
    }
    if (threadIdx.x == 0) { s_counts[0] = n_text; s_counts[1] = n_vis_rows; }
    if ((int)threadIdx.x < p.n_layers) {
      float st, sv;
      backward_scales(p.w, threadIdx.x, n_text, n_vis_rows, p.loss_kind, p.D, st, sv);
      s_scale[2 * threadIdx.x] = st;
      s_scale[2 * threadIdx.x + 1] = sv;
      if (blockIdx.x == 0) {
        p.bwd_scale_out[2 * threadIdx.x] = st;
        p.bwd_scale_out[2 * threadIdx.x + 1] = sv;
      }
    }
  } else {
    for (int i = threadIdx.x; i < 2 * p.n_layers; i += kTmaConsumerThreads) s_scale[i] = __ldg(p.bwd_scale + i);
  }
  named_bar_sync(1, kTmaConsumerThreads);

  const long long tiles_per_layer = (p.n_rows + geo.rows - 1) / geo.rows;
  const long long total = tiles_per_layer * p.n_layers;
  const uint32_t row_bytes = (uint32_t)p.n_chunks * 16u;
  const uint32_t t_row_bytes = row_bytes >> Tch::kShift;
  const long long row_pitch = p.row_stride * (long long)sizeof(T);
  float acc_text = 0.f, acc_vis = 0.f;
  int cur = -1;
  int stage = 0;
  uint32_t phase = 0;
  long long it = 0;
  for (long long t0 = blockIdx.x; t0 < total; t0 += gridDim.x, ++it) {
    mbar_wait(smem_u32(&sm.full[stage]), phase);
    const TmaStageMeta& mt = sm.meta[stage];
    const int l = mt.layer;
    if (FUSED && l != cur) {
      cta_sums_flush(sums, warp, lane, cur, acc_text, acc_vis);
      acc_text = acc_vis = 0.f;
      cur = l;
    }
    char* gb = reinterpret_cast<char*>(p.g[l]);
    const uint32_t s_base = smem_u32(dyn_smem + (size_t)stage * geo.stage_bytes);
    const uint32_t t_base = s_base + (uint32_t)geo.rows * row_bytes;
    const int first =
        (int)((warp + kTmaConsumerWarps - (int)((it * geo.rows) % kTmaConsumerWarps)) % kTmaConsumerWarps);
    if (FUSED || gb != nullptr) {
      for (int r = first; r < mt.n_rows; r += kTmaConsumerWarps) {
        char* grow = gb + (mt.row0 + r) * row_pitch;
        const float w = mt.w[r] * (gout * s_scale[2 * l + mt.mod[r]]);
        if (mt.w[r] == 0.f) {  // padded text row: nothing was fetched; grad = 0 * scale (zero, or NaN if scale is)
          float o[NE];
#pragma unroll
          for (int i = 0; i < NE; ++i) o[i] = w;
          const uint4 fill = Pack<T>::pack(o);
          if (gb != nullptr)
            for (int c = lane; c < p.n_chunks; c += 32) stg_128(grow + (long long)c * 16, fill);
          continue;
        }
        const uint32_t sa = s_base + (uint32_t)r * row_bytes, ta = t_base + (uint32_t)r * t_row_bytes;
        float ch = 0.f, cp = 0.f, rowval = 0.f;
        if constexpr (kSameType) {
          if (LOSS == MAFED_LOSS_COSINE && (p.n_chunks == 96 || p.n_chunks == 128 || p.n_chunks == 192)) {
            // short rows (1.5 / 2 / 3 KB: base and 410M hidden sizes in bf16, base in fp32): fully unrolled forms
            float val;
            if (p.n_chunks == 96) val = cosine_row_unrolled<T, 3, true>(sa, ta, lane, w, gb != nullptr ? grow : nullptr);
            else if (p.n_chunks == 128) val = cosine_row_unrolled<T, 4, false>(sa, ta, lane, w, gb != nullptr ? grow : nullptr);
            else val = cosine_row_unrolled<T, 6, false>(sa, ta, lane, w, gb != nullptr ? grow : nullptr);
            if (FUSED && lane == 0) {
              if (mt.mod[r] == 0) acc_text = fmaf(mt.w[r], val, acc_text);
              else acc_vis = fmaf(mt.w[r], val, acc_vis);
            }
            continue;
          }
        }
        if (LOSS == MAFED_LOSS_COSINE) {
          float x = 0.f, y = 0.f, z = 0.f;
          for (int c = lane; c < p.n_chunks; c += 32) {
            float a[NE], b[NE];
            Pack<T>::unpack(lds_128(sa + (uint32_t)c * 16u), a);
            Tch::unpack(lds_vec<TV>(ta + (uint32_t)c * (uint32_t)Tch::kBytes), b);
            accumulate<LOSS, NE>(a, b, x, y, z);
          }
          x = warp_sum(x); y = warp_sum(y); z = warp_sum(z);
          const float aa = y + kCosEps, den = sqrtf(aa * (z + kCosEps));
          ch = w * (x / den) / aa;
          cp = w / den;
          rowval = (lane == 0) ? 1.f - x / den : 0.f;
        }
        int c = lane;
        for (; c + 96 < p.n_chunks; c += 128) {
          uint4 sv[4];
          TV tv[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            sv[u] = lds_128(sa + (uint32_t)(c + 32 * u) * 16u);
            tv[u] = lds_vec<TV>(ta + (uint32_t)(c + 32 * u) * (uint32_t)Tch::kBytes);
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            float a[NE], b[NE], o[NE];
            Pack<T>::unpack(sv[u], a);
            Tch::unpack(tv[u], b);
            if (FUSED && LOSS == MAFED_LOSS_MSE) {
              float y = 0.f, z = 0.f;
              accumulate<LOSS, NE>(a, b, rowval, y, z);
            }
            grad_elems_tma<LOSS, NE>(a, b, w, ch, cp, o);
            if (gb != nullptr) stg_128(grow + (long long)(c + 32 * u) * 16, Pack<T>::pack(o));
          }
        }
        for (; c < p.n_chunks; c += 32) {
          float a[NE], b[NE], o[NE];
          Pack<T>::unpack(lds_128(sa + (uint32_t)c * 16u), a);
          Tch::unpack(lds_vec<TV>(ta + (uint32_t)c * (uint32_t)Tch::kBytes), b);
          if (FUSED && LOSS == MAFED_LOSS_MSE) {
            float y = 0.f, z = 0.f;
            accumulate<LOSS, NE>(a, b, rowval, y, z);
          }
          grad_elems_tma<LOSS, NE>(a, b, w, ch, cp, o);
          if (gb != nullptr) stg_128(grow + (long long)c * 16, Pack<T>::pack(o));
        }
        if (FUSED) {
          if (mt.mod[r] == 0) acc_text = fmaf(mt.w[r], rowval, acc_text);
          else acc_vis = fmaf(mt.w[r], rowval, acc_vis);
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(smem_u32(&sm.empty[stage]));
    if (++stage == geo.stages) { stage = 0; phase ^= 1u; }
  }
  if (FUSED) {
    cta_sums_flush(sums, warp, lane, cur, acc_text, acc_vis);
    named_bar_sync(1, kTmaConsumerThreads);
    cta_sums_store(sums, p.ws, p.n_layers, 0, kTmaConsumerThreads);
    if (p.tail_done != nullptr) tma_tail<kTmaConsumerThreads>(p, p.inline_scale ? s_counts : p.tail_counts_in, counts_epoch);
  }
}

template <typename T, int LOSS, int MODE, typename TT = T>
__global__ void __launch_bounds__(kTmaConsumerThreads + 32, 1)
k_bwd_tma(const __grid_constant__ PathParams p, const __grid_constant__ TmaGeom geo) {
  bwd_tma_body<T, LOSS, MODE, TT>(p, geo, DenseTeacher());
}

// The same kernel reading the teacher rows straight from the per-task cache (mafed_cached_step.h).
template <typename T, int LOSS, int MODE, typename TT = T>
__global__ void __launch_bounds__(kTmaConsumerThreads + 32, 1)
k_bwd_tma_cached(const __grid_constant__ PathParams p, const __grid_constant__ TmaGeom geo,
                 const __grid_constant__ CacheTeacher c) {
  bwd_tma_body<T, LOSS, MODE, TT>(p, geo, c);
}

}  // namespace MAFED_NS
