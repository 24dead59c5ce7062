// Register-staged kernels: one warp per token row, 128-bit coalesced streaming loads, many loads in
// flight per lane.  Persistent grid (a multiple of the SM count), static round-robin over
// (layer, row-group) work items so that a CTA's warps read consecutive rows.
#pragma once
#include "distill_common.cuh"

namespace MAFED_NS {

constexpr int kLdgThreads = 256;
constexpr int kLdgWarps = kLdgThreads / 32;
constexpr int kLdgMinBlocks = 3;      // forward: <= 80 registers, 24 warps/SM
constexpr int kLdgMinBlocksBwd = 2;   // backward keeps a whole row pair in registers: <= 128 registers

// CPL : 16-byte chunks per lane per pass (a pass covers 32*CPL chunks of a row)
// RPI : rows per warp per iteration (more independent loads in flight for short rows)
// TT: the teacher's element type (TeacherChunk: the teacher's share of a 16-byte student chunk)
template <typename T, int CPL, int RPI, int LOSS, typename TT = T>
__global__ void __launch_bounds__(kLdgThreads, kLdgMinBlocks) k_fwd_ldg(const __grid_constant__ PathParams p) {
  constexpr int NE = Pack<T>::kPer16;
  using Tch = TeacherChunk<T, TT>;
  using TV = typename Tch::Vec;
  __shared__ CtaSums<kLdgWarps> sums;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  cta_sums_zero(sums, p.n_layers);
  __syncthreads();
  pdl_launch_dependents();
  pdl_wait();

  constexpr int kRowsPerIter = kLdgWarps * RPI;
  const long long groups_per_layer = (p.n_rows + kRowsPerIter - 1) / kRowsPerIter;
  const long long total = groups_per_layer * p.n_layers;
  const int n_pass = (CPL == 8) ? (p.n_chunks + 32 * CPL - 1) / (32 * CPL) : 1;
  const long long row_bytes = p.row_stride * (long long)sizeof(T);
  const long long t_row_bytes = p.row_stride * (long long)sizeof(TT);

  float acc_text = 0.f, acc_vis = 0.f;
  int cur = -1;
  for (long long g = blockIdx.x; g < total; g += gridDim.x) {
    const int l = (int)(g / groups_per_layer);
    const long long gi = g - (long long)l * groups_per_layer;
    if (l != cur) {
      cta_sums_flush(sums, warp, lane, cur, acc_text, acc_vis);
      acc_text = acc_vis = 0.f;
      cur = l;
    }
    const char* sb = reinterpret_cast<const char*>(p.s[l]);
    const char* tb = reinterpret_cast<const char*>(p.t[l]);
    const long long row0 = gi * kRowsPerIter + (long long)warp * RPI;

    float w[RPI];
    int m[RPI];
#pragma unroll
    for (int r = 0; r < RPI; ++r) {
      m[r] = 1;
      w[r] = (row0 + r < p.n_rows) ? row_weight(p, row0 + r, m[r]) : 0.f;
    }
    float x[RPI], y[RPI], z[RPI];
#pragma unroll
    for (int r = 0; r < RPI; ++r) x[r] = y[r] = z[r] = 0.f;

    for (int pass = 0; pass < n_pass; ++pass) {
      uint4 sv[RPI][CPL];
      TV tv[RPI][CPL];
#pragma unroll
      for (int r = 0; r < RPI; ++r) {
        const long long off = (row0 + r) * row_bytes;
        const long long t_off = (row0 + r) * t_row_bytes;
#pragma unroll
        for (int i = 0; i < CPL; ++i) {
          const int c = pass * 32 * CPL + lane + 32 * i;
          tv[r][i] = TV{};
          if (w[r] != 0.f && c < p.n_chunks) {
            sv[r][i] = ldg_stream(sb + off + (long long)c * 16);
            if (LOSS != kLossL2Norm) tv[r][i] = Tch::ldg(tb + t_off + (long long)c * Tch::kBytes);
          } else {
            sv[r][i] = make_uint4(0, 0, 0, 0);
          }
        }
      }
#pragma unroll
      for (int r = 0; r < RPI; ++r) {
#pragma unroll
        for (int i = 0; i < CPL; ++i) {
          float a[NE], b[NE];
          Pack<T>::unpack(sv[r][i], a);
          Tch::unpack(tv[r][i], b);
          accumulate<LOSS, NE>(a, b, x[r], y[r], z[r]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < RPI; ++r) {
      if (w[r] == 0.f) continue;
      float val;
      if (LOSS == MAFED_LOSS_MSE) {
        val = x[r];  // lane-partial; summed across lanes at flush time
      } else {
        const float dx = warp_sum(x[r]), dy = warp_sum(y[r]), dz = warp_sum(z[r]);
        val = (lane == 0) ? row_value<LOSS>(dx, dy, dz) : 0.f;
      }
      if (m[r] == 0) acc_text = fmaf(w[r], val, acc_text);
      else acc_vis = fmaf(w[r], val, acc_vis);
    }
  }
  cta_sums_flush(sums, warp, lane, cur, acc_text, acc_vis);
  __syncthreads();
  cta_sums_store(sums, p.ws, p.n_layers, 0, kLdgThreads);
}

// Gradient of the per-row loss w.r.t. the student row, times `scale`.
//   mse   : scale * (h - p)                       (the 2/D lives in bwd_scale)
//   cosine: scale * ((cos/a) * h - p / den)       a = |h|^2+eps, den = sqrt(a*b)
template <int LOSS, int NE>
__device__ __forceinline__ void grad_elems(const float (&a)[NE], const float (&b)[NE], float scale, float ch, float cp,
                                           float (&o)[NE]) {
#pragma unroll
  for (int i = 0; i < NE; ++i) {
    if (LOSS == MAFED_LOSS_MSE) o[i] = scale * (a[i] - b[i]);
    else o[i] = fmaf(ch, a[i], -cp * b[i]);
  }
}

// Upstream gradient seen by a backward-shaped kernel.  Returns false when the kernel has nothing to do
// (fix-up launch after a fused pass whose assumed upstream gradient turned out to be right).
template <int MODE>
__device__ __forceinline__ bool upstream_grad(const PathParams& p, float& gout) {
  if (MODE == kFused) { gout = p.fixed_gout; return true; }
  gout = (p.grad_out ? __ldg(p.grad_out) : 1.f) * p.gout_scale;
  return !(p.skip_if_gout_equals && gout == p.fixed_gout);
}

// MODE = kBackward: gradients only (2 reads + 1 write), work items walked last-to-first so that the pass starts on
// the rows the forward left in L2.  MODE = kFused: the same pass also accumulates the forward's [layer][modality]
// loss sums, so student and teacher are read once per step.
template <typename T, int CPL, int RPI, int LOSS, int MODE, typename TT = T>
__global__ void __launch_bounds__(kLdgThreads, kLdgMinBlocksBwd) k_bwd_ldg(const __grid_constant__ PathParams p) {
  constexpr int NE = Pack<T>::kPer16;
  using Tch = TeacherChunk<T, TT>;
  using TV = typename Tch::Vec;
  constexpr bool FUSED = MODE == kFused;
  __shared__ CtaSums<FUSED ? kLdgWarps : 1> sums;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_launch_dependents();
  pdl_wait();
  float gout;
  if (!upstream_grad<MODE>(p, gout)) return;
  if (FUSED) {
    cta_sums_zero(sums, p.n_layers);
    __syncthreads();
  }
  constexpr int kRowsPerIter = kLdgWarps * RPI;
  const long long groups_per_layer = (p.n_rows + kRowsPerIter - 1) / kRowsPerIter;
  const long long total = groups_per_layer * p.n_layers;
  const int n_pass = (CPL == 8) ? (p.n_chunks + 32 * CPL - 1) / (32 * CPL) : 1;
  const long long row_bytes = p.row_stride * (long long)sizeof(T);
  const long long t_row_bytes = p.row_stride * (long long)sizeof(TT);

  float acc_text = 0.f, acc_vis = 0.f;
  int cur = -1;
  // (the backward steps g itself down: mirroring an ascending index instead costs up to 15 registers per thread and,
  // at short rows, a CTA per SM)
  constexpr bool kReverse = MODE == kBackward;
  const long long step = kReverse ? -(long long)gridDim.x : (long long)gridDim.x;
  for (long long g = kReverse ? total - 1 - blockIdx.x : blockIdx.x; g >= 0 && g < total; g += step) {
    const int l = (int)(g / groups_per_layer);
    const long long gi = g - (long long)l * groups_per_layer;
    char* gb = reinterpret_cast<char*>(p.g[l]);
    if (!FUSED && gb == nullptr) continue;
    if (FUSED && l != cur) {
      cta_sums_flush(sums, warp, lane, cur, acc_text, acc_vis);
      acc_text = acc_vis = 0.f;
      cur = l;
    }
    const char* sb = reinterpret_cast<const char*>(p.s[l]);
    const char* tb = reinterpret_cast<const char*>(p.t[l]);
    const long long row0 = gi * kRowsPerIter + (long long)warp * RPI;

    float w[RPI], wraw[RPI];
    int m[RPI];
    bool live[RPI];
#pragma unroll
    for (int r = 0; r < RPI; ++r) {
      m[r] = 1;
      live[r] = row0 + r < p.n_rows;
      wraw[r] = live[r] ? row_weight(p, row0 + r, m[r]) : 0.f;
      // a zero weight (padded text position) gives 0 * scale: an exact zero row, as autograd's `* mask`
      w[r] = wraw[r] * (gout * __ldg(p.bwd_scale + 2 * l + m[r]));
    }

    // cosine with rows longer than one pass: statistics first, then a second sweep (L2 hits)
    float ch[RPI], cp[RPI], rowval[RPI];
#pragma unroll
    for (int r = 0; r < RPI; ++r) ch[r] = cp[r] = rowval[r] = 0.f;
    if (LOSS == MAFED_LOSS_COSINE && n_pass > 1) {
#pragma unroll
      for (int r = 0; r < RPI; ++r) {
        if (wraw[r] == 0.f) continue;
        float x = 0.f, y = 0.f, z = 0.f;
        const long long off = (row0 + r) * row_bytes;
        const long long t_off = (row0 + r) * t_row_bytes;
        for (int c = lane; c < p.n_chunks; c += 32) {
          float a[NE], b[NE];
          Pack<T>::unpack(ldg_stream(sb + off + (long long)c * 16), a);
          Tch::unpack(Tch::ldg(tb + t_off + (long long)c * Tch::kBytes), b);
          accumulate<LOSS, NE>(a, b, x, y, z);
        }
        x = warp_sum(x); y = warp_sum(y); z = warp_sum(z);
        const float aa = y + kCosEps, den = sqrtf(aa * (z + kCosEps));
        ch[r] = w[r] * (x / den) / aa;
        cp[r] = w[r] / den;
        rowval[r] = (lane == 0) ? 1.f - x / den : 0.f;
      }
    }

    for (int pass = 0; pass < n_pass; ++pass) {
      uint4 sv[RPI][CPL];
      TV tv[RPI][CPL];
#pragma unroll
      for (int r = 0; r < RPI; ++r) {
        const long long off = (row0 + r) * row_bytes;
        const long long t_off = (row0 + r) * t_row_bytes;
#pragma unroll
        for (int i = 0; i < CPL; ++i) {
          const int c = pass * 32 * CPL + lane + 32 * i;
          if (wraw[r] != 0.f && c < p.n_chunks) {
            sv[r][i] = ldg_stream(sb + off + (long long)c * 16);
            tv[r][i] = Tch::ldg(tb + t_off + (long long)c * Tch::kBytes);
          } else {
            sv[r][i] = make_uint4(0, 0, 0, 0);
            tv[r][i] = TV{};
          }
        }
      }
      if (LOSS == MAFED_LOSS_COSINE && n_pass == 1) {
#pragma unroll
        for (int r = 0; r < RPI; ++r) {
          float x = 0.f, y = 0.f, z = 0.f;
#pragma unroll
          for (int i = 0; i < CPL; ++i) {
            float a[NE], b[NE];
            Pack<T>::unpack(sv[r][i], a);
            Tch::unpack(tv[r][i], b);
            accumulate<LOSS, NE>(a, b, x, y, z);
          }
          x = warp_sum(x); y = warp_sum(y); z = warp_sum(z);
          const float aa = y + kCosEps, den = sqrtf(aa * (z + kCosEps));
          ch[r] = w[r] * (x / den) / aa;
          cp[r] = w[r] / den;
          rowval[r] = (lane == 0) ? 1.f - x / den : 0.f;
        }
      }
#pragma unroll
      for (int r = 0; r < RPI; ++r) {
        if (!live[r]) continue;
        const long long off = (row0 + r) * row_bytes;
#pragma unroll
        for (int i = 0; i < CPL; ++i) {
          const int c = pass * 32 * CPL + lane + 32 * i;
          if (c >= p.n_chunks) continue;
          float a[NE], b[NE], o[NE];
          Pack<T>::unpack(sv[r][i], a);
          Tch::unpack(tv[r][i], b);
          if (FUSED && LOSS == MAFED_LOSS_MSE) {
            float y = 0.f, z = 0.f;
            accumulate<LOSS, NE>(a, b, rowval[r], y, z);  // lane-partial sum of (h-p)^2
          }
          if (wraw[r] == 0.f) {
#pragma unroll
            for (int e = 0; e < NE; ++e) o[e] = w[r];  // 0 (or NaN when the scale is NaN, like 0 * NaN upstream)
          } else {
            grad_elems<LOSS, NE>(a, b, w[r], ch[r], cp[r], o);
          }
          if (gb != nullptr) stg_128(gb + off + (long long)c * 16, Pack<T>::pack(o));
        }
      }
    }
    if (FUSED) {
#pragma unroll
      for (int r = 0; r < RPI; ++r) {
        if (wraw[r] == 0.f) continue;
        if (m[r] == 0) acc_text = fmaf(wraw[r], rowval[r], acc_text);
        else acc_vis = fmaf(wraw[r], rowval[r], acc_vis);
      }
    }
  }
  if (FUSED) {
    cta_sums_flush(sums, warp, lane, cur, acc_text, acc_vis);
    __syncthreads();
    cta_sums_store(sums, p.ws, p.n_layers, 0, kLdgThreads);
  }
}

// ---------------------------------------------------------------- generic fallback (any D, any alignment)
// Element-wise loads; used only when a row is not a whole number of aligned 16-byte chunks.
template <typename T, int LOSS, typename TT = T>
__global__ void __launch_bounds__(kLdgThreads) k_fwd_generic(const __grid_constant__ PathParams p) {
  __shared__ CtaSums<kLdgWarps> sums;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  cta_sums_zero(sums, p.n_layers);
  __syncthreads();
  pdl_launch_dependents();
  pdl_wait();
  const long long groups_per_layer = (p.n_rows + kLdgWarps - 1) / kLdgWarps;
  const long long total = groups_per_layer * p.n_layers;
  float acc_text = 0.f, acc_vis = 0.f;
  int cur = -1;
  for (long long g = blockIdx.x; g < total; g += gridDim.x) {
    const int l = (int)(g / groups_per_layer);
    const long long row = (g - (long long)l * groups_per_layer) * kLdgWarps + warp;
    if (l != cur) {
      cta_sums_flush(sums, warp, lane, cur, acc_text, acc_vis);
      acc_text = acc_vis = 0.f;
      cur = l;
    }
    if (row >= p.n_rows) continue;
    int m;
    const float w = row_weight(p, row, m);
    if (w == 0.f) continue;
    float x = 0.f, y = 0.f, z = 0.f;
    for (int d = lane; d < p.D; d += 32) {
      float a[1] = {Pack<T>::load1(p.s[l], row * p.row_stride + d)};
      float b[1] = {Pack<TT>::load1(p.t[l], row * p.row_stride + d)};
      accumulate<LOSS, 1>(a, b, x, y, z);
    }
    x = warp_sum(x); y = warp_sum(y); z = warp_sum(z);
    const float val = (lane == 0) ? row_value<LOSS>(x, y, z) : 0.f;
    if (m == 0) acc_text = fmaf(w, val, acc_text);
    else acc_vis = fmaf(w, val, acc_vis);
  }
  cta_sums_flush(sums, warp, lane, cur, acc_text, acc_vis);
  __syncthreads();
  cta_sums_store(sums, p.ws, p.n_layers, 0, kLdgThreads);
}

template <typename T, int LOSS, typename TT = T>
__global__ void __launch_bounds__(kLdgThreads) k_bwd_generic(const __grid_constant__ PathParams p, int use_fixed_gout) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long groups_per_layer = (p.n_rows + kLdgWarps - 1) / kLdgWarps;
  const long long total = groups_per_layer * p.n_layers;
  pdl_launch_dependents();
  pdl_wait();
  float gout;
  if (use_fixed_gout) gout = p.fixed_gout;
  else if (!upstream_grad<kBackward>(p, gout)) return;
  for (long long g = blockIdx.x; g < total; g += gridDim.x) {
    const int l = (int)(g / groups_per_layer);
    const long long row = (g - (long long)l * groups_per_layer) * kLdgWarps + warp;
    if (row >= p.n_rows || p.g[l] == nullptr) continue;
    int m;
    const float wraw = row_weight(p, row, m);
    const float w = wraw * (gout * __ldg(p.bwd_scale + 2 * l + m));
    float ch = 0.f, cp = 0.f;
    if (LOSS == MAFED_LOSS_COSINE && wraw != 0.f) {
      float x = 0.f, y = 0.f, z = 0.f;
      for (int d = lane; d < p.D; d += 32) {
        float a[1] = {Pack<T>::load1(p.s[l], row * p.row_stride + d)};
        float b[1] = {Pack<TT>::load1(p.t[l], row * p.row_stride + d)};
        accumulate<LOSS, 1>(a, b, x, y, z);
      }
      x = warp_sum(x); y = warp_sum(y); z = warp_sum(z);
      const float aa = y + kCosEps, den = sqrtf(aa * (z + kCosEps));
      ch = w * (x / den) / aa;
      cp = w / den;
    }
    for (int d = lane; d < p.D; d += 32) {
      float o[1] = {w};
      if (wraw != 0.f) {
        float a[1] = {Pack<T>::load1(p.s[l], row * p.row_stride + d)};
        float b[1] = {Pack<TT>::load1(p.t[l], row * p.row_stride + d)};
        grad_elems<LOSS, 1>(a, b, w, ch, cp, o);
      }
      Pack<T>::store1(p.g[l], row * p.row_stride + d, o[0]);
    }
  }
}

}  // namespace MAFED_NS
