// Generic (CUDA-core FFMA/DFMA) A-streaming passes.  Used for float64, for factor widths the tcgen05
// path does not cover, and for ragged/unaligned shards.  Two shapes:
//
//   row_pass : every thread owns RPT rows of the shard; the A tile is staged through padded shared
//              memory (coalesced 128-bit global loads, conflict-free 128-bit shared loads), the H tile
//              is staged transposed so one broadcast LDS.128 feeds VN FMAs per row.
//                 V = A H^T                     (dist_nmf.py:198, :730)
//                 V = (A / (W H + eps)) H^T     (dist_nmf.py:338-339, :806,:810)
//   col_pass : every thread owns CPT adjacent columns and streams rows with coalesced vector loads
//              straight from global memory; W rows are broadcast from shared memory.
//                 Y = W^T A                     (dist_nmf.py:166, :749)
//                 Y = W^T (A / (W H + eps))     (dist_nmf.py:312-313, :806,:808)
//
// Both split the reduced dimension over blockIdx.y into partial buffers that are summed in a fixed
// order by reduce_partials_kernel (deterministic).
#pragma once
#include <type_traits>

#include "common.cuh"

namespace dnmf {

template <typename T, int N>
struct alignas(sizeof(T) * N) Pack {
  T v[N];
};

template <typename T, int N>
__device__ __forceinline__ Pack<T, N> ldpack(const T* p) {
  return *reinterpret_cast<const Pack<T, N>*>(p);
}

constexpr int kRowPassThreads = 128;
constexpr int kRowPassBK = 32;

template <typename T, int KP, bool KL>
struct RowPassCfg {
  static constexpr int VN = 16 / sizeof(T);
  static constexpr int RPT = (sizeof(T) == 4) ? (KL ? (KP <= 16 ? 2 : 1) : (KP <= 32 ? 2 : 1)) : 1;
  static constexpr int BM = kRowPassThreads * RPT;
  static constexpr int AS = kRowPassBK + VN;  // padded strides (elements)
  static constexpr int HS = KP + VN;
  static constexpr size_t smem_bytes = sizeof(T) * ((size_t)BM * AS + (size_t)kRowPassBK * HS);
};

template <typename T, int KP, bool KL, typename TA = T>
__global__ void __launch_bounds__(kRowPassThreads)
row_pass_kernel(const TA* __restrict__ A, int64_t lda, const T* __restrict__ H, int64_t ldh,
                const T* __restrict__ W, int64_t ldw, T* __restrict__ out, int64_t ldo,
                int64_t split_stride, int64_t m, int64_t n, int k, int64_t chunk, T eps, int vec_ok) {
  using Cfg = RowPassCfg<T, KP, KL>;
  constexpr int NT = kRowPassThreads, VN = Cfg::VN, BK = kRowPassBK, RPT = Cfg::RPT, BM = Cfg::BM;
  constexpr int AS = Cfg::AS, HS = Cfg::HS;
  constexpr int HV = (KP < VN) ? KP : VN;  // vector width along kk
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* As = reinterpret_cast<T*>(smem_raw);
  T* Hs = As + (size_t)BM * AS;

  const int t = threadIdx.x;
  const int64_t row0 = (int64_t)blockIdx.x * BM;
  const int64_t c_begin = (int64_t)blockIdx.y * chunk;
  const int64_t c_end = (c_begin + chunk < n) ? (c_begin + chunk) : n;

  T acc[RPT][KP];
#pragma unroll
  for (int i = 0; i < RPT; ++i)
#pragma unroll
    for (int kk = 0; kk < KP; ++kk) acc[i][kk] = T(0);

  T w[RPT][KL ? KP : 1];
  if (KL) {
#pragma unroll
    for (int i = 0; i < RPT; ++i) {
      const int64_t row = row0 + t + i * NT;
#pragma unroll
      for (int kk = 0; kk < KP; ++kk) w[i][kk] = (row < m && kk < k) ? W[row * ldw + kk] : T(0);
    }
  }

  for (int64_t c0 = c_begin; c0 < c_end; c0 += BK) {
    // ---- stage the A tile [BM x BK] ----
    for (int v = t; v < BM * (BK / VN); v += NT) {
      const int r = v / (BK / VN);
      const int cv = (v % (BK / VN)) * VN;
      const int64_t row = row0 + r, col = c0 + cv;
      Pack<T, VN> p;
      if (row < m && vec_ok && col + VN <= c_end) {
        if constexpr (std::is_same<TA, T>::value) {
          p = ldpack<T, VN>(A + row * lda + col);
        } else {
          const Pack<TA, VN> pa = ldpack<TA, VN>(A + row * lda + col);
#pragma unroll
          for (int j = 0; j < VN; ++j) p.v[j] = static_cast<T>(pa.v[j]);
        }
      } else {
#pragma unroll
        for (int j = 0; j < VN; ++j) p.v[j] = (row < m && col + j < c_end) ? static_cast<T>(A[row * lda + col + j]) : T(0);
      }
      *reinterpret_cast<Pack<T, VN>*>(As + r * AS + cv) = p;
    }
    // ---- stage the H tile transposed: Hs[c][kk] ----
    for (int idx = t; idx < KP * BK; idx += NT) {
      const int kk = idx / BK, c = idx % BK;
      const int64_t col = c0 + c;
      Hs[c * HS + kk] = (kk < k && col < c_end) ? H[(int64_t)kk * ldh + col] : T(0);
    }
    __syncthreads();

#pragma unroll 2
    for (int c = 0; c < BK; c += VN) {
      Pack<T, VN> a[RPT];
#pragma unroll
      for (int i = 0; i < RPT; ++i) a[i] = *reinterpret_cast<const Pack<T, VN>*>(As + (t + i * NT) * AS + c);
#pragma unroll
      for (int cc = 0; cc < VN; ++cc) {
        const T* hrow = Hs + (c + cc) * HS;
        if (!KL) {
#pragma unroll
          for (int kk = 0; kk < KP; kk += HV) {
            Pack<T, HV> h = *reinterpret_cast<const Pack<T, HV>*>(hrow + kk);
#pragma unroll
            for (int j = 0; j < HV; ++j)
#pragma unroll
              for (int i = 0; i < RPT; ++i) acc[i][kk + j] = fma(a[i].v[cc], h.v[j], acc[i][kk + j]);
          }
        } else {
          T s[RPT];
#pragma unroll
          for (int i = 0; i < RPT; ++i) s[i] = T(0);
#pragma unroll
          for (int kk = 0; kk < KP; kk += HV) {
            Pack<T, HV> h = *reinterpret_cast<const Pack<T, HV>*>(hrow + kk);
#pragma unroll
            for (int j = 0; j < HV; ++j)
#pragma unroll
              for (int i = 0; i < RPT; ++i) s[i] = fma(w[i][kk + j], h.v[j], s[i]);
          }
          T u[RPT];
#pragma unroll
          for (int i = 0; i < RPT; ++i) u[i] = a[i].v[cc] / (s[i] + eps);
#pragma unroll
          for (int kk = 0; kk < KP; kk += HV) {
            Pack<T, HV> h = *reinterpret_cast<const Pack<T, HV>*>(hrow + kk);
#pragma unroll
            for (int j = 0; j < HV; ++j)
#pragma unroll
              for (int i = 0; i < RPT; ++i) acc[i][kk + j] = fma(u[i], h.v[j], acc[i][kk + j]);
          }
        }
      }
    }
    __syncthreads();
  }

  T* o = out + (int64_t)blockIdx.y * split_stride;
#pragma unroll
  for (int i = 0; i < RPT; ++i) {
    const int64_t row = row0 + t + i * NT;
    if (row < m) {
#pragma unroll
      for (int kk = 0; kk < KP; ++kk)
        if (kk < k) o[row * ldo + kk] = acc[i][kk];
    }
  }
}

constexpr int kColPassThreads = 128;
constexpr int kColPassBR = 64;

template <typename T, int KP, bool KL>
struct ColPassCfg {
  // accumulators (+ the H columns for KL) are register resident: keep KP*CPT*(KL?2:1)*sizeof(T)/4 <= 128 regs
  static constexpr int budget = (sizeof(T) == 4 ? 128 : 64) / (KL ? 2 : 1);
  static constexpr int raw = budget / KP;
  static constexpr int vmax = 16 / sizeof(T);
  static constexpr int CPT = raw >= vmax ? vmax : (raw >= 2 ? 2 : 1);
};

template <typename T, int KP, bool KL, typename TA = T>
__global__ void __launch_bounds__(kColPassThreads)
col_pass_kernel(const TA* __restrict__ A, int64_t lda, const T* __restrict__ W, int64_t ldw,
                const T* __restrict__ H, int64_t ldh, T* __restrict__ out, int64_t ldo,
                int64_t split_stride, int64_t m, int64_t n, int k, int64_t chunk, T eps, int vec_ok) {
  constexpr int NT = kColPassThreads, BR = kColPassBR, RB = 4;
  constexpr int CPT = ColPassCfg<T, KP, KL>::CPT;
  constexpr int VN = 16 / sizeof(T);
  constexpr int WV = (KP < VN) ? KP : VN;
  __shared__ __align__(16) T Ws[BR][KP];

  const int t = threadIdx.x;
  const int64_t col0 = ((int64_t)blockIdx.x * NT + t) * CPT;
  const int64_t r_begin = (int64_t)blockIdx.y * chunk;
  const int64_t r_end = (r_begin + chunk < m) ? (r_begin + chunk) : m;
  const bool full = vec_ok && (col0 + CPT <= n);

  T acc[KP][CPT];
#pragma unroll
  for (int kk = 0; kk < KP; ++kk)
#pragma unroll
    for (int cc = 0; cc < CPT; ++cc) acc[kk][cc] = T(0);

  T h[KL ? KP : 1][CPT];
  if (KL) {
#pragma unroll
    for (int kk = 0; kk < KP; ++kk)
#pragma unroll
      for (int cc = 0; cc < CPT; ++cc)
        h[kk][cc] = (kk < k && col0 + cc < n) ? H[(int64_t)kk * ldh + col0 + cc] : T(0);
  }

  for (int64_t r0 = r_begin; r0 < r_end; r0 += BR) {
    __syncthreads();
    for (int idx = t; idx < BR * KP; idx += NT) {
      const int r = idx / KP, kk = idx % KP;
      const int64_t row = r0 + r;
      Ws[r][kk] = (row < r_end && kk < k) ? W[row * ldw + kk] : T(0);
    }
    __syncthreads();
    const int rows_here = (r_end - r0 < BR) ? (int)(r_end - r0) : BR;
    for (int r = 0; r < rows_here; r += RB) {
      Pack<T, CPT> a[RB];
#pragma unroll
      for (int q = 0; q < RB; ++q) {
        const int64_t row = r0 + r + q;
        if (row < r_end && full) {
          if constexpr (std::is_same<TA, T>::value) {
            a[q] = ldpack<T, CPT>(A + row * lda + col0);
          } else {
            const Pack<TA, CPT> pa = ldpack<TA, CPT>(A + row * lda + col0);
#pragma unroll
            for (int cc = 0; cc < CPT; ++cc) a[q].v[cc] = static_cast<T>(pa.v[cc]);
          }
        } else {
#pragma unroll
          for (int cc = 0; cc < CPT; ++cc)
            a[q].v[cc] = (row < r_end && col0 + cc < n) ? static_cast<T>(A[row * lda + col0 + cc]) : T(0);
        }
      }
#pragma unroll
      for (int q = 0; q < RB; ++q) {
        const T* wrow = &Ws[r + q][0];  // r + q < BR: BR % RB == 0 and r is a multiple of RB
        if (!KL) {
#pragma unroll
          for (int kk = 0; kk < KP; kk += WV) {
            Pack<T, WV> wv = *reinterpret_cast<const Pack<T, WV>*>(wrow + kk);
#pragma unroll
            for (int j = 0; j < WV; ++j)
#pragma unroll
              for (int cc = 0; cc < CPT; ++cc) acc[kk + j][cc] = fma(wv.v[j], a[q].v[cc], acc[kk + j][cc]);
          }
        } else {
          T s[CPT];
#pragma unroll
          for (int cc = 0; cc < CPT; ++cc) s[cc] = T(0);
#pragma unroll
          for (int kk = 0; kk < KP; kk += WV) {
            Pack<T, WV> wv = *reinterpret_cast<const Pack<T, WV>*>(wrow + kk);
#pragma unroll
            for (int j = 0; j < WV; ++j)
#pragma unroll
              for (int cc = 0; cc < CPT; ++cc) s[cc] = fma(wv.v[j], h[kk + j][cc], s[cc]);
          }
          T u[CPT];
#pragma unroll
          for (int cc = 0; cc < CPT; ++cc) u[cc] = a[q].v[cc] / (s[cc] + eps);
#pragma unroll
          for (int kk = 0; kk < KP; kk += WV) {
            Pack<T, WV> wv = *reinterpret_cast<const Pack<T, WV>*>(wrow + kk);
#pragma unroll
            for (int j = 0; j < WV; ++j)
#pragma unroll
              for (int cc = 0; cc < CPT; ++cc) acc[kk + j][cc] = fma(wv.v[j], u[cc], acc[kk + j][cc]);
          }
        }
      }
    }
  }

  T* o = out + (int64_t)blockIdx.y * split_stride;
#pragma unroll
  for (int kk = 0; kk < KP; ++kk) {
    if (kk < k) {
#pragma unroll
      for (int cc = 0; cc < CPT; ++cc)
        if (col0 + cc < n) o[(int64_t)kk * ldo + col0 + cc] = acc[kk][cc];
    }
  }
}

// out[r*so_r + c*so_c] = sum_{s < splits, in order} P[s*split_stride + r*ldp + c]   (ldp >= C: padded partial rows)
template <typename T>
__global__ void __launch_bounds__(256)
reduce_partials_kernel(const T* __restrict__ P, int64_t split_stride, int splits, int64_t R, int64_t C,
                       T* __restrict__ out, int64_t so_r, int64_t so_c, int64_t ldp) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= R * C) return;
  const int64_t r = idx / C, c = idx % C;
  const int64_t src = r * ldp + c;
  T acc = P[src];
  for (int s = 1; s < splits; ++s) acc += P[(int64_t)s * split_stride + src];
  out[r * so_r + c * so_c] = acc;
}

}  // namespace dnmf
