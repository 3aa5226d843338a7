// Factor-sized kernels: Gram products, multiplicative updates, HALS sweeps, BCD steps, norms, shard ops.
// All are negligible next to the A-streaming passes (factor traffic < 0.2 % of an iteration).
#pragma once
#include "common.cuh"
#include "generic_passes.cuh"

namespace dnmf {

// ---------------------------------------------------------------------------------------------
// Gram: partial[b][i*KP+j] = sum_{r in block b} X(r,i) X(r,j);  X(r,kk) = TRANS ? X[kk*ldx+r] : X[r*ldx+kk]
// ---------------------------------------------------------------------------------------------
constexpr int kGramThreads = 256;
constexpr int kGramTR = 32;

template <typename T, int KP, bool TRANS>
__global__ void __launch_bounds__(kGramThreads)
gram_partial_kernel(const T* __restrict__ X, int64_t ldx, int64_t rows, int k, int64_t rows_per_block,
                    T* __restrict__ P) {
  constexpr int NT = kGramThreads, TR = kGramTR;
  constexpr int NO = (KP * KP + NT - 1) / NT;
  __shared__ T Xs[TR][KP + 1];
  const int t = threadIdx.x;
  const int64_t r_begin = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r_end = (r_begin + rows_per_block < rows) ? (r_begin + rows_per_block) : rows;
  T acc[NO];
#pragma unroll
  for (int o = 0; o < NO; ++o) acc[o] = T(0);
  for (int64_t r0 = r_begin; r0 < r_end; r0 += TR) {
    __syncthreads();
    for (int idx = t; idx < TR * KP; idx += NT) {
      int r, kk;
      if (TRANS) { kk = idx / TR; r = idx % TR; } else { r = idx / KP; kk = idx % KP; }
      const int64_t row = r0 + r;
      T v = T(0);
      if (row < r_end && kk < k) v = TRANS ? X[(int64_t)kk * ldx + row] : X[row * ldx + kk];
      Xs[r][kk] = v;
    }
    __syncthreads();
    if (NT % KP == 0) {
      // every output of this thread has the same column j = t % KP (KP divides the block size): load Xs[r][j] once
      // per r and reuse it for the thread's NO outputs (same summation order per output: r ascending)
      const int j = t % KP, i0 = t / KP;
#pragma unroll 8
      for (int r = 0; r < TR; ++r) {
        const T xj = Xs[r][j];
#pragma unroll
        for (int o = 0; o < NO; ++o) {
          const int i = i0 + o * (NT / KP);
          if (i < KP) acc[o] = fma(Xs[r][i], xj, acc[o]);
        }
      }
    } else {
#pragma unroll
      for (int o = 0; o < NO; ++o) {
        const int e = t + o * NT;
        if (e < KP * KP) {
          const int i = e / KP, j = e % KP;
          T a = acc[o];
#pragma unroll 8
          for (int r = 0; r < TR; ++r) a = fma(Xs[r][i], Xs[r][j], a);
          acc[o] = a;
        }
      }
    }
  }
#pragma unroll
  for (int o = 0; o < NO; ++o) {
    const int e = t + o * NT;
    if (e < KP * KP) P[(int64_t)blockIdx.x * (KP * KP) + e] = acc[o];
  }
}

// one warp per output element: lanes stride over the block partials, then a fixed-order shuffle tree (deterministic)
template <typename T>
__global__ void __launch_bounds__(256) gram_reduce_kernel(const T* __restrict__ P, int nblocks, int KP, int k, T* __restrict__ G) {
  const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (e >= k * k) return;
  const int i = e / k, j = e % k;
  T acc = T(0);
  for (int b = lane; b < nblocks; b += 32) acc += P[(int64_t)b * KP * KP + i * KP + j];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) G[e] = acc;
}

// ---------------------------------------------------------------------------------------------
// row-factor updates: out(r,j) = f(X(r,:), G, V(r,j))   MODE 0: MU   W *= V / (W G + eps)
//                                                        MODE 1: BCD  W = max(0, Wm - (Wm G - V)/L)
// ---------------------------------------------------------------------------------------------
constexpr int kRowUpdThreads = 256;
template <typename T, int KP>
struct RowUpdCfg {
  static constexpr int raw = 8192 / (KP * (int)sizeof(T));
  static constexpr int RB = raw > 64 ? 64 : (raw < 16 ? 16 : raw);   // rows per block (static smem <= 48 KB)
};

// Operand given as `splits` partial buffers `sstride` elements apart (the split-K partials an A-streaming pass leaves in
// its workspace): the value is their sum in split order -- the order reduce_partials_kernel uses, so an update that reads
// the partials directly is bit-identical to pass + reduction + update.  splits == 1: a plain operand.
template <typename T>
__device__ __forceinline__ T sum_splits(const T* __restrict__ p, int splits, int64_t sstride) {
  T acc = p[0];
  for (int s = 1; s < splits; ++s) acc += p[(int64_t)s * sstride];
  return acc;
}

template <typename T, int KP, int MODE>
__global__ void __launch_bounds__(kRowUpdThreads)
row_update_kernel(T* __restrict__ W, int64_t ldw, const T* __restrict__ X, int64_t ldx,
                  const T* __restrict__ V, int64_t ldv, const T* __restrict__ G, int64_t m, int k, T p0,
                  const double* __restrict__ p0_dev, int splits, int64_t sstride) {
  // p0_dev != nullptr: the scalar (BCD's Lipschitz bound) lives on the device (no host round trip, graph-capturable)
  if (p0_dev != nullptr) p0 = (T)p0_dev[0];
  constexpr int NT = kRowUpdThreads, RB = RowUpdCfg<T, KP>::RB;
  __shared__ T Gs[KP][KP + 1];
  __shared__ T Xs[RB][KP + 1];
  const int t = threadIdx.x;
  const int64_t row0 = (int64_t)blockIdx.x * RB;
  for (int idx = t; idx < KP * KP; idx += NT) {
    const int l = idx / KP, j = idx % KP;
    Gs[l][j] = (l < k && j < k) ? G[l * k + j] : T(0);
  }
  for (int idx = t; idx < RB * KP; idx += NT) {
    const int r = idx / KP, j = idx % KP;
    const int64_t row = row0 + r;
    Xs[r][j] = (row < m && j < k) ? X[row * ldx + j] : T(0);
  }
  __syncthreads();
  for (int idx = t; idx < RB * KP; idx += NT) {
    const int r = idx / KP, j = idx % KP;
    const int64_t row = row0 + r;
    if (row < m && j < k) {
      T d = T(0);
#pragma unroll
      for (int l = 0; l < KP; ++l) d = fma(Xs[r][l], Gs[l][j], d);
      const T v = sum_splits(V + row * ldv + j, splits, sstride);
      T res;
      if (MODE == 0) {
        res = Xs[r][j] * (v / (d + p0));          // p0 = eps
      } else {
        res = Xs[r][j] - (d - v) / p0;            // p0 = Lipschitz bound
        res = res > T(0) ? res : T(0);
      }
      W[row * ldw + j] = res;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// column-factor updates, one thread per column c, the k values of the column live in registers
//   MODE 0: MU   H(kk,c) *= Y(kk,c) / (sum_l H(l,c) G(l,kk) + eps)     [optional clamp to eps]
//   MODE 1: BCD  H(kk,c) = max(0, Hm(kk,c) - (sum_l G(kk,l) Hm(l,c) - Y(kk,c)) / L)
//   MODE 2: HALS for kk in order: H(kk,c) = max(H(kk,c) + Y(kk,c) - sum_l G(kk,l) H(l,c), eps)  (Gauss-Seidel)
// ---------------------------------------------------------------------------------------------
constexpr int kColUpdThreads = 128;

template <typename T, int KP, int MODE>
__global__ void __launch_bounds__(kColUpdThreads)
col_update_kernel(T* __restrict__ H, int64_t ldh, const T* __restrict__ X, int64_t ldx,
                  const T* __restrict__ Y, int64_t ysk, int64_t ysc, const T* __restrict__ G,
                  int k, int64_t n, T p0, int clamp, const double* __restrict__ p0_dev, int splits, int64_t sstride) {
  if (p0_dev != nullptr) p0 = (T)p0_dev[0];
  __shared__ T Gs[KP * KP];
  const int t = threadIdx.x;
  for (int idx = t; idx < KP * KP; idx += kColUpdThreads) {
    const int l = idx / KP, j = idx % KP;
    Gs[idx] = (l < k && j < k) ? G[l * k + j] : T(0);
  }
  __syncthreads();
  // Y given column-major per column (ysk == 1: the [x][ldp] layout of the split-K partials): a thread would read its
  // column as KP consecutive elements, 128 bytes apart from its neighbour's -- stage the block's columns through shared
  // memory with coalesced loads instead (and add the splits there).
  constexpr bool kStage = sizeof(T) * ((KP + 1) * kColUpdThreads + KP * KP) <= 46 * 1024;    // next to Gs in 48 KB
  __shared__ T Ys[kStage ? kColUpdThreads * (KP + 1) : 1];
  const bool staged = kStage && ysk == 1;
  if (staged) {
    const int64_t c0 = (int64_t)blockIdx.x * kColUpdThreads;
    for (int e = t; e < kColUpdThreads * KP; e += kColUpdThreads) {
      const int col = e / KP, kk = e % KP;
      T v = T(0);
      if (c0 + col < n && kk < k) v = sum_splits(Y + (c0 + col) * ysc + kk, splits, sstride);
      Ys[col * (KP + 1) + kk] = v;
    }
    __syncthreads();
  }
  const int64_t c = (int64_t)blockIdx.x * kColUpdThreads + t;
  if (c >= n) return;
  T h[KP];
#pragma unroll
  for (int l = 0; l < KP; ++l) h[l] = (l < k) ? X[(int64_t)l * ldx + c] : T(0);
  if (MODE == 2) {
#pragma unroll
    for (int kk = 0; kk < KP; ++kk) {
      if (kk < k) {
        T d = T(0);
#pragma unroll
        for (int l = 0; l < KP; ++l) d = fma(Gs[kk * KP + l], h[l], d);
        T v = h[kk] + (staged ? Ys[t * (KP + 1) + kk] : sum_splits(Y + (int64_t)kk * ysk + c * ysc, splits, sstride)) - d;
        h[kk] = v > p0 ? v : p0;
      }
    }
#pragma unroll
    for (int kk = 0; kk < KP; ++kk)
      if (kk < k) H[(int64_t)kk * ldh + c] = h[kk];
  } else {
#pragma unroll
    for (int kk = 0; kk < KP; ++kk) {
      if (kk < k) {
        T d = T(0);
        T res;
        const T y = staged ? Ys[t * (KP + 1) + kk] : sum_splits(Y + (int64_t)kk * ysk + c * ysc, splits, sstride);
        if (MODE == 0) {
#pragma unroll
          for (int l = 0; l < KP; ++l) d = fma(h[l], Gs[l * KP + kk], d);
          res = h[kk] * (y / (d + p0));
          if (clamp) res = res > p0 ? res : p0;
        } else {
#pragma unroll
          for (int l = 0; l < KP; ++l) d = fma(Gs[kk * KP + l], h[l], d);
          res = h[kk] - (d - y) / p0;
          res = res > T(0) ? res : T(0);
        }
        H[(int64_t)kk * ldh + c] = res;
      }
    }
  }
}

// W(r,j) *= V(r,j) / (x[j] + eps)      (KL, W side)
template <typename T>
__global__ void kl_update_w_kernel(T* __restrict__ W, int64_t ldw, const T* __restrict__ V, int64_t ldv,
                                   const T* __restrict__ x, int64_t m, int k, T eps, int splits, int64_t sstride) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= m * k) return;
  const int64_t r = idx / k;
  const int j = (int)(idx % k);
  W[r * ldw + j] *= sum_splits(V + r * ldv + j, splits, sstride) / (x[j] + eps);
}

// H(kk,c) *= Y(kk,c) / (x[kk] + eps)   (KL, H side; optional clamp)
template <typename T>
__global__ void kl_update_h_kernel(T* __restrict__ H, int64_t ldh, const T* __restrict__ Y, int64_t ysk,
                                   int64_t ysc, const T* __restrict__ x, int k, int64_t n, T eps, int clamp, int splits,
                                   int64_t sstride) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)k * n) return;
  const int kk = (int)(idx / n);
  const int64_t c = idx % n;
  T v = H[(int64_t)kk * ldh + c] * (sum_splits(Y + (int64_t)kk * ysk + c * ysc, splits, sstride) / (x[kk] + eps));
  if (clamp) v = v > eps ? v : eps;
  H[(int64_t)kk * ldh + c] = v;
}

// The same update with Y given as split-K partials in the [column][ldp] layout: a block stages 64 columns through shared
// memory (coalesced loads along the factor index, splits added in order) and then updates H with the column index fastest.
template <typename T>
__global__ void __launch_bounds__(256)
kl_update_h_staged_kernel(T* __restrict__ H, int64_t ldh, const T* __restrict__ Yp, int64_t ldp, const T* __restrict__ x,
                          int k, int64_t n, T eps, int clamp, int splits, int64_t sstride) {
  constexpr int CB = 64;
  __shared__ T Ys[CB][DNMF_MAX_K + 1];
  const int64_t c0 = (int64_t)blockIdx.x * CB;
  for (int e = threadIdx.x; e < CB * k; e += 256) {
    const int col = e / k, kk = e % k;
    Ys[col][kk] = (c0 + col < n) ? sum_splits(Yp + (c0 + col) * ldp + kk, splits, sstride) : T(0);
  }
  __syncthreads();
  for (int e = threadIdx.x; e < CB * k; e += 256) {
    const int kk = e / CB, col = e % CB;
    const int64_t c = c0 + col;
    if (c < n) {
      T v = H[(int64_t)kk * ldh + c] * (Ys[col][kk] / (x[kk] + eps));
      if (clamp) v = v > eps ? v : eps;
      H[(int64_t)kk * ldh + c] = v;
    }
  }
}

template <typename T>
__global__ void clamp_min_kernel(T* __restrict__ X, int64_t ldx, int64_t rows, int64_t cols, T lo) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * cols) return;
  T* p = X + (idx / cols) * ldx + (idx % cols);
  const T v = *p;
  *p = v > lo ? v : lo;     // np.maximum(X, lo)
}

// ---------------------------------------------------------------------------------------------
// sums (double accumulation, two deterministic stages)
// ---------------------------------------------------------------------------------------------
// colsum partial: grid (ceil(cols/32), nchunks), block (32, 8): P[chunk][col]
template <typename T>
__global__ void __launch_bounds__(256)
colsum_partial_kernel(const T* __restrict__ X, int64_t ldx, int64_t rows, int64_t cols, int64_t rows_per_chunk,
                      double* __restrict__ P, int sq) {
  __shared__ double red[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int64_t c = (int64_t)blockIdx.x * 32 + tx;
  const int64_t r_begin = (int64_t)blockIdx.y * rows_per_chunk;
  const int64_t r_end = (r_begin + rows_per_chunk < rows) ? (r_begin + rows_per_chunk) : rows;
  double acc = 0.0;
  if (c < cols)
    for (int64_t r = r_begin + ty; r < r_end; r += 8) {
      const double v = (double)X[r * ldx + c];
      acc += sq ? v * v : v;
    }
  red[ty][tx] = acc;
  __syncthreads();
  if (ty == 0 && c < cols) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += red[i][tx];
    P[(int64_t)blockIdx.y * cols + c] = s;
  }
}

// out[c] = (T) sum_chunks P[chunk][c]; one warp per output, fixed-order shuffle tree
template <typename TO>
__global__ void __launch_bounds__(256) sum_partials_kernel(const double* __restrict__ P, int nparts, int64_t count, TO* __restrict__ out) {
  const int64_t idx = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (idx >= count) return;
  double s = 0.0;
  for (int p = lane; p < nparts; p += 32) s += P[(int64_t)p * count + idx];
  s = warp_sum(s);
  if (lane == 0) out[idx] = (TO)s;
}

// rowsum partial: grid (rows, nchunks), block 256: P[chunk][row]   (sq: sum of squares)
template <typename T>
__global__ void __launch_bounds__(256)
rowsum_partial_kernel(const T* __restrict__ X, int64_t ldx, int64_t rows, int64_t cols, int64_t cols_per_chunk,
                      double* __restrict__ P, int sq) {
  __shared__ double red[8];
  const int64_t r = blockIdx.x;
  const int64_t c_begin = (int64_t)blockIdx.y * cols_per_chunk;
  const int64_t c_end = (c_begin + cols_per_chunk < cols) ? (c_begin + cols_per_chunk) : cols;
  double acc = 0.0;
  for (int64_t c = c_begin + threadIdx.x; c < c_end; c += 256) {
    const double v = to_f64(X[r * ldx + c]);
    acc += sq ? v * v : v;
  }
  const double s = block_sum<256>(acc, red);
  if (threadIdx.x == 0) P[(int64_t)blockIdx.y * rows + r] = s;
}

// inner product of two [rows x cols] matrices, stage 1: block b sums the flat elements [b * per_block, (b + 1) * per_block)
// in a fixed order into P[b] (float64)
template <typename T>
__global__ void __launch_bounds__(256)
dot_partial_kernel(const T* __restrict__ X, int64_t ldx, const T* __restrict__ Y, int64_t ldy, int64_t rows, int cols,
                   int64_t per_block, double* __restrict__ P) {
  __shared__ double red[8];
  const int64_t total = rows * cols;
  const int64_t begin = (int64_t)blockIdx.x * per_block;
  const int64_t end = (begin + per_block < total) ? (begin + per_block) : total;
  double acc = 0.0;
  for (int64_t i = begin + threadIdx.x; i < end; i += 256) {
    const int64_t r = i / cols;
    const int c = (int)(i - r * cols);
    acc += (double)X[r * ldx + c] * (double)Y[r * ldy + c];
  }
  const double s = block_sum<256>(acc, red);
  if (threadIdx.x == 0) P[blockIdx.x] = s;
}

// stage 2 of dnmf_trace_terms: out[2 * slot] = sum P[0, n0), out[2 * slot + 1] = sum P[n0, n0 + n1), slot read from (and
// then advanced in) device memory so that a CUDA-graph replay of the step appends to a history instead of overwriting it
static __global__ void __launch_bounds__(256) trace_store_kernel(const double* __restrict__ P, int64_t n0, int64_t n1,
                                                                 double* __restrict__ out, int64_t* __restrict__ slot_counter,
                                                                 int64_t max_slots) {
  __shared__ double red[8];
  double a0 = 0.0, a1 = 0.0;
  for (int64_t i = threadIdx.x; i < n0; i += 256) a0 += P[i];
  for (int64_t i = threadIdx.x; i < n1; i += 256) a1 += P[n0 + i];
  const double s0 = block_sum<256>(a0, red);
  const double s1 = block_sum<256>(a1, red);
  if (threadIdx.x == 0) {
    int64_t slot = 0;
    if (slot_counter != nullptr) {
      slot = *slot_counter;
      *slot_counter = slot + 1;
      if (slot >= max_slots) return;          // history full: keep counting, drop the sample
    }
    out[2 * slot] = s0;
    out[2 * slot + 1] = s1;
  }
}

// final scalar: out[0] = sum_i P[i]  (single block, fixed order)
static __global__ void __launch_bounds__(256) sum_all_kernel(const double* __restrict__ P, int64_t count, double* out) {
  __shared__ double red[8];
  double acc = 0.0;
  for (int64_t i = threadIdx.x; i < count; i += 256) acc += P[i];
  const double s = block_sum<256>(acc, red);
  if (threadIdx.x == 0) out[0] = s;
}

// out[0] = sum_i P[2i], out[1] = sum_i P[2i+1]
static __global__ void __launch_bounds__(256) sum_pairs_kernel(const double* __restrict__ P, int64_t count, double* out) {
  __shared__ double red[8];
  double a0 = 0.0, a1 = 0.0;
  for (int64_t i = threadIdx.x; i < count; i += 256) { a0 += P[2 * i]; a1 += P[2 * i + 1]; }
  const double s0 = block_sum<256>(a0, red);
  const double s1 = block_sum<256>(a1, red);
  if (threadIdx.x == 0) { out[0] = s0; out[1] = s1; }
}

// W(r,j) /= (s[j] + eps)
template <typename T>
__global__ void normalize_w_kernel(T* __restrict__ W, int64_t ldw, int64_t m, int k, const T* __restrict__ s, T eps) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= m * k) return;
  const int64_t r = idx / k;
  const int j = (int)(idx % k);
  W[r * ldw + j] /= (s[j] + eps);
}

// H(j,c) *= s[j]
template <typename T>
__global__ void scale_rows_kernel(T* __restrict__ H, int64_t ldh, int k, int64_t n, const T* __restrict__ s) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)k * n) return;
  const int j = (int)(idx / n);
  const int64_t c = idx % n;
  H[(int64_t)j * ldh + c] *= s[j];
}

// W(r,j) /= s[j]
template <typename T>
__global__ void div_cols_kernel(T* __restrict__ W, int64_t ldw, int64_t m, int k, const T* __restrict__ s) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= m * k) return;
  const int64_t r = idx / k;
  const int j = (int)(idx % k);
  W[r * ldw + j] /= s[j];
}

template <typename T>
__global__ void axpby_kernel(T* __restrict__ out, const T* __restrict__ x, const T* __restrict__ y, T a, T b,
                             int64_t count) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= count) return;
  out[idx] = a * x[idx] + b * y[idx];
}

// ---------------------------------------------------------------------------------------------
// residual: per block partial (||A - W H||^2, ||A||^2) over a [row chunk] x [column block]
// column-owner layout as col_pass (coalesced A, W rows broadcast from shared memory)
// ---------------------------------------------------------------------------------------------
template <typename T, int KP, typename TA = T>
__global__ void __launch_bounds__(kColPassThreads)
residual_kernel(const TA* __restrict__ A, int64_t lda, const T* __restrict__ W, int64_t ldw,
                const T* __restrict__ H, int64_t ldh, int64_t m, int64_t n, int k, int64_t chunk,
                double* __restrict__ P, double* __restrict__ col_num, double* __restrict__ col_den) {
  constexpr int NT = kColPassThreads, BR = kColPassBR;
  __shared__ __align__(16) T Ws[BR][KP];
  __shared__ double red[NT / 32];
  const int t = threadIdx.x;
  const int64_t c = (int64_t)blockIdx.x * NT + t;
  const int64_t r_begin = (int64_t)blockIdx.y * chunk;
  const int64_t r_end = (r_begin + chunk < m) ? (r_begin + chunk) : m;
  T h[KP];
#pragma unroll
  for (int kk = 0; kk < KP; ++kk) h[kk] = (kk < k && c < n) ? H[(int64_t)kk * ldh + c] : T(0);
  double e2 = 0.0, a2 = 0.0;
  for (int64_t r0 = r_begin; r0 < r_end; r0 += BR) {
    __syncthreads();
    for (int idx = t; idx < BR * KP; idx += NT) {
      const int r = idx / KP, kk = idx % KP;
      const int64_t row = r0 + r;
      Ws[r][kk] = (row < r_end && kk < k) ? W[row * ldw + kk] : T(0);
    }
    __syncthreads();
    const int rows_here = (r_end - r0 < BR) ? (int)(r_end - r0) : BR;
    if (c < n) {
      for (int r = 0; r < rows_here; ++r) {
        const T a = static_cast<T>(A[(r0 + r) * lda + c]);
        T s = T(0);
#pragma unroll
        for (int kk = 0; kk < KP; ++kk) s = fma(Ws[r][kk], h[kk], s);
        const T d = a - s;
        e2 += (double)d * (double)d;
        a2 += (double)a * (double)a;
      }
    }
  }
  if (col_num != nullptr) {   // per-column mode (single row chunk): pyDNMF.py:231-233
    if (c < n) { col_num[c] = e2; col_den[c] = a2; }
    return;
  }
  const double s0 = block_sum<NT>(e2, red);
  const double s1 = block_sum<NT>(a2, red);
  if (t == 0) {
    const int64_t b = (int64_t)blockIdx.y * gridDim.x + blockIdx.x;
    P[2 * b] = s0;
    P[2 * b + 1] = s1;
  }
}

// ---------------------------------------------------------------------------------------------
// HALS W sweep, one column:  t = W(r,kk) G(kk,kk) + V(r,kk) - sum_l W(r,l) G(l,kk); W(r,kk) = max(t, eps)
// block partial of sum W(r,kk)^2 -> P[block]
// ---------------------------------------------------------------------------------------------
template <typename T, int KP>
__global__ void __launch_bounds__(256)
hals_w_col_kernel(T* __restrict__ W, int64_t ldw, const T* __restrict__ V, int64_t ldv,
                  const T* __restrict__ G, int64_t m, int k, int kk, T eps, double* __restrict__ P) {
  __shared__ T g[KP];
  __shared__ double red[8];
  if (threadIdx.x < KP) g[threadIdx.x] = (threadIdx.x < k) ? G[threadIdx.x * k + kk] : T(0);
  __syncthreads();
  const int64_t r = (int64_t)blockIdx.x * 256 + threadIdx.x;
  double sq = 0.0;
  if (r < m) {
    T* w = W + r * ldw;
    T d = T(0);
#pragma unroll
    for (int l = 0; l < KP; ++l)
      if (l < k) d = fma(w[l], g[l], d);
    T v = w[kk] * g[kk] + V[r * ldv + kk] - d;
    v = v > eps ? v : eps;
    w[kk] = v;
    sq = (double)v * (double)v;
  }
  const double s = block_sum<256>(sq, red);
  if (threadIdx.x == 0) P[blockIdx.x] = s;
}

// W(:,kk) /= sqrt(ss_sq[0]) when it is > 0        (dist_nmf.py:431-432)
template <typename T>
__global__ void div_col_kernel(T* __restrict__ W, int64_t ldw, int64_t m, int kk, const double* __restrict__ ss_sq) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= m) return;
  const T ss = (T)sqrt(ss_sq[0]);
  if (ss > T(0)) W[r * ldw + kk] /= ss;
}

// ---------------------------------------------------------------------------------------------
// shard ops
// ---------------------------------------------------------------------------------------------
// one warp per row: row_nnz[i] = #(A[i,:] != 0)
template <typename T>
__global__ void __launch_bounds__(256)
row_nnz_kernel(const T* __restrict__ A, int64_t lda, int64_t m, int64_t n, long long* __restrict__ row_nnz) {
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= m) return;
  const int lane = threadIdx.x & 31;
  long long cnt = 0;
  for (int64_t c = lane; c < n; c += 32) cnt += (A[row * lda + c] != T(0)) ? 1 : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if (lane == 0) row_nnz[row] = cnt;
}

// one thread per column over a row chunk; integer atomics (exact, order independent)
template <typename T>
__global__ void __launch_bounds__(256)
col_nnz_kernel(const T* __restrict__ A, int64_t lda, int64_t m, int64_t n, int64_t chunk,
               unsigned long long* __restrict__ col_nnz) {
  const int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (c >= n) return;
  const int64_t r_begin = (int64_t)blockIdx.y * chunk;
  const int64_t r_end = (r_begin + chunk < m) ? (r_begin + chunk) : m;
  unsigned long long cnt = 0;
  for (int64_t r = r_begin; r < r_end; ++r) cnt += (A[r * lda + c] != T(0)) ? 1ull : 0ull;
  if (cnt) atomicAdd(col_nnz + c, cnt);
}

template <typename T>
__global__ void compact_kernel(const T* __restrict__ A, int64_t lda, const long long* __restrict__ row_idx,
                               int64_t mr, const long long* __restrict__ col_idx, int64_t nc,
                               T* __restrict__ out, int64_t ldo) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= mr * nc) return;
  const int64_t i = idx / nc, j = idx % nc;
  out[i * ldo + j] = A[row_idx[i] * lda + col_idx[j]];
}

// out[row_idx[i]][j] = (double) X[i][j]   (ROWS) ; out[i][col_idx[j]] = (double) X[i][j]  (!ROWS)
template <typename T, bool ROWS>
__global__ void scatter_kernel(const T* __restrict__ X, int64_t ldx, const long long* __restrict__ map,
                               int64_t rows, int64_t cols, double* __restrict__ out, int64_t ldo) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * cols) return;
  const int64_t i = idx / cols, j = idx % cols;
  const double v = (double)X[i * ldx + j];
  if (ROWS) out[map[i] * ldo + j] = v; else out[i * ldo + map[j]] = v;
}

// X = A * (((2 nv) u + nv) + 1), every step rounded like numpy's separate ufunc calls (pyDNMFk.py:42-44)
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }

template <typename T>
__global__ void perturb_uniform_kernel(const T* __restrict__ A, const T* __restrict__ U, T* __restrict__ X,
                                       int64_t count, T two_nv, T nv) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= count) return;
  T mfac = mul_rn(two_nv, U[idx]);
  mfac = add_rn(mfac, nv);
  mfac = add_rn(mfac, T(1));
  X[idx] = mul_rn(A[idx], mfac);
}

}  // namespace dnmf
