// Sparse data shards: the A-streaming passes over a compressed (CSR / CSC) shard.  See include/dnmf.h, "sparse shards".
//
// There is one contraction, over the rows of a compressed matrix (ptr, idx, val):
//   out[r, 0:k] = sum_{e in row r} u_e * G[idx_e, 0:k],   u_e = val_e (FRO) or val_e / (F[r,:] . G[idx_e,:] + eps) (KL)
// AH and KL-UHT run it on the CSR of A with G = H^T (F = W); WTA and KL-WTU on the CSC with G = W (F = H^T).  The
// residual mode runs on the CSR like AH and also sums (a - s)^2, s^2 and a^2 over the non-zeros, s = (W H)_ij in float64.
//
// Layout: G and F are copied once per call into the workspace as [rows][KP] arrays, zero-padded to the padded width KP,
// so that a sub-warp of KP / VEC lanes gathers a row of G as 16-byte vectors (VEC = 4 floats or 2 doubles).  The KL dot
// product F[r,:] . G[idx,:] reuses the G row the contraction loads anyway and is reduced across the sub-warp with an XOR
// butterfly, which gives every lane the same bits.
//
// Scheduling: one warp per fixed chunk of kSpChunk non-zeros, not per row, so a row holding a large share of the
// non-zeros does not serialise the pass.  A row that lies inside one chunk is written by that chunk's warp.  A row that
// spans chunks leaves one partial per chunk (tail slot of the chunk where it starts, head slots of the others); the fixup
// kernel adds them in chunk order and writes the zeros of empty rows.  No atomics: repeated calls are bit-identical.
#include "common.cuh"
#include "launch_passes.cuh"

using namespace dnmf;

namespace {

constexpr int64_t kSpChunk = 512;        // non-zeros per warp
constexpr int kSpWarps = 8;              // warps per block of the chunk kernel
constexpr int64_t kSpGramRows = 256;     // rows per block of the float64 Gram partials
constexpr int64_t kSpGramBlocks = 128;   // at most this many Gram partials

enum SpMode { SP_FRO = 0, SP_KL = 1, SP_FRO_RES = 2, SP_RES = 3 };

inline size_t esize(int dtype) { return dtype == DNMF_F64 ? 8 : 4; }

int check_sp(int64_t m, int64_t n, int64_t nnz, int64_t k, int dtype) {
  if (dtype != DNMF_F32 && dtype != DNMF_F64) return fail(DNMF_E_ARG, "dtype must be DNMF_F32 or DNMF_F64");
  if (m < 0 || n < 0 || nnz < 0 || k < 0) return fail(DNMF_E_ARG, "negative dimension");
  if (m >= ((int64_t)1 << 31) || n >= ((int64_t)1 << 31)) return fail(DNMF_E_ARG, "rows and columns of a sparse shard must be < 2^31");
  if (k > DNMF_MAX_K) return fail(DNMF_E_UNSUPPORTED, "k=%lld exceeds DNMF_MAX_K=%d", (long long)k, DNMF_MAX_K);
  return 0;
}

// workspace layout: a pure function of the shape, shared by the size query and the launches
struct SpLayout {
  int64_t chunks, gblocks_m, gblocks_n;
  int64_t off_fm, off_fn, off_head, off_tail, off_res, off_gp, off_g, total;
};

SpLayout sp_layout(int64_t m, int64_t n, int64_t nnz, int64_t k, int dtype) {
  SpLayout L;
  const int64_t kp = padded_k(k), es = (int64_t)esize(dtype);
  L.chunks = ceil_div(nnz, kSpChunk);
  L.gblocks_m = m > 0 ? ceil_div(m, ceil_div(m, kSpGramBlocks * kSpGramRows) * kSpGramRows) : 0;
  L.gblocks_n = n > 0 ? ceil_div(n, ceil_div(n, kSpGramBlocks * kSpGramRows) * kSpGramRows) : 0;
  int64_t o = 0;
  auto take = [&](int64_t bytes) { const int64_t at = o; o += round_up(bytes > 0 ? bytes : 0, 256); return at; };
  L.off_fm = take(m * kp * es);                                     // W, [m][KP]
  L.off_fn = take(n * kp * es);                                     // H^T, [n][KP]
  L.off_head = take(L.chunks * kp * es);
  L.off_tail = take(L.chunks * kp * es);
  L.off_res = take(L.chunks * 3 * (int64_t)sizeof(double));
  L.off_gp = take((L.gblocks_m + L.gblocks_n) * kp * kp * (int64_t)sizeof(double));
  L.off_g = take(2 * kp * kp * (int64_t)sizeof(double));
  L.total = o + 256;
  return L;
}

// dst[r][j] = X[r * sr + j * sc] for j < k, 0 for k <= j < KP
template <typename T>
__global__ void sp_pad_kernel(const T* __restrict__ X, int64_t sr, int64_t sc, int64_t rows, int k, int kp, T* __restrict__ dst) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * kp) return;
  const int64_t r = i / kp;
  const int j = (int)(i % kp);
  dst[i] = j < k ? X[r * sr + (int64_t)j * sc] : T(0);
}

template <typename T, int LANES>
__device__ __forceinline__ T sub_sum(T v) {
#pragma unroll
  for (int o = 1; o < LANES; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <typename T, int KP, int MODE>
__global__ void __launch_bounds__(32 * kSpWarps)
sp_chunk_kernel(const int64_t* __restrict__ ptr, const int* __restrict__ idx, const T* __restrict__ val, int64_t rows,
                int64_t nnz, const T* __restrict__ G, const T* __restrict__ F, T eps, T* __restrict__ out, int64_t ors,
                int64_t ocs, int k, T* __restrict__ head, T* __restrict__ tail, double* __restrict__ res, int64_t chunks) {
  constexpr int VEC = VecOf<T>::N;
  constexpr int LANES = KP / VEC >= 1 ? KP / VEC : 1;
  constexpr int SUB = 32 / LANES;
  constexpr bool KL = MODE == SP_KL;
  constexpr bool RES = MODE == SP_FRO_RES || MODE == SP_RES;
  constexpr bool OUT = MODE != SP_RES;
  const int64_t c = (int64_t)blockIdx.x * kSpWarps + (threadIdx.x >> 5);
  if (c >= chunks) return;
  const int lane = threadIdx.x & 31, sub = lane / LANES, sl = lane % LANES;
  const int64_t cs = c * kSpChunk, ce = cs + kSpChunk < nnz ? cs + kSpChunk : nnz;
  // the row holding non-zero cs: the largest r with ptr[r] <= cs (empty rows share their pointer with the next row)
  int64_t lo = 0, hi = rows - 1;
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) >> 1;
    if (ptr[mid] <= cs) lo = mid; else hi = mid - 1;
  }
  double d2 = 0.0, s2 = 0.0, a2 = 0.0;
  for (int64_t r = lo; r < rows; ++r) {
    const int64_t rb = ptr[r], re = ptr[r + 1];
    if (rb >= ce) break;
    const int64_t e0 = rb > cs ? rb : cs, e1 = re < ce ? re : ce;
    if (e0 >= e1) continue;
    T f[VEC];
    if (KL || RES) vload(F + r * KP + sl * VEC, f);
    T acc[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) acc[v] = T(0);
#pragma unroll 2
    for (int64_t base = e0; base < e1; base += SUB) {
      const int64_t e = base + sub;
      const bool ok = e < e1;
      const int64_t j = ok ? (int64_t)idx[e] : 0;
      const T a = ok ? val[e] : T(0);
      T g[VEC];
      vload(G + j * KP + sl * VEC, g);
      T u = a;
      if (KL) {
        T d = T(0);
#pragma unroll
        for (int v = 0; v < VEC; ++v) d += f[v] * g[v];
        d = sub_sum<T, LANES>(d);
        u = ok ? a / (d + eps) : T(0);
      }
      if (RES) {
        double d = 0.0;
#pragma unroll
        for (int v = 0; v < VEC; ++v) d += (double)f[v] * (double)g[v];
        d = sub_sum<double, LANES>(d);
        if (ok && sl == 0) {
          const double da = (double)a;
          d2 += (da - d) * (da - d);
          s2 += d * d;
          a2 += da * da;
        }
      }
      if (OUT) {
#pragma unroll
        for (int v = 0; v < VEC; ++v) acc[v] += u * g[v];
      }
    }
    if (OUT) {
      // sum over the sub-warps (butterfly: every sub-warp ends with the same bits)
#pragma unroll
      for (int o = LANES; o < 32; o <<= 1) {
#pragma unroll
        for (int v = 0; v < VEC; ++v) acc[v] += __shfl_xor_sync(0xffffffffu, acc[v], o);
      }
      if (sub == 0) {
        if (rb < cs || re > ce) {
          vstore((rb < cs ? head : tail) + c * KP + sl * VEC, acc);
        } else {
#pragma unroll
          for (int v = 0; v < VEC; ++v) {
            const int col = sl * VEC + v;
            if (col < k) out[r * ors + (int64_t)col * ocs] = acc[v];
          }
        }
      }
    }
    if (re > ce) break;
  }
  if (RES) {
    d2 = warp_sum(d2);
    s2 = warp_sum(s2);
    a2 = warp_sum(a2);
    if (lane == 0) {
      res[3 * c] = d2;
      res[3 * c + 1] = s2;
      res[3 * c + 2] = a2;
    }
  }
}

// rows spanning chunks: tail of the first chunk + heads of the following ones, in chunk order; empty rows: zeros
template <typename T>
__global__ void sp_fixup_kernel(const int64_t* __restrict__ ptr, int64_t rows, int k, int kp, const T* __restrict__ head,
                                const T* __restrict__ tail, T* __restrict__ out, int64_t ors, int64_t ocs) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * k) return;
  const int64_t r = i / k;
  const int j = (int)(i % k);
  const int64_t rb = ptr[r], re = ptr[r + 1];
  T* o = out + r * ors + (int64_t)j * ocs;
  if (rb == re) {
    *o = T(0);
    return;
  }
  const int64_t ca = rb / kSpChunk, cb = (re - 1) / kSpChunk;
  if (ca == cb) return;
  T s = tail[ca * kp + j];
  for (int64_t c = ca + 1; c <= cb; ++c) s += head[c * kp + j];
  *o = s;
}

// float64 partial Grams X^T X of [rows][KP] blocks of `per` rows (X zero-padded, so only the k x k corner is nonzero)
template <typename T>
__global__ void __launch_bounds__(256)
sp_gram_partial_kernel(const T* __restrict__ X, int64_t rows, int kp, int64_t per, double* __restrict__ P) {
  __shared__ double tile[32][DNMF_MAX_K + 1];
  const int64_t r0 = (int64_t)blockIdx.x * per;
  const int64_t r1 = r0 + per < rows ? r0 + per : rows;
  const int ne = kp * kp;
  double acc[16];
#pragma unroll
  for (int q = 0; q < 16; ++q) acc[q] = 0.0;
  for (int64_t t0 = r0; t0 < r1; t0 += 32) {
    for (int i = threadIdx.x; i < 32 * kp; i += 256) {
      const int rr = i / kp, j = i % kp;
      tile[rr][j] = t0 + rr < r1 ? (double)X[(t0 + rr) * kp + j] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const int e = threadIdx.x + q * 256;
      if (e < ne) {
        const int a = e / kp, b = e % kp;
        double s = acc[q];
        for (int rr = 0; rr < 32; ++rr) s += tile[rr][a] * tile[rr][b];
        acc[q] = s;
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int q = 0; q < 16; ++q) {
    const int e = threadIdx.x + q * 256;
    if (e < ne) P[(int64_t)blockIdx.x * ne + e] = acc[q];
  }
}

__global__ void sp_gram_reduce_kernel(const double* __restrict__ P, int64_t blocks, int ne, double* __restrict__ Gm) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= ne) return;
  double s = 0.0;
  for (int64_t b = 0; b < blocks; ++b) s += P[b * ne + e];
  Gm[e] = s;
}

// out = [sum (a - s)^2 + (<W^T W, H H^T> - sum s^2), sum a^2]: the zeros of A contribute sum_{a = 0} s^2.  That
// difference of two float64 sums carries an absolute error of ~1e-16 ||W H||^2; a shard without zeros (`full`) has no
// such term, so its residual is the directly summed sum (a - s)^2, as accurate as the dense residual pass.
__global__ void __launch_bounds__(256)
sp_residual_finish_kernel(const double* __restrict__ res, int64_t chunks, const double* __restrict__ Gw,
                          const double* __restrict__ Gh, int ne, int full, double* __restrict__ out) {
  __shared__ double red[8];
  double d2 = 0.0, s2 = 0.0, a2 = 0.0, t = 0.0;
  for (int64_t c = threadIdx.x; c < chunks; c += 256) {
    d2 += res[3 * c];
    s2 += res[3 * c + 1];
    a2 += res[3 * c + 2];
  }
  for (int e = threadIdx.x; e < ne; e += 256) t += Gw[e] * Gh[e];
  d2 = block_sum<256>(d2, red);
  s2 = block_sum<256>(s2, red);
  a2 = block_sum<256>(a2, red);
  t = block_sum<256>(t, red);
  if (threadIdx.x == 0) {
    const double zeros = full ? 0.0 : t - s2;
    out[0] = d2 + (zeros > 0.0 ? zeros : 0.0);
    out[1] = a2;
  }
}

struct SpCall {
  const int64_t* ptr;
  const int* idx;
  const void* val;
  int64_t rows, cols, nnz;   // of the compressed matrix that is walked (CSR: m x n; CSC: n x m)
};

template <typename T>
int sp_pad(const void* X, int64_t sr, int64_t sc, int64_t rows, int k, int kp, T* dst, cudaStream_t st) {
  if (rows * kp == 0) return 0;
  sp_pad_kernel<T><<<(unsigned)ceil_div(rows * kp, 256), 256, 0, st>>>((const T*)X, sr, sc, rows, k, kp, dst);
  DNMF_LAUNCH_CHECK("sp_pad_kernel");
  return 0;
}

template <typename T>
int sp_run(int mode, const SpCall& a, const T* G, const T* F, T eps, T* out, int64_t ors, int64_t ocs, int k,
           const SpLayout& L, char* ws, cudaStream_t st) {
  const int kp = padded_k(k);
  T* head = (T*)(ws + L.off_head);
  T* tail = (T*)(ws + L.off_tail);
  double* res = (double*)(ws + L.off_res);
  if (L.chunks > 0) {
    const unsigned grid = (unsigned)ceil_div(L.chunks, kSpWarps);
    DNMF_DISPATCH_KP(kp, {
      switch (mode) {
        case SP_FRO: sp_chunk_kernel<T, KP, SP_FRO><<<grid, 32 * kSpWarps, 0, st>>>(a.ptr, a.idx, (const T*)a.val, a.rows, a.nnz, G, F, eps, out, ors, ocs, k, head, tail, res, L.chunks); break;
        case SP_KL: sp_chunk_kernel<T, KP, SP_KL><<<grid, 32 * kSpWarps, 0, st>>>(a.ptr, a.idx, (const T*)a.val, a.rows, a.nnz, G, F, eps, out, ors, ocs, k, head, tail, res, L.chunks); break;
        case SP_FRO_RES: sp_chunk_kernel<T, KP, SP_FRO_RES><<<grid, 32 * kSpWarps, 0, st>>>(a.ptr, a.idx, (const T*)a.val, a.rows, a.nnz, G, F, eps, out, ors, ocs, k, head, tail, res, L.chunks); break;
        default: sp_chunk_kernel<T, KP, SP_RES><<<grid, 32 * kSpWarps, 0, st>>>(a.ptr, a.idx, (const T*)a.val, a.rows, a.nnz, G, F, eps, out, ors, ocs, k, head, tail, res, L.chunks); break;
      }
    });
    DNMF_LAUNCH_CHECK("sp_chunk_kernel");
  }
  if (mode != SP_RES && a.rows * k > 0) {
    sp_fixup_kernel<T><<<(unsigned)ceil_div(a.rows * k, 256), 256, 0, st>>>(a.ptr, a.rows, k, kp, head, tail, out, ors, ocs);
    DNMF_LAUNCH_CHECK("sp_fixup_kernel");
  }
  return 0;
}

// float64 <W^T W, H H^T> from the padded copies, then the residual pair
template <typename T>
int sp_residual_finish(const SpLayout& L, int64_t m, int64_t n, int64_t nnz, int k, char* ws, double* out,
                       cudaStream_t st) {
  const int kp = padded_k(k), ne = kp * kp;
  double* P = (double*)(ws + L.off_gp);
  double* Gm = (double*)(ws + L.off_g);
  const int64_t gb[2] = {L.gblocks_m, L.gblocks_n};
  const int64_t rows[2] = {m, n};
  const T* X[2] = {(const T*)(ws + L.off_fm), (const T*)(ws + L.off_fn)};
  for (int s = 0; s < 2; ++s) {
    double* Ps = P + (s == 0 ? 0 : L.gblocks_m * ne);
    if (gb[s] > 0) {
      const int64_t per = ceil_div(rows[s], gb[s] * kSpGramRows) * kSpGramRows;
      sp_gram_partial_kernel<T><<<(unsigned)gb[s], 256, 0, st>>>(X[s], rows[s], kp, per, Ps);
      DNMF_LAUNCH_CHECK("sp_gram_partial_kernel");
    }
    sp_gram_reduce_kernel<<<(unsigned)ceil_div(ne, 256), 256, 0, st>>>(Ps, gb[s], ne, Gm + s * ne);
    DNMF_LAUNCH_CHECK("sp_gram_reduce_kernel");
  }
  sp_residual_finish_kernel<<<1, 256, 0, st>>>((const double*)(ws + L.off_res), L.chunks, Gm, Gm + ne, ne, nnz == m * n ? 1 : 0, out);
  DNMF_LAUNCH_CHECK("sp_residual_finish_kernel");
  return 0;
}

int need_ws(const SpLayout& L, void* ws, int64_t ws_bytes) {
  if (ws == nullptr || ws_bytes < L.total)
    return fail(DNMF_E_WORKSPACE, "sparse pass needs %lld workspace bytes, got %lld", (long long)L.total, (long long)ws_bytes);
  return 0;
}

// the four contractions: rows = true walks the CSR (AH, KL-UHT), false the CSC (WTA, KL-WTU)
int sp_pass(bool rows, bool kl, const int64_t* ptr, const int* idx, const void* val, const void* W, int64_t ldw,
            const void* H, int64_t ldh, void* out, int64_t ldo, int64_t m, int64_t n, int64_t nnz, int64_t k, double eps,
            int transposed_out, int dtype, void* ws, int64_t ws_bytes, cudaStream_t st) {
  const bool need_w = kl || !rows, need_h = kl || rows;
  if (int rc = check_sp(m, n, nnz, k, dtype)) return rc;
  DNMF_CHECK_ARG(ptr && (nnz == 0 || (idx && val)) && out && (!need_w || W) && (!need_h || H), "null pointer");
  DNMF_CHECK_ARG((!need_w || ldw >= k) && (!need_h || ldh >= n) && ldo >= (rows || transposed_out ? k : n),
                 "leading dimension too small");
  const SpLayout L = sp_layout(m, n, nnz, k, dtype);
  if (int rc = need_ws(L, ws, ws_bytes)) return rc;
  if ((rows ? m : n) == 0 || k == 0) return 0;
  char* w = (char*)ws;
  const int kp = padded_k(k);
  const SpCall a{ptr, idx, val, rows ? m : n, rows ? n : m, nnz};
  // output element (r, j) of the walked matrix's row r: V[r][j] (AH), Y^T[r][j] or Y[j][r] (WTA)
  const int64_t ors = rows || transposed_out ? ldo : 1, ocs = rows || transposed_out ? 1 : ldo;
  DNMF_DISPATCH_T(dtype, {
    T* Wp = (T*)(w + L.off_fm);
    T* Hp = (T*)(w + L.off_fn);
    if (need_w) { if (int rc = sp_pad<T>(W, ldw, 1, m, (int)k, kp, Wp, st)) return rc; }
    if (need_h) { if (int rc = sp_pad<T>(H, 1, ldh, n, (int)k, kp, Hp, st)) return rc; }
    return sp_run<T>(kl ? SP_KL : SP_FRO, a, rows ? Hp : Wp, rows ? Wp : Hp, (T)eps, (T*)out, ors, ocs, (int)k, L, w, st);
  });
  return 0;
}

int sp_residual(const int64_t* row_ptr, const int* col_idx, const void* val, const void* W, int64_t ldw, const void* H,
                int64_t ldh, void* V, int64_t ldv, int64_t m, int64_t n, int64_t nnz, int64_t k, double* out, int dtype,
                void* ws, int64_t ws_bytes, cudaStream_t st) {
  if (int rc = check_sp(m, n, nnz, k, dtype)) return rc;
  DNMF_CHECK_ARG(row_ptr && (nnz == 0 || (col_idx && val)) && W && H && out, "null pointer");
  DNMF_CHECK_ARG(ldw >= k && ldh >= n && (V == nullptr || ldv >= k), "leading dimension too small");
  const SpLayout L = sp_layout(m, n, nnz, k, dtype);
  if (int rc = need_ws(L, ws, ws_bytes)) return rc;
  char* w = (char*)ws;
  const int kp = padded_k(k);
  const SpCall a{row_ptr, col_idx, val, m, n, nnz};
  DNMF_DISPATCH_T(dtype, {
    T* Wp = (T*)(w + L.off_fm);
    T* Hp = (T*)(w + L.off_fn);
    if (int rc = sp_pad<T>(W, ldw, 1, m, (int)k, kp, Wp, st)) return rc;
    if (int rc = sp_pad<T>(H, 1, ldh, n, (int)k, kp, Hp, st)) return rc;
    if (m > 0) {
      if (int rc = sp_run<T>(V ? SP_FRO_RES : SP_RES, a, Hp, Wp, T(0), (T*)V, ldv, 1, (int)k, L, w, st)) return rc;
    }
    return sp_residual_finish<T>(L, m, n, nnz, (int)k, w, out, st);
  });
  return 0;
}

}  // namespace

extern "C" {

int64_t dnmf_sp_workspace_bytes(int64_t m, int64_t n, int64_t nnz, int64_t k, int dtype) {
  if (check_sp(m, n, nnz, k, dtype) != 0) return -1;
  return sp_layout(m, n, nnz, k, dtype).total;
}

int dnmf_sp_ah(const int64_t* row_ptr, const int* col_idx, const void* val, const void* H, int64_t ldh, void* V,
               int64_t ldv, int64_t m, int64_t n, int64_t nnz, int64_t k, int dtype, void* ws, int64_t ws_bytes,
               void* stream) {
  return sp_pass(true, false, row_ptr, col_idx, val, nullptr, 0, H, ldh, V, ldv, m, n, nnz, k, 0.0, 0, dtype, ws,
                 ws_bytes, (cudaStream_t)stream);
}

int dnmf_sp_wta(const int64_t* col_ptr, const int* row_idx, const void* val_t, const void* W, int64_t ldw, void* Y,
                int64_t ldy, int64_t m, int64_t n, int64_t nnz, int64_t k, int transposed_out, int dtype, void* ws,
                int64_t ws_bytes, void* stream) {
  return sp_pass(false, false, col_ptr, row_idx, val_t, W, ldw, nullptr, 0, Y, ldy, m, n, nnz, k, 0.0, transposed_out,
                 dtype, ws, ws_bytes, (cudaStream_t)stream);
}

int dnmf_sp_kl_uht(const int64_t* row_ptr, const int* col_idx, const void* val, const void* W, int64_t ldw,
                   const void* H, int64_t ldh, void* V, int64_t ldv, int64_t m, int64_t n, int64_t nnz, int64_t k,
                   double eps, int dtype, void* ws, int64_t ws_bytes, void* stream) {
  return sp_pass(true, true, row_ptr, col_idx, val, W, ldw, H, ldh, V, ldv, m, n, nnz, k, eps, 0, dtype, ws, ws_bytes,
                 (cudaStream_t)stream);
}

int dnmf_sp_kl_wtu(const int64_t* col_ptr, const int* row_idx, const void* val_t, const void* W, int64_t ldw,
                   const void* H, int64_t ldh, void* Y, int64_t ldy, int64_t m, int64_t n, int64_t nnz, int64_t k,
                   double eps, int transposed_out, int dtype, void* ws, int64_t ws_bytes, void* stream) {
  return sp_pass(false, true, col_ptr, row_idx, val_t, W, ldw, H, ldh, Y, ldy, m, n, nnz, k, eps, transposed_out, dtype,
                 ws, ws_bytes, (cudaStream_t)stream);
}

int dnmf_sp_residual_sqnorm(const int64_t* row_ptr, const int* col_idx, const void* val, const void* W, int64_t ldw,
                            const void* H, int64_t ldh, int64_t m, int64_t n, int64_t nnz, int64_t k, double* out,
                            int dtype, void* ws, int64_t ws_bytes, void* stream) {
  return sp_residual(row_ptr, col_idx, val, W, ldw, H, ldh, nullptr, 0, m, n, nnz, k, out, dtype, ws, ws_bytes,
                     (cudaStream_t)stream);
}

int dnmf_sp_ah_residual(const int64_t* row_ptr, const int* col_idx, const void* val, const void* W, int64_t ldw,
                        const void* H, int64_t ldh, void* V, int64_t ldv, int64_t m, int64_t n, int64_t nnz, int64_t k,
                        double* out, int dtype, void* ws, int64_t ws_bytes, void* stream) {
  DNMF_CHECK_ARG(V, "null pointer");
  return sp_residual(row_ptr, col_idx, val, W, ldw, H, ldh, V, ldv, m, n, nnz, k, out, dtype, ws, ws_bytes,
                     (cudaStream_t)stream);
}

}  // extern "C"
