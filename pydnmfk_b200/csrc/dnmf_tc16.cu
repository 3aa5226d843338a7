// tcgen05 kind::f16 path of the A-streaming contractions for a data shard stored in 16 bits (DNMF_A_F16 / DNMF_A_BF16)
// with fp32 factors and fp32 results.
//
//   AH  : V[m x k]   = A[m x n] * H[k x n]^T          (dist_nmf.py:198, :730)
//   WTA : Y^T[n x k] = (W[m x k]^T * A[m x n])^T       (dist_nmf.py:166, :749)
//
// A is an exact operand of the tensor core, so the split warps of the fp32 kernel (dnmf_tc.cu) disappear: TMA streams
// each A tile (128 x 64 elements = 16 KB) and the matching tile of the split factor Bcat into one shared-memory ring,
// the MMA warp contracts both straight from shared memory (4 MMAs of K = 16 per tile), and four drain warps fold the
// TMEM accumulator into fp32 registers every TC16_CHUNK tiles.
//   AH : A tile K-major, TMA box {64, 128}, 128-byte swizzle (one swizzle row per tile row)
//   WTA: A tile MN-major, two TMA boxes {64 columns, 64 rows} side by side, 128-byte swizzle
//
// fp32 accuracy of the factor B (H, or W^T) from 16-bit parts; Bcat stacks NP copies of the kp factor rows (N = NP kp):
//   fp16 A: B 2^s[j] = b_hi + b_lo, both fp16.  s[j] is a power of two per factor row that puts the row's largest
//           magnitude rowmax into [2^14, 2^15): a row of small entries (a dying component near the clamp eps = 1.2e-7)
//           would otherwise fall below fp16's normal range.  Entries >= rowmax 2^-18 keep 22 significant bits; below
//           that b_lo is subnormal and the error is bounded absolutely by 2^-25 2^-s <= rowmax 2^-39 (an entry of 1e-7 in a
//           row whose largest entry is 30 keeps about 11 bits).  The drain undoes the scale exactly.
//   bf16 A: B = b1 + b2 + b3, all bf16 (fp32's exponent range, no scale): 24 significant bits.
// The tensor core accumulates in fp32 with truncation (DESIGN.md section 5.1): draining every TC16_CHUNK tiles (8 MMAs)
// and summing the chunks in registers with round-to-nearest keeps that bias at the level of fp32 arithmetic.
//
// Warp roles (one persistent CTA per SM): w0 TMA producer | w1 MMA issuer + TMEM owner | w2-5 drain.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "generic_passes.cuh"
#include "tc_api.cuh"
#include "tc_common.cuh"

namespace dnmf {

namespace {

constexpr int TC16_BK = 64;       // reduced-dimension tile: 64 16-bit elements = one 128-byte swizzle row = 4 MMA K steps
constexpr int TC16_CHUNK = 2;     // K-tiles accumulated in TMEM before the drain warps fold them into registers
constexpr int TC16_THREADS = 192;

template <int KP, int NP>
struct Tc16Cfg {
  static constexpr int NB = NP * KP;                            // MMA N: the NP parts of the kp factor rows
  static constexpr int A_BYTES = TC_BM * TC16_BK * 2;           // 16 KB
  static constexpr int B_BYTES = NB * TC16_BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = (200 * 1024) / STAGE_BYTES > 12 ? 12 : (200 * 1024) / STAGE_BYTES;
  static constexpr int BUF_COLS = NB <= 64 ? 64 : (NB <= 128 ? 128 : 256);   // TMEM columns per accumulator buffer
  static constexpr int NBUF = 512 / BUF_COLS > 4 ? 4 : 512 / BUF_COLS;
  static constexpr int TMEM_COLS = NBUF * BUF_COLS <= 256 ? 256 : 512;
  static constexpr int BAR_BYTES = 256;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + BAR_BYTES;
  static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB opt-in shared memory limit");
  static_assert((2 * STAGES + 2 * NBUF + 1) * 8 <= BAR_BYTES, "barrier area too small");
  static_assert(NB % 16 == 0 && NB <= 256, "UMMA N for M = 128");
};

// instruction descriptor: D fp32, A and B both fp16 (bf16 = 0) or both bf16 (bf16 = 1), M = 128, N = n, B K-major
__host__ __device__ constexpr uint32_t make_idesc16(int n, int a_mn_major, int bf16) {
  return (1u << 4)                          // c_format = F32
         | ((uint32_t)bf16 << 7)            // a_format: 0 = F16, 1 = BF16
         | ((uint32_t)bf16 << 10)           // b_format
         | ((uint32_t)a_mn_major << 15)     // A major: 0 = K, 1 = MN
         | ((uint32_t)(n >> 3) << 17)       // N >> 3
         | ((uint32_t)(TC_BM >> 4) << 24);  // M >> 4
}

// One K tile (4 MMAs of K = 16) plus the commits that release the ring slot and, at a chunk end, the accumulator; one
// asm block under a single elect.sync, issued by a converged warp (see umma_tile_ts in tc_common.cuh).  ASTEP: the A
// descriptor advance per K step (K-major: 32 bytes; MN-major: two 8-row groups of 1024 bytes).
template <int ASTEP>
__device__ __forceinline__ void umma16_tile(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t acc_first, uint32_t bar_free, uint32_t bar_acc, uint32_t chunk_end) {
  asm volatile(
      "{\n\t"
      ".reg .pred q, p0, p1, pc;\n\t"
      ".reg .b64 a1, a2, a3, b1, b2, b3;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p0, %4, 0;\n\t"
      "setp.eq.b32 p1, 0, 0;\n\t"
      "setp.ne.b32 pc, %7, 0;\n\t"
      "and.pred pc, pc, q;\n\t"
      "add.u64 a1, %1, %8;\n\t"
      "add.u64 a2, %1, %9;\n\t"
      "add.u64 a3, %1, %10;\n\t"
      "add.u64 b1, %2, 2;\n\t"
      "add.u64 b2, %2, 4;\n\t"
      "add.u64 b3, %2, 6;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], a1, b1, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], a2, b2, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], a3, b3, %3, p1;\n\t"
      "@q  tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%5];\n\t"
      "@pc tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%6];\n\t"
      "}\n"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc_first), "r"(bar_free), "r"(bar_acc), "r"(chunk_end),
        "n"(ASTEP), "n"(2 * ASTEP), "n"(3 * ASTEP)
      : "memory");
}

// ---------------------------------------------------------------------------------------------------------
// persistent kernel
//   MODE 0 (AH):  X = rows of A (m), reduced = columns (n);   MODE 1 (WTA): X = columns of A (n), reduced = rows (m)
//   B tile = TMA box {64, NB} of Bcat[NB][reduced], K-major, 128-byte swizzle.
//   Output: P[split][x][KP] (x < x_len), scaled back by 2^-s[j] (fp16) -- the layout of the fp32 kernel's partials.
// ---------------------------------------------------------------------------------------------------------
template <int KP, int NP, int MODE>
__global__ void __launch_bounds__(TC16_THREADS, 1)
tc16_pass_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const int* __restrict__ sexp, float* __restrict__ P, int64_t split_stride, int64_t x_len, int x_blocks,
                 int kt_total, int kt_per_split, int num_units) {
  using Cfg = Tc16Cfg<KP, NP>;
  constexpr int S = Cfg::STAGES, NBUF = Cfg::NBUF;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t bars = base + S * Cfg::STAGE_BYTES;
  auto full = [&](int s) { return bars + 8u * s; };
  auto empty = [&](int s) { return bars + 8u * (S + s); };
  auto accf = [&](int b) { return bars + 8u * (2 * S + b); };
  auto acce = [&](int b) { return bars + 8u * (2 * S + NBUF + b); };
  constexpr int SLOT_IDX = 2 * S + 2 * NBUF;
  const uint32_t tmem_slot = bars + 8u * SLOT_IDX;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(base_ptr + S * Cfg::STAGE_BYTES + 8 * SLOT_IDX);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < S; ++s) { mbar_init(full(s), 1); mbar_init(empty(s), 1); }
    for (int b = 0; b < NBUF; ++b) { mbar_init(accf(b), 1); mbar_init(acce(b), 4); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ===================== producer: A tile + B tile of every (unit, K-tile) into the ring =====================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
        const int xb = unit % x_blocks, sp = unit / x_blocks;
        const int kt0 = sp * kt_per_split;
        const int kt1 = min(kt_total, kt0 + kt_per_split);
        for (int kt = kt0; kt < kt1; ++kt) {
          mbar_wait(empty(s), ph ^ 1u);
          const uint32_t sA = base + s * Cfg::STAGE_BYTES;
          mbar_expect_tx(full(s), Cfg::STAGE_BYTES);
          if (MODE == 0) {
            tma_load_2d(sA, &tmA, full(s), kt * TC16_BK, xb * TC_BM);
          } else {
            tma_load_2d(sA, &tmA, full(s), xb * TC_BM, kt * TC16_BK);
            tma_load_2d(sA + Cfg::A_BYTES / 2, &tmA, full(s), xb * TC_BM + 64, kt * TC16_BK);
          }
          tma_load_2d(sA + Cfg::A_BYTES, &tmB, full(s), kt * TC16_BK, 0);
          if (++s == S) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (the whole warp, converged; one elected lane issues) =====================
    constexpr uint32_t idesc = make_idesc16(Cfg::NB, MODE, NP == 3 ? 1 : 0);
    int s = 0, buf = 0;
    uint32_t ph = 0, accphase = 0;
    for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
      const int sp = unit / x_blocks;
      const int kt0 = sp * kt_per_split;
      const int kt1 = min(kt_total, kt0 + kt_per_split);
      for (int kt = kt0; kt < kt1; ++kt) {
        const int in_chunk = (kt - kt0) % TC16_CHUNK;
        if (in_chunk == 0) mbar_wait(acce(buf), accphase ^ 1u);     // new chunk: the drain warps emptied this buffer
        mbar_wait(full(s), ph);
        tc_fence_after();
        const uint32_t sA = base + s * Cfg::STAGE_BYTES;
        // K-major A: 8-row groups 1024 bytes apart; MN-major A: 64-column halves 8192 bytes apart (leading byte offset),
        // 8-row K groups 1024 bytes apart (stride byte offset)
        const uint64_t adesc = MODE == 0 ? make_smem_desc(sA, 16, 1024) : make_smem_desc(sA, Cfg::A_BYTES / 2, 1024);
        const uint64_t bdesc = make_smem_desc(sA + Cfg::A_BYTES, 16, 1024);
        const bool chunk_end = (in_chunk == TC16_CHUNK - 1) || (kt == kt1 - 1);
        umma16_tile<MODE == 0 ? 2 : 128>(tmem_base + (uint32_t)(buf * Cfg::BUF_COLS), adesc, bdesc, idesc,
                                         in_chunk > 0 ? 1u : 0u, empty(s), accf(buf), chunk_end ? 1u : 0u);
        if (++s == S) { s = 0; ph ^= 1u; }
        if (chunk_end && ++buf == NBUF) { buf = 0; accphase ^= 1u; }
        __syncwarp();
      }
    }
  } else {
    // ===================== drain warps 2-5: TMEM chunk -> fp32 registers -> global partial =====================
    const int q = warp & 3;               // TMEM lane quarter this warp may access
    int buf = 0;
    uint32_t accphase = 0;
    for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
      const int xb = unit % x_blocks, sp = unit / x_blocks;
      const int kt0 = sp * kt_per_split;
      const int kt1 = min(kt_total, kt0 + kt_per_split);
      const int nchunks = (kt1 - kt0 + TC16_CHUNK - 1) / TC16_CHUNK;
      float acc[KP];
#pragma unroll
      for (int j = 0; j < KP; ++j) acc[j] = 0.f;
      for (int c = 0; c < nchunks; ++c) {
        mbar_wait(accf(buf), accphase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * Cfg::BUF_COLS);
#pragma unroll
        for (int j0 = 0; j0 < KP; j0 += 16) {
          uint32_t p0[16], p1[16], p2[16];
          tmem_ld_x16(taddr + j0, p0);
          tmem_ld_x16(taddr + KP + j0, p1);
          if (NP == 3) tmem_ld_x16(taddr + 2 * KP + j0, p2);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float small = NP == 3 ? __uint_as_float(p1[j]) + __uint_as_float(p2[j]) : __uint_as_float(p1[j]);
            acc[j0 + j] += __uint_as_float(p0[j]) + small;
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(acce(buf));   // TMEM buffer may be overwritten
        if (++buf == NBUF) { buf = 0; accphase ^= 1u; }
      }
      const int64_t x = (int64_t)xb * TC_BM + q * 32 + lane;
      if (x < x_len) {
        if (NP == 2) {
#pragma unroll
          for (int j = 0; j < KP; ++j) acc[j] = scalbnf(acc[j], -sexp[j]);
        }
        float* orow = P + (int64_t)sp * split_stride + x * KP;
#pragma unroll
        for (int j = 0; j < KP; j += 4)
          *reinterpret_cast<float4*>(orow + j) = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------------------
// factor split.  B(j, c) = src[j * sj + c * sc] for factor row j < k and reduced index c < len:
//   AH:  B = H (sj = ldh, sc = 1);   WTA: B = W^T (sj = 1, sc = ldw)
// Bcat[p * kp + j][c] (ld = ldb) = part p of B(j, c); rows [k, kp) of every part stay zero (memset by the caller).
// ---------------------------------------------------------------------------------------------------------
// fp16 scale: B(j, :) 2^s has its largest magnitude in [2^14, 2^15)
__device__ __forceinline__ int f16_scale_exp(uint32_t amax_bits) {
  if (amax_bits == 0) return 0;
  const int e = (int)(amax_bits >> 23);           // biased exponent of the row's largest magnitude (0: fp32 subnormal)
  return 14 - (e == 0 ? -126 : e - 127);
}

// row_major: one thread per element in (j, c) order (H) or in (c, j) order (W^T, coalesced reads of W's rows)
__device__ __forceinline__ void split_index(int64_t idx, int k, int64_t len, bool row_major, int& j, int64_t& c) {
  if (row_major) { j = (int)(idx / len); c = idx % len; }
  else { c = idx / k; j = (int)(idx % k); }
}

// largest |B(j, :)| as fp32 bits, atomically max-ed into amax[j] (order independent: deterministic)
__global__ void __launch_bounds__(256) tc16_amax_kernel(const float* __restrict__ src, int64_t sj, int64_t sc, int k,
                                                        int64_t len, int row_major, unsigned* __restrict__ amax) {
  const int64_t total = (int64_t)k * len;
  __shared__ unsigned red[64];
  for (int i = threadIdx.x; i < 64; i += blockDim.x) red[i] = 0u;
  __syncthreads();
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    int j;
    int64_t c;
    split_index(idx, k, len, row_major != 0, j, c);
    atomicMax(&red[j], __float_as_uint(fabsf(src[j * sj + c * sc])));
  }
  __syncthreads();
  for (int i = threadIdx.x; i < k; i += blockDim.x)
    if (red[i]) atomicMax(&amax[i], red[i]);
}

template <int NP>
__global__ void __launch_bounds__(256) tc16_split_kernel(const float* __restrict__ src, int64_t sj, int64_t sc, int k, int kp,
                                                         int64_t len, int row_major, const unsigned* __restrict__ amax,
                                                         int* __restrict__ sexp, uint16_t* __restrict__ Bcat, int64_t ldb) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < kp && NP == 2) sexp[idx] = idx < k ? f16_scale_exp(amax[idx]) : 0;
  if (idx >= (int64_t)k * len) return;
  int j;
  int64_t c;
  split_index(idx, k, len, row_major != 0, j, c);
  const float b = src[j * sj + c * sc];
  uint16_t* out = Bcat + (int64_t)j * ldb + c;
  const int64_t part = (int64_t)kp * ldb;
  if (NP == 2) {
    const float v = scalbnf(b, f16_scale_exp(amax[j]));     // exact
    const __half hi = __float2half_rn(v);
    const __half lo = __float2half_rn(v - __half2float(hi));  // v - hi is exact in fp32
    out[0] = __half_as_ushort(hi);
    out[part] = __half_as_ushort(lo);
  } else {
    const __nv_bfloat16 b1 = __float2bfloat16_rn(b);
    const float r1 = b - __bfloat162float(b1);
    const __nv_bfloat16 b2 = __float2bfloat16_rn(r1);
    const __nv_bfloat16 b3 = __float2bfloat16_rn(r1 - __bfloat162float(b2));
    out[0] = __bfloat16_as_ushort(b1);
    out[part] = __bfloat16_as_ushort(b2);
    out[2 * part] = __bfloat16_as_ushort(b3);
  }
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------
Tc16Layout tc16_layout(int mode, int64_t m, int64_t n, int k, int dtype) {
  Tc16Layout L;
  const int64_t x_len = mode == 0 ? m : n;
  const int64_t r_len = mode == 0 ? n : m;
  L.kp = tc_padded_k(k);
  L.np = dtype == DNMF_A_F16 ? 2 : 3;
  L.pl = tc_plan(x_len, r_len, L.kp, TC16_BK);
  L.ldb = round_up(r_len > 0 ? r_len : 1, 8);                   // 16-byte rows for TMA
  L.bcat_bytes = round_up((int64_t)L.np * L.kp * L.ldb * 2, 1024);
  L.aux_bytes = 1024;
  L.total = L.bcat_bytes + L.aux_bytes + L.pl.partial_bytes;
  return L;
}

namespace {

template <int KP, int NP, int MODE>
int launch16(const CUtensorMap& tmA, const CUtensorMap& tmB, const int* sexp, float* P, int64_t split_stride,
             int64_t x_len, const TcPlan& pl, cudaStream_t st) {
  using Cfg = Tc16Cfg<KP, NP>;
  if (int rc = smem_attr_once<tc16_pass_kernel<KP, NP, MODE>>(Cfg::SMEM_BYTES, "tc16_pass_kernel smem attribute")) return rc;
  tc16_pass_kernel<KP, NP, MODE><<<pl.grid, TC16_THREADS, Cfg::SMEM_BYTES, st>>>(
      tmA, tmB, sexp, P, split_stride, x_len, pl.x_blocks, pl.kt_total, pl.kt_per_split, pl.num_units);
  DNMF_LAUNCH_CHECK("tc16_pass_kernel");
  return 0;
}

template <int NP, int MODE>
int launch16_k(int kp, const CUtensorMap& tmA, const CUtensorMap& tmB, const int* sexp, float* P, int64_t split_stride,
               int64_t x_len, const TcPlan& pl, cudaStream_t st) {
  switch (kp) {
    case 16: return launch16<16, NP, MODE>(tmA, tmB, sexp, P, split_stride, x_len, pl, st);
    case 32: return launch16<32, NP, MODE>(tmA, tmB, sexp, P, split_stride, x_len, pl, st);
    case 64: return launch16<64, NP, MODE>(tmA, tmB, sexp, P, split_stride, x_len, pl, st);
  }
  return fail(DNMF_E_UNSUPPORTED, "tcgen05 kind::f16 path: k must be padded to 16, 32 or 64");
}

}  // namespace

int tc16_run(int mode, const void* A, int64_t lda, const float* B, int64_t ldbsrc, float* out, int64_t ldo, int64_t m,
             int64_t n, int k, int transposed_out, int dtype, void* ws, int64_t ws_bytes, cudaStream_t st,
             TcPartials* defer) {
  const Tc16Layout L = tc16_layout(mode, m, n, k, dtype);
  const TcPlan& pl = L.pl;
  const int64_t x_len = mode == 0 ? m : n;
  const int64_t r_len = mode == 0 ? n : m;
  if (int rc = tc_begin(ws, ws_bytes, L.total, L.bcat_bytes, L.kp != k, st)) return rc;
  uint8_t* w8 = reinterpret_cast<uint8_t*>(ws);
  uint16_t* Bcat = reinterpret_cast<uint16_t*>(w8);
  unsigned* amax = reinterpret_cast<unsigned*>(w8 + L.bcat_bytes);
  int* sexp = reinterpret_cast<int*>(w8 + L.bcat_bytes + 256);
  float* P = reinterpret_cast<float*>(w8 + L.bcat_bytes + L.aux_bytes);
  const int64_t sj = mode == 0 ? ldbsrc : 1, sc = mode == 0 ? 1 : ldbsrc;
  const int row_major = mode == 0 ? 1 : 0;
  const int64_t total = (int64_t)k * r_len;
  if (L.np == 2) {
    cudaError_t e = cudaMemsetAsync(amax, 0, 256, st);
    if (e != cudaSuccess) return cuda_fail(e, "amax memset");
    const int64_t blocks = ceil_div(total, 256);
    tc16_amax_kernel<<<(unsigned)(blocks < 4 * sm_count() ? blocks : 4 * sm_count()), 256, 0, st>>>(B, sj, sc, k, r_len,
                                                                                                   row_major, amax);
    DNMF_LAUNCH_CHECK("tc16_amax_kernel");
    tc16_split_kernel<2><<<(unsigned)ceil_div(total > L.kp ? total : L.kp, 256), 256, 0, st>>>(B, sj, sc, k, L.kp, r_len,
                                                                                             row_major, amax, sexp, Bcat, L.ldb);
  } else {
    tc16_split_kernel<3><<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(B, sj, sc, k, L.kp, r_len, row_major, amax,
                                                                        sexp, Bcat, L.ldb);
  }
  DNMF_LAUNCH_CHECK("tc16_split_kernel");
  alignas(64) CUtensorMap tmA, tmB;
  const CUtensorMapDataType type = dtype == DNMF_A_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  int rc = mode == 0 ? tc_make_map(&tmA, type, A, m, n, lda, TC16_BK, TC_BM)
                     : tc_make_map(&tmA, type, A, m, n, lda, 64, TC16_BK);
  if (rc || (rc = tc_make_map(&tmB, type, Bcat, (int64_t)L.np * L.kp, r_len, L.ldb, TC16_BK, L.np * L.kp))) return rc;
  const int64_t split_stride = x_len * L.kp;
  if (L.np == 2) rc = mode == 0 ? launch16_k<2, 0>(L.kp, tmA, tmB, sexp, P, split_stride, x_len, pl, st)
                                : launch16_k<2, 1>(L.kp, tmA, tmB, sexp, P, split_stride, x_len, pl, st);
  else rc = mode == 0 ? launch16_k<3, 0>(L.kp, tmA, tmB, sexp, P, split_stride, x_len, pl, st)
                      : launch16_k<3, 1>(L.kp, tmA, tmB, sexp, P, split_stride, x_len, pl, st);
  if (rc) return rc;
  return tc_finish(P, x_len, L.kp, pl.splits, mode, k, transposed_out, out, ldo, st, defer);
}

}  // namespace dnmf
