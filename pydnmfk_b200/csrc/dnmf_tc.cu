// tcgen05 / TMA / TMEM path of the A-streaming contractions (fp32 data, k in {16, 32, 64}).
//
//   AH  : V[m x k]   = A[m x n] * H[k x n]^T          (dist_nmf.py:198, :730)
//   WTA : Y^T[n x k] = (W[m x k]^T * A[m x n])^T       (dist_nmf.py:166, :749)
//
// Both stream the resident shard A exactly once from HBM with TMA (cp.async.bulk.tensor) into a shared-memory ring
// and contract it on the 5th-generation tensor cores (tcgen05.mma kind::tf32, accumulators in TMEM).  fp32 accuracy
// comes from the 3-term split  A*B ~= Ah*Bh + Ah*Bl + Al*Bh :
//   - the small operand (H or W) is split once per call into Bcat = [B_hi | B_lo]  (2k "N" rows, K-major, smem),
//   - four "splitter" warps pull every A tile from shared memory into registers and store BOTH the raw tile (the
//     tensor core uses its top 19 bits = A_hi) and A_lo = A - A_hi into TENSOR MEMORY (tcgen05.st): the MMA's A
//     operand then comes from TMEM, which is what makes a skinny (N = 2k) tf32 MMA cheap -- with A in shared
//     memory the tensor core is bound by its 32 B/clk A-operand fetch (measured: 128 clk per K=8 step at any N),
//   - per 32-wide K tile the MMA warp issues 4 x { D[:, 0:2k] += Ah * Bcat^T ;  D[:, k:2k] += Al * Bh^T },
//   - the tensor core accumulates in fp32 with truncation, so every TC_CHUNK tiles four "drain" warps fold the
//     TMEM accumulator into fp32 registers (round-to-nearest) and finally write a per-split partial; the splits
//     are summed in a fixed order by reduce_partials_kernel (deterministic).
//
// Warp roles (one persistent CTA per SM):  w0 A-TMA | w1 MMA issuer + TMEM owner | w2-5 splitters | w6-9 drain |
// w10 B-TMA | w11-14 second splitter group | w15-18 second drain set (k = 64: columns 32-63).
#include "generic_passes.cuh"
#include "tc_api.cuh"
#include "tc_common.cuh"

namespace dnmf {
namespace {

constexpr int TC_THREADS_BASE = 352;  // 11 warps: A producer | MMA | 4 splitters | 4 drain | B producer (+4 splitters)
constexpr int TC_CHUNK = 4;      // K-tiles accumulated in TMEM before the drain warps fold them into registers

// Three decoupled rings:
//   A ring   (shared memory, SA slots x 16 KB): TMA -> splitter warps; freed as soon as the tile is in registers
//   B ring   (shared memory, SB slots x 2K*128 B): TMA -> tensor core (B operand); freed by a splitter warp once the
//            tile's MMAs have completed (see umma_tile_ts)
//   operand ring (TENSOR memory, NT slots x 64 columns): raw A (= A_hi for the tensor core) and A_lo, written by the
//            splitters with tcgen05.st, read by tcgen05.mma as the A operand; freed by tcgen05.commit
// plus NBUF accumulator buffers of 2K TMEM columns.  The tensor core therefore reads only B from shared memory.
template <int K>
struct TcCfg {
  static constexpr int N2 = 2 * K;
  static constexpr int A_BYTES = TC_BM * TC_BK * 4;   // 16 KB
  static constexpr int B_BYTES = N2 * TC_BK * 4;
  static constexpr int SA = (K == 16) ? 10 : (K == 32) ? 8 : 7;
  static constexpr int SB = (K == 16) ? 12 : (K == 32) ? 10 : 6;
  static constexpr int NBUF = (K == 16) ? 4 : (K == 32) ? 3 : 2;
  // two splitter groups work on alternate tiles (hides the tcgen05.st round trip).  The K = 64 drain needs 64 accumulator
  // registers per thread on top of the load buffers -- too many for the 600-thread CTA that two groups make -- so there
  // TWO drain warps share each tensor-memory lane quarter, each folding 32 of the 64 output columns (DW = 2).
  static constexpr int SG = 2;
  static constexpr int DW = (K <= 32) ? 1 : 2;
  static constexpr int KD = K / DW;                   // output columns per drain warp
  static constexpr int THREADS = TC_THREADS_BASE + 128 * (SG - 1) + 128 * (DW - 1);
  static constexpr int OP_COL0 = NBUF * N2;
  static constexpr int NT = (512 - OP_COL0) / 64;
  static constexpr int TMEM_COLS = 512;
  static constexpr int BAR_BYTES = 1024;
  static constexpr int SMEM_BYTES = SA * A_BYTES + SB * B_BYTES + 1024 + BAR_BYTES;
  static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB opt-in shared memory limit");
  static_assert((2 * SA + 2 * SB + 2 * NT + 2 * NBUF + 1) * 8 <= BAR_BYTES, "barrier area too small");
};

// ---------------------------------------------------------------------------------------------------------
// persistent tcgen05 kernel
//   MODE 0 (AH):  X = rows of A (m), reduced = columns (n);  A tile = TMA box {32 cols, 128 rows}, 128B swizzle
//                 (so that a thread can read "its" row with conflict-free 128-bit loads)
//   MODE 1 (WTA): X = columns of A (n), reduced = rows (m);  A tile = TMA box {128 cols, 32 rows}, no swizzle
//                 (a thread reads "its" column, one coalesced 32-bit load per K row)
//   B tile = TMA box {32, 2K} of Bcat[2K][reduced], K-major, 128B swizzle (UMMA B operand).
//   Output: P[split][x][K] (ld = K), x < x_len.
// ---------------------------------------------------------------------------------------------------------
template <int K, int MODE>
__global__ void __launch_bounds__(TcCfg<K>::THREADS, 1)
tc_pass_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               float* __restrict__ P, int64_t split_stride, int64_t x_len, int x_blocks, int kt_total,
               int kt_per_split, int num_units) {
  using Cfg = TcCfg<K>;
  constexpr int SA = Cfg::SA, SB = Cfg::SB, NT = Cfg::NT, NBUF = Cfg::NBUF, N2 = Cfg::N2;
  constexpr int chunk = TC_CHUNK;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sA0 = base, sB0 = base + SA * Cfg::A_BYTES;
  const uint32_t bars = sB0 + SB * Cfg::B_BYTES;
  auto a_full = [&](int s) { return bars + 8u * s; };
  auto a_free = [&](int s) { return bars + 8u * (SA + s); };
  auto b_full = [&](int s) { return bars + 8u * (2 * SA + s); };
  auto b_free = [&](int s) { return bars + 8u * (2 * SA + SB + s); };
  auto t_full = [&](int s) { return bars + 8u * (2 * SA + 2 * SB + s); };
  auto t_free = [&](int s) { return bars + 8u * (2 * SA + 2 * SB + NT + s); };
  auto accf_bar = [&](int b) { return bars + 8u * (2 * SA + 2 * SB + 2 * NT + b); };
  auto acce_bar = [&](int b) { return bars + 8u * (2 * SA + 2 * SB + 2 * NT + NBUF + b); };
  constexpr int SLOT_IDX = 2 * SA + 2 * SB + 2 * NT + 2 * NBUF;
  const uint32_t tmem_slot = bars + 8u * SLOT_IDX;
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(base_ptr + SA * Cfg::A_BYTES + SB * Cfg::B_BYTES + 8 * SLOT_IDX);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < SA; ++s) { mbar_init(a_full(s), 1); mbar_init(a_free(s), 4); }
    for (int s = 0; s < SB; ++s) { mbar_init(b_full(s), 1); mbar_init(b_free(s), 1); }
    for (int s = 0; s < NT; ++s) { mbar_init(t_full(s), 4); mbar_init(t_free(s), 1); }
    for (int b = 0; b < NBUF; ++b) { mbar_init(accf_bar(b), 1); mbar_init(acce_bar(b), 4 * Cfg::DW); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ===================== A producer (TMA) =====================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
        const int xb = unit % x_blocks, sp = unit / x_blocks;
        const int kt0 = sp * kt_per_split;
        const int kt1 = min(kt_total, kt0 + kt_per_split);
        for (int kt = kt0; kt < kt1; ++kt) {
          mbar_wait(a_free(s), ph ^ 1u);
          mbar_expect_tx(a_full(s), Cfg::A_BYTES);
          if (MODE == 0) tma_load_2d(sA0 + s * Cfg::A_BYTES, &tmA, a_full(s), kt * TC_BK, xb * TC_BM);
          else tma_load_2d(sA0 + s * Cfg::A_BYTES, &tmA, a_full(s), xb * TC_BM, kt * TC_BK);
          if (++s == SA) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 10) {
    // ===================== B producer (TMA) =====================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
        const int sp = unit / x_blocks;
        const int kt0 = sp * kt_per_split;
        const int kt1 = min(kt_total, kt0 + kt_per_split);
        for (int kt = kt0; kt < kt1; ++kt) {
          mbar_wait(b_free(s), ph ^ 1u);
          mbar_expect_tx(b_full(s), Cfg::B_BYTES);
          tma_load_2d(sB0 + s * Cfg::B_BYTES, &tmB, b_full(s), kt * TC_BK, 0);
          if (++s == SB) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (both A operands come from tensor memory) =====================
    // the whole warp runs this loop converged; one elected lane issues each tcgen05 instruction
    {
      constexpr uint32_t idesc_full = make_idesc(N2, 0);
      constexpr uint32_t idesc_half = make_idesc(K, 0);
      int sb = 0, ts = 0, buf = 0;
      uint32_t pb = 0, pt = 0, accphase = 0;
      for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
        const int sp = unit / x_blocks;
        const int kt0 = sp * kt_per_split;
        const int kt1 = min(kt_total, kt0 + kt_per_split);
        for (int kt = kt0; kt < kt1; ++kt) {
          const int in_chunk = (kt - kt0) % chunk;
          if (in_chunk == 0) {                      // new accumulation chunk: wait for the drain warps
            mbar_wait(acce_bar(buf), accphase ^ 1u);
          }
          mbar_wait(t_full(ts), pt);
          mbar_wait(b_full(sb), pb);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + (uint32_t)(buf * N2);
          const uint32_t a_raw = tmem_base + (uint32_t)(Cfg::OP_COL0 + ts * 64);
          const uint32_t sB = sB0 + sb * Cfg::B_BYTES;
          const bool chunk_end = (in_chunk == chunk - 1) || (kt == kt1 - 1);
          // cols [0,K): Ah*Bh (large term, alone in its accumulator);  cols [K,2K): Ah*Bl + Al*Bh (small terms)
          umma_tile_ts<K>(d_tmem, a_raw, make_smem_desc(sB, 16, 1024), in_chunk > 0 ? 1u : 0u, idesc_full, idesc_half,
                          t_free(ts), accf_bar(buf), chunk_end ? 1u : 0u);
          if (++ts == NT) { ts = 0; pt ^= 1u; }
          if (++sb == SB) { sb = 0; pb ^= 1u; }
          if (chunk_end) {
            if (++buf == NBUF) { buf = 0; accphase ^= 1u; }
          }
          __syncwarp();
        }
      }
    }
  } else if (warp < 6 || (warp >= 11 && warp < 15)) {
    // ===================== splitters (warps 2-5 [+ 11-14]): smem A tile -> registers -> {A, A - hi(A)} in TMEM =====
    // Thread (q, lane) owns accumulator row q*32+lane: a row of A (AH) or a column of A (WTA).  With two groups,
    // group g takes the tiles whose running index is congruent to g (mod 2).
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const int group = (warp >= 11) ? 1 : 0;
    int tile = 0;
    for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
      const int sp = unit / x_blocks;
      const int kt0 = sp * kt_per_split;
      const int kt1 = min(kt_total, kt0 + kt_per_split);
      const int tile0 = tile;                      // this group's tiles of the unit, stepping by the group count
      for (int kt = kt0 + ((group - tile0) & (Cfg::SG - 1)); kt < kt1; kt += Cfg::SG) {
        tile = tile0 + (kt - kt0);
        const int sa = tile % SA, ts = tile % NT;
        const uint32_t pa = (uint32_t)(tile / SA) & 1u, pt = (uint32_t)(tile / NT) & 1u;
        mbar_wait(a_full(sa), pa);
        const uint8_t* tile_smem = base_ptr + sa * Cfg::A_BYTES;
        uint32_t raw[32], lo[32];
        if (MODE == 0) {
          // row r = 128 contiguous bytes, 16-byte chunk c stored at position c ^ (r & 7)  (SWIZZLE_128B)
          const uint8_t* row = tile_smem + r * 128;
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const uint4 v = *reinterpret_cast<const uint4*>(row + ((c ^ (r & 7)) << 4));
            raw[4 * c + 0] = v.x; raw[4 * c + 1] = v.y; raw[4 * c + 2] = v.z; raw[4 * c + 3] = v.w;
          }
        } else {
          // [32 K rows][128 columns] row-major: one coalesced 32-bit load per K row
          const uint8_t* col = tile_smem + r * 4;
#pragma unroll
          for (int j = 0; j < 32; ++j) raw[j] = *reinterpret_cast<const uint32_t*>(col + j * 512);
        }
        // a - hi(a) is exact; rounding it to tf32 here (nearest) instead of letting the tensor core truncate it
        // removes the one-sided error of the third term
#pragma unroll
        for (int j = 0; j < 32; j += 2) tf32_lo_bits2(raw[j], raw[j + 1], lo[j], lo[j + 1]);
        mbar_wait(t_free(ts), pt ^ 1u);
        // the MMAs of tile (tile - NT) have completed (this operand slot is free again): so is that tile's B slot
        if (q == 0 && lane == 0 && tile >= NT) mbar_arrive(b_free((tile - NT) % SB));
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(Cfg::OP_COL0 + ts * 64);
        tmem_st_x32(taddr, raw);
        tmem_st_x32(taddr + 32, lo);
        // Release the smem slot only now: the tcgen05.st instructions above consume every loaded register, so all
        // shared-memory loads of this tile have completed (an arrive placed right after the loads could overtake
        // loads still in flight and let TMA overwrite the tile under them).
        __syncwarp();
        if (lane == 0) mbar_arrive(a_free(sa));
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(t_full(ts));
      }
      tile = tile0 + max(0, kt1 - kt0);
    }
  } else {
    // ===================== drain warps 6-9: TMEM chunk -> fp32 register accumulators -> global partial ==========
    // The tensor core adds into its fp32 accumulator with truncation; draining every TC_CHUNK K-tiles and summing the
    // chunks here with round-to-nearest keeps that bias at the level of plain fp32 arithmetic.
    const int q = warp & 3;               // TMEM lane quarter this warp may access
    constexpr int KD = Cfg::KD;
    const int c0 = (Cfg::DW == 2 && warp >= 15) ? KD : 0;     // first output column of this drain warp
    int buf = 0;
    uint32_t accphase = 0;
    constexpr int CH = 16;
    for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
      const int xb = unit % x_blocks, sp = unit / x_blocks;
      const int kt0 = sp * kt_per_split;
      const int kt1 = min(kt_total, kt0 + kt_per_split);
      const int nchunks = (kt1 - kt0 + TC_CHUNK - 1) / TC_CHUNK;
      float acc[KD];
#pragma unroll
      for (int j = 0; j < KD; ++j) acc[j] = 0.f;
      for (int c = 0; c < nchunks; ++c) {
        mbar_wait(accf_bar(buf), accphase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * N2 + c0);
        constexpr int HALF = (Cfg::DW == 2) ? 16 : ((KD >= 32) ? 32 : KD);       // columns folded per batch of loads
#pragma unroll
        for (int h0 = 0; h0 < KD; h0 += HALF) {
          uint32_t a[HALF], b[HALF];
#pragma unroll
          for (int j0 = 0; j0 < HALF; j0 += CH) {
            tmem_ld_x16(taddr + h0 + j0, *reinterpret_cast<uint32_t(*)[CH]>(&a[j0]));          // Ah*Bh
            tmem_ld_x16(taddr + K + h0 + j0, *reinterpret_cast<uint32_t(*)[CH]>(&b[j0]));      // Ah*Bl + Al*Bh
          }
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < HALF; ++j) acc[h0 + j] += __uint_as_float(a[j]) + __uint_as_float(b[j]);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(acce_bar(buf));   // TMEM buffer may be overwritten
        if (++buf == NBUF) { buf = 0; accphase ^= 1u; }
      }
      const int64_t x = (int64_t)xb * TC_BM + q * 32 + lane;
      if (x < x_len) {
        float* orow = P + (int64_t)sp * split_stride + x * K + c0;
#pragma unroll
        for (int j = 0; j < KD; j += 4)
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
// small-operand split: Bcat = [hi(B) ; B - hi(B)] with the reduced dimension contiguous (K-major)
// ---------------------------------------------------------------------------------------------------------
// AH: B = H [k x n] (already K-major)
// (k real factor rows, kp = padded count the kernel is instantiated for: rows [k, kp) of both halves stay zero)
__global__ void __launch_bounds__(256) tc_split_h_kernel(const float* __restrict__ H, int64_t ldh, float* __restrict__ Bcat,
                                                         int64_t ldb, int k, int kp, int64_t n) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)k * n) return;
  const int j = (int)(idx / n);
  const int64_t c = idx % n;
  const float h = H[(int64_t)j * ldh + c];
  const float hi = tf32_rn(h);     // nearest: the low part is then signed and half as large
  Bcat[(int64_t)j * ldb + c] = hi;
  Bcat[(int64_t)(kp + j) * ldb + c] = h - hi;
}
// WTA: B = W^T, W is [m x k]: transpose through shared memory (coalesced both ways)
__global__ void __launch_bounds__(256) tc_split_wt_kernel(const float* __restrict__ W, int64_t ldw, float* __restrict__ Bcat,
                                                          int64_t ldb, int k, int kp, int64_t m) {
  __shared__ float tile[64][65];
  const int64_t r0 = (int64_t)blockIdx.x * 64;
  for (int idx = threadIdx.x; idx < 64 * k; idx += 256) {
    const int r = idx / k, j = idx % k;
    tile[r][j] = (r0 + r < m) ? W[(r0 + r) * ldw + j] : 0.f;
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < 64 * k; idx += 256) {
    const int j = idx / 64, r = idx % 64;
    if (r0 + r < m) {
      const float w = tile[r][j];
      const float hi = tf32_rn(w);
      Bcat[(int64_t)j * ldb + r0 + r] = hi;
      Bcat[(int64_t)(kp + j) * ldb + r0 + r] = w - hi;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
    else
      cudaGetLastError();
  }
  return fn;
}

}  // namespace

int tc_padded_k(int k) { return k <= 16 ? 16 : (k <= 32 ? 32 : 64); }

TcPlan tc_plan(int64_t x_len, int64_t r_len, int k, int bk) {
  TcPlan p;
  p.x_blocks = (int)ceil_div(x_len, TC_BM);
  p.kt_total = (int)ceil_div(r_len, bk);
  const int sms = sm_count();
  // Number of K splits: units = x_blocks * splits are dealt to the CTAs round-robin (unit % grid), so the pass lasts
  // ceil(units / sms) * (tiles per unit + fill / drain of the unit's pipeline), plus the traffic of the partials every
  // split adds (written by the pass, read by the consumer).  Pick the split count that minimises that estimate instead
  // of a fixed 12 units per SM: for a short x (8192 rows on 8 GPUs: 64 x-blocks) the old rule gave 28 splits -- 8.6 % over
  // the ideal time and 28 MiB of partials -- where 9 splits are 3 % over with a third of the partial traffic.
  const int64_t kUnitOverhead = 4;                                   // tile-times to fill + drain one unit
  const double tile_bytes = (double)sms * TC_BM * TC_BK * 4.0;       // A bytes the machine streams per tile-time (128-byte
                                                                     // tile rows: 32 fp32 or 64 16-bit elements)
  const double split_cost = 2.0 * (double)x_len * k * 4.0 / tile_bytes;   // tile-times per extra split (write + read)
  int best_s = 1;
  double best = 1e300;
  for (int s = 1; s <= 32; ++s) {
    const int per_s = (int)ceil_div(p.kt_total, s);
    if (s > 1 && per_s < 16) break;                                  // >= 512 reduced elements per unit
    const int real_s = (int)ceil_div(p.kt_total, per_s);
    if (real_s != s) continue;                                       // same schedule as a smaller s
    const int64_t waves = ceil_div((int64_t)p.x_blocks * s, sms);
    const double cost = (double)waves * (double)(per_s + kUnitOverhead) + split_cost * s;
    if (cost < best - 1e-9) { best = cost; best_s = s; }
  }
  p.kt_per_split = (int)ceil_div(p.kt_total, best_s);
  p.splits = (int)ceil_div(p.kt_total, p.kt_per_split);
  p.num_units = p.x_blocks * p.splits;
  p.grid = p.num_units < sms ? p.num_units : sms;
  p.ldb = round_up(r_len, 4);
  p.bcat_bytes = round_up((int64_t)2 * k * p.ldb * 4, 1024);
  p.partial_bytes = (int64_t)p.splits * x_len * k * 4;
  return p;
}

int tc_begin(void* ws, int64_t ws_bytes, int64_t need, int64_t bcat_bytes, bool padded, cudaStream_t st) {
  if (ws == nullptr || ws_bytes < need)
    return fail(DNMF_E_WORKSPACE, "tcgen05 pass needs %lld workspace bytes, got %lld", (long long)need, (long long)ws_bytes);
  if (((uintptr_t)ws % 256) != 0) return fail(DNMF_E_ARG, "workspace must be 256-byte aligned");
  if (padded) {
    cudaError_t e = cudaMemsetAsync(ws, 0, (size_t)bcat_bytes, st);
    if (e != cudaSuccess) return cuda_fail(e, "Bcat memset");
  }
  return 0;
}

int tc_make_map(CUtensorMap* map, CUtensorMapDataType type, const void* ptr, int64_t rows, int64_t cols, int64_t ld,
                int box_cols, int box_rows, CUtensorMapSwizzle swz) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(DNMF_E_UNSUPPORTED, "cuTensorMapEncodeTiled is not available from this driver");
  const int64_t esize = type == CU_TENSOR_MAP_DATA_TYPE_FLOAT32 ? 4 : 2;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)(ld * esize)};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, type, 2, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(DNMF_E_ARG, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return 0;
}

int tc_map_a(CUtensorMap* map, const void* A, int dtype, int64_t lda, int64_t m, int64_t n, int mode) {
  const CUtensorMapDataType type = dtype == DNMF_A_F16    ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                   : dtype == DNMF_A_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                                          : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  if (mode == 1) return tc_make_map(map, type, A, m, n, lda, TC_BM, TC_BK, CU_TENSOR_MAP_SWIZZLE_NONE);
  return tc_make_map(map, type, A, m, n, lda, TC_BK, TC_BM,
                     dtype == DNMF_F32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B);
}

int tc_launch_split_h(const float* H, int64_t ldh, float* Bcat, int64_t ldb, int k, int kp, int64_t n, cudaStream_t st) {
  tc_split_h_kernel<<<(unsigned)ceil_div((int64_t)k * n, 256), 256, 0, st>>>(H, ldh, Bcat, ldb, k, kp, n);
  DNMF_LAUNCH_CHECK("tc_split_h_kernel");
  return 0;
}
int tc_launch_split_wt(const float* W, int64_t ldw, float* Bcat, int64_t ldb, int k, int kp, int64_t m, cudaStream_t st) {
  tc_split_wt_kernel<<<(unsigned)ceil_div(m, 64), 256, 0, st>>>(W, ldw, Bcat, ldb, k, kp, m);
  DNMF_LAUNCH_CHECK("tc_split_wt_kernel");
  return 0;
}

namespace {

int g_tc_usable = -1;   // -1 not probed yet, 1 the tensor core truncates tf32 operands as the splitters assume, 0 it does not
int64_t g_min_elems = -1;

template <int K, int MODE>
int launch_pass(const CUtensorMap& tmA, const CUtensorMap& tmB, float* P, int64_t split_stride, int64_t x_len,
                const TcPlan& pl, cudaStream_t st) {
  if (int rc = smem_attr_once<tc_pass_kernel<K, MODE>>(TcCfg<K>::SMEM_BYTES, "tc_pass_kernel smem attribute")) return rc;
  tc_pass_kernel<K, MODE><<<pl.grid, TcCfg<K>::THREADS, TcCfg<K>::SMEM_BYTES, st>>>(
      tmA, tmB, P, split_stride, x_len, pl.x_blocks, pl.kt_total, pl.kt_per_split, pl.num_units);
  DNMF_LAUNCH_CHECK("tc_pass_kernel");
  return 0;
}

template <int MODE>
int launch_pass_k(int k, const CUtensorMap& tmA, const CUtensorMap& tmB, float* P, int64_t split_stride, int64_t x_len,
                  const TcPlan& pl, cudaStream_t st) {
  switch (k) {
    case 16: return launch_pass<16, MODE>(tmA, tmB, P, split_stride, x_len, pl, st);
    case 32: return launch_pass<32, MODE>(tmA, tmB, P, split_stride, x_len, pl, st);
    case 64: return launch_pass<64, MODE>(tmA, tmB, P, split_stride, x_len, pl, st);
  }
  return fail(DNMF_E_UNSUPPORTED, "tcgen05 path: k must be 16, 32 or 64");
}

// ws = [Bcat | partials].  The kernels exist for 16 / 32 / 64 factor columns: smaller k ride along zero-padded.
struct FroLayout {
  TcPlan pl;
  int kp;
  int64_t total;
};
FroLayout fro_layout(int mode, int64_t m, int64_t n, int k) {
  FroLayout L;
  L.kp = tc_padded_k(k);
  L.pl = mode == 0 ? tc_plan(m, n, L.kp) : tc_plan(n, m, L.kp);
  L.total = L.pl.bcat_bytes + L.pl.partial_bytes;
  return L;
}

// V (AH, mode 0) or Y / Y^T (WTA, mode 1) through the tensor path
int tc_run(int mode, const float* A, int64_t lda, const float* B, int64_t ldbsrc, float* out, int64_t ldo,
           int64_t m, int64_t n, int k, int transposed_out, void* ws, int64_t ws_bytes, cudaStream_t st,
           TcPartials* defer) {
  const FroLayout L = fro_layout(mode, m, n, k);
  const TcPlan& pl = L.pl;
  const int64_t x_len = mode == 0 ? m : n;
  const int64_t r_len = mode == 0 ? n : m;
  if (int rc = tc_begin(ws, ws_bytes, L.total, pl.bcat_bytes, L.kp != k, st)) return rc;
  float* Bcat = reinterpret_cast<float*>(ws);
  float* P = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(ws) + pl.bcat_bytes);
  int rc = mode == 0 ? tc_launch_split_h(B, ldbsrc, Bcat, pl.ldb, k, L.kp, n, st)
                     : tc_launch_split_wt(B, ldbsrc, Bcat, pl.ldb, k, L.kp, m, st);
  if (rc) return rc;
  alignas(64) CUtensorMap tmA, tmB;
  if ((rc = tc_map_a(&tmA, A, DNMF_F32, lda, m, n, mode)) ||
      (rc = tc_make_map(&tmB, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, Bcat, 2 * L.kp, r_len, pl.ldb, TC_BK, 2 * L.kp)))
    return rc;
  const int64_t split_stride = x_len * L.kp;
  rc = mode == 0 ? launch_pass_k<0>(L.kp, tmA, tmB, P, split_stride, x_len, pl, st)
                 : launch_pass_k<1>(L.kp, tmA, tmB, P, split_stride, x_len, pl, st);
  if (rc) return rc;
  return tc_finish(P, x_len, L.kp, pl.splits, mode, k, transposed_out, out, ldo, st, defer);
}

// One-time probe: does kind::tf32 truncate the fp32 bits it reads, as the splitters assume?  A = 1 + 1.5 * 2^-11
// everywhere, H = 1: V = 32 * (1 + 1.5 * 2^-11) exactly iff the splitter's notion of A_hi matches the hardware's.
void calibrate() {
  if (g_tc_usable >= 0) return;
  g_tc_usable = 0;
  const int m = 128, n = 32, k = 16;
  const int64_t wsb = fro_layout(0, m, n, k).total;
  float *dA = nullptr, *dH = nullptr, *dV = nullptr;
  void* dws = nullptr;
  if (cudaMalloc(&dA, m * n * 4) != cudaSuccess || cudaMalloc(&dH, k * n * 4) != cudaSuccess ||
      cudaMalloc(&dV, m * k * 4) != cudaSuccess || cudaMalloc(&dws, wsb) != cudaSuccess) {
    cudaGetLastError();
    return;
  }
  const float aval = 1.0f + 1.5f * 0.00048828125f;   // 1 + 1.5 * 2^-11
  float* hA = new float[m * n];
  float* hH = new float[k * n];
  float* hV = new float[m * k];
  for (int i = 0; i < m * n; ++i) hA[i] = aval;
  for (int i = 0; i < k * n; ++i) hH[i] = 1.0f;
  cudaMemcpy(dA, hA, m * n * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dH, hH, k * n * 4, cudaMemcpyHostToDevice);
  const float expect = 32.0f * aval;
  cudaMemset(dV, 0, m * k * 4);
  const int64_t saved = tls().launches;
  const int rc = tc_run(0, dA, n, dH, n, dV, k, m, n, k, 0, dws, wsb, 0, nullptr);
  tls().launches = saved;
  if (rc != 0 || cudaDeviceSynchronize() != cudaSuccess) {
    cudaGetLastError();
  } else {
    cudaMemcpy(hV, dV, m * k * 4, cudaMemcpyDeviceToHost);
    bool ok = true;
    for (int i = 0; i < m * k; ++i) ok = ok && (hV[i] == expect);
    g_tc_usable = ok ? 1 : 0;
  }
  if (getenv("DNMF_VERBOSE")) fprintf(stderr, "[libdnmf] tcgen05 tf32 path: %s\n", g_tc_usable ? "usable" : "off");
  delete[] hA; delete[] hH; delete[] hV;
  cudaFree(dA); cudaFree(dH); cudaFree(dV); cudaFree(dws);
}

bool device_is_sm100() {
  static int cached = -1;
  if (cached < 0) {
    int dev = 0, major = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) == cudaSuccess)
      cached = (major == 10) ? 1 : 0;
    else {
      cudaGetLastError();
      cached = 0;
    }
  }
  return cached == 1;
}

}  // namespace

bool tc_eligible(int op, const void* A, int64_t lda, int64_t m, int64_t n, int64_t k, int dtype) {
  if (tls().force_generic) return false;
  const bool kl = (op == DNMF_OP_KL_UHT || op == DNMF_OP_KL_WTU);
  if (op != DNMF_OP_AH && op != DNMF_OP_WTA && !kl) return false;
  if (g_min_elems < 0) {
    const char* env = getenv("DNMF_TC_MIN_ELEMS");
    g_min_elems = env ? atoll(env) : (int64_t)1 << 20;
  }
  if (dtype == DNMF_A_F16 || dtype == DNMF_A_BF16) {
    if (k < 1 || k > 64) return false;
    if (((uintptr_t)A % 16) != 0 || (lda % 8) != 0) return false;
    if (m * n < g_min_elems || !device_is_sm100()) return false;
    // AH / WTA: the kind::f16 kernel of dnmf_tc16.cu (an exact operand, no tf32 calibration involved)
    if (!kl) return true;
    // KL: the 16-bit build of the fused KL kernel, whose two GEMMs are kind::tf32 like the fp32 path's
    calibrate();
    return g_tc_usable == 1;
  }
  if (dtype != DNMF_F32) return false;
  if (k < 1 || k > 64) return false;
  if (((uintptr_t)A % 16) != 0 || (lda % 4) != 0) return false;
  if (m * n < g_min_elems) return false;
  if (!device_is_sm100()) return false;
  calibrate();
  return g_tc_usable == 1;    // the splitters assume a truncating kind::tf32 (what B200 does); anything else: generic path
}

void tc_set_min_elems(int64_t elems) { g_min_elems = elems < 0 ? 0 : elems; }

int64_t tc_workspace_bytes(int op, int64_t m, int64_t n, int64_t k, int dtype) {
  const bool a16 = dtype == DNMF_A_F16 || dtype == DNMF_A_BF16;
  if (op == DNMF_OP_AH_RESIDUAL) return (dtype == DNMF_F32 || a16) && k <= 32 ? tc_kl_layout(3, m, n).total : 0;
  if ((dtype != DNMF_F32 && !a16) || k < 1 || k > 64) return 0;
  const int mode = (op == DNMF_OP_AH || op == DNMF_OP_KL_UHT) ? 0 : 1;
  if (op == DNMF_OP_AH || op == DNMF_OP_WTA)
    return a16 ? tc16_layout(mode, m, n, (int)k, dtype).total : fro_layout(mode, m, n, (int)k).total;
  if (op == DNMF_OP_KL_UHT || op == DNMF_OP_KL_WTU)
    return k > 32 ? tc_kl_layout_k64(mode, m, n).total : tc_kl_layout(mode, m, n).total;
  return 0;
}

int tc_pass(int op, int dtype, const void* A, int64_t lda, const float* W, int64_t ldw, const float* H, int64_t ldh,
            float* out, int64_t ldo, int64_t m, int64_t n, int k, float eps, int transposed_out, void* ws,
            int64_t ws_bytes, cudaStream_t st, TcPartials* defer) {
  const int mode = (op == DNMF_OP_AH || op == DNMF_OP_KL_UHT) ? 0 : 1;
  if (op == DNMF_OP_KL_UHT || op == DNMF_OP_KL_WTU)
    return (k > 32 ? tc_kl_run_k64 : tc_kl_run)(mode, A, dtype, lda, W, ldw, H, ldh, out, ldo, m, n, k, eps,
                                                 transposed_out, ws, ws_bytes, st, defer);
  const float* B = mode == 0 ? H : W;          // the small operand: H (AH) or W (WTA)
  const int64_t ldbsrc = mode == 0 ? ldh : ldw;
  if (dtype == DNMF_A_F16 || dtype == DNMF_A_BF16)
    return tc16_run(mode, A, lda, B, ldbsrc, out, ldo, m, n, k, transposed_out, dtype, ws, ws_bytes, st, defer);
  return tc_run(mode, (const float*)A, lda, B, ldbsrc, out, ldo, m, n, k, transposed_out, ws, ws_bytes, st, defer);
}

}  // namespace dnmf
