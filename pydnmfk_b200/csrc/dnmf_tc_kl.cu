// Fused KL contractions on the tcgen05 path (fp32 or 16-bit data, k <= 64):
//
//   UHT : V[m x k]   = (A / (W H + eps)) * H^T          (dist_nmf.py:338-339, :806,:810)
//   WTU : Y^T[n x k] = (W^T * (A / (W H + eps)))^T      (dist_nmf.py:312-313, :806,:808)
//
// W H is never materialised.  Flash-attention-like structure per 128 x 32 tile of A (x = accumulator row: a row of A
// for UHT, a column of A for WTU; r = the 32 reduced indices of the tile):
//   GEMM1  S[x, r] = Fx[x, :] . Fr[r, :]        Fx = the x-side factor block (128 x k), resident in TENSOR MEMORY
//                                                for the whole unit; Fr tile (64 x k, hi|lo) streamed by TMA
//   U[x, r] = A[x, r] / (S[x, r] + eps)          splitter warps: A tile from smem, S from TMEM (tcgen05.ld)
//   GEMM2  D[x, :] += U[x, r] . B[:, r]^T        exactly the FRO contraction with A replaced by U
// Both GEMMs use the 3-term tf32 split (see dnmf_tc.cu) so the result is fp32-accurate; U and U_lo go to the TMEM
// operand ring like A and A_lo do on the FRO path.  GEMM1 works on PAIRS of tiles (64 reduced indices): its three split
// terms are K-concatenated into ONE accumulator of N = 64 MMAs (umma_tile_cat), whose columns [0,32) hold the S tile of
// the even tile and [32,64) the odd one's.  N = 64 runs at the tensor pipe's full rate (an N = 32 MMA costs 22 cycles
// instead of 16), the splitters load 32 S columns per tile, and one S slot / one factor-tile slot serves two tiles
// (round 2: -6 % UHT / -0 % WTU isolated, -3 % sustained against two separate accumulators per tile).  The MMA warp
// issues GEMM1 ahead of GEMM2.
//
// MODE 3 (A H^T AND residual in one pass, tc_ah_residual_run; the BCD iteration's second pass, dist_nmf.py:1023-1024):
// rows of A like MODE 0, U = A itself (so GEMM2 yields V = A H^T exactly as the FRO kernel does), and the splitters
// accumulate the residual terms on the side.
//
// Warp roles (one persistent CTA per SM), see KlCfg::GROUPS:
//   KK = 32: w0-11 three splitter groups | w12-15 drain | w16 A-TMA | w17 Bcat-TMA (lane 0) + Fr-TMA (lane 1) |
//            w18 GEMM2 issuer | w19 GEMM1 issuer
//   KK = 64: w0 A-TMA | w1 GEMM2 issuer | w2-5, w11-14 two splitter groups | w6-9 drain | w10 Bcat-TMA + Fr-TMA |
//            w15 GEMM1 issuer
// Barrier waits spin on try_wait without the suspend-time hint (mbar_wait_spin, see tc_common.cuh).
//
// A 16-bit A (fp16 / bf16, DNMF_A_F16 / DNMF_A_BF16) is read in one place only: the splitters widen their row (column) of
// the smem tile to fp32 exactly, and everything after that -- U, the tf32 split, both GEMMs, the summation order -- is
// the fp32 kernel's.  A 16-bit pass is therefore bit-identical to the fp32 pass on the widened matrix; only the tile
// bytes (8 KB instead of 16 KB) and the swizzle of the MODE 0 / 3 tile (64-byte rows) differ.
#include "generic_passes.cuh"
#include "tc_common.cuh"
#include "tc_api.cuh"

namespace dnmf {
namespace {

// KL_KK: factor width this translation unit is built for.  32 (default: any k <= 32, zero-padded) or 64 (32 < k <= 64,
// dnmf_tc_kl64.cu includes this file with KL_KK = 64: two splitter groups, single-buffered accumulator, see KlCfg).
#ifndef KL_KK
#define KL_KK 32
#endif
constexpr int KK = KL_KK;         // factor width handled by this kernel
constexpr int KATOMS = KK / 32;   // 128-byte swizzle atoms along k of one factor-tile row
static_assert(KK == 32 || KK == 64, "KL_KK must be 32 or 64");
#if KL_KK == 64
#define KL_FN(name) name##_k64
#else
#define KL_FN(name) name
#endif

template <typename TA>
struct KlCfg {
  // GROUPS splitter groups of 4 warps work on tiles round-robin; the per-tile chain (A tile -> S load -> divide -> split ->
  // tensor-memory store -> GEMM2 -> slot free) is latency-bound, so the number of tiles in flight sets the pass time.
  // KK = 32: 3 groups are 10-17 % faster than 2 (profiles/r02_kl_lab.md).  KK = 64: tensor memory holds 128
  // (accumulator) + 2 x 64 (U ring) + 2 x 64 (S pair ring) + 128 (Fx) = 512 columns, which leaves room for two.
  static constexpr int GROUPS = (KK == 32) ? 3 : 2;
  static constexpr int THREADS = 512 + 128 * (GROUPS - 2);
  static constexpr int PAIRS = GROUPS * 128;         // residual pairs per CTA (one per splitter thread)
  static constexpr int CHUNK = 4;                    // K-tiles accumulated in TMEM before the drain warps fold them
  static constexpr int N2 = 2 * KK;                    // 64
  static constexpr int A_BYTES = TC_BM * TC_BK * (int)sizeof(TA);   // 16 KB fp32, 8 KB 16-bit
  static constexpr int B_BYTES = N2 * TC_BK * 4;       // 8 KB  Bcat tile  [2k][32 r]
  static constexpr int F_ROWS = 2 * TC_BK;             // reduced indices per factor tile: a pair of tiles
  static constexpr int F_ATOM_BYTES = F_ROWS * 128;    // F_ROWS rows of one 128-byte swizzle atom (32 factor columns)
  static constexpr int F_BYTES = 2 * KATOMS * F_ATOM_BYTES;   // FrCat tile [hi: KATOMS atoms | lo: KATOMS atoms]: 16 / 32 KB
  // ring depths, in tiles for every element type of A; KK = 64, fp32: 80 KB A ring + 3 x 16 KB Bcat + 2 x 32 KB FrCat
  // pairs = 192 KB
  static constexpr int SA = (KK == 32) ? 8 : 5, SB = (KK == 32) ? 4 : 3, SF = 2;
  static constexpr int NBUF = (KK == 32) ? 2 : 1, NT = (KK == 32) ? 3 : 2;
  static constexpr int NS = 2, S_COLS = 64;            // one S slot = the S tiles of a pair
  static constexpr int NSF = 2 * NS;                   // S-full barriers: pair p fills slot p % NS, signals p % NSF
  static constexpr int ACC_COL0 = 0;
  static constexpr int OP_COL0 = NBUF * N2;            // 128
  static constexpr int S_COL0 = OP_COL0 + NT * 64;
  static constexpr int FX_COL0 = S_COL0 + NS * S_COLS; // 448 (384 for KK = 64)
  static_assert(FX_COL0 + 2 * KK <= 512, "TMEM has 512 columns");
  // A splitter group waits on a full barrier by phase PARITY, which is only unambiguous while the barrier's previous
  // phase has completed.  The group knows that for every tile up to its own previous one (tile - GROUPS; GEMM1 and GEMM2
  // complete in tile order).  Operand ring: the barrier's previous use is tile - NT.  S ring: pair p's barrier was last
  // used by pair p - NSF, and the group only knows pair(tile - GROUPS) >= p - GROUPS complete: a unit of odd tile count
  // ends in a lone-tile pair, so with one-tile units every pair holds one tile.  With one full barrier per S slot
  // (NSF = NS = 2, 3 groups) such units let a group pass the wait for pair p while pair p - 2 was still outstanding and
  // read the S tile of pair p - 4 (tall UHT / residual passes with n <= 32, WTU with m <= 32).  Too shallow a ring also
  // hangs (observed with one S slot per tile, NS = 2 and 3 groups).
  static_assert(NSF >= GROUPS && NT >= GROUPS, "S barriers and operand ring too shallow for the splitter groups");
  static constexpr int NBARS = 2 * SA + 2 * SB + 2 * SF + 2 * NT + NSF + NS + 2 * NBUF + 2;
  static constexpr int BAR_BYTES = 1024;
  static_assert((NBARS + 1) * 8 <= BAR_BYTES, "barrier area too small");
  static constexpr int SMEM_BYTES = SA * A_BYTES + SB * B_BYTES + SF * F_BYTES + 1024 + BAR_BYTES;
  static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB opt-in shared memory limit");
};

// fp32 bits of a 16-bit element of A (fp16 or bf16; both widen exactly)
template <typename TA>
__device__ __forceinline__ uint32_t widen_bits(uint32_t b) {
  if constexpr (std::is_same<TA, __half>::value) return __float_as_uint(__half2float(__ushort_as_half((unsigned short)b)));
  else return b << 16;
}

// MODE 0 (UHT): x = rows of A, A tile = TMA box {32 cols, 128 rows} with 128B swizzle (64B for a 16-bit A), Fx = W rows
// MODE 1 (WTU): x = columns of A, A tile = TMA box {128 cols, 32 rows} unswizzled,                      Fx = H^T rows
// TA: element type of A (float, __half, __nv_bfloat16)
template <int MODE, typename TA>
__global__ void __launch_bounds__(KlCfg<TA>::THREADS, 1)
tc_kl_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
             const __grid_constant__ CUtensorMap tmF, const float* __restrict__ Fx, int64_t ldfx, int64_t fr_rows_pad,
             float* __restrict__ P, int64_t split_stride, int64_t x_len, int x_blocks, int kt_total, int kt_per_split,
             int num_units, int k_real, float eps, double* __restrict__ pairs_out) {
  using Cfg = KlCfg<TA>;
  constexpr int SA = Cfg::SA, SB = Cfg::SB, SF = Cfg::SF, NT = Cfg::NT, NS = Cfg::NS, NSF = Cfg::NSF, NBUF = Cfg::NBUF;
  constexpr int N2 = Cfg::N2;
  constexpr int GROUPS = Cfg::GROUPS, CHUNK = Cfg::CHUNK;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sA0 = base, sB0 = sA0 + SA * Cfg::A_BYTES, sF0 = sB0 + SB * Cfg::B_BYTES;
  const uint32_t bars = sF0 + SF * Cfg::F_BYTES;
  int bi = 0;
  const int iAF = bi; bi += SA;  const int iAE = bi; bi += SA;
  const int iBF = bi; bi += SB;  const int iBE = bi; bi += SB;
  const int iFF = bi; bi += SF;  const int iFE = bi; bi += SF;
  const int iTF = bi; bi += NT;  const int iTE = bi; bi += NT;
  const int iSF = bi; bi += NSF; const int iSE = bi; bi += NS;
  const int iCF = bi; bi += NBUF; const int iCE = bi; bi += NBUF;
  const int iXF = bi; bi += 1;   const int iXE = bi; bi += 1;
  const int iSLOT = bi;
  auto bar = [&](int idx) { return bars + 8u * idx; };
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(
      base_ptr + SA * Cfg::A_BYTES + SB * Cfg::B_BYTES + SF * Cfg::F_BYTES + 8 * iSLOT);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmF);
    for (int s = 0; s < SA; ++s) { mbar_init(bar(iAF + s), 1); mbar_init(bar(iAE + s), 4); }
    for (int s = 0; s < SB; ++s) { mbar_init(bar(iBF + s), 1); mbar_init(bar(iBE + s), 1); }
    for (int s = 0; s < SF; ++s) { mbar_init(bar(iFF + s), 1); mbar_init(bar(iFE + s), 1); }
    for (int s = 0; s < NT; ++s) { mbar_init(bar(iTF + s), 4); mbar_init(bar(iTE + s), 1); }
    for (int s = 0; s < NSF; ++s) mbar_init(bar(iSF + s), 1);
    for (int s = 0; s < NS; ++s) mbar_init(bar(iSE + s), 8);
    for (int b = 0; b < NBUF; ++b) { mbar_init(bar(iCF + b), 1); mbar_init(bar(iCE + b), 4); }
    mbar_init(bar(iXF), 4);
    mbar_init(bar(iXE), 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(bar(iSLOT), 512);      // (allocation and release by the same warp; any role)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  // Warp-role placement.  The SM's issue arbiter prefers the higher warp id, and setmaxnreg moves registers per warpgroup.
  // With three splitter groups the CTA has 640 threads = 96 registers per thread at launch; the producer / issuer
  // warpgroup needs far fewer and hands the rest to the splitter warpgroups (setmaxnreg works per warpgroup, hence the
  // warpgroup-aligned roles, control at the top).  setmaxnreg.inc can only draw on what the CTA's own warpgroups released
  // (the CTA's pool is its launch allocation, 640 x 96): 4 x 32 + 4 x 80 + 12 x 120 registers x 32 lanes = 60416 <= 61440.
  // With two groups (KK = 64) the round-1 placement stays, without register moves.
  constexpr bool WG_ALIGNED = (GROUPS == 3);
  constexpr int W_CTRL0 = 4 * GROUPS + 4;
  constexpr int W_APROD = WG_ALIGNED ? W_CTRL0 : 0, W_BPROD = WG_ALIGNED ? W_CTRL0 + 1 : 10;
  constexpr int W_G1 = WG_ALIGNED ? W_CTRL0 + 3 : 15;    // GEMM2 issuer: the remaining control warp (W_CTRL0 + 2 or 1)
  const bool is_ctrl = WG_ALIGNED ? warp >= W_CTRL0 : (warp < 2 || warp == W_BPROD || warp == W_G1);
  const bool is_split = WG_ALIGNED ? warp < 4 * GROUPS : ((warp >= 2 && warp < 6) || (warp >= 11 && warp < 15));
  const int split_group = WG_ALIGNED ? warp >> 2 : (warp >= 11 ? 1 : 0);
  if (is_ctrl) {
  if constexpr (WG_ALIGNED) asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");
  if (warp == W_APROD) {
    // ===================== A producer =====================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
        const int xb = unit % x_blocks, sp = unit / x_blocks;
        const int kt0 = sp * kt_per_split, kt1 = min(kt_total, kt0 + kt_per_split);
        for (int kt = kt0; kt < kt1; ++kt) {
          mbar_wait_spin(bar(iAE + s), ph ^ 1u);
          mbar_expect_tx(bar(iAF + s), Cfg::A_BYTES);
          if (MODE != 1) tma_load_2d(sA0 + s * Cfg::A_BYTES, &tmA, bar(iAF + s), kt * TC_BK, xb * TC_BM);
          else tma_load_2d(sA0 + s * Cfg::A_BYTES, &tmA, bar(iAF + s), xb * TC_BM, kt * TC_BK);
          if (++s == SA) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == W_BPROD) {
    // ===================== Bcat producer (lane 0, GEMM2 B operand) and FrCat producer (lane 1, GEMM1 B operand) =====
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
        const int sp = unit / x_blocks;
        const int kt0 = sp * kt_per_split, kt1 = min(kt_total, kt0 + kt_per_split);
        for (int kt = kt0; kt < kt1; ++kt) {
          mbar_wait_spin(bar(iBE + s), ph ^ 1u);
          mbar_expect_tx(bar(iBF + s), Cfg::B_BYTES);
          tma_load_2d(sB0 + s * Cfg::B_BYTES, &tmB, bar(iBF + s), kt * TC_BK, 0);
          if (++s == SB) { s = 0; ph ^= 1u; }
        }
      }
    } else if (lane == 1) {
      // hi rows then lo rows of the 64 reduced indices of a PAIR of K tiles (the TMA box has 64 rows)
      int s = 0;
      uint32_t ph = 0;
      for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
        const int sp = unit / x_blocks;
        const int kt0 = sp * kt_per_split, kt1 = min(kt_total, kt0 + kt_per_split);
        for (int kt = kt0; kt < kt1; kt += 2) {
          mbar_wait_spin(bar(iFE + s), ph ^ 1u);
          mbar_expect_tx(bar(iFF + s), Cfg::F_BYTES);
#pragma unroll
          for (int a = 0; a < KATOMS; ++a) {      // one TMA box per 128-byte swizzle atom along k
            tma_load_2d(sF0 + s * Cfg::F_BYTES + a * Cfg::F_ATOM_BYTES, &tmF, bar(iFF + s), a * 32, kt * TC_BK);
            tma_load_2d(sF0 + s * Cfg::F_BYTES + Cfg::F_BYTES / 2 + a * Cfg::F_ATOM_BYTES, &tmF, bar(iFF + s), a * 32,
                        (int)fr_rows_pad + kt * TC_BK);
          }
          if (++s == SF) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == W_G1) {
    // ===================== GEMM1 issuer: S = Fx . Fr^T on tile pairs, runs ahead of GEMM2 by up to NS pairs ==========
    //   cols [0,64) = Fx_hi*Fr_hi + Fx_hi*Fr_lo + Fx_lo*Fr_hi
    constexpr uint32_t idesc_pair = make_idesc(64, 0);      // N = 64 reduced indices
    int sf = 0, ss = 0, sfull = 0;
    uint32_t pf = 0, ps = 0, pxu = 0;
    const uint32_t fx_tmem = tmem_base + (uint32_t)Cfg::FX_COL0;
    for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
      const int sp = unit / x_blocks;
      const int kt0 = sp * kt_per_split, kt1 = min(kt_total, kt0 + kt_per_split);
      const int ntiles = kt1 - kt0;
      mbar_wait_spin(bar(iXF), pxu);                     // this unit's Fx block is in tensor memory
      for (int j = 0; j < ntiles; j += 2) {
        mbar_wait_spin(bar(iFF + sf), pf);
        mbar_wait_spin(bar(iSE + ss), ps ^ 1u);
        tc_fence_after();
        if constexpr (KK == 64)
          umma_tile_cat64(tmem_base + (uint32_t)(Cfg::S_COL0 + ss * Cfg::S_COLS), fx_tmem,
                          make_smem_desc(sF0 + sf * Cfg::F_BYTES, 16, 1024), idesc_pair,
                          bar(iSF + sfull), bar(iFE + sf), bar(iXE), (j + 2 >= ntiles) ? 1u : 0u);
        else
          umma_tile_cat<64>(tmem_base + (uint32_t)(Cfg::S_COL0 + ss * Cfg::S_COLS), fx_tmem,
                            make_smem_desc(sF0 + sf * Cfg::F_BYTES, 16, 1024), idesc_pair,
                            bar(iSF + sfull), bar(iFE + sf), bar(iXE), (j + 2 >= ntiles) ? 1u : 0u);
        if (++sf == SF) { sf = 0; pf ^= 1u; }
        if (++ss == NS) { ss = 0; ps ^= 1u; }
        if (++sfull == NSF) sfull = 0;
        __syncwarp();
      }
      pxu ^= 1u;
    }
  } else {
    // ===================== GEMM2 issuer (converged warp, elected lane inside the asm block) ======================
    constexpr uint32_t idesc_full = make_idesc(N2, 0);
    constexpr uint32_t idesc_half = make_idesc(KK, 0);
    int sb = 0, ts = 0, buf = 0;
    uint32_t pb = 0, pt = 0, accphase = 0;
    for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
      const int sp = unit / x_blocks;
      const int kt0 = sp * kt_per_split, kt1 = min(kt_total, kt0 + kt_per_split);
      const int ntiles = kt1 - kt0;
      for (int i = 0; i < ntiles; ++i) {
        const int in_chunk = i % CHUNK;
        if (in_chunk == 0) mbar_wait_spin(bar(iCE + buf), accphase ^ 1u);
        mbar_wait_spin(bar(iTF + ts), pt);
        mbar_wait_spin(bar(iBF + sb), pb);
        tc_fence_after();
        const bool chunk_end = (in_chunk == CHUNK - 1) || (i == ntiles - 1);
        umma_tile_ts<KK>(tmem_base + (uint32_t)(Cfg::ACC_COL0 + buf * N2), tmem_base + (uint32_t)(Cfg::OP_COL0 + ts * 64),
                         make_smem_desc(sB0 + sb * Cfg::B_BYTES, 16, 1024), in_chunk > 0 ? 1u : 0u, idesc_full, idesc_half,
                         bar(iTE + ts), bar(iCF + buf), chunk_end ? 1u : 0u);
        if (++ts == NT) { ts = 0; pt ^= 1u; }
        if (++sb == SB) { sb = 0; pb ^= 1u; }
        if (chunk_end) { if (++buf == NBUF) { buf = 0; accphase ^= 1u; } }
        __syncwarp();
      }
    }
  }
  } else if (is_split) {
    if constexpr (WG_ALIGNED) asm volatile("setmaxnreg.inc.sync.aligned.u32 120;");
    // ===================== splitters: A tile + S tile -> U = A / (S + eps) -> {U, U_lo} in TMEM ====================
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const int group = split_group;
    int tile = 0;
    int pair_base = 0;                      // tile pairs of the units this CTA has finished
    uint32_t pxe = 0;
    double res_sum = 0.0, a_sum = 0.0;      // MODE 3 only
    for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
      const int xb = unit % x_blocks, sp = unit / x_blocks;
      const int kt0 = sp * kt_per_split, kt1 = min(kt_total, kt0 + kt_per_split);
      if (group == 0) {
        // x-side factor row of this thread -> tensor memory (hi | lo), once per unit
        mbar_wait_spin(bar(iXE), pxe ^ 1u);              // the previous unit's GEMM1s have finished reading Fx
        tc_fence_after();
        const int64_t x = (int64_t)xb * TC_BM + r;
        const float* frow = Fx + x * ldfx;
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)Cfg::FX_COL0;
#pragma unroll
        for (int c0 = 0; c0 < KK; c0 += 32) {       // hi columns [0, KK), lo columns [KK, 2 KK), 32 at a time
          uint32_t hi[32], lo[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float w = (x < x_len && c0 + j < k_real) ? frow[c0 + j] : 0.f;      // factor columns beyond k: zero padding
            const float h = tf32_rn(w);
            hi[j] = __float_as_uint(h);
            lo[j] = __float_as_uint(tf32_round_up(w - h));
          }
          tmem_st_x32(taddr + c0, hi);
          tmem_st_x32(taddr + KK + c0, lo);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(iXF));
        pxe ^= 1u;
      }
      // this group's tiles of the unit, stepping by the group count (the walk over every tile with a modulo test per
      // tile cost 10 % of the kernel's warp samples, profiles/r02_ncu_source_hotspots.txt)
      const int tile0 = tile;
      int first = group - tile0 % GROUPS;
      if (first < 0) first += GROUPS;
      for (int kt = kt0 + first; kt < kt1; kt += GROUPS) {
        tile = tile0 + (kt - kt0);
        const int sa = tile % SA, ts = tile % NT;
        const uint32_t pa = (uint32_t)(tile / SA) & 1u, pt = (uint32_t)(tile / NT) & 1u;
        // S slots hold PAIRS of tiles: pair index inside this CTA's sequence, which half of the slot is this tile's, and
        // whether the tile has no partner (odd tile count of the unit: it then releases the slot for both)
        const int jt = kt - kt0;
        const uint32_t pairid = (uint32_t)(pair_base + (jt >> 1));
        const int ss = (int)(pairid % NS), s_half = jt & 1;
        const int sfull = (int)(pairid % NSF);
        const uint32_t psf = (pairid / NSF) & 1u;
        const bool s_lone = (s_half == 0) && (kt == kt1 - 1);
        mbar_wait_spin(bar(iAF + sa), pa);
        const uint8_t* tl = base_ptr + sa * Cfg::A_BYTES;
        uint32_t u[32], lo[32];
        if constexpr (sizeof(TA) == 4) {
          if (MODE != 1) {
            const uint8_t* row = tl + r * 128;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              const uint4 v = *reinterpret_cast<const uint4*>(row + ((c ^ (r & 7)) << 4));
              u[4 * c + 0] = v.x; u[4 * c + 1] = v.y; u[4 * c + 2] = v.z; u[4 * c + 3] = v.w;
            }
          } else {
            const uint8_t* col = tl + r * 4;
#pragma unroll
            for (int j = 0; j < 32; ++j) u[j] = *reinterpret_cast<const uint32_t*>(col + j * 512);
          }
        } else {
          // 16-bit A, widened to fp32 exactly (u then holds the bits of A16.float())
          if (MODE != 1) {
            // row r = 64 contiguous bytes, 16-byte chunk c stored at position c ^ ((r >> 1) & 3)  (SWIZZLE_64B): the
            // eight threads of a quarter warp cover all 32 banks, as the fp32 read does
            const uint8_t* row = tl + r * 64;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const uint4 v = *reinterpret_cast<const uint4*>(row + ((c ^ ((r >> 1) & 3)) << 4));
              const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                u[8 * c + 2 * e] = widen_bits<TA>(w[e] & 0xFFFFu);
                u[8 * c + 2 * e + 1] = widen_bits<TA>(w[e] >> 16);
              }
            }
          } else {
            const uint8_t* col = tl + r * 2;
#pragma unroll
            for (int j = 0; j < 32; ++j) u[j] = widen_bits<TA>(*reinterpret_cast<const uint16_t*>(col + j * 256));
          }
        }
        // S tile of this accumulator row
        mbar_wait_spin(bar(iSF + sfull), psf);
        tc_fence_after();
        const uint32_t saddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(Cfg::S_COL0 + ss * Cfg::S_COLS + s_half * 32);
        {
          uint32_t s0[32];
          tmem_ld_x32(saddr, s0);         // Fx_hi * Fr_hi + Fx_hi * Fr_lo + Fx_lo * Fr_hi
          tmem_ld_wait();
          if (MODE == 3) {
            // residual: this row's 32 elements of (A - W H)^2 and A^2, fp32 within the tile, float64 across tiles
            float t_res = 0.f, t_a = 0.f;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const float a = __uint_as_float(u[j]);
              const float d = a - __uint_as_float(s0[j]);
              t_res = fmaf(d, d, t_res);
              t_a = fmaf(a, a, t_a);
            }
            res_sum += (double)t_res;
            a_sum += (double)t_a;
          }
          // U = A / (S + eps), two elements per FADD2 / FMUL2 (sm_100 packed fp32).  den >= eps > 0 and far from
          // overflow: one MUFU.RCP (1 ulp) and one multiply, no range handling.  The rounding errors of the 65536
          // quotients of a row are independent and average out in the contraction.
#pragma unroll
          for (int j = 0; MODE != 3 && j < 32; j += 2) {
            const float2 den = __fadd2_rn(make_float2(__uint_as_float(s0[j]), __uint_as_float(s0[j + 1])), make_float2(eps, eps));
            const float2 q2 = make_float2(rcp_approx(den.x), rcp_approx(den.y));
            const float2 uu = __fmul2_rn(make_float2(__uint_as_float(u[j]), __uint_as_float(u[j + 1])), q2);
            u[j] = __float_as_uint(uu.x);
            u[j + 1] = __float_as_uint(uu.y);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(bar(iSE + ss));                       // S slot may be overwritten
          if (s_lone) mbar_arrive(bar(iSE + ss));           // ... on behalf of the missing odd tile as well
        }
#pragma unroll
        for (int j = 0; j < 32; j += 2) tf32_lo_bits2(u[j], u[j + 1], lo[j], lo[j + 1]);
        mbar_wait_spin(bar(iTE + ts), pt ^ 1u);
        // GEMM2 of tile (tile - NT) has completed (this operand slot is free again): so is that tile's Bcat slot
        if (q == 0 && lane == 0 && tile >= NT) mbar_arrive(bar(iBE + (tile - NT) % SB));
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(Cfg::OP_COL0 + ts * 64);
        tmem_st_x32(taddr, u);
        tmem_st_x32(taddr + 32, lo);
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(iAE + sa));          // smem tile fully consumed (see dnmf_tc.cu)
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(iTF + ts));
      }
      tile = tile0 + max(0, kt1 - kt0);
      pair_base += (kt1 - kt0 + 1) >> 1;
    }
    if (MODE == 3) {
      // one (residual, norm) pair per splitter thread; summed in a fixed order by the caller
      double* pairs = pairs_out + ((int64_t)blockIdx.x * Cfg::PAIRS + (group * 4 + q) * 32 + lane) * 2;
      pairs[0] = res_sum;
      pairs[1] = a_sum;
    }
  } else {
    if constexpr (WG_ALIGNED) asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
    // ===================== drain warps =====================
    const int q = warp & 3;
    int buf = 0;
    uint32_t accphase = 0;
    for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
      const int xb = unit % x_blocks, sp = unit / x_blocks;
      const int kt0 = sp * kt_per_split, kt1 = min(kt_total, kt0 + kt_per_split);
      const int nchunks = (kt1 - kt0 + CHUNK - 1) / CHUNK;
      float acc[KK];
#pragma unroll
      for (int j = 0; j < KK; ++j) acc[j] = 0.f;
      for (int c = 0; c < nchunks; ++c) {
        mbar_wait_spin(bar(iCF + buf), accphase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(Cfg::ACC_COL0 + buf * N2);
        constexpr int DCH = (KK > 32) ? 16 : KK;      // columns folded per batch of loads (register budget at KK = 64)
#pragma unroll
        for (int h0 = 0; h0 < KK; h0 += DCH) {
          uint32_t a[DCH], b[DCH];
#pragma unroll
          for (int j0 = 0; j0 < DCH; j0 += 16) {
            tmem_ld_x16(taddr + h0 + j0, *reinterpret_cast<uint32_t(*)[16]>(&a[j0]));
            tmem_ld_x16(taddr + KK + h0 + j0, *reinterpret_cast<uint32_t(*)[16]>(&b[j0]));
          }
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < DCH; ++j) acc[h0 + j] += __uint_as_float(a[j]) + __uint_as_float(b[j]);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(iCE + buf));
        if (++buf == NBUF) { buf = 0; accphase ^= 1u; }
      }
      const int64_t x = (int64_t)xb * TC_BM + q * 32 + lane;
      if (x < x_len) {
        float* orow = P + (int64_t)sp * split_stride + x * KK;
#pragma unroll
        for (int j = 0; j < KK; j += 4)
          *reinterpret_cast<float4*>(orow + j) = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// FrCat = [hi(F) ; lo(F)] for an r-side factor given as F[r][k] (rows = reduced indices), each half padded to r_pad rows
// TRANS: the source is H [k x r] (row-major) and is transposed on the fly.
template <bool TRANS>
__global__ void __launch_bounds__(256) kl_split_fr_kernel(const float* __restrict__ src, int64_t lds, float* __restrict__ FrCat,
                                                          int64_t r_len, int64_t r_pad, int k) {
  __shared__ float tile[64][KK + 1];
  const int64_t r0 = (int64_t)blockIdx.x * 64;
  if (TRANS) {
    for (int idx = threadIdx.x; idx < 64 * k; idx += 256) {
      const int j = idx / 64, r = idx % 64;                 // coalesced along r
      tile[r][j] = (r0 + r < r_len) ? src[(int64_t)j * lds + r0 + r] : 0.f;
    }
  } else {
    for (int idx = threadIdx.x; idx < 64 * k; idx += 256) {
      const int r = idx / k, j = idx % k;
      tile[r][j] = (r0 + r < r_len) ? src[(r0 + r) * lds + j] : 0.f;
    }
  }
  __syncthreads();
  // rows of KK entries: the k real factor columns, then zero padding
  for (int idx = threadIdx.x; idx < 64 * KK; idx += 256) {
    const int r = idx / KK, j = idx % KK;
    if (r0 + r < r_pad) {
      const float w = j < k ? tile[r][j] : 0.f;
      const float hi = tf32_rn(w);
      FrCat[(r0 + r) * KK + j] = hi;
      FrCat[(r_pad + r0 + r) * KK + j] = tf32_round_up(w - hi);
    }
  }
}

// Ht[c][j] = H[j][c] for j < k, 0 for k <= j < KK
__global__ void __launch_bounds__(256) kl_transpose_kernel(const float* __restrict__ H, int64_t ldh, float* __restrict__ Ht,
                                                           int64_t n, int k) {
  __shared__ float tile[64][KK + 1];
  const int64_t c0 = (int64_t)blockIdx.x * 64;
  for (int idx = threadIdx.x; idx < 64 * k; idx += 256) {
    const int j = idx / 64, c = idx % 64;
    tile[c][j] = (c0 + c < n) ? H[(int64_t)j * ldh + c0 + c] : 0.f;
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < 64 * KK; idx += 256) {
    const int c = idx / KK, j = idx % KK;
    if (c0 + c < n) Ht[(c0 + c) * KK + j] = j < k ? tile[c][j] : 0.f;
  }
}

template <int MODE, typename TA>
int kl_launch(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmF, const float* Fx, int64_t ldfx,
              const KlLayout& L, float* P, int64_t x_len, int k_real, float eps, double* pairs, cudaStream_t st) {
  using Cfg = KlCfg<TA>;
  if (int rc = smem_attr_once<tc_kl_kernel<MODE, TA>>(Cfg::SMEM_BYTES, "tc_kl_kernel smem attribute")) return rc;
  tc_kl_kernel<MODE, TA><<<L.pl.grid, Cfg::THREADS, Cfg::SMEM_BYTES, st>>>(
      tmA, tmB, tmF, Fx, ldfx, L.r_pad, P, x_len * KK, x_len, L.pl.x_blocks, L.pl.kt_total, L.pl.kt_per_split,
      L.pl.num_units, k_real, eps, pairs);
  DNMF_LAUNCH_CHECK("tc_kl_kernel");
  return 0;
}

// the instantiation for A's storage type (dtype: DNMF_F32, DNMF_A_F16 or DNMF_A_BF16)
template <int MODE>
int kl_launch_a(int dtype, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmF, const float* Fx,
                int64_t ldfx, const KlLayout& L, float* P, int64_t x_len, int k_real, float eps, double* pairs,
                cudaStream_t st) {
  switch (dtype) {
    case DNMF_F32: return kl_launch<MODE, float>(tmA, tmB, tmF, Fx, ldfx, L, P, x_len, k_real, eps, pairs, st);
    case DNMF_A_F16: return kl_launch<MODE, __half>(tmA, tmB, tmF, Fx, ldfx, L, P, x_len, k_real, eps, pairs, st);
    case DNMF_A_BF16: return kl_launch<MODE, __nv_bfloat16>(tmA, tmB, tmF, Fx, ldfx, L, P, x_len, k_real, eps, pairs, st);
  }
  return fail(DNMF_E_UNSUPPORTED, "tcgen05 KL path: no kernel for dtype %d", dtype);
}

}  // namespace

// every size is for the padded factor width KK
KlLayout KL_FN(tc_kl_layout)(int mode, int64_t m, int64_t n) {
  KlLayout L;
  const int64_t x_len = mode == 1 ? n : m, r_len = mode == 1 ? m : n;
  L.pl = tc_plan(x_len, r_len, KK);
  L.r_pad = round_up(r_len, 64);
  L.frcat_bytes = round_up(2 * L.r_pad * KK * 4, 1024);
  L.ht_bytes = mode == 3 ? 0 : round_up(n * (int64_t)KK * 4, 1024);      // plain H^T (Fx of WTU)
  L.pairs_bytes = mode == 3 ? round_up((int64_t)L.pl.grid * KlCfg<float>::PAIRS * 2 * (int64_t)sizeof(double), 1024) : 0;
  L.total = L.pl.bcat_bytes + L.frcat_bytes + L.ht_bytes + L.pl.partial_bytes + L.pairs_bytes;
  return L;
}

// The kernel is written for KK factor columns; smaller k ride along zero-padded (zero columns of W / rows of H add nothing
// to S = W H, and their output columns are dropped by the final reduction).
int KL_FN(tc_kl_run)(int mode, const void* A, int dtype, int64_t lda, const float* W, int64_t ldw, const float* H,
                     int64_t ldh, float* out, int64_t ldo, int64_t m, int64_t n, int k, float eps, int transposed_out,
                     void* ws, int64_t ws_bytes, cudaStream_t st, TcPartials* defer) {
  if (k < 1 || k > KK) return fail(DNMF_E_UNSUPPORTED, "tcgen05 KL path: k must be in [1, %d]", KK);
  const KlLayout L = KL_FN(tc_kl_layout)(mode, m, n);
  const TcPlan& pl = L.pl;
  const int64_t x_len = mode == 1 ? n : m, r_len = mode == 1 ? m : n;
  if (int rc = tc_begin(ws, ws_bytes, L.total, pl.bcat_bytes, k != KK, st)) return rc;
  uint8_t* wsb = reinterpret_cast<uint8_t*>(ws);
  float* Bcat = reinterpret_cast<float*>(wsb);
  float* FrCat = reinterpret_cast<float*>(wsb + pl.bcat_bytes);
  float* Ht = reinterpret_cast<float*>(wsb + pl.bcat_bytes + L.frcat_bytes);
  float* P = reinterpret_cast<float*>(wsb + pl.bcat_bytes + L.frcat_bytes + L.ht_bytes);
  double* pairs = mode == 3 ? reinterpret_cast<double*>(wsb + L.total - L.pairs_bytes) : nullptr;
  const unsigned fr_blocks = (unsigned)ceil_div(L.r_pad, 64);
  const float* Fx;
  int64_t ldfx;
  int rc;
  if (mode != 1) {
    // UHT (and mode 3): GEMM2 B = split(H); GEMM1 r-side factor = H^T rows (columns of A); x-side factor = W rows
    if ((rc = tc_launch_split_h(H, ldh, Bcat, pl.ldb, k, KK, n, st))) return rc;
    kl_split_fr_kernel<true><<<fr_blocks, 256, 0, st>>>(H, ldh, FrCat, r_len, L.r_pad, k);
    DNMF_LAUNCH_CHECK("kl_split_fr_kernel<T>");
    Fx = W;
    ldfx = ldw;
  } else {
    // WTU: GEMM2 B = split(W^T); GEMM1 r-side factor = W rows; x-side factor = H^T rows (columns of A)
    if ((rc = tc_launch_split_wt(W, ldw, Bcat, pl.ldb, k, KK, m, st))) return rc;
    kl_split_fr_kernel<false><<<fr_blocks, 256, 0, st>>>(W, ldw, FrCat, r_len, L.r_pad, k);
    DNMF_LAUNCH_CHECK("kl_split_fr_kernel<N>");
    kl_transpose_kernel<<<(unsigned)ceil_div(n, 64), 256, 0, st>>>(H, ldh, Ht, n, k);    // H^T [n x KK], zero padded
    DNMF_LAUNCH_CHECK("kl_transpose_kernel");
    Fx = Ht;
    ldfx = KK;
  }
  alignas(64) CUtensorMap tmA, tmB, tmF;
  if ((rc = tc_map_a(&tmA, A, dtype, lda, m, n, mode)) ||
      (rc = tc_make_map(&tmB, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, Bcat, 2 * KK, r_len, pl.ldb, TC_BK, 2 * KK)) ||
      (rc = tc_make_map(&tmF, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, FrCat, 2 * L.r_pad, KK, KK, 32, KlCfg<float>::F_ROWS)))
    return rc;
  // (for UHT the x-side factor rows are read straight from W with its own leading dimension: only k_real columns exist)
  const int k_real = mode == 1 ? KK : k;
  switch (mode) {
    case 0: rc = kl_launch_a<0>(dtype, tmA, tmB, tmF, Fx, ldfx, L, P, x_len, k_real, eps, pairs, st); break;
    case 1: rc = kl_launch_a<1>(dtype, tmA, tmB, tmF, Fx, ldfx, L, P, x_len, k_real, eps, pairs, st); break;
#if KL_KK == 32      // the residual variant (BCD, k <= 32) exists in the 32-wide build only
    case 3: rc = kl_launch_a<3>(dtype, tmA, tmB, tmF, Fx, ldfx, L, P, x_len, k_real, eps, pairs, st); break;
#endif
    default: return fail(DNMF_E_UNSUPPORTED, "tcgen05 KL path: no kernel for mode %d", mode);
  }
  if (rc) return rc;
  return tc_finish(P, x_len, KK, pl.splits, mode == 1 ? 1 : 0, k, transposed_out, out, ldo, st, defer);
}

#if KL_KK == 32
// ---- V = A H^T together with ||A - W H||^2 and ||A||^2 in ONE pass over A (MODE 3) -------------------------------------
int tc_ah_residual_run(const void* A, int dtype, int64_t lda, const float* W, int64_t ldw, const float* H, int64_t ldh,
                       float* V, int64_t ldv, int64_t m, int64_t n, int k, void* ws, int64_t ws_bytes, double** out_pairs,
                       int64_t* n_pairs, cudaStream_t st) {
  if (int rc = tc_kl_run(3, A, dtype, lda, W, ldw, H, ldh, V, ldv, m, n, k, 0.f, 0, ws, ws_bytes, st, nullptr)) return rc;
  const KlLayout L = tc_kl_layout(3, m, n);
  *out_pairs = reinterpret_cast<double*>(reinterpret_cast<uint8_t*>(ws) + L.total - L.pairs_bytes);
  *n_pairs = (int64_t)L.pl.grid * KlCfg<float>::PAIRS;
  return 0;
}
#endif  // KL_KK == 32

}  // namespace dnmf
