// Shared device-side PTX wrappers and host-side helpers of the tcgen05 / TMA / TMEM kernels
// (dnmf_tc.cu: FRO contractions, dnmf_tc_kl.cu: fused KL contractions).
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace dnmf {

constexpr int TC_BM = 128;      // outer tile (rows of A for AH/UHT, columns of A for WTA/WTU) = UMMA M
constexpr int TC_BK = 32;       // reduced-dimension tile: 32 fp32 = one 128-byte swizzle row = 4 UMMA K steps

namespace {

// ---------------------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Blocking wait.  try_wait suspends the warp in hardware until the phase completes or a time limit expires; with the
// default limit the waiting roles (producers, issuers, drain warps) re-issued YIELD / TRYWAIT / BRA triplets often enough
// to make up 28 % of all executed warp instructions of the KL pass (ncu source page, round 1).  The explicit
// suspend-time hint keeps a waiting warp parked until the barrier actually flips.
#ifndef DNMF_WAIT_HINT
#define DNMF_WAIT_HINT 1
#endif
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
#if DNMF_WAIT_HINT
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}"
      ::"r"(bar), "r"(parity), "r"(0x989680u)
      : "memory");
#else
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
#endif
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// DRAM -> L2 only: issued TC_PF tiles ahead of the shared-memory ring so that the ring's own loads find their tile
// in L2.  The A ring holds 6-9 tiles (96-144 KB) per SM; at the loaded DRAM latency that many bytes in flight cap a
// pass near 8.7 TB/s of TMA traffic whatever the kernel computes (round-2 ablations: removing every MMA or all of the
// splitter arithmetic left the pass time unchanged).  Prefetching decouples the DRAM latency from the ring depth.
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* map, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(map), "r"(c0), "r"(c1) : "memory");
}
#ifndef TC_PF_DEFAULT
#define TC_PF_DEFAULT 0
#endif
// prefetch distance in tiles from the debug word (bits 8-15: 0 = default, v = v - 1 tiles)
__device__ __forceinline__ int tc_pf_dist(int dbg) {
  const int v = (dbg >> 8) & 0xFF;
  return v ? v - 1 : TC_PF_DEFAULT;
}
// XOR of a tile row held in registers.  Reading every register makes the warp wait for the shared-memory loads that
// fill them, so the A slot can be handed back to TMA right afterwards (instead of after the tensor-memory store
// that consumes the registers much later); the value is folded into the barrier address through a mask that is zero at
// run time but opaque to the compiler.
__device__ __forceinline__ uint32_t xor_all(const uint32_t (&r)[32]) {
  uint32_t x = 0;
#pragma unroll
  for (int j = 0; j < 32; ++j) x ^= r[j];
  return x;
}
#ifndef TC_EARLY_RELEASE
#define TC_EARLY_RELEASE 0
#endif
// 1: a splitter group steps through its own tiles of a unit; 0 (rounds 1-2 until the last profile): it walks every tile
// and skips the other groups' -- bit-identical results, 5-13 % slower passes (profiles/r02_ab_step.txt)
#ifndef TC_STEP_GROUPS
#define TC_STEP_GROUPS 1
#endif

// (unit, k-tile) sequence of one persistent CTA, used by the producers' prefetch cursor
struct TileCursor {
  int unit, kt, kt1;
  int x_blocks, kt_total, kt_per_split, num_units, stride;
  __device__ __forceinline__ void init(int first_unit, int stride_, int x_blocks_, int kt_total_, int kt_per_split_, int num_units_) {
    x_blocks = x_blocks_; kt_total = kt_total_; kt_per_split = kt_per_split_; num_units = num_units_; stride = stride_;
    unit = first_unit;
    load_unit();
  }
  __device__ __forceinline__ void load_unit() {
    if (unit < num_units) {
      const int sp = unit / x_blocks;
      kt = sp * kt_per_split;
      kt1 = min(kt_total, kt + kt_per_split);
    }
  }
  __device__ __forceinline__ bool valid() const { return unit < num_units; }
  __device__ __forceinline__ int xb() const { return unit % x_blocks; }
  __device__ __forceinline__ void next() {
    if (++kt >= kt1) { unit += stride; load_unit(); }
  }
};

__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc]^T, kind::tf32, issued by ONE thread
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// A operand in tensor memory (lane = row, one 32-bit column per K element).  MUST be executed by a fully converged
// warp: the elect.sync predicate inside the asm block picks the issuing lane.  Issuing from a divergent
// `if (lane == 0)` region makes ptxas wrap every UTCHMMA in an ELECT / BRA.U.ANY loop that costs ~60-100 cycles
// per MMA (measured, tools/umma_bench.cu) -- more than a skinny N <= 64 MMA itself (N/2 cycles).
__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives once every tcgen05 op issued so far by this thread has completed
// (converged warp, elected lane -- see umma_tf32_ts)
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
      ::"r"(bar) : "memory");
}

// TC_SOFT_FREE = 1: the B-operand slot of a tile is handed back to its TMA producer by a splitter warp (a plain
// mbarrier.arrive once it has seen the barrier that the tile's MMAs committed to) instead of by a second
// tcgen05.commit; every commit costs the tensor pipe's front end ~40 cycles (tools/umma_bench.cu) and the KL pass is
// bound by that front end (round-2 role timers: both issuers busy 47 % each).  bar_b == 0 skips the commit.
#ifndef TC_SOFT_FREE
#define TC_SOFT_FREE 1
#endif

// One K tile (4 K=8 steps) of the 3-term split, plus the tcgen05.commits that release the operand slot, the B slot
// and (at a chunk end) the accumulator, issued from ONE asm block under a single elect.sync: the uniform-datapath
// set-up (ELECT, R2UR of every operand) is paid once per tile instead of once per instruction.
//   D[:, 0:2K] (+)= A_raw[tmem] * Bcat^T        (N = 2K)      D[:, K:2K] += A_lo[tmem] * B_hi^T     (N = K)
template <int K>
__device__ __forceinline__ void umma_tile_ts(uint32_t d_tmem, uint32_t a_raw, uint64_t bdesc, uint32_t acc_first,
                                             uint32_t idesc_full, uint32_t idesc_half, uint32_t bar_t, uint32_t bar_b,
                                             uint32_t bar_acc, uint32_t chunk_end, uint32_t skip_lo) {
  asm volatile(
      "{\n\t"
      ".reg .pred q, p0, p1, pc, pl, pb;\n\t"
      ".reg .b32 dl, a1, a2, a3, l0, l1, l2, l3;\n\t"
      ".reg .b64 b1, b2, b3;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p0, %3, 0;\n\t"
      "setp.eq.b32 p1, 0, 0;\n\t"
      "setp.ne.b32 pc, %9, 0;\n\t"
      "and.pred pc, pc, q;\n\t"
      "setp.eq.b32 pl, %10, 0;\n\t"
      "and.pred pl, pl, q;\n\t"
      "setp.ne.b32 pb, %7, 0;\n\t"
      "and.pred pb, pb, q;\n\t"
      "add.u32 dl, %0, %11;\n\t"
      "add.u32 l0, %1, 32;\n\t"
      "add.u32 a1, %1, 8;\n\t"
      "add.u32 l1, %1, 40;\n\t"
      "add.u32 a2, %1, 16;\n\t"
      "add.u32 l2, %1, 48;\n\t"
      "add.u32 a3, %1, 24;\n\t"
      "add.u32 l3, %1, 56;\n\t"
      "add.u64 b1, %2, 2;\n\t"
      "add.u64 b2, %2, 4;\n\t"
      "add.u64 b3, %2, 6;\n\t"
      "@q  tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %4, p0;\n\t"
      "@pl tcgen05.mma.cta_group::1.kind::tf32 [dl], [l0], %2, %5, p1;\n\t"
      "@q  tcgen05.mma.cta_group::1.kind::tf32 [%0], [a1], b1, %4, p1;\n\t"
      "@pl tcgen05.mma.cta_group::1.kind::tf32 [dl], [l1], b1, %5, p1;\n\t"
      "@q  tcgen05.mma.cta_group::1.kind::tf32 [%0], [a2], b2, %4, p1;\n\t"
      "@pl tcgen05.mma.cta_group::1.kind::tf32 [dl], [l2], b2, %5, p1;\n\t"
      "@q  tcgen05.mma.cta_group::1.kind::tf32 [%0], [a3], b3, %4, p1;\n\t"
      "@pl tcgen05.mma.cta_group::1.kind::tf32 [dl], [l3], b3, %5, p1;\n\t"
      "@q  tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%6];\n\t"
      "@pb tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%7];\n\t"
      "@pc tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%8];\n\t"
      "}\n"
      ::"r"(d_tmem), "r"(a_raw), "l"(bdesc), "r"(acc_first), "r"(idesc_full), "r"(idesc_half), "r"(bar_t), "r"(bar_b),
        "r"(bar_acc), "r"(chunk_end), "r"(skip_lo), "n"(K)
      : "memory");
}

// One K tile of the 3-term split K-CONCATENATED into a single accumulator (12 MMAs of N = K):
//   D[:, 0:K] = A_hi[tmem] * B_hi^T + A_hi * B_lo^T + A_lo[tmem + 32] * B_hi^T
// B tile = [K hi rows | K lo rows] of 128 bytes (LO_OFF = K * 128 / 16 descriptor units).  Used where an accumulator
// lives for ONE tile only (the KL path's S = W H): the truncating accumulation of the tensor core then adds 12 terms,
// far below the bias that made the long-lived accumulators keep the large term apart (see dnmf_tc.cu).
template <int K>
__device__ __forceinline__ void umma_tile_cat(uint32_t d_tmem, uint32_t a_hi, uint64_t bdesc, uint32_t idesc_n, uint32_t bar_t,
                                              uint32_t bar_b, uint32_t bar_acc, uint32_t chunk_end) {
  asm volatile(
      "{\n\t"
      ".reg .pred q, p0, p1, pc;\n\t"
      ".reg .b32 a1, a2, a3, l0, l1, l2, l3;\n\t"
      ".reg .b64 b1, b2, b3, c0, c1, c2, c3;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p0, 0, 0;\n\t"
      "setp.eq.b32 p1, 0, 0;\n\t"
      "setp.ne.b32 pc, %7, 0;\n\t"
      "and.pred pc, pc, q;\n\t"
      "add.u32 a1, %1, 8;\n\t"
      "add.u32 a2, %1, 16;\n\t"
      "add.u32 a3, %1, 24;\n\t"
      "add.u32 l0, %1, 32;\n\t"
      "add.u32 l1, %1, 40;\n\t"
      "add.u32 l2, %1, 48;\n\t"
      "add.u32 l3, %1, 56;\n\t"
      "add.u64 b1, %2, 2;\n\t"
      "add.u64 b2, %2, 4;\n\t"
      "add.u64 b3, %2, 6;\n\t"
      "add.u64 c0, %2, %8;\n\t"
      "add.u64 c1, c0, 2;\n\t"
      "add.u64 c2, c0, 4;\n\t"
      "add.u64 c3, c0, 6;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [a1], b1, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [a2], b2, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [a3], b3, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], c0, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [a1], c1, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [a2], c2, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [a3], c3, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [l0], %2, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [l1], b1, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [l2], b2, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [l3], b3, %3, p1;\n\t"
      "@q  tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%4];\n\t"
      "@q  tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%5];\n\t"
      "@pc tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%6];\n\t"
      "}\n"
      ::"r"(d_tmem), "r"(a_hi), "l"(bdesc), "r"(idesc_n), "r"(bar_t), "r"(bar_b), "r"(bar_acc), "r"(chunk_end),
        "n"(K * 8)
      : "memory");
}

// One PAIR of K tiles of the 3-term split for a 64-wide factor (K = 64 = 8 tf32 K-steps, two 128-byte swizzle atoms along
// K), K-concatenated into a single N = 64 accumulator: 24 MMAs + the commits under one elect.sync.
//   B tile layout: [hi: atom 0 | atom 1][lo: atom 0 | atom 1], each atom = 64 rows x 128 B (ATOM = 512 descriptor units)
__device__ __forceinline__ void umma_tile_cat64(uint32_t d_tmem, uint32_t a_hi, uint64_t bdesc, uint32_t idesc_n, uint32_t bar_t,
                                                uint32_t bar_b, uint32_t bar_acc, uint32_t chunk_end) {
  asm volatile(
      "{\n\t"
      ".reg .pred q, p0, p1, pc;\n\t"
      ".reg .b32 ah0, ah1, ah2, ah3, ah4, ah5, ah6, ah7, al0, al1, al2, al3, al4, al5, al6, al7;\n\t"
      ".reg .b64 bh0, bh1, bh2, bh3, bh4, bh5, bh6, bh7, bl0, bl1, bl2, bl3, bl4, bl5, bl6, bl7;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p0, 0, 0;\n\t"
      "setp.eq.b32 p1, 0, 0;\n\t"
      "setp.ne.b32 pc, %7, 0;\n\t"
      "and.pred pc, pc, q;\n\t"
      "add.u32 ah0, %1, 0;\n\t"
      "add.u32 al0, %1, 64;\n\t"
      "add.u64 bh0, %2, 0;\n\t"
      "add.u64 bl0, %2, 1024;\n\t"
      "add.u32 ah1, %1, 8;\n\t"
      "add.u32 al1, %1, 72;\n\t"
      "add.u64 bh1, %2, 2;\n\t"
      "add.u64 bl1, %2, 1026;\n\t"
      "add.u32 ah2, %1, 16;\n\t"
      "add.u32 al2, %1, 80;\n\t"
      "add.u64 bh2, %2, 4;\n\t"
      "add.u64 bl2, %2, 1028;\n\t"
      "add.u32 ah3, %1, 24;\n\t"
      "add.u32 al3, %1, 88;\n\t"
      "add.u64 bh3, %2, 6;\n\t"
      "add.u64 bl3, %2, 1030;\n\t"
      "add.u32 ah4, %1, 32;\n\t"
      "add.u32 al4, %1, 96;\n\t"
      "add.u64 bh4, %2, 512;\n\t"
      "add.u64 bl4, %2, 1536;\n\t"
      "add.u32 ah5, %1, 40;\n\t"
      "add.u32 al5, %1, 104;\n\t"
      "add.u64 bh5, %2, 514;\n\t"
      "add.u64 bl5, %2, 1538;\n\t"
      "add.u32 ah6, %1, 48;\n\t"
      "add.u32 al6, %1, 112;\n\t"
      "add.u64 bh6, %2, 516;\n\t"
      "add.u64 bl6, %2, 1540;\n\t"
      "add.u32 ah7, %1, 56;\n\t"
      "add.u32 al7, %1, 120;\n\t"
      "add.u64 bh7, %2, 518;\n\t"
      "add.u64 bl7, %2, 1542;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah0], bh0, %3, p0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah1], bh1, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah2], bh2, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah3], bh3, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah4], bh4, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah5], bh5, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah6], bh6, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah7], bh7, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah0], bl0, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah1], bl1, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah2], bl2, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah3], bl3, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah4], bl4, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah5], bl5, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah6], bl6, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [ah7], bl7, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [al0], bh0, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [al1], bh1, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [al2], bh2, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [al3], bh3, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [al4], bh4, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [al5], bh5, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [al6], bh6, %3, p1;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [al7], bh7, %3, p1;\n\t"
      "@q  tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%4];\n\t"
      "@q  tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%5];\n\t"
      "@pc tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%6];\n\t"
      "}\n"
      ::"r"(d_tmem), "r"(a_hi), "l"(bdesc), "r"(idesc_n), "r"(bar_t), "r"(bar_b), "r"(bar_acc), "r"(chunk_end)
      : "memory");
}

// the commits of a tile without its MMAs (timing ablations only)
__device__ __forceinline__ void umma_commits_only(uint32_t bar_t, uint32_t bar_b, uint32_t bar_acc, uint32_t chunk_end) {
  asm volatile(
      "{\n\t"
      ".reg .pred q, pc;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 pc, %3, 0;\n\t"
      "and.pred pc, pc, q;\n\t"
      "@q  tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
      "@q  tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%1];\n\t"
      "@pc tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%2];\n\t"
      "}\n"
      ::"r"(bar_t), "r"(bar_b), "r"(bar_acc), "r"(chunk_end)
      : "memory");
}

__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st_x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,"
      "%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
        "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
        "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,"
      "%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// a / d for d > 0 on the FMA pipe only (no MUFU): magic-constant seed (12 % error) + 3 Newton steps (4e-8).  Used for
// every other element so the division work is spread over the SFU and FMA pipes.
__device__ __forceinline__ float div_newton(float a, float d) {
  float r = __uint_as_float(0x7EF311C7u - __float_as_uint(d));
  r = r * fmaf(-d, r, 2.0f);
  r = r * fmaf(-d, r, 2.0f);
  r = r * fmaf(-d, r, 2.0f);
  return a * r;
}
__device__ __forceinline__ float rcp_approx(float d) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d));
  return r;
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// shared-memory matrix descriptor, 128-byte swizzle (cute::UMMA::SmemDescriptor bit layout)
// layout_type: 2 = SWIZZLE_128B (16-byte chunks, 8-row period), 1 = SWIZZLE_128B_BASE32B (32-byte chunks, 4-row
// period) -- the only shared-memory layout the tensor core accepts for MN-major 32-bit operands
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                                   uint32_t layout_type = 2) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);               // [0,14)  start address >> 4
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;      // [16,30) leading byte offset >> 4
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;      // [32,46) stride byte offset >> 4
  d |= (uint64_t)1 << 46;                                 // [46,48) descriptor version (Blackwell)
  d |= (uint64_t)layout_type << 61;                       // [61,64) layout type
  return d;
}

// instruction descriptor (cute::UMMA::InstrDescriptor): D fp32, A/B tf32, M = 128, N = n
__host__ __device__ constexpr uint32_t make_idesc(int n, int a_mn_major) {
  return (1u << 4)                       // c_format = F32
         | (2u << 7)                     // a_format = TF32
         | (2u << 10)                    // b_format = TF32
         | ((uint32_t)a_mn_major << 15)  // A major: 0 = K, 1 = MN
         | (0u << 16)                    // B major: K
         | ((uint32_t)(n >> 3) << 17)    // N >> 3
         | ((uint32_t)(TC_BM >> 4) << 24);  // M >> 4
}

__device__ __forceinline__ float tf32_hi(float x, int mode) {
  uint32_t u = __float_as_uint(x);
  if (mode) u += 0x0FFFu + ((u >> 13) & 1u);   // round to nearest even (calibration fallback)
  return __uint_as_float(u & 0xFFFFE000u);      // default: the tensor core drops the low 13 mantissa bits
}

// nearest tf32 with ties away from zero: 2 integer ops (the tie bias is ~3e-8 relative, see DESIGN.md)
__device__ __forceinline__ float tf32_round_up(float x) {
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
}

// The splitters' hot loop, 3 instructions per element (LOP3, FADD, IADD): the low part a - trunc_tf32(a) (exact), biased by
// half a tf32 ulp so that the tensor core's own truncation of the operand rounds it to nearest.  Only valid on hardware
// whose kind::tf32 truncates (checked once by calibrate(); otherwise the tensor path is switched off).
__device__ __forceinline__ uint32_t tf32_lo_bits(uint32_t raw) {
  const float v = __uint_as_float(raw);
  return __float_as_uint(v - __uint_as_float(raw & 0xFFFFE000u)) + 0x1000u;
}
// the same for two elements with one packed subtraction (FADD2, sm_100): one LOP3 per element forms -trunc_tf32(a), one
// FADD2 per pair adds it (exact), one integer add per element applies the half-ulp bias
__device__ __forceinline__ void tf32_lo_bits2(uint32_t raw0, uint32_t raw1, uint32_t& lo0, uint32_t& lo1) {
  const float2 nh = make_float2(__uint_as_float((raw0 & 0xFFFFE000u) ^ 0x80000000u),
                                __uint_as_float((raw1 & 0xFFFFE000u) ^ 0x80000000u));
  const float2 l = __fadd2_rn(make_float2(__uint_as_float(raw0), __uint_as_float(raw1)), nh);
  lo0 = __float_as_uint(l.x) + 0x1000u;
  lo1 = __float_as_uint(l.y) + 0x1000u;
}


// DNMF_TC_LAB = 1 (tools/build_variant.sh, tools/kl_lab.py, tools/prof_tc.py --roles): the kernels honour the
// timing-ablation word (dnmf_set_tc_debug) and the per-role cycle counters (dnmf_set_tc_profile).  The production build
// (0) compiles both out: the flag tests, the register copies that join their alternative code paths and the predicated
// clock reads cost the splitter warps ~15 % of their issue slots (round-2 ncu source page).
#ifndef DNMF_TC_LAB
#define DNMF_TC_LAB 0
#endif
#if DNMF_TC_LAB
#define TC_LAB_ARGS(dbg_arg, prof_arg) const int dbg = (dbg_arg); unsigned long long* const prof = (prof_arg);
#else
// DNMF_TC_DBG_CONST: ablation word fixed at compile time (lab builds that remove one stage without paying for the
// run-time flag tests); 0 in production
#ifndef DNMF_TC_DBG_CONST
#define DNMF_TC_DBG_CONST 0
#endif
#define TC_LAB_ARGS(dbg_arg, prof_arg) constexpr int dbg = DNMF_TC_DBG_CONST; constexpr unsigned long long* prof = nullptr; (void)(dbg_arg); (void)(prof_arg);
#endif
// cycle accounting (dnmf_set_tc_profile): per-role time split written to a debug buffer; off in production
#define TC_T(var) do { if (prof) { const long long _n = clock64(); var += _n - tprev; tprev = _n; } } while (0)

}  // namespace

// ---- host helpers defined in dnmf_tc.cu ------------------------------------------------------------------
// 2-D fp32 row-major tensor map [rows][cols] with leading dimension ld, box {box_cols, box_rows}; OOB reads are zero
int tc_make_map(CUtensorMap* map, const float* ptr, int64_t rows, int64_t cols, int64_t ld, int box_cols, int box_rows,
                CUtensorMapSwizzle swz);
struct TcPlan {
  int x_blocks, kt_total, kt_per_split, splits, num_units, grid;
  int64_t ldb;            // leading dimension of Bcat (reduced length rounded up to 4)
  int64_t bcat_bytes, partial_bytes;
};
int tc_padded_k(int k);
// bk: reduced-dimension elements per tile (TC_BK fp32, TC16_BK for a 16-bit A)
TcPlan tc_plan(int64_t x_len, int64_t r_len, int k, int bk = TC_BK);
int tc_hi_mode();                       // 0: the tensor core truncates fp32 -> tf32, 1: rounds to nearest (calibrated)
unsigned long long* tc_prof_ptr();      // debug buffer or nullptr
int tc_dbg_flags();

// small-operand split kernels (dnmf_tc.cu)
void tc_launch_split_h(const float* H, int64_t ldh, float* Bcat, int64_t ldb, int k, int kp, int64_t n, cudaStream_t st);
void tc_launch_split_wt(const float* W, int64_t ldw, float* Bcat, int64_t ldb, int k, int kp, int64_t m, cudaStream_t st);

// fused KL contractions (dnmf_tc_kl.cu)
int64_t tc_kl_workspace_bytes(int op, int64_t m, int64_t n, int64_t k);
bool tc_kl_supported(int64_t k);
// the 64-wide build (dnmf_tc_kl64.cu): 32 < k <= 64
int64_t tc_kl_workspace_bytes_k64(int op, int64_t m, int64_t n, int64_t k);
bool tc_kl_supported_k64(int64_t k);
struct TcPartials;
int tc_kl_run(int mode, const float* A, int64_t lda, const float* W, int64_t ldw, const float* H, int64_t ldh, float* out,
              int64_t ldo, int64_t m, int64_t n, int k, float eps, int transposed_out, void* ws, int64_t ws_bytes,
              cudaStream_t st, TcPartials* defer = nullptr);
int tc_kl_run_k64(int mode, const float* A, int64_t lda, const float* W, int64_t ldw, const float* H, int64_t ldh, float* out,
                  int64_t ldo, int64_t m, int64_t n, int k, float eps, int transposed_out, void* ws, int64_t ws_bytes,
                  cudaStream_t st, TcPartials* defer = nullptr);

}  // namespace dnmf
