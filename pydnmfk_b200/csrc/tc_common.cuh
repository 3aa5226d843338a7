// Shared device-side PTX wrappers and host-side helpers of the tcgen05 / TMA / TMEM kernels
// (dnmf_tc.cu: FRO contractions, dnmf_tc_kl.cu: fused KL contractions).
#pragma once
#include <cuda.h>

#include "common.cuh"
#include "launch_passes.cuh"
#include "tc_api.cuh"

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
// Blocking waits, in two flavours chosen per kernel by measurement.  try_wait suspends the warp in hardware until the
// phase completes or a time limit expires.
// mbar_wait (FRO and 16-bit kernels): an explicit suspend-time hint keeps a waiting warp parked until the barrier actually
// flips.  With the default limit the waiting roles (producers, issuers, drain warps) re-issued YIELD / TRYWAIT / BRA
// triplets often enough to make up 28 % of all executed warp instructions of the KL pass (ncu source page, round 1);
// the hint is worth 5 % on the FRO passes.
// mbar_wait_spin (KL kernels): try_wait with the default limit, re-issued in a loop -- measured 2-4 % faster than the
// hinted wait on the KL passes (tools/kl_lab.py, profiles/r02_kl_lab.md).
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}"
      ::"r"(bar), "r"(parity), "r"(0x989680u)
      : "memory");
}
__device__ __forceinline__ void mbar_wait_spin(uint32_t bar, uint32_t parity) {
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
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
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

// One K tile (4 K=8 steps) of the 3-term split, plus the tcgen05.commits that release the operand slot and (at a chunk
// end) the accumulator, issued from ONE asm block under a single elect.sync: the uniform-datapath set-up (ELECT, R2UR of
// every operand) is paid once per tile instead of once per instruction.  Both A operands come from tensor memory (lane =
// row, one 32-bit column per K element).
//   D[:, 0:2K] (+)= A_raw[tmem] * Bcat^T        (N = 2K)      D[:, K:2K] += A_lo[tmem] * B_hi^T     (N = K)
// MUST be executed by a fully converged warp: the elect.sync predicate inside the asm block picks the issuing lane.
// Issuing from a divergent `if (lane == 0)` region makes ptxas wrap every UTCHMMA in an ELECT / BRA.U.ANY loop that costs
// ~60-100 cycles per MMA (measured, tools/umma_bench.cu) -- more than a skinny N <= 64 MMA itself (N/2 cycles).
// The B-operand slot of the tile is not released here: a splitter warp hands it back to its TMA producer (a plain
// mbarrier.arrive once it has seen the barrier bar_t that the tile's MMAs committed to) instead of a second
// tcgen05.commit; every commit costs the tensor pipe's front end ~40 cycles (tools/umma_bench.cu) and the KL pass is
// bound by that front end (round-2 role timers: both issuers busy 47 % each).
template <int K>
__device__ __forceinline__ void umma_tile_ts(uint32_t d_tmem, uint32_t a_raw, uint64_t bdesc, uint32_t acc_first,
                                             uint32_t idesc_full, uint32_t idesc_half, uint32_t bar_t, uint32_t bar_acc,
                                             uint32_t chunk_end) {
  asm volatile(
      "{\n\t"
      ".reg .pred q, p0, p1, pc;\n\t"
      ".reg .b32 dl, a1, a2, a3, l0, l1, l2, l3;\n\t"
      ".reg .b64 b1, b2, b3;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p0, %3, 0;\n\t"
      "setp.eq.b32 p1, 0, 0;\n\t"
      "setp.ne.b32 pc, %8, 0;\n\t"
      "and.pred pc, pc, q;\n\t"
      "add.u32 dl, %0, %9;\n\t"
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
      "@q  tcgen05.mma.cta_group::1.kind::tf32 [dl], [l0], %2, %5, p1;\n\t"
      "@q  tcgen05.mma.cta_group::1.kind::tf32 [%0], [a1], b1, %4, p1;\n\t"
      "@q  tcgen05.mma.cta_group::1.kind::tf32 [dl], [l1], b1, %5, p1;\n\t"
      "@q  tcgen05.mma.cta_group::1.kind::tf32 [%0], [a2], b2, %4, p1;\n\t"
      "@q  tcgen05.mma.cta_group::1.kind::tf32 [dl], [l2], b2, %5, p1;\n\t"
      "@q  tcgen05.mma.cta_group::1.kind::tf32 [%0], [a3], b3, %4, p1;\n\t"
      "@q  tcgen05.mma.cta_group::1.kind::tf32 [dl], [l3], b3, %5, p1;\n\t"
      "@q  tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%6];\n\t"
      "@pc tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%7];\n\t"
      "}\n"
      ::"r"(d_tmem), "r"(a_raw), "l"(bdesc), "r"(acc_first), "r"(idesc_full), "r"(idesc_half), "r"(bar_t), "r"(bar_acc),
        "r"(chunk_end), "n"(K)
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

// nearest tf32, ties to even: the high part of a factor split (the low part x - tf32_rn(x) is then signed and at most
// half a tf32 ulp)
__device__ __forceinline__ float tf32_rn(float x) {
  const uint32_t u = __float_as_uint(x);
  return __uint_as_float((u + 0x0FFFu + ((u >> 13) & 1u)) & 0xFFFFE000u);
}

// nearest tf32 with ties away from zero: 2 integer ops (the tie bias is ~3e-8 relative, see DESIGN.md)
__device__ __forceinline__ float tf32_round_up(float x) {
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
}

// The splitters' hot loop: the low part a - trunc_tf32(a) (exact), biased by half a tf32 ulp so that the tensor core's own
// truncation of the operand rounds it to nearest.  Only valid on hardware whose kind::tf32 truncates (checked once by
// calibrate(); otherwise the tensor path is switched off).  Two elements per packed subtraction (FADD2, sm_100): one LOP3
// per element forms -trunc_tf32(a), one FADD2 per pair adds it (exact), one integer add per element applies the bias.
__device__ __forceinline__ void tf32_lo_bits2(uint32_t raw0, uint32_t raw1, uint32_t& lo0, uint32_t& lo1) {
  const float2 nh = make_float2(__uint_as_float((raw0 & 0xFFFFE000u) ^ 0x80000000u),
                                __uint_as_float((raw1 & 0xFFFFE000u) ^ 0x80000000u));
  const float2 l = __fadd2_rn(make_float2(__uint_as_float(raw0), __uint_as_float(raw1)), nh);
  lo0 = __float_as_uint(l.x) + 0x1000u;
  lo1 = __float_as_uint(l.y) + 0x1000u;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------
// host side: planning and the launch skeleton shared by the drivers tc_run (dnmf_tc.cu), tc16_run (dnmf_tc16.cu),
// tc_kl_run (dnmf_tc_kl.cu; also the A H^T + residual pass) -- defined in dnmf_tc.cu unless inline
// ---------------------------------------------------------------------------------------------------------
struct TcPlan {
  int x_blocks, kt_total, kt_per_split, splits, num_units, grid;
  int64_t ldb;            // leading dimension of Bcat (reduced length rounded up to 4)
  int64_t bcat_bytes, partial_bytes;
};
int tc_padded_k(int k);
// bk: reduced-dimension elements per tile (TC_BK fp32, TC16_BK for a 16-bit A)
TcPlan tc_plan(int64_t x_len, int64_t r_len, int k, int bk = TC_BK);

// Start of a pass: the workspace must hold `need` bytes at 256-byte alignment; its first `bcat_bytes` (the split factor
// Bcat) are zeroed when the kernel runs on zero-padded factor rows.
int tc_begin(void* ws, int64_t ws_bytes, int64_t need, int64_t bcat_bytes, bool padded, cudaStream_t st);
// 2-D row-major tensor map [rows][cols] of `type` (fp32, fp16 or bf16) elements with leading dimension ld, box
// {box_cols, box_rows}; out-of-bounds elements read as zero (ragged edges need no special casing in the kernels)
int tc_make_map(CUtensorMap* map, CUtensorMapDataType type, const void* ptr, int64_t rows, int64_t cols, int64_t ld,
                int box_cols, int box_rows, CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B);
// the map of A (dtype DNMF_F32, or DNMF_A_F16 / DNMF_A_BF16 for the KL kernels) in TC_BK-element tiles: mode 1 (WTA /
// WTU, x = columns of A) MN-major tiles, box {TC_BM, TC_BK}, no swizzle; any other mode (x = rows of A) K-major tiles,
// box {TC_BK, TC_BM}, one swizzle row per tile row (128-byte swizzle for fp32, 64-byte for 16-bit elements)
int tc_map_a(CUtensorMap* map, const void* A, int dtype, int64_t lda, int64_t m, int64_t n, int mode);
// End of a pass: the split partials P[split][x][kp] are described in *defer, or summed in a fixed order into the k real
// columns of out: V[x][kk] (mode 0), Y[kk][x] (mode 1) or Y^T[x][kk] (mode 1, transposed_out).  Inline, so that every
// driver's translation unit keeps its own reduce_partials_kernel.
inline int tc_finish(float* P, int64_t x_len, int kp, int splits, int mode, int k, int transposed_out, float* out,
                     int64_t ldo, cudaStream_t st, TcPartials* defer) {
  const int64_t split_stride = x_len * kp;
  if (defer != nullptr) {
    defer->P = P; defer->ldp = kp; defer->split_stride = split_stride; defer->splits = splits;
    return 0;
  }
  const bool x_rows = mode == 0 || transposed_out;   // x indexes the rows of out
  return launch_reduce<float>(P, split_stride, splits, x_len, k, kp, out, x_rows ? ldo : 1, x_rows ? 1 : ldo, st);
}

// small-operand split kernels (dnmf_tc.cu)
int tc_launch_split_h(const float* H, int64_t ldh, float* Bcat, int64_t ldb, int k, int kp, int64_t n, cudaStream_t st);
int tc_launch_split_wt(const float* W, int64_t ldw, float* Bcat, int64_t ldb, int k, int kp, int64_t m, cudaStream_t st);

// 16-bit A (dtype DNMF_A_F16 / DNMF_A_BF16), fp32 factors and outputs (dnmf_tc16.cu).  ws = [Bcat | amax + s | partials]
struct Tc16Layout {
  TcPlan pl;
  int kp, np;
  int64_t ldb, bcat_bytes, aux_bytes, total;
};
Tc16Layout tc16_layout(int mode, int64_t m, int64_t n, int k, int dtype);
int tc16_run(int mode, const void* A, int64_t lda, const float* B, int64_t ldbsrc, float* out, int64_t ldo, int64_t m,
             int64_t n, int k, int transposed_out, int dtype, void* ws, int64_t ws_bytes, cudaStream_t st,
             TcPartials* defer);

// fused KL contractions (dnmf_tc_kl.cu: k <= 32; the _k64 build, dnmf_tc_kl64.cu: 32 < k <= 64).  mode 0 UHT, 1 WTU,
// 3 A H^T + residual (32-wide build only).  A is fp32 or 16-bit (dtype); the layout does not depend on it.
// ws = [Bcat | FrCat | Ht (modes 0, 1) | partials | residual pairs (mode 3)]
struct KlLayout {
  TcPlan pl;
  int64_t r_pad, frcat_bytes, ht_bytes, pairs_bytes, total;
};
KlLayout tc_kl_layout(int mode, int64_t m, int64_t n);
KlLayout tc_kl_layout_k64(int mode, int64_t m, int64_t n);
int tc_kl_run(int mode, const void* A, int dtype, int64_t lda, const float* W, int64_t ldw, const float* H, int64_t ldh,
              float* out, int64_t ldo, int64_t m, int64_t n, int k, float eps, int transposed_out, void* ws,
              int64_t ws_bytes, cudaStream_t st, TcPartials* defer);
int tc_kl_run_k64(int mode, const void* A, int dtype, int64_t lda, const float* W, int64_t ldw, const float* H,
                  int64_t ldh, float* out, int64_t ldo, int64_t m, int64_t n, int k, float eps, int transposed_out,
                  void* ws, int64_t ws_bytes, cudaStream_t st, TcPartials* defer);

}  // namespace dnmf
