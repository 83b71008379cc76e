// tcgen05 implicit-GEMM convolution kernel shared by the forward (conv_umma.cu) and the backward
// data-gradient pass (conv_bwd.cu).  See conv_umma.cu for the design notes.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>

#include <type_traits>

#include "common.cuh"

namespace wn {

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// Bounded wait: a pipeline bug becomes a trap ("unspecified launch failure"), never a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  for (uint32_t it = 0; it < (1u << 26); it++) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (done) return;
  }
  __trap();
}
// One non-blocking probe of a barrier phase; lets a waiter look at the NEXT stage's barrier while
// it still has work to issue for the current one (the probe's ~100-cycle latency is then hidden).
__device__ __forceinline__ bool mbar_try(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return done != 0;
}
// CTA-pair kernels: arrival on the barrier at the same shared-memory offset in CTA `rank` of the cluster.
// Waiters use the plain mbar_wait: what they order is asynchronous-proxy work (TMA writes that have
// completed on a barrier before the arrival was sent; MMAs issued after the wait), and a cluster-scope
// acquire on every stage costs the issuer ~600 cycles (measured: 3x3 layers got 30 % slower with it).
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t rank) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(rank));
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* tmap, uint64_t* bar, int c0,
                                            int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_u32(dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
// shared-memory matrix descriptor: no swizzle, K-major.  LBO = byte distance between the two
// 8-element K halves of a K=16 step, SBO = byte distance between 8-row groups.
__device__ __forceinline__ uint64_t make_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((addr >> 4) & 0x3fff);
  d |= (uint64_t)((lbo >> 4) & 0x3fff) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3fff) << 32;
  d |= 1ull << 46;
  return d;
}
__host__ __device__ constexpr uint32_t make_idesc(int M, int N) {
  // c=f32 (bit 4), a=b=bf16 (bits 7, 10), K-major both, N>>3 at 17, M>>4 at 24
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same, descriptors given as (lo, hi) 32-bit halves so that the per-MMA work is one add.
__device__ __forceinline__ void umma_bf16_split(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo,
                                                uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem),
      "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
// CTA-pair forms: one M=256 MMA over both CTAs' shared memory / TMEM (issued by the leader CTA only);
// the commit arrives on the barrier at this offset in BOTH CTAs.
__device__ __forceinline__ void umma2_bf16_split(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo,
                                                 uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem),
      "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma2_commit(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"((uint16_t)3)
      : "memory");
}
template <int CG>
__device__ __forceinline__ void umma_issue(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo,
                                           uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
  if constexpr (CG == 2) umma2_bf16_split(d_tmem, a_lo, a_hi, b_lo, b_hi, idesc, accumulate);
  else umma_bf16_split(d_tmem, a_lo, a_hi, b_lo, b_hi, idesc, accumulate);
}
// A operand from tensor memory (lane = M row, one 32-bit column = two consecutive bf16 K elements), B from shared
// memory: the fused tail layer's GEMM reads the activation tile the epilogue wrote back with tcgen05.st.
template <int CG>
__device__ __forceinline__ void umma_issue_ts(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi,
                                              uint32_t idesc, uint32_t accumulate) {
  if constexpr (CG == 2)
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\t"
        "setp.ne.b32 p, %5, 0;\n\t"
        "mov.b64 db, {%2, %3};\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], db, %4, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\t"
        "setp.ne.b32 p, %5, 0;\n\t"
        "mov.b64 db, {%2, %3};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// kind::f8f6f4 (K = 32 fp8 values per instruction): the fp8 correction pass.  Same descriptors as the bf16
// form -- a core-matrix row is 16 bytes either way (8 bf16 or 16 fp8 values).
template <int CG>
__device__ __forceinline__ void umma_issue_f8(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo,
                                              uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
  if constexpr (CG == 2)
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "mov.b64 da, {%1, %2};\n\t"
        "mov.b64 db, {%3, %4};\n\t"
        "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "mov.b64 da, {%1, %2};\n\t"
        "mov.b64 db, {%3, %4};\n\t"
        "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
// instruction descriptor of the fp8 pass: A = B = e4m3 (format 0), D = f32.  (e5m2 activations -- format 1,
// range-safe like fp16 -- were measured too: twice the error, 4.4-7.2e-4 at the network output with the stress
// weights; with e4m3 an activation above 448 merely saturates its *correction* term, i.e. degrades that
// element to single-pass bf16 accuracy, and one below 2^-9 loses a correction of < 4e-6 absolute.)
__host__ __device__ constexpr uint32_t make_idesc_f8(int M, int N) {
  return (1u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// four floats -> four e4m3 bytes, f0 at the lowest address
__device__ __forceinline__ uint32_t pack_e4m3x4(float f0, float f1, float f2, float f3) {
  uint16_t lo, hi;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(lo) : "f"(f1), "f"(f0));
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(hi) : "f"(f3), "f"(f2));
  return (uint32_t)lo | ((uint32_t)hi << 16);
}
__device__ __forceinline__ uint16_t pack_e4m3x2(float f0, float f1) {
  uint16_t v;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(v) : "f"(f1), "f"(f0));
  return v;
}
template <int CG>
__device__ __forceinline__ void umma_done(uint64_t* bar) {
  if constexpr (CG == 2) umma2_commit(bar);
  else umma_commit(bar);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),
        "=r"(v[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ------------------------------------------------------------------------------------------
// Kernel configuration
// ------------------------------------------------------------------------------------------
// kEpiAct: bias + ReLU -> bf16 hi/lo planes.  kEpiSigmoid: bias + sigmoid -> 3 fp32 maps.
// kEpiGate: bias + ReLU, gated sum with the confidence maps -> fp32 NCHW output.
// kEpiDgrad (backward): no bias; zero where the saved forward activation is zero (ReLU'), -> planes.
enum Epilogue { kEpiAct = 0, kEpiSigmoid = 1, kEpiGate = 2, kEpiDgrad = 3 };

constexpr int kSubW = 8, kSubH = 16;  // one M=128 sub-tile: 8 px wide, 16 px tall
// warps 0-7: epilogue (two groups); 8: A producer; 9: B producer; 10: TMEM allocator; 11: MMA issuer.
// The issuer has the highest warp id (the sub-partition arbiter serves higher warp ids first, so its few
// instructions per stage do not queue behind the epilogue warps).  Measured effect: ~4 % when the GPU runs
// at full clocks, none in the power-capped steady state of a long step.
constexpr int kThreads = 384;
constexpr int kWarpA = 8, kWarpB = 9, kWarpTmem = 10, kWarpMma = 11;

// NPAD   output channels per diagonal block (UMMA N of the lo*hi pass)
// CONCAT weight stage rows are [hi rows | lo rows]: a_hi x [w_hi|w_lo] is ONE MMA of N = 2*NPAD (the
//        activation tile is read from shared memory once for two products), then a_lo x w_hi with
//        N = NPAD.  Pays when NPAD <= 64, where an MMA is bound by the 4 KB A-operand read.
// NBLK   number of diagonal blocks (the three refiners run as one block-diagonal layer): input
//        chunk c only feeds block c / (NCHUNK / NBLK), so only that block's weights are staged.
// TPS    filter taps per weight stage: small-N layers batch a kernel row (or all taps) per stage so
//        that the per-stage pipeline cost (barrier wait, commit, bulk-copy latency) is amortised.
// CG     CTAs per MMA (tcgen05 cta_group).  2: a cluster of two CTAs works on two adjacent tiles; the leader
//        issues M=256 MMAs over both CTAs' halo tiles, and each CTA stages only HALF of the weight rows
//        (the N dimension is split over the pair) -- the shared-memory operand traffic per MMA, which
//        bounds N<=128 layers (tools/umma_rate_probe.cu), drops from 128+N to 128+N/2 rows.
// FMT    bit 0 (kFmtIn8): fp8 correction scheme on the input side.  v = hi (bf16) + lo; instead of the two
//        bf16 correction passes (a_lo x w_hi, a_hi x w_lo) ONE kind::f8f6f4 MMA of K = 32 multiplies
//        [e4m3(lo * 2^9) | e4m3(v)] (the two fp8 planes the producing layer wrote where the bf16 lo planes
//        used to be) by [e4m3(w * ws) ; e4m3(w_lo * ws * 2^9)]: 2 pass-equivalents instead of 3 at half the
//        operand bytes.  Both MMAs accumulate into the SAME fp32 accumulator: the bf16 weights of such a layer
//        are packed pre-scaled by the power of two ws * 2^9 (exact), so the two products carry the same scale
//        and the epilogue multiplies the sum by 2^-9 / ws once.  (A separate correction accumulator, as in
//        round 1, doubles the TMEM columns and forces single-buffered or single-sub-tile configurations.)
//        bit 1 (kFmtOut8): the epilogue writes that hi + fp8-planes format (its consumer has bit 0 set).
constexpr int kFmtIn8 = 1, kFmtOut8 = 2;
// TN     fused "tail" layer (0 = none): a 1x1 convolution of TN output channels applied to this layer's output tile
//        before it ever leaves the SM.  The epilogue writes the tile's activations (bias, ReLU, bf16 hi/lo split) back
//        into TENSOR MEMORY as packed bf16 pairs (tcgen05.st: lane = pixel row, one 32-bit column = two channels --
//        exactly the K-major A operand of a tcgen05.mma that takes A from TMEM), the issuer runs a second, small
//        GEMM (K = this layer's output channels, bf16x3 in the CONCAT form, weights resident in shared memory) into
//        the accumulator columns the epilogue has just drained, and a second epilogue pass stores the tail layer's
//        output.  cmg.conv3 -> conv4 (net.py:20-27): conv3's 512 B/px write, conv4's 512 B/px read and its launch
//        disappear; no shared memory is spent on the intermediate tile.
// KP     K-packed first layer (inference).  The 12 input channels fill only 12 of a K = 16 step's 16 slots.  A UMMA
//        descriptor addresses the two 8-element K halves of a step independently (start address + LBO), so a step
//        can pair ANY two 16-byte rows of the halo tile: channels 0-7 of one tap (plane 0), or a row of plane 1 that
//        holds channels 8-11 of TWO neighbouring pixels [c8..11 @ x | c8..11 @ x+1] and so serves two taps of a
//        kernel row at once.  A 7-tap row needs 7 + 4 = 11 halves instead of 14: 77 halves = 39 (padded: kKpSteps =
//        40) K-steps per tile instead of 49.  The pairs and their LBOs come from a table (ConvArgs::kp_off / kp_lbo;
//        l1k_table()); the weights are packed to match.  Plane 1's "next pixel" half makes the planes one column
//        wider: column x + 1 holds pixel x, so that TMA zero fill left of the image stays correct.
constexpr int kKpSteps = 40;
template <int KS, int CIN_PAD, int NPAD, int S, int AS, int CONCAT = 0, int NBLK = 1, int TPS = 1, int CG = 1,
          int FMT = 0, int TN = 0, int KP = 0, int A2S = 0>
struct UmmaCfg {
  static constexpr int KSTEPS = KP ? kKpSteps : KS * KS;   // weight "taps" (K = 16 steps per chunk) per tile
  static constexpr int K2 = NPAD * NBLK;                                 // tail GEMM K = this layer's output channels
  // the tail GEMM's A operand (bf16 hi/lo copy of the tile): in tensor memory (A2S == 0), K2 columns per sub-tile (K2/2
  // hi pairs | K2/2 lo pairs), or in shared memory (A2S != 0), per sub-tile [hi|lo][k8 group][128 rows][16 B]
  static constexpr int A2_COLS = (TN && !A2S) ? K2 : 0;
  static constexpr int A2_SUB = 2 * (K2 / 8) * 2048;
  static constexpr int A2_BYTES = (TN && A2S) ? S * A2_SUB : 0;
  // tail weights per K=16 step and rank.  One block (NBLK == 1), CONCAT form: [k8][TN | TN/2 rows][16 B] (a_hi x [w_hi|w_lo],
  // a_lo x w_hi).  Block-diagonal (the three refiners): TN / NBLK columns per block, three passes into the same
  // columns, [hi|lo][k8][TN / NBLK / 2 rows][16 B]
  static constexpr bool TAIL_BLK = NBLK > 1;
  static constexpr int TNB = TN / NBLK;                                  // tail output columns per block
  static constexpr int WT_TAP = TAIL_BLK ? TNB * 32 : TN * 48;
  static constexpr int WT_BYTES = TN ? (K2 / 16) * WT_TAP : 0;
  static constexpr int TAIL_BYTES = (A2_BYTES + WT_BYTES + 1023) / 1024 * 1024;

  static constexpr bool F8IN = (FMT & kFmtIn8) != 0;
  static constexpr bool DUAL = CONCAT != 0;  // two accumulator halves per block: [a x w_hi | a_hi x w_lo]
  static constexpr int TILE_W = kSubW * S, TILE_H = kSubH;
  static constexpr int HALO_W = TILE_W + KS - 1, HALO_H = TILE_H + KS - 1;
  static constexpr int NCHUNK = CIN_PAD / 16;
  static constexpr int PLANE_BYTES = HALO_W * HALO_H * 16;
  static constexpr int A_STAGE = (4 * PLANE_BYTES + 1023) / 1024 * 1024;  // hi k0, hi k1, lo k0, lo k1
  // one tap of weights.  CG=1: [hi|lo][k8 0|1][NPAD][16 B] (CONCAT: [k8][hi rows | lo rows]).
  // CG=2, per CTA: [hi|lo][k8][NPAD/2 rows of this rank]; CONCAT: [k8][NPAD rows (rank 0: w_hi, rank 1:
  // w_lo) | NPAD/2 rows of w_hi for the a_lo pass] -- the same descriptor serves both CTAs.
  static constexpr int B_TAP = CG == 1 ? NPAD * 64 : CONCAT ? NPAD * 48 : NPAD * 32;
  static constexpr int B_STAGE = TPS * B_TAP;
  static_assert(KSTEPS % TPS == 0, "a weight stage holds whole taps of one chunk");
  static constexpr int NSTAGE_PER_CHUNK = KSTEPS / TPS;
  static_assert(!KP || (KS == 7 && CIN_PAD == 16 && CG == 2 && !CONCAT && TN == 0), "K-packing: the 7x7 first layer");
  static constexpr int BUDGET = 225 * 1024 - 2048 - TAIL_BYTES;
  // halo ring: enough stages to prefetch the next chunk (or the next tile when there is one chunk)
  // (a 1x1 layer is HBM-bound and its stages are small: keep more loads in flight)
  static constexpr int NA_WANT = NCHUNK == 1 ? 2 : KS == 1 ? 6 : 3;
  // weight ring: whatever is left after the halo ring, 2..8 stages; deep rings hide the L2 latency of
  // the bulk copies when a stage carries only a few MMAs (first layer: 14 KB per 4-6 MMAs)
  // CTA pairs: a halo stage is handed to the leader through one more hop (the peer's relay warp), and a
  // chunk of a 3x3 layer lasts only ~2k cycles -- up to 6 halo stages after 4 weight stages are set aside
  static constexpr int NA_PAIR_FIT = (BUDGET - 4 * B_STAGE) / A_STAGE;
  static constexpr int NA_PAIR = NA_PAIR_FIT > 6 ? 6 : NA_PAIR_FIT < 2 ? 2 : NA_PAIR_FIT;
  static constexpr int NA_TARGET = CG == 2 ? NA_PAIR : NA_WANT;
  static constexpr int NB_FIT = (BUDGET - NA_TARGET * A_STAGE) / B_STAGE;
  static constexpr int NB = NB_FIT > 8 ? 8 : NB_FIT < 2 ? 2 : NB_FIT;
  static constexpr int NA_FIT = (BUDGET - NB * B_STAGE) / A_STAGE;
  static constexpr int NA = NA_FIT > NA_TARGET ? NA_TARGET : NA_FIT;
  static_assert(CG == 1 || (CG == 2 && NPAD % 32 == 0), "CTA pairs: each CTA stages half of the weight rows");
  static_assert(!F8IN || (CG == 2 && !CONCAT), "fp8 corrections: CTA-pair layers with the [hi | second part] layout");
  static constexpr int CPB = NCHUNK / NBLK;                // chunks per diagonal block
  static constexpr int N1 = CONCAT ? 2 * NPAD : NPAD;      // UMMA N of the a_hi pass
  static constexpr int BLK_COLS = DUAL ? 2 * NPAD : NPAD;   // accumulator columns per block
  static constexpr int SUB_COLS = NBLK * BLK_COLS;         // accumulator columns per sub-tile
  static constexpr int A2_COL0 = AS * S * SUB_COLS;        // tail: first TMEM column of the activation tile(s)
  // A2_SHARED: no room for one bf16 copy per sub-tile -> the sub-tiles take turns on ONE region (sub-tile s writes it
  // after the tail GEMM of sub-tile s - 1 has read it; barriers t2_sub[])
  static constexpr bool A2_SHARED = TN != 0 && AS * S * SUB_COLS + S * A2_COLS > 512;
  static constexpr int A2_REGIONS = A2_SHARED ? 1 : S;
  static constexpr int TMEM_COLS_USED = AS * S * SUB_COLS + A2_REGIONS * A2_COLS;
  static_assert(NCHUNK % NBLK == 0, "chunks must split evenly over the diagonal blocks");
  static_assert(N1 % 16 == 0 && N1 <= 256, "invalid UMMA N for the a_hi pass");
  static constexpr int TMEM_COLS = TMEM_COLS_USED <= 32 ? 32 : TMEM_COLS_USED <= 64 ? 64
                                   : TMEM_COLS_USED <= 128 ? 128 : TMEM_COLS_USED <= 256 ? 256 : 512;
  static constexpr int SMEM_BYTES = NA * A_STAGE + NB * B_STAGE + TAIL_BYTES + 2048 + 1024;  // + barriers/bias + align slack
  static_assert(NA >= 1, "halo tile does not fit in shared memory");
  static_assert(TMEM_COLS_USED <= 512, "accumulators do not fit in TMEM");
  static_assert(NPAD % 16 == 0 && NPAD >= 16 && NPAD <= 256, "invalid UMMA N");
  static_assert(TN == 0 || (CG == 2 && AS >= 2 && TNB % 32 == 0 && (TAIL_BLK ? 1 : 2) * TN <= SUB_COLS),
                "tail layer: CTA pairs, multi-buffered accumulators, and its accumulators fit the drained columns");
};

struct ActDst {
  uint4* base;   // [n][2*planes_half][H][W] of 16-byte (8 x bf16) units
  int planes_half;
};

struct ConvArgs {
  const uint8_t* wpk;   // packed weight stages
  const float* bias;    // [NPAD]
  int N, H, W;
  int in_planes_half;   // C_in_pad / 8
  int tiles_x, tiles_y;
  // kEpiAct
  ActDst dst0, dst1;
  int split_c;          // channels [0, split_c) -> dst0, [split_c, cout) -> dst1
  int cout;             // valid output channels
  // kEpiSigmoid / kEpiGate
  float* out_f32;       // [n][3][H][W] (gate: optional)
  const float* cm;      // [n][3][H][W] (gate; null = no gated sum, only refined_out is produced)
  uint8_t* out_u8;      // gate, optional: ten2arr of the result (clip [0,1], *255, truncate), uint8 NHWC
  // optional: *skip_lo != 0 means every input value is exactly representable in the hi plane
  // (8-bit image levels), so the a_lo x w_hi pass contributes nothing and is not issued
  const int* skip_lo;
  // the input planes hold exact 8-bit levels and only the hi planes exist (written by the preprocess kernel):
  // the halo loads fetch two planes per chunk instead of four and the a_lo pass is never issued
  int a_hi_only;
  // kEpiGate, training only: also store the three refined images (post-ReLU), fp32 [n][9][H][W]
  float* refined_out;
  // kEpiDgrad: saved forward activation (planes) whose zeros gate the gradient
  const uint4* mask_base;
  int mask_planes_half;
  // fp8 correction scheme (FMT bit 0): dequantisation factor 2^-9 / ws of the second accumulator
  const float* f8_scale;
  // FMT bit 1: sticky device flag raised when an activation leaves the e4m3 range (its correction terms would
  // saturate in the consumer's fp8 pass); the host side then re-runs the batch with the bf16x3 kernels
  int* f8_overflow;
  // fused tail layer (UmmaCfg TN): packed weights (two per-rank images, CG=2 CONCAT layout) and bias; dst0 / dst1 /
  // split_c / cout then describe the TAIL layer's output
  const uint8_t* wtail;
  const float* bias2;
  // K-packed first layer (UmmaCfg KP): per K step the start offset (16-byte units inside the halo stage) of its
  // lower half and the distance to the other one
  uint16_t kp_off[kKpSteps], kp_lbo[kKpSteps];
  // conditional launch: when non-null and *run_if == 0 the kernel returns at once (the bf16x3 re-run of a
  // batch is enqueued unconditionally behind the fp8-correction pass and only does work if the flag is up)
  const int* run_if;
};

__device__ __forceinline__ uint32_t pack_bf16x2(__nv_bfloat16 a, __nv_bfloat16 b) {
  return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}
// v = hi + lo with hi = bf16(v), lo = bf16(v - hi), for two values at once: two packed conversions
// (F2FP.BF16.PACK_AB) instead of four scalar F2F, and the back-conversion is a shift.
__device__ __forceinline__ void split_bf16x2(float f0, float f1, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(f0, f1);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  const float h0 = __uint_as_float(hi << 16), h1 = __uint_as_float(hi & 0xffff0000u);
  const __nv_bfloat162 l = __floats2bfloat162_rn(f0 - h0, f1 - h1);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

// TEPI   what the tail layer's epilogue stores: kTailAct = bias, ReLU, activation planes (conv4 behind conv3);
//        kTailTaps = the raw fp32 sums as planes [n][cout][H][W].  The latter serves a 3x3 layer with very few
//        output channels (cmg.conv8: 64 -> 3) in "tap-stacked" form: its 9 x 3 = 27 (tap, channel) filters are 27
//        output columns of a 1x1 tail GEMM on the UNSHIFTED tile -- column 3*tap + c of pixel q is tap's
//        contribution to output pixel q - shift(tap) -- and a small gather kernel adds the nine shifted planes.
//        Bit 1 (kTailSmem): the bf16 copy of the tile -- the tail GEMM's A operand -- goes through SHARED memory
//        (UMMA K-major layout, st.shared + fence.proxy.async) instead of tensor memory.  A tcgen05.mma that takes A from
//        TMEM costs ~150-200 cycles here whatever its N (same-box A/B, profiles/r2_ab_fused_tails.log), one from
//        shared memory 36-64; layers whose operand rings leave 64-96 KB of shared memory free (conv7, the refiners'
//        conv2) use this form, conv3 (rings need the space) the tensor-memory form.
enum TailEpilogue { kTailAct = 0, kTailTaps = 1, kTailSmem = 2 };
template <int KS, int CIN_PAD, int NPAD, int S, int AS, int EPI, int CONCAT, int NBLK, int TPS, int CG = 1, int FMT = 0,
          int TN = 0, int TEPI = kTailAct, int KP = 0>
__global__ void __launch_bounds__(kThreads, 1)
conv_umma_kernel(const __grid_constant__ CUtensorMap tmap_in, const ConvArgs g) {
  using C = UmmaCfg<KS, CIN_PAD, NPAD, S, AS, CONCAT, NBLK, TPS, CG, FMT, TN, KP, (TEPI & kTailSmem) != 0>;
  constexpr bool A2SMEM = (TEPI & kTailSmem) != 0, TAPS = (TEPI & kTailTaps) != 0;
  static_assert(TN == 0 || EPI == kEpiAct, "a tail layer follows an activation layer");
  constexpr bool F8IN = C::F8IN, DUAL = C::DUAL, OUT8 = (FMT & kFmtOut8) != 0;
  static_assert(!OUT8 || EPI == kEpiAct, "fp8 planes are written by the activation epilogue only");
  if (g.run_if != nullptr && *reinterpret_cast<const volatile int*>(g.run_if) == 0) return;  // whole grid alike
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* a_stages = smem;
  uint8_t* b_stages = smem + C::NA * C::A_STAGE;
  uint8_t* a2_tiles = b_stages + C::NB * C::B_STAGE;    // tail layer, shared-memory form: the tile(s) in operand layout
  uint8_t* wt_smem = a2_tiles + C::A2_BYTES;            // tail layer: its weights, resident for the whole launch
  uint8_t* tail = a2_tiles + C::TAIL_BYTES;
  uint64_t* a_full = reinterpret_cast<uint64_t*>(tail);
  uint64_t* a_empty = a_full + C::NA;
  uint64_t* b_full = a_empty + C::NA;
  uint64_t* b_empty = b_full + C::NB;
  uint64_t* t_full = b_empty + C::NB;
  uint64_t* t_empty = t_full + AS;
  uint64_t* a_full_peer = t_empty + AS;        // CG=2, leader: "the peer CTA's stage is full too"
  uint64_t* b_full_peer = a_full_peer + C::NA;
  uint64_t* a2_full = b_full_peer + C::NB;     // [S] tail: "sub-tile s is back in TMEM as bf16 operand" (leader's barrier counts both CTAs)
  uint64_t* t2_full = a2_full + S;             // [AS] tail: "the tail GEMM of this accumulator stage has completed"
  uint64_t* t2_sub = t2_full + AS;             // [S] tail, shared operand region: "the tail GEMM of sub-tile s has completed"
  uint64_t* wt_full = t2_sub + S;              // tail weights landed (own CTA) / (leader) in the peer CTA
  uint64_t* wt_full_peer = wt_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wt_full_peer + 1);
  float* s_bias = reinterpret_cast<float*>(tail + 512);
  float* s_bias2 = s_bias + NBLK * NPAD;
  static_assert(AS <= 4 && S <= 4 && (3 * 6 + 3 * 8 + 2 * AS + S + AS + S + 2) * 8 + 4 <= 512, "barrier area");
  static_assert((NBLK * NPAD + TN) * 4 <= 2048 - 512, "bias area");

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int num_tiles = g.tiles_x * g.tiles_y * g.N;
  // a cluster of CG CTAs takes CG adjacent tiles at a time; an odd tail repeats the last tile in the
  // peer CTA (computed, not stored) so that both CTAs walk the same pipeline sequence
  const uint32_t rank = CG == 2 ? cluster_ctarank() : 0u;
  const int cid = (int)blockIdx.x / CG, ncl = (int)gridDim.x / CG;
  const int num_ptiles = (num_tiles + CG - 1) / CG;

  if (tid == 0) {
    for (int i = 0; i < C::NA; i++) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1); mbar_init(&a_full_peer[i], 1); }
    for (int i = 0; i < C::NB; i++) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); mbar_init(&b_full_peer[i], 1); }
    for (int i = 0; i < AS; i++) { mbar_init(&t_full[i], 1); mbar_init(&t_empty[i], 8 * CG); }
    if constexpr (TN > 0) {
      for (int i = 0; i < S; i++) mbar_init(&a2_full[i], (S == 1 ? 8 : 4) * CG);
      for (int i = 0; i < AS; i++) mbar_init(&t2_full[i], 1);
      for (int i = 0; i < S; i++) mbar_init(&t2_sub[i], 1);
      mbar_init(wt_full, 1);
      mbar_init(wt_full_peer, 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = tid; i < NBLK * NPAD; i += kThreads) s_bias[i] = g.bias[i];
  if constexpr (TN > 0 && !TAPS)
    for (int i = tid; i < TN; i += kThreads) s_bias2[i] = g.bias2[i];
  if (warp == kWarpTmem) {
    if constexpr (CG == 2) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                   "r"((uint32_t)C::TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                   "r"((uint32_t)C::TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CG == 2) cluster_sync_all();  // the peer's barriers are initialised before anyone arrives on them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (tmem_base != 0) __trap();  // see the MMA issuer: accumulators are addressed from column 0

  if (warp == kWarpA) {
    // ===================== A producer: halo tiles by TMA =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int pt = cid; pt < num_ptiles; pt += ncl) {
        const int tile = min(pt * CG + (int)rank, num_tiles - 1);
        const int n = tile / (g.tiles_x * g.tiles_y);
        const int rem = tile - n * g.tiles_x * g.tiles_y;
        const int ty = rem / g.tiles_x, tx = rem - ty * g.tiles_x;
        const int x0 = tx * C::TILE_W - KS / 2 + (KP ? 1 : 0), y0 = ty * C::TILE_H - KS / 2;  // KP: column x + 1 = pixel x
        for (int c = 0; c < C::NCHUNK; c++) {
          mbar_wait(&a_empty[stage], phase ^ 1);
          uint8_t* dst = a_stages + stage * C::A_STAGE;
          mbar_expect_tx(&a_full[stage], (g.a_hi_only ? 2 : 4) * C::PLANE_BYTES);
          tma_load_5d(dst, &tmap_in, &a_full[stage], 0, x0, y0, 2 * c, n);
          if (!g.a_hi_only)
            tma_load_5d(dst + 2 * C::PLANE_BYTES, &tmap_in, &a_full[stage], 0, x0, y0,
                        g.in_planes_half + 2 * c, n);
          if (++stage == C::NA) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == kWarpB) {
    // ===================== B producer: packed weight stages =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      if constexpr (TN > 0) {  // the tail layer's weights: this rank's image, once
        mbar_expect_tx(wt_full, C::WT_BYTES);
        bulk_load(wt_smem, g.wtail + (size_t)rank * C::WT_BYTES, C::WT_BYTES, wt_full);
      }
      // CG=2: this rank's half of the weight rows (second image right after the first)
      const uint8_t* wpk = g.wpk + (size_t)rank * ((size_t)C::NCHUNK * C::NSTAGE_PER_CHUNK * C::B_STAGE);
      for (int pt = cid; pt < num_ptiles; pt += ncl) {
        for (int it = 0; it < C::NCHUNK * C::NSTAGE_PER_CHUNK; it++) {
          mbar_wait(&b_empty[stage], phase ^ 1);
          mbar_expect_tx(&b_full[stage], C::B_STAGE);
          bulk_load(b_stages + stage * C::B_STAGE, wpk + (size_t)it * C::B_STAGE, C::B_STAGE, &b_full[stage]);
          if (++stage == C::NB) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == kWarpMma && CG == 2 && rank != 0) {
    // ===================== peer CTA of a pair: relay "stage full" to the leader =====================
    // The leader issues the MMAs for both CTAs; it learns that THIS CTA's halo / weight stage has landed
    // from an arrival on its a_full_peer / b_full_peer barrier, sent here in the leader's consumption order.
    if (lane == 0) {
      int astage = 0, bstage = 0;
      uint32_t aphase = 0, bphase = 0;
      if constexpr (TN > 0) {
        mbar_wait(wt_full, 0);
        mbar_arrive_remote(wt_full_peer, 0);
      }
      for (int pt = cid; pt < num_ptiles; pt += ncl) {
        for (int c = 0; c < C::NCHUNK; c++) {
          mbar_wait(&a_full[astage], aphase);
          mbar_arrive_remote(&a_full_peer[astage], 0);
          for (int tg = 0; tg < C::NSTAGE_PER_CHUNK; tg++) {
            mbar_wait(&b_full[bstage], bphase);
            mbar_arrive_remote(&b_full_peer[bstage], 0);
            if (++bstage == C::NB) { bstage = 0; bphase ^= 1; }
          }
          if (++astage == C::NA) { astage = 0; aphase ^= 1; }
        }
      }
    }
  } else if (warp == kWarpMma) {
    // ===================== MMA issuer =====================
    // The whole warp walks the pipeline (converged, so every operand stays in uniform registers);
    // one elected lane issues the MMAs and commits.
    {
      constexpr uint32_t idesc1 = make_idesc(128 * CG, C::N1);  // a_hi pass
      constexpr uint32_t idesc2 = make_idesc(128 * CG, NPAD);   // a_lo x w_hi (and a_hi x w_lo without CONCAT)
      constexpr uint32_t idesc8 = make_idesc_f8(128 * CG, NPAD);  // fp8 correction pass
      // descriptor halves: hi = SBO | version, lo = start address | LBO
      constexpr uint32_t a_hi32 = ((uint32_t)(C::HALO_W * 16) >> 4) | (1u << 14);
      constexpr uint32_t b_hi32 = (128u >> 4) | (1u << 14);
      // weight stage: CONCAT [k8][hi rows | lo rows][16 B] (LBO = 2*NPAD*16), else [hi|lo][k8][rows][16 B]
      // CG=2 (per CTA): CONCAT [k8][NPAD rows | NPAD/2 rows of w_hi][16 B], else [hi|lo][k8][NPAD/2 rows][16 B]
      constexpr uint32_t b_lbo =
          CG == 2 ? (uint32_t)((CONCAT ? NPAD * 24 : NPAD * 8)) : (uint32_t)((CONCAT ? 2 * NPAD : NPAD) * 16);
      // start of the rows the a_lo pass multiplies (16-byte units, inside a tap)
      constexpr uint32_t b_lopass_off = (CG == 2 && CONCAT) ? (uint32_t)NPAD : 0u;
      // start of the w_lo rows for the a_hi x w_lo pass without CONCAT (16-byte units)
      constexpr uint32_t b_wlo_off = CG == 2 ? (uint32_t)NPAD : (uint32_t)(2 * NPAD * 16 >> 4);
      int astage = 0, bstage = 0, acc = 0;
      uint32_t aphase = 0, bphase = 0, tphase = 0;
      const bool skip_lo = (g.skip_lo != nullptr && *g.skip_lo != 0) || g.a_hi_only;
      bool b_ready = false;  // result of the early probe of the upcoming weight stage
      // ---- fused tail layer (UmmaCfg TN): the second GEMM of a tile is issued early in the NEXT tile's main loop:
      // polled for at the first weight stages, waited for before stage kTailForceAt.  MMAs execute in issue order,
      // so a tail GEMM issued behind a deep queue of the next tile's MMAs would hold the (single-buffered) bf16 copy
      // of its tile -- and with it the epilogue's next first pass -- for the whole queue; issued after two stages it
      // runs ~2 stages after its tile completed, while those two stages keep the tensor pipe busy during the
      // epilogue's first pass.  (ncu, conv7 + tap-stacked conv8: 12.4k -> ~8.6k cycles per tile.)
      // The tail GEMM is polled for at every weight stage of the next tile and waited for only when 3/4 of that tile's
      // stages have been issued (a safety net, not the schedule).
      constexpr int kStagesPerTile = C::NCHUNK * C::NSTAGE_PER_CHUNK;
      constexpr int kTailForceAt = kStagesPerTile * 3 / 4 < kStagesPerTile - 1 ? kStagesPerTile * 3 / 4 : kStagesPerTile - 1;
      int pend_acc = -1;            // accumulator stage whose tail GEMM is still to be issued
      int pend_sub = 0;             // shared operand region: the next sub-tile of that tile
      uint32_t a2phase = 0;
      // the tail GEMM of sub-tile sb of accumulator stage `acc`
      auto tail_mmas = [&](int tacc, int sb) {
        if constexpr (TN > 0) {
          constexpr uint32_t wt_hi32 = (128u >> 4) | (1u << 14);
          const uint32_t d2 = (uint32_t)((tacc * S + sb) * C::SUB_COLS);
          // A operand of K step `step`, hi (lo = 0) or lo (lo = 1) parts.  Tensor-memory form: 8 columns per step
          // (K = 16 bf16 pairs), lo parts K2/2 columns further.  Shared-memory form: a descriptor over
          // [k8 group][128 rows][16 B] -- LBO (the step's second k8 group) 2048 B, SBO (8-row groups) 128 B.
          const uint32_t a2_col = (uint32_t)(C::A2_COL0 + (C::A2_SHARED ? 0 : sb) * C::A2_COLS);
          const uint32_t a2_desc = A2SMEM ? (smem_u32(a2_tiles + sb * C::A2_SUB) >> 4) | ((2048u >> 4) << 16) : 0u;
          auto mma = [&](uint32_t d, int step, int lo, uint32_t w, uint32_t idesc, uint32_t accumulate) {
            if constexpr (A2SMEM)
              umma_issue<CG>(d, a2_desc + (uint32_t)((lo * (C::K2 / 8) * 2048 + step * 4096) >> 4), wt_hi32, w, wt_hi32, idesc,
                             accumulate);
            else
              umma_issue_ts<CG>(d, a2_col + (uint32_t)(lo * (C::K2 / 2) + 8 * step), w, wt_hi32, idesc, accumulate);
          };
          if constexpr (C::TAIL_BLK) {
            // block-diagonal tail (three refiners): block b = channels [K2/NBLK * b, ...) -> columns [TNB * b, ...),
            // three bf16 passes per K = 16 step into the same columns
            constexpr uint32_t idesc_b = make_idesc(128 * CG, C::TNB);
            constexpr int SPB = C::K2 / 16 / NBLK;  // K = 16 steps per block
            const uint32_t wt_lo32 = (smem_u32(wt_smem) >> 4) | ((uint32_t)(C::TNB * 8 >> 4) << 16);  // LBO: k8 halves
#pragma unroll
            for (int blk = 0; blk < NBLK; blk++)
#pragma unroll
              for (int j = 0; j < SPB; j++) {
                const int step = blk * SPB + j;
                const uint32_t w = wt_lo32 + (uint32_t)(step * (C::WT_TAP >> 4));
                const uint32_t d = d2 + (uint32_t)(blk * C::TNB);
                mma(d, step, 0, w, idesc_b, j == 0 ? 0u : 1u);                      // a_hi x w_hi
                mma(d, step, 1, w, idesc_b, 1u);                                    // a_lo x w_hi
                mma(d, step, 0, w + (uint32_t)(C::TNB * 16 >> 4), idesc_b, 1u);     // a_hi x w_lo
              }
          } else {
            constexpr uint32_t idesc_t1 = make_idesc(128 * CG, 2 * TN);   // a_hi x [w_hi | w_lo]
            constexpr uint32_t idesc_t2 = make_idesc(128 * CG, TN);       // a_lo x w_hi
            const uint32_t wt_lo32 = (smem_u32(wt_smem) >> 4) | ((uint32_t)(TN * 24 >> 4) << 16);
#pragma unroll
            for (int j = 0; j < C::K2 / 16; j++) mma(d2, j, 0, wt_lo32 + (uint32_t)(j * (C::WT_TAP >> 4)), idesc_t1, j == 0 ? 0u : 1u);
#pragma unroll
            for (int j = 0; j < C::K2 / 16; j++)
              mma(d2, j, 1, wt_lo32 + (uint32_t)(j * (C::WT_TAP >> 4)) + (uint32_t)TN, idesc_t2, 1u);
          }
        }
      };
      // stage_idx: index of the weight stage (of the NEXT tile's main loop) about to be issued; < 0 = flush
      auto tail_step = [&](int stage_idx) {
        if constexpr (TN > 0) {
          if (pend_acc < 0) return;
          if constexpr (C::A2_SHARED) {
            // one sub-tile at a time (they share the operand region): polled for at every stage, waited for from
            // stage kTailForceAt on
            const bool force = stage_idx < 0 || stage_idx >= kTailForceAt;
            if (!force && __shfl_sync(0xffffffffu, (int)mbar_try(&a2_full[pend_sub], a2phase), 0) == 0) return;
            mbar_wait(&a2_full[pend_sub], a2phase);
            tc_fence_after();
            if (elect_one_sync()) {
              tail_mmas(pend_acc, pend_sub);
              umma_done<CG>(&t2_sub[pend_sub]);
            }
            __syncwarp();
            if (++pend_sub == S) { pend_sub = 0; pend_acc = -1; a2phase ^= 1; }
          } else {
            // All sub-tiles of the tile go in ONE batch.  The decision is warp-uniform (lane 0 probes): the lanes must
            // stay converged for the election below.
            const bool force = stage_idx < 0 || stage_idx >= kTailForceAt;
            if (!force) {
              int ready = 1;
#pragma unroll
              for (int sb = 0; sb < S; sb++) ready &= (int)mbar_try(&a2_full[sb], a2phase);
              if (__shfl_sync(0xffffffffu, ready, 0) == 0) return;
            }
#pragma unroll
            for (int sb = 0; sb < S; sb++) mbar_wait(&a2_full[sb], a2phase);
            tc_fence_after();
            if (elect_one_sync()) {
#pragma unroll
              for (int sb = 0; sb < S; sb++) tail_mmas(pend_acc, sb);
              umma_done<CG>(&t2_full[pend_acc]);
            }
            __syncwarp();
            pend_acc = -1;
            a2phase ^= 1;
          }
        }
      };
      if constexpr (TN > 0) {  // the tail weights of both CTAs are in place
        mbar_wait(wt_full, 0);
        mbar_wait(wt_full_peer, 0);
      }
      for (int pt = cid; pt < num_ptiles; pt += ncl) {
        if constexpr (CG == 2) mbar_wait(&t_empty[acc], tphase ^ 1);  // both CTAs' epilogues arrive here
        else mbar_wait(&t_empty[acc], tphase ^ 1);
        tc_fence_after();
        // TMEM addresses are compile-time column offsets: this CTA is alone on its SM (shared memory
        // footprint) and owns the allocation at column 0 (checked after the allocation).
        const uint32_t d_tile = (uint32_t)(acc * S * C::SUB_COLS);
        for (int c = 0; c < C::NCHUNK; c++) {
          mbar_wait(&a_full[astage], aphase);
          if constexpr (CG == 2) mbar_wait(&a_full_peer[astage], aphase);
          tc_fence_after();
          const uint32_t a_lo32 = (smem_u32(a_stages + astage * C::A_STAGE) >> 4) | ((uint32_t)(C::PLANE_BYTES >> 4) << 16);
          const int blk = NBLK > 1 ? c / C::CPB : 0;
          const uint32_t d_base = d_tile + (uint32_t)(blk * C::BLK_COLS);
          for (int tg = 0; tg < C::NSTAGE_PER_CHUNK; tg++) {
            tail_step(c * C::NSTAGE_PER_CHUNK + tg);
            if constexpr (TN > 0) {  // nothing of the previous tile may be left when this tile's main loop ends
              if (c == C::NCHUNK - 1 && tg == C::NSTAGE_PER_CHUNK - 1)
                while (pend_acc >= 0) tail_step(-1);
            }
            if (!b_ready) mbar_wait(&b_full[bstage], bphase);
            if constexpr (CG == 2) mbar_wait(&b_full_peer[bstage], bphase);
            tc_fence_after();
            {  // probe the next stage's barrier now; its latency overlaps the MMA issue below
              const int nstage = bstage + 1 == C::NB ? 0 : bstage + 1;
              b_ready = mbar_try(&b_full[nstage], nstage == 0 ? bphase ^ 1 : bphase);
            }
            const uint32_t b_stage32 = (smem_u32(b_stages + bstage * C::B_STAGE) >> 4) | ((b_lbo >> 4) << 16);
            if (elect_one_sync()) {
              constexpr uint32_t a_lo_off = (uint32_t)(2 * C::PLANE_BYTES >> 4);
#pragma unroll
              for (int t = 0; t < TPS; t++) {
                const int tap = tg * TPS + t;
                const int ky = tap / KS, kx = tap - ky * KS;
                const uint32_t b_lo32 = b_stage32 + (uint32_t)(t * (C::B_TAP >> 4));
                // K-packed: "tap" is a K step whose two halves are any two rows of the stage (table-driven)
                const uint32_t a_tap = KP ? (a_lo32 & 0xffffu) + (uint32_t)g.kp_off[tap] + ((uint32_t)g.kp_lbo[tap] << 16)
                                          : a_lo32 + (uint32_t)(ky * C::HALO_W + kx);
                const uint32_t first = ((NBLK > 1 ? c % C::CPB : c) | tap) == 0 ? 0u : 1u;
                // pass-major order: consecutive MMAs target different accumulators
#pragma unroll
                for (int s = 0; s < S; s++)  // a_hi x w_hi (CONCAT: x [w_hi | w_lo])
                  umma_issue<CG>(d_base + (uint32_t)(s * C::SUB_COLS), a_tap + (uint32_t)(s * kSubW), a_hi32, b_lo32,
                                 b_hi32, idesc1, first);
                if constexpr (F8IN) {
#pragma unroll
                  for (int s = 0; s < S; s++)  // [e4m3(lo*2^9) | e4m3(v)] x [e4m3(w*ws) ; e4m3(w_lo*ws*2^9)], K = 32
                    umma_issue_f8<CG>(d_base + (uint32_t)(s * C::SUB_COLS), a_tap + (uint32_t)(s * kSubW) + a_lo_off,
                                      a_hi32, b_lo32 + b_wlo_off, b_hi32, idesc8, 1u);
                } else if (!skip_lo) {
#pragma unroll
                  for (int s = 0; s < S; s++)  // a_lo x w_hi
                    umma_issue<CG>(d_base + (uint32_t)(s * C::SUB_COLS), a_tap + (uint32_t)(s * kSubW) + a_lo_off,
                                   a_hi32, b_lo32 + b_lopass_off, b_hi32, idesc2, 1u);
                }
                if (!CONCAT && !F8IN) {
#pragma unroll
                  for (int s = 0; s < S; s++)  // a_hi x w_lo
                    umma_issue<CG>(d_base + (uint32_t)(s * C::SUB_COLS), a_tap + (uint32_t)(s * kSubW), a_hi32,
                                   b_lo32 + b_wlo_off, b_hi32, idesc2, 1u);
                }
              }
              umma_done<CG>(&b_empty[bstage]);
              if (tg == C::NSTAGE_PER_CHUNK - 1) {
                umma_done<CG>(&a_empty[astage]);
                if (c == C::NCHUNK - 1) umma_done<CG>(&t_full[acc]);
              }
            }
            __syncwarp();
            if (++bstage == C::NB) { bstage = 0; bphase ^= 1; }
          }
          if (++astage == C::NA) { astage = 0; aphase ^= 1; }
        }
        if constexpr (TN > 0) pend_acc = acc;
        if (++acc == AS) { acc = 0; tphase ^= 1; }
      }
      while (pend_acc >= 0) tail_step(-1);  // the last tile's tail GEMM(s)
    }
  } else if (warp < 8) {
    // ===================== epilogue =====================
    // a warp may only touch TMEM lanes 32*(warp%4)..+31; the two groups take alternate sub-tiles
    int acc = 0;
    uint32_t tphase = 0;
    uint32_t tile_phase = 0;   // fused tail, shared operand region: parity of the per-tile barriers t2_sub[]
    const int egroup = warp >> 2, quarter = warp & 3;
    const int row = quarter * 32 + lane;      // TMEM lane == pixel row of the sub-tile
    const int px = row & 7, py = row >> 3;
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    const float dscale = F8IN ? *g.f8_scale : 1.f;
    for (int pt = cid; pt < num_ptiles; pt += ncl) {
      const bool tile_valid = pt * CG + (int)rank < num_tiles;  // the odd tail's repeat is not stored
      const int tile = min(pt * CG + (int)rank, num_tiles - 1);
      const int n = tile / (g.tiles_x * g.tiles_y);
      const int rem = tile - n * g.tiles_x * g.tiles_y;
      const int ty = rem / g.tiles_x, tx = rem - ty * g.tiles_x;
      mbar_wait(&t_full[acc], tphase);
      tc_fence_after();
      const int gy = ty * C::TILE_H + py;
      // the two epilogue groups take alternate sub-tiles; a single sub-tile (S == 1) is split by channel
      // groups instead (a warp may read any columns of its own 32 TMEM lanes)
      static_assert(S > 1 || EPI == kEpiAct || EPI == kEpiDgrad, "S == 1 needs the channel-group split");
      if constexpr (TN > 0) {
        // ===== fused tail layer =====
        // pass 1: this layer's activations (bias, ReLU, bf16 hi/lo) -> tensor memory as packed bf16 pairs
        //         (K2/2 columns of hi parts, K2/2 of lo parts); then "sub-tile ready" to the issuer
        constexpr int GC = 32, NG = NBLK * NPAD / GC, STEP = S == 1 ? 2 : 1;
        static_assert(S <= 2 && !DUAL && (NBLK * NPAD) % GC == 0, "tail layer: tile shape (one accumulator per channel)");
        static_assert(!C::A2_SHARED || S == 2, "shared operand region: one epilogue group per sub-tile");
#pragma unroll 1
        for (int s = (S == 1 ? 0 : egroup); s < S; s += 2) {
          const uint32_t t_addr = tmem_base + lane_base + (uint32_t)((acc * S + s) * C::SUB_COLS);
          const uint32_t a2_addr = tmem_base + lane_base + (uint32_t)(C::A2_COL0 + (C::A2_SHARED ? 0 : s) * C::A2_COLS);
          if constexpr (C::A2_SHARED) {
            // the sub-tiles take turns on one operand region: wait until the tail GEMM of the previous user has
            // read it -- sub-tile s - 1 of this tile, or (s == 0) the last sub-tile of the previous tile
            if (s > 0) mbar_wait(&t2_sub[s - 1], tile_phase);
            else if (pt != cid) mbar_wait(&t2_sub[S - 1], tile_phase ^ 1);
            tc_fence_after();
          }
          uint32_t vb[2][GC], wb[2][DUAL ? GC : 1];
          auto issue1 = [&](int ch0, uint32_t* v, uint32_t* w) {
#pragma unroll
            for (int q = 0; q < GC; q += 16) tmem_ld16(t_addr + (uint32_t)(ch0 + q), v + q);
            if constexpr (DUAL) {
#pragma unroll
              for (int q = 0; q < GC; q += 16) tmem_ld16(t_addr + (uint32_t)(ch0 + NPAD + q), w + q);
            }
          };
          const int first = S == 1 ? egroup : 0;
          const int cnt = (NG - first + STEP - 1) / STEP;   // S == 1: the two epilogue groups take alternate channel groups
          if (cnt > 0) issue1(first * GC, vb[0], wb[0]);
#pragma unroll
          for (int k = 0; k < (NG + STEP - 1) / STEP; k++) {
            if (k >= cnt) break;
            const int c0 = (first + k * STEP) * GC;
            tmem_ld_wait();
            if (k + 1 < cnt) issue1(c0 + STEP * GC, vb[(k + 1) & 1], wb[(k + 1) & 1]);
            uint32_t hi[GC / 2], lo[GC / 2];   // bf16 pairs (channel c in the low half, c + 1 in the high half)
#pragma unroll
            for (int j = 0; j < GC; j += 2) {
              const float a0 = F8IN ? __uint_as_float(vb[k & 1][j]) * dscale
                                    : __uint_as_float(vb[k & 1][j]) + (DUAL ? __uint_as_float(wb[k & 1][DUAL ? j : 0]) : 0.f);
              const float a1 = F8IN ? __uint_as_float(vb[k & 1][j + 1]) * dscale
                                    : __uint_as_float(vb[k & 1][j + 1]) + (DUAL ? __uint_as_float(wb[k & 1][DUAL ? j + 1 : 0]) : 0.f);
              split_bf16x2(fmaxf(a0 + s_bias[c0 + j], 0.f), fmaxf(a1 + s_bias[c0 + j + 1], 0.f), hi[j >> 1], lo[j >> 1]);
            }
            if constexpr (A2SMEM) {
              // [k8 group][row][16 B]: group g of this row holds channels 8g..8g+7 = four bf16 pairs
              uint4* a2_hi = reinterpret_cast<uint4*>(a2_tiles + s * C::A2_SUB) + row;
              uint4* a2_lo = a2_hi + (C::K2 / 8) * 128;
#pragma unroll
              for (int q = 0; q < GC / 8; q++) {
                a2_hi[((c0 >> 3) + q) * 128] = make_uint4(hi[4 * q], hi[4 * q + 1], hi[4 * q + 2], hi[4 * q + 3]);
                a2_lo[((c0 >> 3) + q) * 128] = make_uint4(lo[4 * q], lo[4 * q + 1], lo[4 * q + 2], lo[4 * q + 3]);
              }
            } else {
              tmem_st16(a2_addr + (uint32_t)(c0 >> 1), hi);
              tmem_st16(a2_addr + (uint32_t)(C::K2 / 2 + (c0 >> 1)), lo);
            }
          }
          if constexpr (A2SMEM) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy stores -> tensor core
          else tmem_st_wait();
          // the tail GEMM reads the columns just written and overwrites the accumulator columns just read
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            // plain arrival: what is handed over lives in tensor memory (tcgen05.st + wait::st + fence above), not in
            // generic memory -- a cluster-scope release here compiles to MEMBAR.ALL.GPU and waits ~1 us for the previous
            // tile's global stores, on the path every tail GEMM waits for (ncu source page: ERRBAR / MEMBAR stalls)
            if constexpr (CG == 2) mbar_arrive_remote(&a2_full[s], 0);
            else mbar_arrive(&a2_full[s]);
          }
        }
        // pass 2: the tail layer's accumulators (CONCAT: [a x w_hi | a_hi x w_lo]) -> bias, ReLU -> planes in HBM
        if constexpr (C::A2_SHARED) mbar_wait(&t2_sub[S == 1 ? 0 : egroup], tile_phase);  // this group's sub-tile
        else mbar_wait(&t2_full[acc], tphase);
        tc_fence_after();
        constexpr int NG2 = TN / GC;
        static_assert(!TAPS || !OUT8, "the tap-stacked tail stores raw sums");
#pragma unroll 1
        for (int s = (S == 1 ? 0 : egroup); s < S; s += 2) {
          const int gx = tx * C::TILE_W + s * kSubW + px;
          const bool inside = gx < g.W && gy < g.H && tile_valid;
          const uint32_t t_addr = tmem_base + lane_base + (uint32_t)((acc * S + s) * C::SUB_COLS);
          const size_t pix = (size_t)gy * g.W + gx;
          const size_t hw = (size_t)g.H * g.W;
#pragma unroll
          for (int k = 0; k < NG2; k++) {
            if (S == 1 && (k & 1) != egroup) continue;   // S == 1: alternate channel groups per epilogue group
            const int c0 = k * GC;
            uint32_t v[GC], w[C::TAIL_BLK ? 1 : GC];
#pragma unroll
            for (int q = 0; q < GC; q += 16) tmem_ld16(t_addr + (uint32_t)(c0 + q), v + q);
            if constexpr (!C::TAIL_BLK) {   // CONCAT form: the a_hi x w_lo products sit TN columns further
#pragma unroll
              for (int q = 0; q < GC; q += 16) tmem_ld16(t_addr + (uint32_t)(TN + c0 + q), w + q);
            }
            tmem_ld_wait();
            if constexpr (!C::TAIL_BLK) {
#pragma unroll
              for (int j = 0; j < GC; j++) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(w[j]));
            }
            if (!inside) continue;
            if constexpr (TAPS) {
              // group k = one 3x3 layer with 3 output channels, tap-stacked: 27 of its 32 columns are in use
              float* o = g.out_f32 + ((size_t)n * (NG2 * 27) + k * 27) * hw + pix;
#pragma unroll
              for (int j = 0; j < 27; j++) o[(size_t)j * hw] = __uint_as_float(v[j]);
            } else if (c0 >= g.cout) {
              continue;
            } else if constexpr (OUT8) {
#pragma unroll
              for (int q = 0; q < GC; q += 16) {
                const int ch = c0 + q;
                uint32_t hi[8], l8[4], h8[4];
                float vmax = 0.f;
#pragma unroll
                for (int j = 0; j < 16; j += 4) {
                  float x[4], r[4];
#pragma unroll
                  for (int t = 0; t < 4; t++) {
                    x[t] = fmaxf(__uint_as_float(v[q + j + t]) + s_bias2[ch + j + t], 0.f);
                    vmax = fmaxf(vmax, x[t]);
                  }
#pragma unroll
                  for (int t = 0; t < 4; t += 2) {
                    const __nv_bfloat162 hh = __floats2bfloat162_rn(x[t], x[t + 1]);
                    const uint32_t hb = *reinterpret_cast<const uint32_t*>(&hh);
                    hi[(j + t) >> 1] = hb;
                    r[t] = (x[t] - __uint_as_float(hb << 16)) * 512.f;
                    r[t + 1] = (x[t + 1] - __uint_as_float(hb & 0xffff0000u)) * 512.f;
                  }
                  l8[j >> 2] = pack_e4m3x4(r[0], r[1], r[2], r[3]);
                  h8[j >> 2] = pack_e4m3x4(x[0], x[1], x[2], x[3]);
                }
                if (!(vmax <= 448.f) && g.f8_overflow) atomicOr(g.f8_overflow, 1);
                const ActDst& d = g.dst0;
                uint4* p_hi = d.base + ((size_t)n * 2 * d.planes_half + (ch >> 3)) * hw + pix;
                uint4* p_f8 = d.base + ((size_t)n * 2 * d.planes_half + d.planes_half + 2 * (ch >> 4)) * hw + pix;
                p_hi[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                p_hi[hw] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
                p_f8[0] = make_uint4(l8[0], l8[1], l8[2], l8[3]);
                p_f8[hw] = make_uint4(h8[0], h8[1], h8[2], h8[3]);
              }
            } else {
#pragma unroll
              for (int q = 0; q < GC; q += 8) {
                const int ch = c0 + q;
                uint32_t hi[4], lo[4];
#pragma unroll
                for (int j = 0; j < 8; j += 2)
                  split_bf16x2(fmaxf(__uint_as_float(v[q + j]) + s_bias2[ch + j], 0.f),
                               fmaxf(__uint_as_float(v[q + j + 1]) + s_bias2[ch + j + 1], 0.f), hi[j >> 1], lo[j >> 1]);
                const ActDst& d = g.dst0;
                uint4* p_hi = d.base + ((size_t)n * 2 * d.planes_half + (ch >> 3)) * hw + pix;
                p_hi[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                p_hi[(size_t)d.planes_half * hw] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
              }
            }
          }
        }
      } else {
#pragma unroll 1
      for (int s = (S == 1 ? 0 : egroup); s < S; s += 2) {
        const int gx = tx * C::TILE_W + s * kSubW + px;
        const bool inside = gx < g.W && gy < g.H && tile_valid;
        const uint32_t t_addr = tmem_base + lane_base + (uint32_t)((acc * S + s) * C::SUB_COLS);
        // Issue the TMEM loads of NC accumulator columns starting at output channel ch0 (+ the
        // a_hi x w_lo half when CONCAT); the caller waits once, later, so loads overlap ALU work.
        auto issue_cols = [&](int ch0, uint32_t* v, uint32_t* w, auto nc_tag) {
          constexpr int NC = decltype(nc_tag)::value;
          const int blk = NBLK > 1 ? ch0 / NPAD : 0;
          const uint32_t col = (uint32_t)(blk * C::BLK_COLS + (NBLK > 1 ? ch0 % NPAD : ch0));
#pragma unroll
          for (int q = 0; q < NC; q += 16) tmem_ld16(t_addr + col + q, v + q);
          if constexpr (DUAL) {
#pragma unroll
            for (int q = 0; q < NC; q += 16) tmem_ld16(t_addr + col + NPAD + q, w + q);
          }
        };
        if constexpr (EPI == kEpiAct || EPI == kEpiDgrad) {
          constexpr int GC = 32;  // channels per group
          constexpr int NG = NBLK * NPAD / GC;
          static_assert((NBLK * NPAD) % GC == 0 && (NBLK == 1 || NPAD % GC == 0), "channel groups of 32");
          auto act_groups = [&](auto first_tag) {
          constexpr int FIRST = decltype(first_tag)::value;
          constexpr int STEP = S == 1 ? 2 : 1;
          constexpr int CNT = (NG - FIRST + STEP - 1) / STEP;
          uint32_t vb[2][GC], wb[2][DUAL ? GC : 1];
          if constexpr (CNT > 0) issue_cols(FIRST * GC, vb[0], wb[0], std::integral_constant<int, GC>{});
#pragma unroll
          for (int k = 0; k < CNT; k++) {
            const int gi = FIRST + k * STEP;
            const int c0 = gi * GC;
            tmem_ld_wait();
            if (k + 1 < CNT)
              issue_cols(c0 + STEP * GC, vb[(k + 1) & 1], wb[(k + 1) & 1], std::integral_constant<int, GC>{});
            float f[GC];
#pragma unroll
            for (int j = 0; j < GC; j++)
              f[j] = F8IN ? __uint_as_float(vb[k & 1][j]) * dscale
                          : __uint_as_float(vb[k & 1][j]) + (DUAL ? __uint_as_float(wb[k & 1][DUAL ? j : 0]) : 0.f);
            if (c0 < g.cout && inside) {
              const size_t pix = (size_t)gy * g.W + gx;
              const size_t hw = (size_t)g.H * g.W;
              if constexpr (OUT8) {
                // hi planes as usual; where the bf16 lo planes would be: per 16 channels one plane of
                // e4m3((v - hi) * 2^9) and one of e4m3(v) -- the K = 32 operand of the consumer's fp8 pass
#pragma unroll
                for (int q = 0; q < GC; q += 16) {
                  const int ch = c0 + q;
                  uint32_t hi[8], l8[4], h8[4];
                  float vmax = 0.f;
#pragma unroll
                  for (int j = 0; j < 16; j += 4) {
                    float v[4], r[4];
#pragma unroll
                    for (int t = 0; t < 4; t++) {
                      v[t] = fmaxf(f[q + j + t] + s_bias[ch + j + t], 0.f);
                      vmax = fmaxf(vmax, v[t]);
                    }
#pragma unroll
                    for (int t = 0; t < 4; t += 2) {
                      const __nv_bfloat162 h = __floats2bfloat162_rn(v[t], v[t + 1]);
                      const uint32_t hb = *reinterpret_cast<const uint32_t*>(&h);
                      hi[(j + t) >> 1] = hb;
                      r[t] = (v[t] - __uint_as_float(hb << 16)) * 512.f;
                      r[t + 1] = (v[t + 1] - __uint_as_float(hb & 0xffff0000u)) * 512.f;
                    }
                    l8[j >> 2] = pack_e4m3x4(r[0], r[1], r[2], r[3]);
                    h8[j >> 2] = pack_e4m3x4(v[0], v[1], v[2], v[3]);
                  }
                  // e4m3 range guard (|v| <= 448); written as !(<=) so that a NaN raises the flag too
                  if (!(vmax <= 448.f) && g.f8_overflow) atomicOr(g.f8_overflow, 1);
                  const bool second = ch >= g.split_c;
                  const ActDst& d = second ? g.dst1 : g.dst0;
                  const int chl = second ? ch - g.split_c : ch;
                  uint4* p_hi = d.base + ((size_t)n * 2 * d.planes_half + (chl >> 3)) * hw + pix;
                  uint4* p_f8 = d.base + ((size_t)n * 2 * d.planes_half + d.planes_half + 2 * (chl >> 4)) * hw + pix;
                  p_hi[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                  p_hi[hw] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
                  p_f8[0] = make_uint4(l8[0], l8[1], l8[2], l8[3]);
                  p_f8[hw] = make_uint4(h8[0], h8[1], h8[2], h8[3]);
                }
              } else {
#pragma unroll
              for (int q = 0; q < GC; q += 8) {  // one 8-channel plane at a time
                const int ch = c0 + q;
                uint32_t hi[4], lo[4];
                uint32_t mask[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
                if constexpr (EPI == kEpiDgrad) {
                  if (g.mask_base) {  // no mask: gradient with respect to the network input (no ReLU in front)
                    const uint4 m = g.mask_base[((size_t)n * 2 * g.mask_planes_half + (ch >> 3)) * hw + pix];
                    mask[0] = m.x; mask[1] = m.y; mask[2] = m.z; mask[3] = m.w;
                  }
                }
#pragma unroll
                for (int j = 0; j < 8; j += 2) {
                  float f0, f1;
                  if constexpr (EPI == kEpiDgrad) {  // ReLU': pass the gradient where the activation was > 0
                    f0 = (mask[j >> 1] & 0x0000ffffu) ? f[q + j] : 0.f;
                    f1 = (mask[j >> 1] & 0xffff0000u) ? f[q + j + 1] : 0.f;
                  } else {
                    f0 = fmaxf(f[q + j] + s_bias[ch + j], 0.f);
                    f1 = fmaxf(f[q + j + 1] + s_bias[ch + j + 1], 0.f);
                  }
                  split_bf16x2(f0, f1, hi[j >> 1], lo[j >> 1]);
                }
                const bool second = ch >= g.split_c;
                const ActDst& d = second ? g.dst1 : g.dst0;
                const int plane = (second ? ch - g.split_c : ch) >> 3;
                uint4* p_hi = d.base + ((size_t)n * 2 * d.planes_half + plane) * hw + pix;
                p_hi[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                p_hi[(size_t)d.planes_half * hw] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
              }
              }
            }
          }
          };  // act_groups
          if constexpr (S == 1) {
            if (egroup == 0) act_groups(std::integral_constant<int, 0>{});
            else act_groups(std::integral_constant<int, 1>{});
          } else {
            act_groups(std::integral_constant<int, 0>{});
          }
        } else {
          uint32_t v16[16], w16[DUAL ? 16 : 1];
          issue_cols(0, v16, w16, std::integral_constant<int, 16>{});
          tmem_ld_wait();
          float f[16];
#pragma unroll
          for (int j = 0; j < 16; j++)
            f[j] = F8IN ? __uint_as_float(v16[j]) * dscale
                        : __uint_as_float(v16[j]) + (DUAL ? __uint_as_float(w16[DUAL ? j : 0]) : 0.f);
          if (inside) {
            const size_t hw = (size_t)g.H * g.W;
            const size_t o = (size_t)n * 3 * hw + (size_t)gy * g.W + gx;
            if constexpr (EPI == kEpiSigmoid) {
#pragma unroll
              for (int c = 0; c < 3; c++) g.out_f32[o + c * hw] = 1.0f / (1.0f + expf(-(f[c] + s_bias[c])));
            } else {  // kEpiGate: columns 3r+c = refiner r, colour c  (net.py:104-108)
              float r[9];
#pragma unroll
              for (int j = 0; j < 9; j++) r[j] = fmaxf(f[j] + s_bias[j], 0.f);
              if (g.refined_out) {
#pragma unroll
                for (int j = 0; j < 9; j++) g.refined_out[(size_t)n * 9 * hw + (size_t)gy * g.W + gx + j * hw] = r[j];
              }
              if (g.cm) {
                const float c0 = g.cm[o], c1 = g.cm[o + hw], c2 = g.cm[o + 2 * hw];
                float v[3];
#pragma unroll
                for (int c = 0; c < 3; c++)
                  v[c] = __fadd_rn(__fadd_rn(__fmul_rn(r[c], c0), __fmul_rn(r[3 + c], c1)), __fmul_rn(r[6 + c], c2));
                if (g.out_f32) {
#pragma unroll
                  for (int c = 0; c < 3; c++) g.out_f32[o + c * hw] = v[c];
                }
                if (g.out_u8) {  // ten2arr (hubconf.py:24-34): clip to [0,1], *255, truncate; NHWC
                  uint8_t* q = g.out_u8 + ((size_t)n * hw + (size_t)gy * g.W + gx) * 3;
#pragma unroll
                  for (int c = 0; c < 3; c++) q[c] = (uint8_t)(int)__fmul_rn(fminf(fmaxf(v[c], 0.0f), 1.0f), 255.0f);
                }
              }
            }
          }
        }
      }
      }  // TN == 0
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (CG == 2) mbar_arrive_remote(&t_empty[acc], 0);  // the leader's barrier counts both CTAs
        else mbar_arrive(&t_empty[acc]);
      }
      if (++acc == AS) { acc = 0; tphase ^= 1; }
      tile_phase ^= 1;
    }
  }

  tc_fence_before();
  __syncthreads();
  if constexpr (CG == 2) cluster_sync_all();  // nobody leaves (or frees TMEM) while the pair still works
  if (warp == kWarpTmem) {
    tc_fence_after();
    if constexpr (CG == 2)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                   "r"((uint32_t)C::TMEM_COLS)
                   : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                   "r"((uint32_t)C::TMEM_COLS)
                   : "memory");
  }
}

// ------------------------------------------------------------------------------------------
// Operand packing kernels
// ------------------------------------------------------------------------------------------
// scatter one OIHW fp32 tensor into a dense [npad][cinpad][ks*ks] fp32 block-matrix
static __global__ void scatter_weights_kernel(const float* __restrict__ src, float* __restrict__ dense, int co, int ci,
                                       int kk, int cinpad, int row_off, int split, int base0, int base1,
                                       float divisor) {
  const int total = co * ci * kk;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int t = i % kk;
    int c = (i / kk) % ci;
    int o = i / (kk * ci);
    int cd = c < split ? base0 + c : base1 + (c - split);
    dense[((size_t)(row_off + o) * cinpad + cd) * kk + t] = __fdiv_rn(src[i], divisor);
  }
}
static __global__ void scatter_bias_kernel(const float* __restrict__ src, float* __restrict__ dst, int co, int row_off) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < co; i += gridDim.x * blockDim.x) dst[row_off + i] = src[i];
}
// dense fp32 [nblk*npad][cinpad][kk] -> weight stages, one per (chunk, tap), holding the rows of the
// diagonal block the chunk feeds:  concat ? [k8][hi rows | lo rows][8] : [hi|lo][k8][rows][8]   (bf16)
static __global__ void pack_stages_kernel(const float* __restrict__ dense, __nv_bfloat16* __restrict__ out, int npad,
                                   int cinpad, int kk, int concat, int nblk) {
  const int nchunk = cinpad / 16, cpb = nchunk / nblk;
  const size_t total = (size_t)nchunk * kk * 2 * 2 * npad * 8;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int e = (int)(i % 8);
    size_t r = i / 8;
    int k8, split, nrow;
    if (concat) {
      int row2 = (int)(r % (2 * npad)); r /= 2 * npad;
      k8 = (int)(r % 2); r /= 2;
      split = row2 >= npad;
      nrow = row2 - split * npad;
    } else {
      nrow = (int)(r % npad); r /= npad;
      k8 = (int)(r % 2); r /= 2;
      split = (int)(r % 2); r /= 2;
    }
    int tap = (int)(r % kk);
    int chunk = (int)(r / kk);
    int cin = chunk * 16 + k8 * 8 + e;
    int row = (chunk / cpb) * npad + nrow;
    float w = dense[((size_t)row * cinpad + cin) * kk + tap];
    __nv_bfloat16 hi = __float2bfloat16_rn(w);
    out[i] = split == 0 ? hi : __float2bfloat16_rn(w - __bfloat162float(hi));
  }
}

// CTA-pair (CG=2) weight stages: two images, one per cluster rank, each holding that rank's half of the
// N dimension per (chunk, tap) -- see UmmaCfg::B_TAP.  dense is [nblk*npad][cinpad][kk]; a chunk only
// carries the rows of the diagonal block it feeds.
static __global__ void pack_stages_cg2_kernel(const float* __restrict__ dense, __nv_bfloat16* __restrict__ out,
                                              int npad, int cinpad, int kk, int concat, int nblk) {
  const int nchunk = cinpad / 16, cpb = nchunk / nblk;
  const int rows = concat ? npad + npad / 2 : npad / 2;        // rows per k8 group (per hi/lo part)
  const int parts = concat ? 1 : 2;                            // non-concat: hi part then lo part
  const size_t per_rank = (size_t)nchunk * kk * parts * 2 * rows * 8;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < 2 * per_rank; i += (size_t)gridDim.x * blockDim.x) {
    const int rank = (int)(i / per_rank);
    size_t r = i % per_rank;
    const int e = (int)(r % 8); r /= 8;
    const int q = (int)(r % rows); r /= rows;
    const int k8 = (int)(r % 2); r /= 2;
    const int part = (int)(r % parts); r /= parts;
    const int tap = (int)(r % kk);
    const int chunk = (int)(r / kk);
    int row, lo;
    if (concat) {
      if (q < npad) { row = q; lo = rank; }                      // hi pass: rank 0 supplies w_hi, rank 1 w_lo
      else { row = rank * (npad / 2) + (q - npad); lo = 0; }     // a_lo pass: this rank's half of w_hi
    } else {
      row = rank * (npad / 2) + q;
      lo = part;
    }
    const int cin = chunk * 16 + k8 * 8 + e;
    const float w = dense[((size_t)((chunk / cpb) * npad + row) * cinpad + cin) * kk + tap];
    const __nv_bfloat16 hi = __float2bfloat16_rn(w);
    out[i] = lo == 0 ? hi : __float2bfloat16_rn(w - __bfloat162float(hi));
  }
}

// fp8 correction scheme (UmmaCfg FMT bit 0), CTA pairs: per rank, per (chunk, tap):
//   part 0  [k8 0|1][rows][8 bf16]            w_hi * ws * 2^9              (K = 16 bf16 MMA)
//   part 1  [k16 0|1][rows][16 fp8 (e4m3)]    w * ws  |  w_lo * ws * 2^9   (K = 32 fp8 MMA)
// with rows = npad/2 of this rank.  scale[0] = ws (a power of two placing max|w| in [112, 224]),
// scale[1] = 2^-9 / ws (what the epilogue multiplies the second accumulator with); scale[2] = max|w|.
// scale[2] (as unsigned bits) accumulates max|w| over the grid (bit patterns of non-negative floats are
// ordered like the floats); f8_scale_finish_kernel turns it into scale[0], scale[1].
static __global__ void f8_absmax_kernel(const float* __restrict__ dense, size_t n, float* __restrict__ scale) {
  __shared__ float smax[256];
  float m = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(dense[i]));
  smax[threadIdx.x] = m;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) smax[threadIdx.x] = fmaxf(smax[threadIdx.x], smax[threadIdx.x + o]);
    __syncthreads();
  }
  if (threadIdx.x == 0) atomicMax(reinterpret_cast<unsigned int*>(scale + 2), __float_as_uint(smax[0]));
}
static __global__ void f8_scale_finish_kernel(float* __restrict__ scale) {
  const float mx = fmaxf(scale[2], 1e-30f);
  const float ws = exp2f(floorf(log2f(224.f / mx)));
  scale[0] = ws;
  scale[1] = 1.f / (512.f * ws);
}
static __global__ void pack_stages_f8_cg2_kernel(const float* __restrict__ dense, uint8_t* __restrict__ out,
                                                 const float* __restrict__ scale, int npad, int cinpad, int kk,
                                                 int nblk) {
  const int nchunk = cinpad / 16, cpb = nchunk / nblk, rows = npad / 2;
  const size_t tap_bytes = (size_t)rows * 64;
  const size_t per_rank = (size_t)nchunk * kk * tap_bytes;
  const float ws = scale[0];
  // one thread per (rank, chunk, tap, row, channel pair of the chunk)
  const size_t total = (size_t)2 * nchunk * kk * rows * 8;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    size_t r = i;
    const int cp = (int)(r % 8); r /= 8;            // channels 2cp, 2cp+1 of the chunk
    const int row = (int)(r % rows); r /= rows;
    const int tap = (int)(r % kk); r /= kk;
    const int chunk = (int)(r % nchunk);
    const int rank = (int)(r / nchunk);
    const int wrow = (chunk / cpb) * npad + rank * rows + row;
    float w[2], wl[2];
    uint16_t hb[2];
#pragma unroll
    for (int t = 0; t < 2; t++) {
      w[t] = dense[((size_t)wrow * cinpad + chunk * 16 + 2 * cp + t) * kk + tap];
      const __nv_bfloat16 h = __float2bfloat16_rn(w[t]);
      hb[t] = __bfloat16_as_ushort(h);
      wl[t] = w[t] - __bfloat162float(h);
    }
    uint8_t* base = out + (size_t)rank * per_rank + ((size_t)chunk * kk + tap) * tap_bytes;
    // part 0: channel c = 2cp+t -> k8 = c / 8, element c % 8.  bf16(w) * (ws * 2^9): an exact power-of-two scaling
    // that puts the bf16 product on the scale of the fp8 correction product (one shared accumulator)
    const int c = 2 * cp;
#pragma unroll
    for (int t = 0; t < 2; t++)
      hb[t] = __bfloat16_as_ushort(__float2bfloat16_rn(__bfloat162float(__ushort_as_bfloat16(hb[t])) * ws * 512.f));
    *reinterpret_cast<uint32_t*>(base + ((size_t)(c / 8) * rows + row) * 16 + (c % 8) * 2) =
        (uint32_t)hb[0] | ((uint32_t)hb[1] << 16);
    // part 1: K half 0 = e4m3(w * ws), K half 1 = e4m3(w_lo * ws * 512), 16 channels per row
    uint8_t* p1 = base + (size_t)rows * 32;
    *reinterpret_cast<uint16_t*>(p1 + ((size_t)0 * rows + row) * 16 + c) = pack_e4m3x2(w[0] * ws, w[1] * ws);
    *reinterpret_cast<uint16_t*>(p1 + ((size_t)1 * rows + row) * 16 + c) =
        pack_e4m3x2(wl[0] * ws * 512.f, wl[1] * ws * 512.f);
  }
}

// ------------------------------------------------------------------------------------------
// K-packed first layer (UmmaCfg KP): the table of K steps and the matching weight images
// ------------------------------------------------------------------------------------------
// One 8-element K half: plane 0 row = channels 0-7 of tap (ky, kx); plane 1 row = channels 8-11 of taps (ky, kx) and
// (ky, kx + 1); type 2 = padding (zero weights).
struct KpHalf {
  int8_t type, ky, kx;
};
struct KpTable {
  KpHalf half[2 * kKpSteps];   // half[2 * step + k8]: the step's lower-address / higher-address half
  uint16_t off[kKpSteps], lbo[kKpSteps];
};
// halo_w, plane_units: geometry of the halo stage (16-byte units).  Halves in kernel-row order: plane 0 at kx = 0..6,
// plane 1 at kx = 0, 2, 4, 6 (77 halves), padded to 80; consecutive halves pair up, lower address first.
static KpTable l1k_table(int halo_w, int plane_units) {
  KpTable t;
  KpHalf seq[2 * kKpSteps];
  int n = 0;
  for (int ky = 0; ky < 7; ky++) {
    for (int kx = 0; kx < 7; kx++) seq[n++] = KpHalf{0, (int8_t)ky, (int8_t)kx};
    for (int kx = 0; kx < 7; kx += 2) seq[n++] = KpHalf{1, (int8_t)ky, (int8_t)kx};
  }
  // padding halves: distinct valid rows (their weights are zero)
  seq[n++] = KpHalf{2, 0, 0};
  seq[n++] = KpHalf{2, 0, 1};
  seq[n++] = KpHalf{2, 0, 2};
  auto addr = [&](const KpHalf& hf) { return (hf.type == 1 ? plane_units : 0) + hf.ky * halo_w + hf.kx; };
  for (int s = 0; s < kKpSteps; s++) {
    KpHalf a = seq[2 * s], b = seq[2 * s + 1];
    if (addr(a) > addr(b)) { KpHalf tmp = a; a = b; b = tmp; }
    t.half[2 * s] = a;
    t.half[2 * s + 1] = b;
    t.off[s] = (uint16_t)addr(a);
    t.lbo[s] = (uint16_t)(addr(b) - addr(a));
  }
  return t;
}
// dense fp32 [npad rows][16 channels][49 taps] -> per rank [step][hi|lo][k8][npad/2 rows][8] bf16 (the CG=2 non-CONCAT
// stage layout with K steps in place of taps)
static __global__ void pack_l1k_kernel(const float* __restrict__ dense, __nv_bfloat16* __restrict__ out, int npad,
                                       const KpTable t) {
  const int rows = npad / 2;
  const size_t per_rank = (size_t)kKpSteps * 2 * 2 * rows * 8;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < 2 * per_rank; i += (size_t)gridDim.x * blockDim.x) {
    const int rank = (int)(i / per_rank);
    size_t r = i % per_rank;
    const int e = (int)(r % 8); r /= 8;
    const int q = (int)(r % rows); r /= rows;
    const int k8 = (int)(r % 2); r /= 2;
    const int part = (int)(r % 2); r /= 2;
    const int step = (int)r;
    const KpHalf hf = t.half[2 * step + k8];
    int ch = -1, tap = 0;
    if (hf.type == 0) { ch = e; tap = hf.ky * 7 + hf.kx; }
    else if (hf.type == 1) {
      ch = 8 + (e & 3);
      const int kx = hf.kx + (e >> 2);
      tap = hf.ky * 7 + kx;
      if (kx > 6) ch = -1;
    }
    float w = 0.f;
    if (ch >= 0) w = dense[((size_t)(rank * rows + q) * 16 + ch) * 49 + tap];
    const __nv_bfloat16 hi = __float2bfloat16_rn(w);
    out[i] = part == 0 ? hi : __float2bfloat16_rn(w - __bfloat162float(hi));
  }
}

// ------------------------------------------------------------------------------------------
// Host helpers
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;

static int get_encoder() {
  if (g_encode) return WN_OK;
  cudaDriverEntryPointQueryResult q;
  void* fn = nullptr;
  WN_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
  if (!fn || q != cudaDriverEntryPointSuccess) {
    set_error("cuTensorMapEncodeTiled is not available from this driver");
    return WN_E_UNSUPPORTED;
  }
  g_encode = (EncodeTiledFn)fn;
  return WN_OK;
}

static int make_tmap(CUtensorMap* tm, void* base, int planes_total, int N, int H, int W, int halo_w, int halo_h) {
  cuuint64_t dims[5] = {8, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)planes_total, (cuuint64_t)N};
  cuuint64_t strides[4] = {16, (cuuint64_t)W * 16, (cuuint64_t)H * W * 16, (cuuint64_t)planes_total * H * W * 16};
  cuuint32_t box[5] = {8, (cuuint32_t)halo_w, (cuuint32_t)halo_h, 2, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, base, dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with %d (planes=%d N=%d H=%d W=%d box=%dx%d)", (int)r, planes_total, N, H,
              W, halo_w, halo_h);
    return WN_E_CUDA;
  }
  return WN_OK;
}

// Launch one convolution.  `slot` is the timing slot (common.cuh).
template <int KS, int CIN_PAD, int NPAD, int S, int AS, int EPI, int CONCAT = 0, int NBLK = 1, int TPS = 1, int CG = 1,
          int FMT = 0, int TN = 0, int TEPI = 0, int KP = 0>
static int launch_conv(wn_handle* h, int slot, const uint8_t* wpk, const float* bias, void* in_base, ConvArgs a,
                       cudaStream_t stream) {
  using C = UmmaCfg<KS, CIN_PAD, NPAD, S, AS, CONCAT, NBLK, TPS, CG, FMT, TN, KP, (TEPI & kTailSmem) != 0>;
  int rc = get_encoder();
  if (rc) return rc;
  CUtensorMap tm;
  rc = make_tmap(&tm, in_base, (a.a_hi_only ? 1 : 2) * (CIN_PAD / 8), a.N, a.H, a.W + (KP ? 1 : 0), C::HALO_W, C::HALO_H);
  if (rc) return rc;
  a.wpk = wpk;
  a.bias = bias;
  a.in_planes_half = CIN_PAD / 8;
  a.tiles_x = (a.W + C::TILE_W - 1) / C::TILE_W;
  a.tiles_y = (a.H + C::TILE_H - 1) / C::TILE_H;
  const long long tiles = (long long)a.tiles_x * a.tiles_y * a.N;
  auto kern = conv_umma_kernel<KS, CIN_PAD, NPAD, S, AS, EPI, CONCAT, NBLK, TPS, CG, FMT, TN, TEPI, KP>;
  WN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
  TimedScope ts(h, slot, stream);
  if constexpr (CG == 2) {  // clusters of two CTAs (one TPC each); every pair takes two adjacent tiles at a time
    const long long pairs = (tiles + 1) / 2;
    const int max_pairs = h->sm_count / 2;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(2 * (pairs < max_pairs ? pairs : max_pairs)));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = C::SMEM_BYTES;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    WN_CUDA(cudaLaunchKernelEx(&cfg, kern, tm, a));
  } else {
    int grid = (int)(tiles < h->sm_count ? tiles : h->sm_count);
    kern<<<grid, kThreads, C::SMEM_BYTES, stream>>>(tm, a);
  }
  WN_LAUNCH_CHECK(h);
  return WN_OK;
}

}  // namespace wn
