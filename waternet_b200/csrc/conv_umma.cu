// Tensor-core path of WaterNet.forward (WN_MODE_BF16X3, WN_MODE_BF16_FP8): tcgen05 implicit-GEMM convolutions.
//
// Replaces /root/reference/waternet/net.py:45-56, :75-80, :99-108.  Every
// convolution is a dense contraction (SURVEY.md 2.1), so it runs on the 5th-gen
// tensor cores -- but the 1e-3 parity bar rules out single-pass bf16/tf32 operands
// (SURVEY.md section 0).  Each fp32 operand is split into bf16 hi + lo and
// hi*hi + lo*w + hi*w_lo accumulates in fp32 in TMEM: as three bf16 MMAs ("bf16x3",
// ~2^-16 relative operand error), or -- the default for the tensor-bound layers -- as
// one bf16 MMA plus ONE fp8 (e4m3) MMA of K = 32 for both correction terms
// (UmmaCfg FMT in umma_conv.cuh; DESIGN.md 4.2).
//
// Data layout in HBM: activations are bf16 planes of 8 channels,
//     act[n][plane][y][x][8]   planes [0, C/8) = hi parts, [C/8, 2C/8) = lo parts,
// so that ONE 5-D TMA box (8 ch, x, y, planes, n) drops a halo tile into shared
// memory as [plane][y][x][16 B] -- exactly the no-swizzle K-major UMMA operand
// layout with "8 consecutive pixels of a row" as the 8x16B core matrix.  A filter
// tap (ky,kx) is then just a different descriptor start address into the SAME halo
// tile: the activations are read from L2/HBM once per tile, not once per tap, and
// out-of-image pixels come back as zeros from the TMA (padding="same").
//
// One persistent CTA per SM (most layers: clusters of two CTAs that share every MMA, cta_group::2, each
// staging half of the weight rows), warp-specialised:
//   warps 0-7  epilogue, two groups that split a tile's sub-tiles
//              (TMEM -> registers -> bias/act -> bf16 hi/lo planes or fp32)
//   warp 8     A producer (TMA halo tiles, one 16-channel chunk per stage)
//   warp 9     B producer (bulk copies of pre-packed weight stages, 1-9 taps of a chunk per stage)
//   warp 10    TMEM allocator
//   warp 11    MMA issuer (converged warp, one elected lane issues; highest warp id = scheduling priority);
//              in the peer CTA of a pair: relays "stage full" to the leader's barriers
// A CTA tile is S sub-tiles of 8x16 pixels (M = 128 each) sharing every weight stage.
#include "umma_conv.cuh"

namespace wn {

// torch.cat([x, wb, ce, gc], 1) (net.py:46) -> act planes: 16 channels (12 + 4 zero), bf16 hi/lo of
// v*255.  Inputs that came from 8-bit images (arr2ten: u/255) give integers 0..255, exact in the
// 8-bit bf16 significand: then lo == 0 and the first layer can drop its a_lo pass (flag stays set).
struct PackInArgs {
  const float* p[4];
  long long s[4][4];
};
// kp != 0: the K-packed first layer's layout (UmmaCfg KP): planes are W + 1 columns wide, column x + 1 = pixel x, and
// plane 1 holds [c8..11 @ x | c8..11 @ x + 1] (each pixel writes its four channels into two half rows).
__global__ void __launch_bounds__(256) pack_inputs_kernel(PackInArgs a, uint4* __restrict__ out, int H, int W,
                                                          int* __restrict__ exact_flag, int kp) {
  const int n = blockIdx.y;
  const int pix = blockIdx.x * 256 + threadIdx.x;
  const int hw = H * W;
  bool exact = true;
  if (pix < hw) {
    const int y = pix / W, x = pix - y * W;
    float v[16];
#pragma unroll
    for (int t = 0; t < 4; t++)
#pragma unroll
      for (int c = 0; c < 3; c++) {
        float f = __fmul_rn(a.p[t][n * a.s[t][0] + c * a.s[t][1] + y * a.s[t][2] + x * a.s[t][3]], 255.0f);
        float r = rintf(f);
        // (u/255)*255 lands within ~2e-5 of u; anything within 2^-14 of a level is treated as that level
        if (fabsf(f - r) <= 6.103515625e-5f && r >= 0.f && r <= 255.f) f = r; else exact = false;
        v[t * 3 + c] = f;
      }
    v[12] = v[13] = v[14] = v[15] = 0.f;
    uint32_t hi[8], lo[8];
#pragma unroll
    for (int j = 0; j < 16; j += 2) {
      split_bf16x2(v[j], v[j + 1], hi[j >> 1], lo[j >> 1]);
    }
    if (kp) {
      const size_t plane = (size_t)H * (W + 1);
      uint4* o = out + (size_t)n * 4 * plane + (size_t)y * (W + 1) + x + 1;   // planes: hi0, hi1, lo0, lo1
      store_kp_pixel(o, plane, x, W, make_uint4(hi[0], hi[1], hi[2], hi[3]), make_uint2(hi[4], hi[5]));
      store_kp_pixel(o + 2 * plane, plane, x, W, make_uint4(lo[0], lo[1], lo[2], lo[3]), make_uint2(lo[4], lo[5]));
    } else {
    uint4* o = out + (size_t)n * 4 * hw + pix;  // planes: hi0, hi1, lo0, lo1
    o[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    o[hw] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
    o[2 * (size_t)hw] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    o[3 * (size_t)hw] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
    }
  }
  if (!__syncthreads_and(exact) && threadIdx.x == 0) atomicExch(exact_flag, 0);
}

// ------------------------------------------------------------------------------------------
// Host side
// ------------------------------------------------------------------------------------------
// The ten tensor-core launches of one forward (fused layer list).
enum UmmaLayer {
  kL1 = 0,    // cmg.conv1 (12->128) + the three refiner conv1 (6->32 each): 16 -> 224, 7x7
  kC2, kC3, kC4, kC5, kC6, kC7,
  kC8,        // 64 -> 3 (pad 16), sigmoid
  kR2,        // three refiner conv2 as one block-diagonal 96 -> 96, 5x5
  kR3,        // three refiner conv3 as block-diagonal 96 -> 9 (pad 16), ReLU, gated sum
  kNumUmmaLayers
};
// Weight layout of each layer's packed images.  The tensor-bound layers run as CTA pairs (cta_group::2, the
// single-CTA form measured slower: profiles/r1_ab_cta_pairs.log); conv2/conv3 use the non-CONCAT layout.
struct UmmaLayerSpec {
  int ks, cinpad, npad, cout, slot, concat, nblk;  // npad = output columns per diagonal block
  int cg;                                           // CTAs per MMA: 2 = weight rows split over a CTA pair
  bool f8;                                          // has an fp8-correction weight image (UmmaCfg FMT bit 0)
};
static constexpr UmmaLayerSpec kSpecs[kNumUmmaLayers] = {
    {7, 16, 224, 224, 0, 0, 1, 2, false},
    {5, 128, 128, 128, 1, 0, 1, 2, true},
    {3, 128, 128, 128, 2, 0, 1, 2, true},
    {1, 128, 64, 64, 3, 1, 1, 1, false},
    {7, 64, 64, 64, 4, 1, 1, 2, true},
    {5, 64, 64, 64, 5, 1, 1, 2, true},
    {3, 64, 64, 64, 6, 1, 1, 2, true},
    {3, 64, 16, 3, 7, 1, 1, 1, false},
    {5, 96, 32, 96, 9, 1, 3, 2, true},
    {3, 96, 16, 9, 10, 1, 1, 1, false}};

// The weight image a launch reads: the layer's bf16 stages, its fp8-correction stages (stages8: [hi | fp8] layout,
// CTA pairs, whatever the layer's own CONCAT / CG) or the K-packed first layer (stages_l1k).
enum WeightImage { kImgPlain, kImgF8, kImgKPacked };
struct UmmaLaunch {
  int layer;  // UmmaLayer: KS, CIN_PAD, NPAD, NBLK, CONCAT and CG come from its kSpecs row
  int s, as, epi, tps, fmt, tn, tepi;
  WeightImage img;
};
// Every tensor-core launch of a forward, one row each.
enum UmmaLaunchId {
  // fp8-correction scheme (inference)
  kF8L1K, kF8L1, kF8C2, kF8C34, kF8C3, kF8C4, kF8C5, kF8C6, kF8C78, kF8C7, kF8R23, kF8R2,
  // bf16x3 (training, the fp8 scheme's range-guard re-run, and the bf16x3 mode)
  kX3L1K, kX3L1, kX3C2, kX3C3, kX3C4, kX3C5, kX3C6, kX3C7, kX3R2,
  // the last layers of the unfused forms (both schemes)
  kC8Sigmoid, kR3Gate,
  kNumUmmaLaunches
};
constexpr int IN8 = kFmtIn8, OUT8 = kFmtOut8;
static constexpr UmmaLaunch kLaunches[kNumUmmaLaunches] = {
    // layer  S  AS  EPI          TPS  FMT          TN  TEPI                    image
    // first layer, S = 1: its 224 accumulator columns fill TMEM at S = 2, so the epilogue could not overlap the next
    // tile; S = 1 double-buffers them (21.7 -> 17.8 ms per batch; the refiners' conv2, in the same situation, is slower
    // that way: profiles/r1_ab_cta_pairs.log)
    {kL1, 1, 2, kEpiAct, 5, OUT8, 0, 0, kImgKPacked},
    {kL1, 1, 2, kEpiAct, 7, OUT8, 0, 0, kImgPlain},
    // conv2: one shared accumulator of 128 columns per sub-tile (round 1 kept the correction product in a second one):
    // S = 2 double-buffered fills TMEM exactly and halves the weight-stage fill traffic per MMA, which competes with the
    // operand reads for the 128 B/clk port
    {kC2, 2, 2, kEpiAct, 5, IN8 | OUT8, 0, 0, kImgF8},
    // conv3 with the fused conv4 tail: 9 taps per stage (24 KB of shared memory hold the tail's weights); one sub-tile
    // = 128 columns and the bf16 copy of the tile (the tail GEMM's A operand) another 128, so three accumulator stages
    // fill tensor memory; the tile's second epilogue pass (after the tail GEMM) then has two tiles of slack before its
    // accumulator stage is needed again
    {kC3, 1, 3, kEpiAct, 9, IN8 | OUT8, 64, kTailAct, kImgF8},
    {kC3, 2, 2, kEpiAct, 9, IN8, 0, 0, kImgF8},
    {kC4, 2, 2, kEpiAct, 1, OUT8, 0, 0, kImgPlain},
    // conv5 / conv6 (64 -> 64): one accumulator of 64 columns per sub-tile, S = 4 double-buffered fills TMEM; more
    // sub-tiles per weight stage = less weight-stage fill traffic on the shared-memory port these layers are bound by.
    // conv5 (7x7): 22.5 -> 22.0 ms per batch with four sub-tiles; conv6 (5x5) is slower that way (11.6 -> 11.9)
    {kC5, 4, 2, kEpiAct, 7, IN8 | OUT8, 0, 0, kImgF8},
    {kC6, 2, 2, kEpiAct, 5, IN8 | OUT8, 0, 0, kImgF8},
    // conv7 with the tap-stacked conv8 tail: 2 x 64 accumulator columns per stage (+ 2 x 64 for the bf16 tiles in the
    // tensor-memory form).  The tail's operand in tensor memory: measured equal to the shared-memory form, and it keeps
    // conv7's halo ring at 6 stages
    {kC7, 2, 3, kEpiAct, 9, IN8, 32, kTailTaps, kImgF8},
    {kC7, 2, 2, kEpiAct, 9, IN8, 0, 0, kImgF8},
    // the refiners' conv2 with the tap-stacked conv3 tail: S = 2, AS = 2 = 384 accumulator columns + ONE 96-column bf16
    // operand region the two sub-tiles take turns on (UmmaCfg::A2_SHARED), the operand in shared memory; 5 taps per
    // weight stage = one kernel row.  Unfused: 96 accumulator columns per sub-tile, S = 2 double-buffered = 384
    {kR2, 2, 2, kEpiAct, 5, IN8, 96, kTailTaps | kTailSmem, kImgF8},
    {kR2, 2, 2, kEpiAct, 5, IN8, 0, 0, kImgF8},

    {kL1, 1, 2, kEpiAct, 5, 0, 0, 0, kImgKPacked},
    {kL1, 1, 2, kEpiAct, 7, 0, 0, 0, kImgPlain},
    {kC2, 2, 2, kEpiAct, 5, 0, 0, 0, kImgPlain},
    {kC3, 2, 2, kEpiAct, 3, 0, 0, 0, kImgPlain},
    {kC4, 2, 2, kEpiAct, 1, 0, 0, 0, kImgPlain},
    {kC5, 2, 2, kEpiAct, 7, 0, 0, 0, kImgPlain},
    {kC6, 2, 2, kEpiAct, 5, 0, 0, 0, kImgPlain},
    {kC7, 2, 2, kEpiAct, 9, 0, 0, 0, kImgPlain},
    {kR2, 2, 1, kEpiAct, 5, 0, 0, 0, kImgPlain},  // 5 taps per stage = one kernel row (25 = a whole chunk)

    {kC8, 4, 2, kEpiSigmoid, 9, 0, 0, 0, kImgPlain},
    {kR3, 4, 2, kEpiGate, 9, 0, 0, 0, kImgPlain}};

// The kernel configuration of launch row R.
template <int R>
struct UmmaRow {
  static constexpr UmmaLaunch r = kLaunches[R];
  static constexpr UmmaLayerSpec l = kSpecs[r.layer];
  static constexpr bool F8 = r.img == kImgF8;
  static constexpr int CONCAT = F8 ? 0 : l.concat, CG = F8 ? 2 : l.cg, KP = r.img == kImgKPacked ? 1 : 0;
  static_assert(F8 == ((r.fmt & kFmtIn8) != 0), "the fp8-correction form reads the fp8 weight image");
  static_assert(!F8 || (l.f8 && CONCAT == 0 && CG == 2), "fp8 weight images: CTA pairs, [hi | fp8] layout");
  static_assert(!KP || (r.layer == kL1 && l.cg == 2), "the K-packed image is the first layer's, for CTA pairs");
  static_assert(r.tn == 0 || F8, "the fused tail layer exists for the fp8-correction form only");
  using Cfg = UmmaCfg<l.ks, l.cinpad, l.npad, r.s, r.as, CONCAT, l.nblk, r.tps, CG, r.fmt, r.tn, KP,
                      (r.tepi & kTailSmem) != 0>;
};

// OIHW [co][ci][kk] -> dense [kk * co rows][ld]: row co * tap + c holds tap's filter of output channel c
static __global__ void scatter_tapstack_kernel(const float* __restrict__ src, float* __restrict__ dense, int co, int ci, int kk,
                                               int ld) {
  const int total = co * ci * kk;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int t = i % kk, c = (i / kk) % ci, o = i / (kk * ci);
    dense[(size_t)(t * co + o) * ld + c] = src[i];
  }
}
// The second half of the three refiners' tap-stacked conv3 + the gated sum (net.py:68-70, 79, 104-108):
//   refined[r][c] = relu(bias[3r + c] + sum over the 3x3 taps of taps[n][27 r + 3 tap + c][y + ky - 1][x + kx - 1])
//   out[c]        = refined[0][c] * cm[0] + refined[1][c] * cm[1] + refined[2][c] * cm[2]
// written as fp32 NCHW and/or ten2arr'd uint8 NHWC; refined_out optionally receives the nine refined planes.
// HBM-bound: 324 B/px of partial sums read exactly once, 12 B/px of maps, 3..48 B/px written.
static __global__ void __launch_bounds__(256, 8)  // 8 blocks = all 2048 threads of an SM: the kernel lives on loads in flight
gather_gate_kernel(const float* __restrict__ taps, const float* __restrict__ bias, const float* __restrict__ cm,
                   float* __restrict__ out_f32, uint8_t* __restrict__ out_u8, float* __restrict__ refined_out, int H, int W,
                   PeerOut peers) {
  const int x = blockIdx.x * 64 + threadIdx.x, y = blockIdx.y * 4 + threadIdx.y, n = blockIdx.z;
  if (y >= H) return;  // warp-uniform (a warp is 32 consecutive x of one row)
  const bool inside = x < W;
  const size_t hw = (size_t)H * W, pix = (size_t)y * W + x;
  uint32_t rgb = 0;  // this pixel's three output bytes
  if (inside) {
    const float* t = taps + (size_t)n * 81 * hw;
    float r[9];
#pragma unroll
    for (int j = 0; j < 9; j++) r[j] = bias[j];
#pragma unroll
    for (int ky = 0; ky < 3; ky++) {
      const int yy = y + ky - 1;
      if (yy < 0 || yy >= H) continue;
#pragma unroll
      for (int kx = 0; kx < 3; kx++) {
        const int xx = x + kx - 1;
        if (xx < 0 || xx >= W) continue;
        const float* p = t + (size_t)((ky * 3 + kx) * 3) * hw + (size_t)yy * W + xx;
#pragma unroll
        for (int rr = 0; rr < 3; rr++)
#pragma unroll
          for (int c = 0; c < 3; c++) r[3 * rr + c] += p[(size_t)(27 * rr + c) * hw];
      }
    }
#pragma unroll
    for (int j = 0; j < 9; j++) r[j] = fmaxf(r[j], 0.f);
    if (refined_out) {
#pragma unroll
      for (int j = 0; j < 9; j++) refined_out[((size_t)n * 9 + j) * hw + pix] = r[j];
    }
    if (cm) {
      const size_t o = (size_t)n * 3 * hw + pix;
      const float c0 = cm[o], c1 = cm[o + hw], c2 = cm[o + 2 * hw];
      float v[3];
#pragma unroll
      for (int c = 0; c < 3; c++)
        v[c] = __fadd_rn(__fadd_rn(__fmul_rn(r[c], c0), __fmul_rn(r[3 + c], c1)), __fmul_rn(r[6 + c], c2));
      if (out_f32) {
#pragma unroll
        for (int c = 0; c < 3; c++) out_f32[o + c * hw] = v[c];
      }
#pragma unroll
      for (int c = 0; c < 3; c++)  // ten2arr (hubconf.py:24-34)
        rgb |= (uint32_t)(int)__fmul_rn(fminf(fmaxf(v[c], 0.0f), 1.0f), 255.0f) << (8 * c);
    }
  }
  if (!cm || !out_u8) return;
  // uint8 NHWC: the warp's 32 pixels are 96 contiguous bytes.  With peer addresses (the all-gather of the output fused
  // here) lane l < 24 assembles 32-bit word l of them from its neighbours' bytes, so a full segment leaves as one
  // coalesced 96-byte store per (4-byte aligned) destination: NVLink wants whole sectors, not bytes.  Without peers the
  // three byte stores per pixel merge in L2 and cost less than the shuffles.
  const int lane = threadIdx.x & 31;
  const int xw = x - lane;  // the warp's first pixel
  const size_t off = ((size_t)n * hw + (size_t)y * W + xw) * 3;
  const bool words = peers.n > 0 && xw + 32 <= W;  // warp-uniform
  uint32_t word = 0;
  if (words) {
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int k = 4 * lane + j;  // byte k of the segment = component k % 3 of pixel k / 3 (lanes >= 24: unused)
      word |= ((__shfl_sync(0xffffffffu, rgb, (k / 3) & 31) >> (8 * (k % 3))) & 0xffu) << (8 * j);
    }
  }
  auto put = [&](uint8_t* dst) {  // this warp's segment -> dst (the same for every lane)
    if (words && (reinterpret_cast<uintptr_t>(dst + off) & 3) == 0) {
      if (lane < 24) reinterpret_cast<uint32_t*>(dst + off)[lane] = word;
    } else if (inside) {
#pragma unroll
      for (int c = 0; c < 3; c++) dst[off + 3 * lane + c] = (uint8_t)(rgb >> (8 * c));
    }
  };
  put(out_u8);
#pragma unroll
  for (int i = 0; i < WN_MAX_PEERS; i++)  // unrolled: the addresses stay kernel parameters (no local copy)
    if (i < peers.n) put(peers.p[i]);
}
// out -> every peer address (the paths whose uint8 output leaves a convolution epilogue: bf16x3 mode, the range guard's
// re-run -- then conditional on *run_if like every launch of that chain -- and the A/B switches)
static __global__ void __launch_bounds__(256)
mirror_u8_kernel(const uint8_t* __restrict__ src, PeerOut peers, size_t bytes, const int* __restrict__ run_if) {
  if (run_if && *run_if == 0) return;
  const size_t stride = (size_t)gridDim.x * blockDim.x, i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
#pragma unroll
  for (int k = 0; k < WN_MAX_PEERS; k++) {
    if (k >= peers.n) continue;
    uint8_t* dst = peers.p[k];
    // 16-byte copies where source and destination allow it (the batches of a 16-byte aligned buffer); bytes otherwise
    const size_t vecs = (((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0) ? bytes / 16 : 0;
    for (size_t i = i0; i < vecs; i += stride) reinterpret_cast<uint4*>(dst)[i] = reinterpret_cast<const uint4*>(src)[i];
    for (size_t i = vecs * 16 + i0; i < bytes; i += stride) dst[i] = src[i];
  }
}
int mirror_u8(wn_handle* h, const uint8_t* src, const PeerOut& peers, size_t bytes, const int* run_if, cudaStream_t stream) {
  if (peers.n <= 0 || bytes == 0) return WN_OK;
  mirror_u8_kernel<<<592, 256, 0, stream>>>(src, peers, bytes, run_if);
  WN_LAUNCH_CHECK(h);
  return WN_OK;
}
// cm[n][c][y][x] = sigmoid(bias[c] + sum over the 3x3 taps of taps[n][3 * tap + c][y + ky - 1][x + kx - 1]), zero outside
// the image ("same" padding): the second half of the tap-stacked cmg.conv8 (net.py:40-43, 54).  HBM-bound: 108 B/px
// read (every partial sum exactly once), 12 B/px written.
static __global__ void __launch_bounds__(256)
gather_sigmoid_kernel(const float* __restrict__ taps, const float* __restrict__ bias, float* __restrict__ cm, int H, int W) {
  const int x = blockIdx.x * 64 + threadIdx.x, y = blockIdx.y * 4 + threadIdx.y, n = blockIdx.z;
  if (x >= W || y >= H) return;
  const size_t hw = (size_t)H * W;
  const float* t = taps + (size_t)n * 27 * hw;
  float acc[3] = {bias[0], bias[1], bias[2]};
#pragma unroll
  for (int ky = 0; ky < 3; ky++) {
    const int yy = y + ky - 1;
    if (yy < 0 || yy >= H) continue;
#pragma unroll
    for (int kx = 0; kx < 3; kx++) {
      const int xx = x + kx - 1;
      if (xx < 0 || xx >= W) continue;
      const float* p = t + (size_t)((ky * 3 + kx) * 3) * hw + (size_t)yy * W + xx;
#pragma unroll
      for (int c = 0; c < 3; c++) acc[c] += p[(size_t)c * hw];
    }
  }
  float* o = cm + (size_t)n * 3 * hw + (size_t)y * W + x;
#pragma unroll
  for (int c = 0; c < 3; c++) o[(size_t)c * hw] = 1.0f / (1.0f + expf(-acc[c]));
}

// halo-stage geometry of the first layer's kernel (S = 1: 8 + 6 columns, 16 + 6 rows), in 16-byte units
static constexpr int kL1HaloW = 14, kL1PlaneUnits = 14 * 22;
static size_t stage8_bytes_total(const UmmaLayerSpec& s) {
  return (size_t)2 * (s.cinpad / 16) * s.ks * s.ks * (s.npad / 2) * 64;  // two per-rank images
}
struct UmmaWeights {
  uint8_t* stages8[kNumUmmaLayers];  // fp8-correction weight images (kSpecs f8 layers)
  float* scale8[kNumUmmaLayers];     // {ws, 2^-9 / ws, max|w|, -}
  uint8_t* stages_l1k;               // the first layer K-packed (UmmaCfg KP): two per-rank images of kKpSteps stages of 224 x 32 B
  uint8_t* tailr3;                   // the three refiners' conv3 tap-stacked (block-diagonal, 3 x 27 columns) as the tail of their conv2
  uint8_t* tail8;                    // cmg.conv8 tap-stacked (27 = 9 taps x 3 channels columns) as the tail layer of conv7
  uint8_t* tail4;                    // cmg.conv4 as the tail layer of conv3: two per-rank images, CG=2 CONCAT layout
  int* overflow_dev;                 // sticky: an activation left the e4m3 range in the fp8-correction mode
  int* overflow_host;                // pinned mirror, refreshed at the end of every forward of that mode
  uint8_t* stages[kNumUmmaLayers];
  float* bias[kNumUmmaLayers];
  float* dense;  // scratch for packing
};

static size_t stage_bytes_total(const UmmaLayerSpec& s) {
  if (s.cg == 2)  // two per-rank images (UmmaCfg::B_TAP per tap each)
    return (size_t)2 * (s.cinpad / 16) * s.ks * s.ks * s.npad * (s.concat ? 48 : 32);
  return (size_t)(s.cinpad / 16) * s.ks * s.ks * s.npad * 64;  // one block's rows per stage
}

int umma_pack_weights(wn_handle* h, const float* const* params, cudaStream_t stream) {
  if (!h->umma) h->umma = (UmmaWeights*)calloc(1, sizeof(UmmaWeights));
  for (int i = 0; i < kNumUmmaLayers; i++) {  // (re)allocate whatever an earlier, failed call left unallocated
    if (!h->umma->stages[i]) WN_CUDA(cudaMalloc(&h->umma->stages[i], stage_bytes_total(kSpecs[i])));
    if (!h->umma->bias[i]) WN_CUDA(cudaMalloc(&h->umma->bias[i], kSpecs[i].npad * kSpecs[i].nblk * sizeof(float)));
    if (kSpecs[i].f8) {
      if (!h->umma->stages8[i]) WN_CUDA(cudaMalloc(&h->umma->stages8[i], stage8_bytes_total(kSpecs[i])));
      if (!h->umma->scale8[i]) WN_CUDA(cudaMalloc(&h->umma->scale8[i], 4 * sizeof(float)));
    }
  }
  // the tail images as packed below (two per-rank images each) are what the fused launches read
  static_assert(2 * 8 * 64 * 48 == 2 * UmmaRow<kF8C34>::Cfg::WT_BYTES, "tail4 layout");
  static_assert(2 * 4 * 32 * 48 == 2 * UmmaRow<kF8C78>::Cfg::WT_BYTES, "tail8 layout");
  static_assert(2 * 6 * 32 * 32 == 2 * UmmaRow<kF8R23>::Cfg::WT_BYTES, "tailr3 layout");
  if (!h->umma->dense) WN_CUDA(cudaMalloc(&h->umma->dense, (size_t)224 * 128 * 49 * sizeof(float)));
  if (!h->umma->tail4) WN_CUDA(cudaMalloc(&h->umma->tail4, (size_t)2 * 8 * 64 * 48));
  if (!h->umma->stages_l1k) WN_CUDA(cudaMalloc(&h->umma->stages_l1k, (size_t)kKpSteps * 224 * 32 * 2));
  if (!h->umma->tail8) WN_CUDA(cudaMalloc(&h->umma->tail8, (size_t)2 * 4 * 32 * 48));
  if (!h->umma->tailr3) WN_CUDA(cudaMalloc(&h->umma->tailr3, (size_t)2 * 6 * 32 * 32));
  if (!h->umma->overflow_dev) WN_CUDA(cudaMalloc(&h->umma->overflow_dev, sizeof(int)));
  if (!h->umma->overflow_host) WN_CUDA(cudaHostAlloc(&h->umma->overflow_host, sizeof(int), cudaHostAllocDefault));
  UmmaWeights* u = h->umma;
  *u->overflow_host = 0;  // new weights: the fp8-correction mode gets a fresh chance
  WN_CUDA(cudaMemsetAsync(u->overflow_dev, 0, sizeof(int), stream));
  auto W = [&](int conv) { return params[2 * conv]; };
  auto B = [&](int conv) { return params[2 * conv + 1]; };
  for (int li = 0; li < kNumUmmaLayers; li++) {
    const UmmaLayerSpec& s = kSpecs[li];
    const int kk = s.ks * s.ks;
    const int rows = s.npad * s.nblk;
    WN_CUDA(cudaMemsetAsync(u->dense, 0, (size_t)rows * s.cinpad * kk * sizeof(float), stream));
    WN_CUDA(cudaMemsetAsync(u->bias[li], 0, rows * sizeof(float), stream));
    auto scatter = [&](int conv, int co, int ci, int row_off, int split, int base0, int base1) -> int {
      // the first layer consumes image levels 0..255 (see pack_inputs_kernel): fold the /255 into its weights
      scatter_weights_kernel<<<128, 256, 0, stream>>>(W(conv), u->dense, co, ci, kk, s.cinpad, row_off, split,
                                                      base0, base1, li == kL1 ? 255.0f : 1.0f);
      WN_LAUNCH_CHECK(h);
      scatter_bias_kernel<<<1, 256, 0, stream>>>(B(conv), u->bias[li], co, row_off);
      WN_LAUNCH_CHECK(h);
      return WN_OK;
    };
    int rc = WN_OK;
    if (li == kL1) {
      rc = scatter(0, 128, 12, 0, 12, 0, 0);
      for (int r = 0; r < 3 && !rc; r++)  // refiner r sees cat[x, input r+1]: channels 0..2 and 3(r+1)..3(r+1)+2
        rc = scatter(8 + 3 * r, 32, 6, 128 + 32 * r, 3, 0, 3 * (r + 1));
    } else if (li >= kC2 && li <= kC8) {
      const int conv = li;  // cmg.conv2..conv8 are convs 1..7
      const LayerDesc& d = kCmg[conv];
      rc = scatter(conv, d.cout, d.cin, 0, d.cin, 0, 0);
    } else if (li == kR2) {
      for (int r = 0; r < 3 && !rc; r++) rc = scatter(8 + 3 * r + 1, 32, 32, 32 * r, 32, 32 * r, 0);
    } else {
      for (int r = 0; r < 3 && !rc; r++) rc = scatter(8 + 3 * r + 2, 3, 32, 3 * r, 32, 32 * r, 0);
    }
    if (rc) return rc;
    if (s.cg == 2)
      pack_stages_cg2_kernel<<<256, 256, 0, stream>>>(u->dense, (__nv_bfloat16*)u->stages[li], s.npad, s.cinpad, kk,
                                                      s.concat, s.nblk);
    else
      pack_stages_kernel<<<256, 256, 0, stream>>>(u->dense, (__nv_bfloat16*)u->stages[li], s.npad, s.cinpad, kk,
                                                  s.concat, s.nblk);
    WN_LAUNCH_CHECK(h);
    if (li == kL1) {  // the K-packed form of the first layer (inference): K steps pair arbitrary halo rows (l1k_table)
      pack_l1k_kernel<<<256, 256, 0, stream>>>(u->dense, (__nv_bfloat16*)u->stages_l1k, s.npad, l1k_table(kL1HaloW, kL1PlaneUnits));
      WN_LAUNCH_CHECK(h);
    }
    if (li == kC4) {  // the same weights as conv3's fused tail layer (UmmaCfg TN): per rank [chunk][k8][64 | 32 rows][8]
      pack_stages_cg2_kernel<<<256, 256, 0, stream>>>(u->dense, (__nv_bfloat16*)u->tail4, s.npad, s.cinpad, kk, 1, 1);
      WN_LAUNCH_CHECK(h);
    }
    if (li == kC8) {  // tap-stacked form: dense [32 rows = 3 * tap + channel (27 used)][64 input channels], a 1x1 layer
      float* stacked = u->dense + (size_t)16 * 64 * 9;  // behind conv8's own [16][64][9] matrix
      WN_CUDA(cudaMemsetAsync(stacked, 0, (size_t)32 * 64 * sizeof(float), stream));
      scatter_tapstack_kernel<<<8, 256, 0, stream>>>(W(7), stacked, 3, 64, 9, 64);
      WN_LAUNCH_CHECK(h);
      pack_stages_cg2_kernel<<<64, 256, 0, stream>>>(stacked, (__nv_bfloat16*)u->tail8, 32, 64, 1, 1, 1);
      WN_LAUNCH_CHECK(h);
    }
    if (li == kR3) {  // tap-stacked, block-diagonal: dense [96 rows: 32 r + 3 tap + c][96 channels: 32 r + ci], a 1x1 layer
      float* stacked = u->dense + (size_t)16 * 96 * 9;  // behind the refiners' own [16][96][9] matrix
      WN_CUDA(cudaMemsetAsync(stacked, 0, (size_t)96 * 96 * sizeof(float), stream));
      for (int r = 0; r < 3; r++) {
        scatter_tapstack_kernel<<<8, 256, 0, stream>>>(W(8 + 3 * r + 2), stacked + ((size_t)32 * r * 96 + 32 * r), 3, 32, 9, 96);
        WN_LAUNCH_CHECK(h);
      }
      pack_stages_cg2_kernel<<<64, 256, 0, stream>>>(stacked, (__nv_bfloat16*)u->tailr3, 32, 96, 1, 0, 3);
      WN_LAUNCH_CHECK(h);
    }
    if (s.f8) {
      WN_CUDA(cudaMemsetAsync(u->scale8[li], 0, 4 * sizeof(float), stream));
      f8_absmax_kernel<<<64, 256, 0, stream>>>(u->dense, (size_t)rows * s.cinpad * kk, u->scale8[li]);
      WN_LAUNCH_CHECK(h);
      f8_scale_finish_kernel<<<1, 1, 0, stream>>>(u->scale8[li]);
      WN_LAUNCH_CHECK(h);
      pack_stages_f8_cg2_kernel<<<256, 256, 0, stream>>>(u->dense, u->stages8[li], u->scale8[li], s.npad, s.cinpad, kk,
                                                         s.nblk);
      WN_LAUNCH_CHECK(h);
    }
  }
  return WN_OK;
}

void umma_free(wn_handle* h) {
  if (!h->umma) return;
  for (int i = 0; i < kNumUmmaLayers; i++) {
    if (h->umma->stages[i]) cudaFree(h->umma->stages[i]);
    if (h->umma->bias[i]) cudaFree(h->umma->bias[i]);
    if (h->umma->stages8[i]) cudaFree(h->umma->stages8[i]);
    if (h->umma->scale8[i]) cudaFree(h->umma->scale8[i]);
  }
  if (h->umma->dense) cudaFree(h->umma->dense);
  if (h->umma->tail4) cudaFree(h->umma->tail4);
  if (h->umma->stages_l1k) cudaFree(h->umma->stages_l1k);
  if (h->umma->tail8) cudaFree(h->umma->tail8);
  if (h->umma->tailr3) cudaFree(h->umma->tailr3);
  if (h->umma->overflow_dev) cudaFree(h->umma->overflow_dev);
  if (h->umma->overflow_host) cudaFreeHost(h->umma->overflow_host);
  free(h->umma);
  h->umma = nullptr;
}

// bytes per pixel: act0 (16 ch) 64 | cmg ping/pong (128 ch) 512 each | ref ping/pong (96 ch) 384 each | cm 12
static constexpr size_t kUmmaBytesPerPixel = 64 + 512 + 512 + 384 + 384 + 12;

// Images per pass: <= 8 Mi pixels (~15 GB of workspace) by default; wn_set_chunk_pixels lowers the cap
// (tests force the multi-pass path on small batches with it; it never raises the workspace need).
static constexpr long long kDefaultChunkPixels = 8ll << 20;
static int umma_chunk(long long cap, int n, int h, int w) {
  if (cap <= 0 || cap > kDefaultChunkPixels) cap = kDefaultChunkPixels;
  long long per = (long long)h * w;
  long long nb = cap / (per > 0 ? per : 1);
  if (nb < 1) nb = 1;
  return nb < n ? (int)nb : n;
}
int umma_chunk_images(const wn_handle* h, int n, int height, int width) {
  return umma_chunk(h ? h->chunk_pixels : 0, n, height, width);
}

size_t umma_forward_workspace_bytes(int n, int h, int w) {
  const size_t nb = (size_t)umma_chunk(0, n, h, w);
  return nb * h * w * kUmmaBytesPerPixel + nb * h * 64 + 4096;
}

// Launch row R of kLaunches on the weight image it reads.
template <int R>
static int launch(wn_handle* h, void* in_base, ConvArgs a, cudaStream_t stream) {
  using Row = UmmaRow<R>;
  constexpr UmmaLaunch r = Row::r;
  constexpr UmmaLayerSpec l = Row::l;
  const uint8_t* w = h->umma->stages[r.layer];
  if constexpr ((r.fmt & kFmtOut8) != 0) a.f8_overflow = h->umma->overflow_dev;
  if constexpr (Row::F8) {
    w = h->umma->stages8[r.layer];
    a.f8_scale = h->umma->scale8[r.layer] + 1;
  }
  if constexpr (Row::KP) {  // K-packed first layer: its own weight images and the table of K steps
    static_assert(Row::Cfg::HALO_W == kL1HaloW && Row::Cfg::PLANE_BYTES / 16 == kL1PlaneUnits, "l1k_table geometry");
    w = h->umma->stages_l1k;
    const KpTable t = l1k_table(kL1HaloW, kL1PlaneUnits);
    for (int i = 0; i < kKpSteps; i++) { a.kp_off[i] = t.off[i]; a.kp_lbo[i] = t.lbo[i]; }
  }
  return launch_conv<l.ks, l.cinpad, l.npad, r.s, r.as, r.epi, Row::CONCAT, l.nblk, r.tps, Row::CG, r.fmt, r.tn, r.tepi,
                     Row::KP>(h, l.slot, w, h->umma->bias[r.layer], in_base, a, stream);
}

// bf16 hi/lo planes -> fp32 NCHW (test aid)
__global__ void decode_planes_kernel(const uint4* __restrict__ src, float* __restrict__ dst, int planes_half, int hw,
                                     int f8) {
  const int n = blockIdx.z, plane = blockIdx.y;
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= hw) return;
  const uint4 h4 = src[((size_t)n * 2 * planes_half + plane) * hw + pix];
  if (f8) {  // hi planes + per 16 channels {e4m3((v - hi) * 2^9), e4m3(v)}: v ~ hi + lo8 / 512
    const uint4 l4 = src[((size_t)n * 2 * planes_half + planes_half + 2 * (plane >> 1)) * hw + pix];
    const uint32_t hs[4] = {h4.x, h4.y, h4.z, h4.w}, ls[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const float hi = __uint_as_float(((hs[j >> 1] >> ((j & 1) * 16)) & 0xffffu) << 16);
      const int byte = (plane & 1) * 8 + j;
      const uint32_t b8 = (ls[byte >> 2] >> ((byte & 3) * 8)) & 0xffu;  // e4m3: sign, 4 exponent bits (bias 7), 3 mantissa
      const int e = (int)((b8 >> 3) & 15), m = (int)(b8 & 7);
      const float mag = e == 0 ? ldexpf((float)m, -9) : ldexpf((float)(8 + m), e - 10);
      const float lo = ((b8 & 0x80u) ? -mag : mag) * (1.f / 512.f);
      dst[((size_t)n * planes_half * 8 + plane * 8 + j) * hw + pix] = hi + lo;
    }
    return;
  }
  const uint4 l4 = src[((size_t)n * 2 * planes_half + planes_half + plane) * hw + pix];
  const uint32_t hs[4] = {h4.x, h4.y, h4.z, h4.w}, ls[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
  for (int j = 0; j < 8; j++) {
    float hi = __uint_as_float(((hs[j >> 1] >> ((j & 1) * 16)) & 0xffffu) << 16);
    float lo = __uint_as_float(((ls[j >> 1] >> ((j & 1) * 16)) & 0xffffu) << 16);
    dst[((size_t)n * planes_half * 8 + plane * 8 + j) * hw + pix] = hi + lo;
  }
}

// Where every layer's output lives.  Inference ping-pongs two buffers per stack; the training
// forward (conv_bwd.cu) gives every activation its own buffer because the backward pass needs them.
int umma_forward_layers(wn_handle* h, const float* const in[4], const int64_t st[4][4], float* out, int n, int H,
                        int W, const FwdBuffers& b, cudaStream_t stream, const FwdOpts& o) {
  const int dbg_layer = o.dbg_layer;
  float* const dbg_dst = o.dbg_dst;
  if (!o.packed) {
    PackInArgs pa;
    for (int t = 0; t < 4; t++) {
      pa.p[t] = in[t];
      for (int k = 0; k < 4; k++) pa.s[t][k] = st[t][k];
    }
    TimedScope ts(h, kSlotPack, stream);
    WN_CUDA(cudaMemsetAsync(b.exact_flag, 1, sizeof(int), stream));  // nonzero = "all inputs are 8-bit levels"
    pack_inputs_kernel<<<dim3((H * W + 255) / 256, n), 256, 0, stream>>>(pa, b.act0, H, W, b.exact_flag, o.kpack ? 1 : 0);
    WN_LAUNCH_CHECK(h);
  }
  ConvArgs a;
  memset(&a, 0, sizeof(a));
  a.N = n; a.H = H; a.W = W;
  a.run_if = o.run_if;
  int rc;
  auto dump = [&](int layer, const uint4* buf, int channels, int f8 = 0) -> bool {
    if (dbg_layer != layer) return false;
    decode_planes_kernel<<<dim3((H * W + 255) / 256, channels / 8, n), 256, 0, stream>>>(buf, dbg_dst, channels / 8,
                                                                                     H * W, f8);
    h->launches++;
    return true;
  };
  auto act = [&](uint4* d0, int c0, uint4* d1, int c1) {
    a.dst0.base = d0; a.dst0.planes_half = c0 / 8;
    a.dst1.base = d1; a.dst1.planes_half = c1 / 8;
    a.split_c = c0; a.cout = c0 + c1;
  };
  // the last launch: refiner conv3 + ReLU, then (when the maps are given) the gated sum -> fp32 NCHW and/or
  // ten2arr'd uint8 NHWC; refined_out optionally receives the three refined images
  auto last = [&]() {
    a.out_f32 = out;
    a.out_u8 = o.out_u8;
    a.cm = o.stack == kStackRefiners ? nullptr : b.cm;
    a.refined_out = b.refined;
  };
  const bool want_cmg = o.stack != kStackRefiners, want_ref = o.stack != kStackCmg;
  if (o.scheme == 1) {
    // fp8-correction scheme (inference): the tensor-bound layers replace the two bf16 correction passes by one
    // fp8 MMA (UmmaCfg FMT); a layer whose consumer is such a layer writes the hi + fp8-planes format
    act(b.a[1], 128, b.r[1], 96);
    a.skip_lo = b.exact_flag;
    a.a_hi_only = o.hi_only ? 1 : 0;
    if (o.kpack) {
      if ((rc = launch<kF8L1K>(h, b.act0, a, stream))) return rc;
    } else if ((rc = launch<kF8L1>(h, b.act0, a, stream))) return rc;
    a.skip_lo = nullptr;
    a.a_hi_only = 0;
    if (dump(0, b.a[1], 128, 1) || dump(8, b.r[1], 96, 1)) return WN_OK;
    if (want_cmg) {
      act(b.a[2], 128, nullptr, 0);
      if ((rc = launch<kF8C2>(h, b.a[1], a, stream))) return rc;
      if (dump(1, b.a[2], 128, 1)) return WN_OK;
      // where conv4..conv7 write: the ping-pong assignment of carve() has conv4's output in conv2's buffer, which
      // the fused conv3+conv4 launch is still reading (halos of tiles to come) -- with conv4 fused, conv4..7 take
      // the buffers of conv3..6 instead
      const bool fuse34 = dbg_layer != 2 && !(h->dbg_flags & 256);
      uint4* const a4 = fuse34 ? b.a[3] : b.a[4];
      uint4* const a5 = fuse34 ? b.a[4] : b.a[5];
      uint4* const a6 = fuse34 ? b.a[5] : b.a[6];
      uint4* const a7 = fuse34 ? b.a[6] : b.a[7];
      if (fuse34) {
        // conv3 with conv4 (1x1) as its fused tail layer: conv3's output tile goes back into tensor memory as the
        // A operand of a second GEMM; only conv4's 64 channels reach HBM (net.py:20-27)
        act(a4, 64, nullptr, 0);
        a.wtail = h->umma->tail4;
        a.bias2 = h->umma->bias[kC4];
        if ((rc = launch<kF8C34>(h, b.a[2], a, stream))) return rc;
        a.wtail = nullptr;
        a.bias2 = nullptr;
      } else {
        act(b.a[3], 128, nullptr, 0);
        if ((rc = launch<kF8C3>(h, b.a[2], a, stream))) return rc;
        if (dump(2, b.a[3], 128)) return WN_OK;
        act(a4, 64, nullptr, 0);
        if ((rc = launch<kF8C4>(h, b.a[3], a, stream))) return rc;
      }
      if (dump(3, a4, 64, 1)) return WN_OK;
      act(a5, 64, nullptr, 0);
      if ((rc = launch<kF8C5>(h, a4, a, stream))) return rc;
      if (dump(4, a5, 64, 1)) return WN_OK;
      act(a6, 64, nullptr, 0);
      if ((rc = launch<kF8C6>(h, a5, a, stream))) return rc;
      if (dump(5, a6, 64, 1)) return WN_OK;
      float* const cm_dst = dbg_layer == 7 ? dbg_dst : b.cm;
      if (dbg_layer != 6 && !(h->dbg_flags & 512)) {
        // conv7 with conv8 (3x3, 64 -> 3) tap-stacked as its fused tail layer: the 27 per-tap partial sums of every
        // pixel (fp32 planes, 108 B/px, in the buffer conv7's activations would have taken) instead of conv7's 64
        // channels (256 B/px); gather_sigmoid_kernel then adds the nine shifted planes, the bias, and applies the
        // sigmoid (net.py:36-43, 54)
        float* taps = reinterpret_cast<float*>(a7);
        a.out_f32 = taps;
        a.cout = 27;
        a.wtail = h->umma->tail8;
        a.bias2 = h->umma->bias[kC8];  // unused by the tap-stacked epilogue (the gather adds the bias)
        if ((rc = launch<kF8C78>(h, a6, a, stream))) return rc;
        a.wtail = nullptr;
        a.bias2 = nullptr;
        {
          TimedScope ts(h, kSpecs[kC8].slot, stream);
          gather_sigmoid_kernel<<<dim3((W + 63) / 64, (H + 3) / 4, n), dim3(64, 4), 0, stream>>>(taps, h->umma->bias[kC8], cm_dst, H, W);
          WN_LAUNCH_CHECK(h);
        }
      } else {
        act(a7, 64, nullptr, 0);
        if ((rc = launch<kF8C7>(h, a6, a, stream))) return rc;
        if (dump(6, a7, 64)) return WN_OK;
        a.out_f32 = cm_dst;
        if ((rc = launch<kC8Sigmoid>(h, a7, a, stream))) return rc;
      }
      if (dbg_layer == 7) return WN_OK;
    }
    if (!want_ref) return WN_OK;
    if (dbg_layer != 9 && !(h->dbg_flags & 1024)) {
      // the refiners' conv2 with their conv3 (3x3, 32 -> 3 each) tap-stacked as a block-diagonal fused tail layer:
      // 81 partial-sum planes (324 B/px, in the buffer conv2's activations would have taken) instead of 96 channels
      // (384 B/px); gather_gate_kernel adds the nine shifted planes per output, bias, ReLU and the gated sum
      // (net.py:65-70, 104-108).  The tail GEMM's operand goes through shared memory here (kTailSmem: the refiners'
      // small rings leave 96 KB free).  Same-box: 16.0 + 6.3 -> 19.8 + 1.9 ms per batch, +0.8 % images/s
      // (profiles/r2_ab_fused_tails.log) -- the tail costs the conv2 launch more than its 36 small MMAs per tile
      // suggest, see DESIGN.md 4.2.
      float* taps = reinterpret_cast<float*>(b.r[2]);
      a.out_f32 = taps;
      a.wtail = h->umma->tailr3;
      a.bias2 = nullptr;
      if ((rc = launch<kF8R23>(h, b.r[1], a, stream))) return rc;
      a.wtail = nullptr;
      TimedScope ts(h, kSpecs[kR3].slot, stream);
      gather_gate_kernel<<<dim3((W + 63) / 64, (H + 3) / 4, n), dim3(64, 4), 0, stream>>>(
          taps, h->umma->bias[kR3], o.stack == kStackRefiners ? nullptr : b.cm, out, o.out_u8, b.refined, H, W,
          o.out_u8 ? o.peers : PeerOut());
      WN_LAUNCH_CHECK(h);
      return WN_OK;
    }
    act(b.r[2], 96, nullptr, 0);
    if ((rc = launch<kF8R2>(h, b.r[1], a, stream))) return rc;
    if (dump(9, b.r[2], 96)) return WN_OK;
    last();
    if ((rc = launch<kR3Gate>(h, b.r[2], a, stream))) return rc;
    return o.out_u8 ? mirror_u8(h, o.out_u8, o.peers, (size_t)n * H * W * 3, o.run_if, stream) : WN_OK;
  }
  // L1: 16 -> 128 (cmg) + 96 (refiners)
  act(b.a[1], 128, b.r[1], 96);
  a.skip_lo = b.exact_flag;
  a.a_hi_only = o.hi_only ? 1 : 0;
  if (o.kpack) {
    if ((rc = launch<kX3L1K>(h, b.act0, a, stream))) return rc;
  } else if ((rc = launch<kX3L1>(h, b.act0, a, stream))) return rc;
  a.skip_lo = nullptr;
  a.a_hi_only = 0;
  if (dump(0, b.a[1], 128) || dump(8, b.r[1], 96)) return WN_OK;
  if (want_cmg) {
    act(b.a[2], 128, nullptr, 0);
    if ((rc = launch<kX3C2>(h, b.a[1], a, stream))) return rc;
    if (dump(1, b.a[2], 128)) return WN_OK;
    act(b.a[3], 128, nullptr, 0);
    if ((rc = launch<kX3C3>(h, b.a[2], a, stream))) return rc;
    if (dump(2, b.a[3], 128)) return WN_OK;
    act(b.a[4], 64, nullptr, 0);
    if ((rc = launch<kX3C4>(h, b.a[3], a, stream))) return rc;
    if (dump(3, b.a[4], 64)) return WN_OK;
    act(b.a[5], 64, nullptr, 0);
    if ((rc = launch<kX3C5>(h, b.a[4], a, stream))) return rc;
    if (dump(4, b.a[5], 64)) return WN_OK;
    act(b.a[6], 64, nullptr, 0);
    if ((rc = launch<kX3C6>(h, b.a[5], a, stream))) return rc;
    if (dump(5, b.a[6], 64)) return WN_OK;
    act(b.a[7], 64, nullptr, 0);
    if ((rc = launch<kX3C7>(h, b.a[6], a, stream))) return rc;
    if (dump(6, b.a[7], 64)) return WN_OK;
    a.out_f32 = dbg_layer == 7 ? dbg_dst : b.cm;
    if ((rc = launch<kC8Sigmoid>(h, b.a[7], a, stream))) return rc;
    if (dbg_layer == 7) return WN_OK;
  }
  if (!want_ref) return WN_OK;
  act(b.r[2], 96, nullptr, 0);
  if ((rc = launch<kX3R2>(h, b.r[1], a, stream))) return rc;
  if (dump(9, b.r[2], 96)) return WN_OK;
  last();
  if ((rc = launch<kR3Gate>(h, b.r[2], a, stream))) return rc;
  return o.out_u8 ? mirror_u8(h, o.out_u8, o.peers, (size_t)n * H * W * 3, o.run_if, stream) : WN_OK;
}

// Workspace carve-up of one pass (<= umma_chunk images).
static FwdBuffers carve(void* workspace, int n, int H, int W) {
  const size_t px = (size_t)n * H * W;
  uint8_t* ws = (uint8_t*)(((uintptr_t)workspace + 1023) / 1024 * 1024);
  uint4* cmgAB[2];
  uint4* refAB[2];
  FwdBuffers b;
  memset(&b, 0, sizeof(b));
  b.act0 = (uint4*)ws;     ws += (px + (size_t)n * H) * 64;   // + one column per row: the K-packed layout is W + 1 wide
  cmgAB[0] = (uint4*)ws;   ws += px * 512;
  cmgAB[1] = (uint4*)ws;   ws += px * 512;
  refAB[0] = (uint4*)ws;   ws += px * 384;
  refAB[1] = (uint4*)ws;   ws += px * 384;
  b.cm = (float*)ws;       ws += px * 12;
  b.exact_flag = (int*)(((uintptr_t)ws + 255) / 256 * 256);
  for (int l = 1; l <= 7; l++) b.a[l] = cmgAB[(l - 1) & 1];
  b.r[1] = refAB[0];
  b.r[2] = refAB[1];
  return b;
}

// One pass in `scheme`; in the fp8-correction scheme the bf16x3 chain of the same batch is enqueued right behind
// it, every launch conditional on the sticky e4m3 range flag (ConvArgs::run_if): a batch whose activations left
// the e4m3 range is recomputed within the same call, nobody ever sees the degraded result.
static int umma_pass(wn_handle* h, const float* const in[4], const int64_t st[4][4], float* out, int n, int H, int W,
                     const FwdBuffers& b, cudaStream_t stream, FwdOpts o) {
  int rc = umma_forward_layers(h, in, st, out, n, H, W, b, stream, o);
  if (rc || o.scheme != 1 || o.dbg_layer >= 0) return rc;
  o.scheme = 0;
  o.packed = true;  // act0 (and the exact-levels flag) of this batch are still in place
  o.run_if = h->umma->overflow_dev;
  Timing* timing = h->timing;  // the conditional launches are not part of the per-kernel timing record
  h->timing = nullptr;
  rc = umma_forward_layers(h, in, st, out, n, H, W, b, stream, o);
  h->timing = timing;
  return rc;
}

int umma_debug_layer(wn_handle* h, const float* const in[4], const int64_t in_strides[4][4], int n, int H, int W,
                     int layer, float* dst, void* workspace, size_t workspace_bytes, cudaStream_t stream, int scheme) {
  if (!h->umma || umma_chunk(0, n, H, W) != n || workspace_bytes < umma_forward_workspace_bytes(n, H, W)) {
    set_error("debug layer dump: weights not packed, batch too large for one pass or workspace too small");
    return WN_E_WORKSPACE;
  }
  int rc = get_encoder();
  if (rc) return rc;
  FwdOpts o;
  o.scheme = scheme;
  o.dbg_layer = layer;
  o.dbg_dst = dst;
  o.kpack = !(h->dbg_flags & 2048);
  return umma_forward_layers(h, in, in_strides, nullptr, n, H, W, carve(workspace, n, H, W), stream, o);
}

// fp8-correction mode: once an activation has left the e4m3 range (sticky flag, mirrored to the host at the end
// of every call) this handle keeps to the bf16x3 kernels until new weights are packed.
static int effective_scheme(wn_handle* h, int scheme) {
  return (scheme == 1 && *h->umma->overflow_host) ? 0 : scheme;
}
static int mirror_overflow(wn_handle* h, int scheme, cudaStream_t stream) {
  if (scheme == 1)
    WN_CUDA(cudaMemcpyAsync(h->umma->overflow_host, h->umma->overflow_dev, sizeof(int), cudaMemcpyDeviceToHost, stream));
  return WN_OK;
}

int umma_forward(wn_handle* h, const float* const in[4], const int64_t in_strides[4][4], float* out, int n, int H,
                 int W, void* workspace, size_t workspace_bytes, cudaStream_t stream, int scheme, int stack,
                 float* refined) {
  if (!h->umma) {
    set_error("tensor-core weights have not been packed");
    return WN_E_STATE;
  }
  if (workspace_bytes < umma_forward_workspace_bytes(n, H, W)) {
    set_error("forward workspace too small: %zu < %zu", workspace_bytes, umma_forward_workspace_bytes(n, H, W));
    return WN_E_WORKSPACE;
  }
  int rc = get_encoder();
  if (rc) return rc;
  scheme = effective_scheme(h, scheme);
  const int nb = umma_chunk(h->chunk_pixels, n, H, W);
  for (int n0 = 0; n0 < n; n0 += nb) {
    const int cur = n - n0 < nb ? n - n0 : nb;
    const float* sub[4];
    for (int t = 0; t < 4; t++) sub[t] = in[t] + (long long)n0 * in_strides[t][0];
    FwdBuffers b = carve(workspace, cur, H, W);
    FwdOpts o;
    o.scheme = scheme;
    o.stack = stack;
    o.kpack = !(h->dbg_flags & 2048);
    float* dst = out + (size_t)n0 * 3 * H * W;
    if (stack == kStackCmg) b.cm = dst;                                   // the maps are the result
    if (stack == kStackRefiners) { b.refined = refined + (size_t)n0 * 9 * H * W; dst = nullptr; }
    rc = umma_pass(h, sub, in_strides, dst, cur, H, W, b, stream, o);
    if (rc) return rc;
  }
  return mirror_overflow(h, scheme, stream);
}

// preprocess -> forward -> ten2arr without materialising the four fp32 input tensors or the fp32 output:
// the per-pixel preprocess kernel writes the first layer's operand planes (8-bit levels are exact in bf16: hi
// planes only), the last launch's epilogue writes uint8 NHWC (hubconf.py:8-34, SURVEY 8f.2).
size_t umma_enhance_workspace_bytes(int n, int h, int w) {
  const int nb = umma_chunk(0, n, h, w);
  return umma_forward_workspace_bytes(n, h, w) + (preprocess_workspace_bytes(nb, h, w) + 255) / 256 * 256 + 1024;
}

int umma_enhance_u8(wn_handle* h, const uint8_t* rgb, uint8_t* out_u8, float* out_f32, int n, int H, int W,
                    void* workspace, size_t workspace_bytes, cudaStream_t stream, int scheme, const PeerOut& peers) {
  if (!h->umma) {
    set_error("tensor-core weights have not been packed");
    return WN_E_STATE;
  }
  if (workspace_bytes < umma_enhance_workspace_bytes(n, H, W)) {
    set_error("enhance workspace too small: %zu < %zu", workspace_bytes, umma_enhance_workspace_bytes(n, H, W));
    return WN_E_WORKSPACE;
  }
  int rc = get_encoder();
  if (rc) return rc;
  scheme = effective_scheme(h, scheme);
  const int nb = umma_chunk(h->chunk_pixels, n, H, W);
  uint8_t* pre_ws = (uint8_t*)(((uintptr_t)workspace + 255) / 256 * 256);
  const size_t pre_b = (preprocess_workspace_bytes(nb, H, W) + 255) / 256 * 256;
  void* fwd_ws = pre_ws + pre_b;
  const int64_t none[4][4] = {};
  const float* no_in[4] = {nullptr, nullptr, nullptr, nullptr};
  for (int n0 = 0; n0 < n; n0 += nb) {
    const int cur = n - n0 < nb ? n - n0 : nb;
    FwdBuffers b = carve(fwd_ws, cur, H, W);
    WN_CUDA(cudaMemsetAsync(b.exact_flag, 1, sizeof(int), stream));
    const bool kpack = !(h->dbg_flags & 2048);
    rc = preprocess_u8_planes(h, rgb + (size_t)n0 * H * W * 3, cur, H, W, b.act0, pre_ws, pre_b, stream, kpack ? 1 : 0);
    if (rc) return rc;
    FwdOpts o;
    o.scheme = scheme;
    o.packed = true;
    o.hi_only = true;
    o.kpack = kpack;
    o.out_u8 = out_u8 + (size_t)n0 * H * W * 3;
    o.peers.n = peers.n;
    for (int k = 0; k < peers.n; k++) o.peers.p[k] = peers.p[k] + (size_t)n0 * H * W * 3;
    rc = umma_pass(h, no_in, none, out_f32 ? out_f32 + (size_t)n0 * 3 * H * W : nullptr, cur, H, W, b, stream, o);
    if (rc) return rc;
  }
  return mirror_overflow(h, scheme, stream);
}

int umma_f8_overflowed(const wn_handle* h) { return h->umma && h->umma->overflow_host ? *h->umma->overflow_host : 0; }

}  // namespace wn
