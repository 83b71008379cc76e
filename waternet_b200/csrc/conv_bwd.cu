// Backward pass of WaterNet on the tensor cores (SURVEY.md section 8f.1): the training hot loop
// of /root/reference/train.py:100-133 (loss.backward() through waternet/net.py:99-108).
//
//   gate_bwd_kernel      d(out)/d(refined), d(out)/d(cm) and sigmoid'/ReLU' -> gradient planes
//   conv_umma_kernel     data gradient = the forward implicit-GEMM kernel run on flipped,
//   <..., kEpiDgrad>     transposed weights; the epilogue applies ReLU' from the saved activation
//   wgrad_umma_kernel    weight gradient: dW[co][ci][tap] = sum_px g[px][co] * a[px+tap][ci], a
//                        GEMM whose K dimension is PIXELS.  Both operands are read straight from
//                        the activation-plane layout act[plane][y][x][8ch], which is exactly the
//                        no-swizzle MN-major UMMA layout (8 channels contiguous, 16 consecutive
//                        pixels of a row = one K=16 step); a tap is again only a start-address
//                        shift of the B operand.  Every CTA stores its fp32 partial sums; a second kernel adds
//                        them in a fixed order (bit-reproducible gradients, no atomics).
//   bias_grad_kernel     db[co] = sum_px g[px][co]
//
// All three GEMM-shaped pieces use the same bf16x3 split as the forward (gradient error ~1e-5).
#include "umma_conv.cuh"

namespace wn {

// ------------------------------------------------------------------------------------------
// Weight-gradient kernel
// ------------------------------------------------------------------------------------------
template <int KS, int NCI, int TPG>
struct WgradCfg {
  static constexpr int TX = 16;  // one K=16 step = 16 consecutive pixels of a row
  static constexpr int HALO_W = TX + KS - 1;
  static constexpr int A_PLANES = NCI / 8;
  static constexpr int stage_bytes(int ty) {
    return (2 * 16 * ty * TX * 16 + 2 * A_PLANES * (ty + KS - 1) * HALO_W * 16 + 1023) / 1024 * 1024;
  }
  // two pipeline stages (the TMA of the next tile overlaps the MMAs of this one): 8 rows per tile
  // when that fits in shared memory, else 4
  static constexpr int TY = 2 * stage_bytes(8) + 2048 <= 227 * 1024 ? 8 : 4;
  static constexpr int HALO_H = TY + KS - 1;
  static constexpr int G_PLANE = TY * TX * 16;            // one 8-channel plane of the gradient tile
  static constexpr int G_HALF = 16 * G_PLANE;             // M = 128 output channels = 16 planes
  static constexpr int G_BYTES = 2 * G_HALF;              // hi | lo
  static constexpr int A_PLANE = HALO_W * HALO_H * 16;
  static constexpr int A_HALF = A_PLANES * A_PLANE;
  static constexpr int STAGE = stage_bytes(TY);
  static constexpr int NSTAGE = 2;
  static constexpr int SMEM_BYTES = NSTAGE * STAGE + 1024 + 1024;
  static constexpr int NGROUPS = (KS * KS + TPG - 1) / TPG;
  static constexpr int COLS = TPG * NCI;
  static constexpr int TMEM_COLS = COLS <= 32 ? 32 : COLS <= 64 ? 64 : COLS <= 128 ? 128 : COLS <= 256 ? 256 : 512;
  static_assert(COLS <= 512, "tap group does not fit in TMEM");
  static_assert(NCI % 16 == 0 && NCI <= 256, "invalid UMMA N");
  static_assert(SMEM_BYTES <= 227 * 1024, "tiles do not fit in shared memory");
};

struct WgradArgs {
  float* partial;  // [CTA = split * NGROUPS + group][TPG][128][NCI] fp32 partial sums (reduced by reduce_wgrad_kernel)
  int N, H, W;
  int co_planes;    // 8-channel planes of the gradient to load (per hi/lo half)
  int planes_half;  // planes per half in the gradient buffer (lo parts start there)
  int co_valid;     // valid output channels
  int tiles_x, tiles_y;
};

constexpr int kWgradThreads = 192;  // warps 0-3 epilogue, 4 TMA producer, 5 MMA issuer

template <int KS, int NCI, int TPG>
__global__ void __launch_bounds__(kWgradThreads, 1)
wgrad_umma_kernel(const __grid_constant__ CUtensorMap tmap_g, const __grid_constant__ CUtensorMap tmap_a,
                  const WgradArgs g) {
  using C = WgradCfg<KS, NCI, TPG>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  // stage s: [gradient tile hi | lo][activation halo hi | lo]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::NSTAGE * C::STAGE);
  uint64_t* full = bars;                 // [NSTAGE]
  uint64_t* empty = bars + C::NSTAGE;    // [NSTAGE]
  uint64_t* done = bars + 2 * C::NSTAGE;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * C::NSTAGE + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int group = blockIdx.x;
  const int num_tiles = g.tiles_x * g.tiles_y * g.N;
  const int my_tiles = num_tiles > (int)blockIdx.y ? (num_tiles - 1 - (int)blockIdx.y) / (int)gridDim.y + 1 : 0;
  if (my_tiles == 0) return;
  const int tap0 = group * TPG;
  const int ntaps = min(TPG, KS * KS - tap0);

  // planes the TMA never writes (output channels beyond co_planes*8) must read as zero
  for (int st = 0; st < C::NSTAGE; st++)
    for (int i = tid; i < C::G_BYTES / 16; i += kWgradThreads)
      reinterpret_cast<uint4*>(smem + st * C::STAGE)[i] = make_uint4(0, 0, 0, 0);
  if (tid == 0) {
    for (int st = 0; st < C::NSTAGE; st++) { mbar_init(&full[st], 1); mbar_init(&empty[st], 1); }
    mbar_init(done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)C::TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (tmem_base != 0) __trap();  // one CTA per SM: the allocation starts at column 0

  if (warp == 4) {
    if (lane == 0) {
      int st = 0;
      uint32_t phase = 0;
      for (int i = 0; i < my_tiles; i++) {
        const int tile = blockIdx.y + i * gridDim.y;
        const int n = tile / (g.tiles_x * g.tiles_y);
        const int rem = tile - n * g.tiles_x * g.tiles_y;
        const int ty = rem / g.tiles_x, tx = rem - ty * g.tiles_x;
        const int x0 = tx * C::TX, y0 = ty * C::TY;
        uint8_t* g_tile = smem + st * C::STAGE;
        uint8_t* a_tile = g_tile + C::G_BYTES;
        mbar_wait(&empty[st], phase ^ 1);
        mbar_expect_tx(&full[st], (uint32_t)(2 * g.co_planes * C::G_PLANE + 2 * C::A_HALF));
        tma_load_5d(g_tile, &tmap_g, &full[st], 0, x0, y0, 0, n);
        tma_load_5d(g_tile + C::G_HALF, &tmap_g, &full[st], 0, x0, y0, g.planes_half, n);
        tma_load_5d(a_tile, &tmap_a, &full[st], 0, x0 - KS / 2, y0 - KS / 2, 0, n);
        tma_load_5d(a_tile + C::A_HALF, &tmap_a, &full[st], 0, x0 - KS / 2, y0 - KS / 2, C::A_PLANES, n);
        if (++st == C::NSTAGE) { st = 0; phase ^= 1; }
      }
    }
  } else if (warp == 5) {
    // MN-major operands (bits 15, 16): K = pixels along x, LBO = 128 B between the two 8-pixel halves
    constexpr uint32_t idesc = make_idesc(128, NCI) | (1u << 15) | (1u << 16);
    constexpr uint32_t g_hi32 = ((uint32_t)C::G_PLANE >> 4) | (1u << 14);
    constexpr uint32_t a_hi32 = ((uint32_t)C::A_PLANE >> 4) | (1u << 14);
    constexpr uint32_t lbo = (128u >> 4) << 16;
    int st = 0;
    uint32_t phase = 0;
    for (int i = 0; i < my_tiles; i++) {
      mbar_wait(&full[st], phase);
      tc_fence_after();
      const uint32_t g_lo32 = (smem_u32(smem + st * C::STAGE) >> 4) | lbo;
      const uint32_t a_lo32 = (smem_u32(smem + st * C::STAGE + C::G_BYTES) >> 4) | lbo;
      if (elect_one_sync()) {
        for (int tl = 0; tl < ntaps; tl++) {
          const int tap = tap0 + tl;
          const int ky = tap / KS, kx = tap - ky * KS;
          const uint32_t d = (uint32_t)(tl * NCI);
#pragma unroll
          for (int y = 0; y < C::TY; y++) {
            const uint32_t g_row = g_lo32 + (uint32_t)(y * C::TX);
            const uint32_t a_row = a_lo32 + (uint32_t)((y + ky) * C::HALO_W + kx);
            const uint32_t first = (i | y) == 0 ? 0u : 1u;
            umma_bf16_split(d, g_row, g_hi32, a_row, a_hi32, idesc, first);                                   // g_hi x a_hi
            umma_bf16_split(d, g_row + (uint32_t)(C::G_HALF >> 4), g_hi32, a_row, a_hi32, idesc, 1u);         // g_lo x a_hi
            umma_bf16_split(d, g_row, g_hi32, a_row + (uint32_t)(C::A_HALF >> 4), a_hi32, idesc, 1u);         // g_hi x a_lo
          }
        }
        umma_commit(&empty[st]);
        if (i == my_tiles - 1) umma_commit(done);
      }
      __syncwarp();
      if (++st == C::NSTAGE) { st = 0; phase ^= 1; }
    }
  } else if (warp < 4) {
    mbar_wait(done, 0);
    tc_fence_after();
    const int co = warp * 32 + lane;  // TMEM lane == output channel
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    float* base = g.partial + (size_t)(blockIdx.y * gridDim.x + blockIdx.x) * (TPG * 128 * NCI);
    for (int tl = 0; tl < ntaps; tl++) {
      float4* dst = reinterpret_cast<float4*>(base + ((size_t)tl * 128 + co) * NCI);
#pragma unroll 1
      for (int c0 = 0; c0 < NCI; c0 += 16) {
        uint32_t v[16];
        tmem_ld16(tmem_base + lane_base + (uint32_t)(tl * NCI + c0), v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; j += 4)
          dst[(c0 + j) >> 2] = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]),
                                           __uint_as_float(v[j + 3]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"((uint32_t)C::TMEM_COLS)
                 : "memory");
  }
}

// dense[tap][co][c] = sum over the pixel splits, in split order, of the CTAs' partial sums (deterministic)
__global__ void __launch_bounds__(256)
reduce_wgrad_kernel(const float* __restrict__ partial, float* __restrict__ dense, int kk, int tpg, int ngroups,
                    int splits, int nci, int co_valid) {
  const int per_tap = 128 * nci;
  const long long total = (long long)kk * per_tap;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int tap = (int)(i / per_tap);
    const int rem = (int)(i - (long long)tap * per_tap);
    const int grp = tap / tpg, tl = tap - grp * tpg;
    float acc = 0.f;
    if (rem / nci < co_valid) {
      const float* p = partial + ((size_t)grp * tpg + tl) * per_tap + rem;
      for (int s = 0; s < splits; s++) acc += p[(size_t)s * ngroups * tpg * per_tap];
    }
    dense[i] = acc;
  }
}
// db[c] = sum of the per-block partial sums, in block order
__global__ void reduce_bias_kernel(const float* __restrict__ part, float* __restrict__ db, int nsplit, int stride,
                                   int co_valid) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= co_valid) return;
  float acc = 0.f;
  for (int s = 0; s < nsplit; s++) acc += part[(size_t)s * stride + c];
  db[c] = acc;
}

// part[split][c] = sum over this block's images and pixels of (hi + lo).  grid = (planes, splits), 256 threads.
__global__ void __launch_bounds__(256)
bias_grad_kernel(const uint4* __restrict__ gplanes, float* __restrict__ db, int planes_half, int n_img, int hw,
                 int co_valid) {
  __shared__ float s_part[8][256];
  const int plane = blockIdx.x;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  const long long total = (long long)n_img * hw;
  for (long long i = (long long)blockIdx.y * 256 + threadIdx.x; i < total; i += (long long)gridDim.y * 256) {
    const int n = (int)(i / hw);
    const int pix = (int)(i - (long long)n * hw);
    const uint4 h4 = gplanes[((size_t)n * 2 * planes_half + plane) * hw + pix];
    const uint4 l4 = gplanes[((size_t)n * 2 * planes_half + planes_half + plane) * hw + pix];
    const uint32_t hs[4] = {h4.x, h4.y, h4.z, h4.w}, ls[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
    for (int j = 0; j < 8; j++) {
      acc[j] += __uint_as_float(((hs[j >> 1] >> ((j & 1) * 16)) & 0xffffu) << 16) +
                __uint_as_float(((ls[j >> 1] >> ((j & 1) * 16)) & 0xffffu) << 16);
    }
  }
#pragma unroll
  for (int j = 0; j < 8; j++) s_part[j][threadIdx.x] = acc[j];
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o)
#pragma unroll
      for (int j = 0; j < 8; j++) s_part[j][threadIdx.x] += s_part[j][threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x < 8) db[(size_t)blockIdx.y * gridDim.x * 8 + plane * 8 + threadIdx.x] = s_part[threadIdx.x][0];
}

// dense [kk][128][nci] -> OIHW gradient tensor:  dst[o][c][t] = scale * dense[t][row_off + o][cd(c)]
__global__ void extract_wgrad_kernel(const float* __restrict__ dense, float* __restrict__ dst, int co, int ci, int kk,
                                     int nci, int row_off, int split, int base0, int base1, float scale) {
  const int total = co * ci * kk;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int t = i % kk;
    int c = (i / kk) % ci;
    int o = i / (kk * ci);
    int cd = c < split ? base0 + c : base1 + (c - split);
    dst[i] = scale * dense[((size_t)t * 128 + row_off + o) * nci + cd];
  }
}

// Backward of out = sum_r refined_r * cm_r, refined = relu(z_r3), cm = sigmoid(z_8)   (net.py:100-108)
//   g_zr3[3r+c] = g_out[c] * cm[r]            where refined[3r+c] > 0
//   g_z8[r]     = (sum_c g_out[c] * refined[3r+c]) * cm[r] * (1 - cm[r])
// Both are written as 16-channel gradient planes (bf16 hi/lo), unused channels zero.
__global__ void __launch_bounds__(256)
gate_bwd_kernel(const float* __restrict__ g_out, const float* __restrict__ cm, const float* __restrict__ refined,
                uint4* __restrict__ g8, uint4* __restrict__ gr3, int hw) {
  const int n = blockIdx.y;
  const int pix = blockIdx.x * 256 + threadIdx.x;
  if (pix >= hw) return;
  float go[3], c[3], v8[16], v9[16];
#pragma unroll
  for (int k = 0; k < 3; k++) {
    go[k] = g_out[((size_t)n * 3 + k) * hw + pix];
    c[k] = cm[((size_t)n * 3 + k) * hw + pix];
  }
#pragma unroll
  for (int j = 0; j < 16; j++) v8[j] = v9[j] = 0.f;
#pragma unroll
  for (int r = 0; r < 3; r++) {
    float dot = 0.f;
#pragma unroll
    for (int k = 0; k < 3; k++) {
      const float rf = refined[((size_t)n * 9 + 3 * r + k) * hw + pix];
      dot += go[k] * rf;
      v9[3 * r + k] = rf > 0.f ? go[k] * c[r] : 0.f;
    }
    v8[r] = dot * c[r] * (1.0f - c[r]);
  }
  auto store = [&](uint4* base, const float* v) {
    uint32_t hi[8], lo[8];
#pragma unroll
    for (int j = 0; j < 16; j += 2) {
      split_bf16x2(v[j], v[j + 1], hi[j >> 1], lo[j >> 1]);
    }
    uint4* o = base + (size_t)n * 4 * hw + pix;  // planes: hi0, hi1, lo0, lo1
    o[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    o[hw] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
    o[2 * (size_t)hw] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    o[3 * (size_t)hw] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
  };
  store(g8, v8);
  store(gr3, v9);
}

// data-gradient weights: dense_d[row_off + c][col(o)][kk-1-t] = W[o][c][t]   (transpose + spatial flip)
// input channel c lands in row  row_off + c  (c < split)  or  row_off + c + shift  (c >= split)
__global__ void scatter_weights_T_kernel(const float* __restrict__ src, float* __restrict__ dense, int co, int ci,
                                         int kk, int kpad, int row_off, int col_off, int split, int shift) {
  const int total = co * ci * kk;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int t = i % kk;
    int c = (i / kk) % ci;
    int o = i / (kk * ci);
    int row = row_off + c + (c >= split ? shift : 0);
    dense[((size_t)row * kpad + col_off + o) * kk + (kk - 1 - t)] = src[i];
  }
}

// d(loss)/d(input images) from the two 32-channel gradient buffers of the first layers (12 real channels:
// x, wb, he, gc): sum them (hi + lo each) and write the four fp32 (N,3,H,W) tensors.
struct InputGrads {
  float* p[4];
};
__global__ void __launch_bounds__(256)
input_grads_kernel(const uint4* __restrict__ ga, const uint4* __restrict__ gb, InputGrads out, int hw) {
  const int n = blockIdx.y;
  const int pix = blockIdx.x * 256 + threadIdx.x;
  if (pix >= hw) return;
  float v[16];
#pragma unroll
  for (int j = 0; j < 16; j++) v[j] = 0.f;
  const uint4* bufs[2] = {ga, gb};
#pragma unroll
  for (int b = 0; b < 2; b++) {
#pragma unroll
    for (int plane = 0; plane < 2; plane++) {
#pragma unroll
      for (int half = 0; half < 2; half++) {  // 32-channel buffers: 4 planes per half
        const uint4 q = bufs[b][((size_t)n * 8 + half * 4 + plane) * hw + pix];
        const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int j = 0; j < 8; j++)
          v[plane * 8 + j] += __uint_as_float(((w[j >> 1] >> ((j & 1) * 16)) & 0xffffu) << 16);
      }
    }
  }
#pragma unroll
  for (int t = 0; t < 4; t++)
#pragma unroll
    for (int c = 0; c < 3; c++) out.p[t][((size_t)n * 3 + c) * hw + pix] = v[t * 3 + c];
}

// ------------------------------------------------------------------------------------------
// Host side
// ------------------------------------------------------------------------------------------
enum DgradLayer { kD8 = 0, kD7, kD6, kD5, kD4, kD3, kD2, kDR3, kDR2, kD1, kDR1, kNumDgrad };
// The data-gradient launches, one row each: the weight layout they are packed in and the kernel configuration.
// All but the HBM-bound 1x1 run as CTA pairs, like the forward.
struct DgradSpec {
  int ks, kpad, npad, nblk, concat, conv;  // K = forward Cout (padded), N per block = forward Cin
  int cg;
  int s, as, tps;                          // sub-tiles per tile, accumulator stages, taps per weight stage
};
static constexpr DgradSpec kDSpecs[kNumDgrad] = {
    {3, 16, 64, 1, 1, 7, 2, 2, 2, 9},
    {3, 64, 64, 1, 1, 6, 2, 2, 2, 9},
    {5, 64, 64, 1, 1, 5, 2, 2, 2, 5},
    {7, 64, 64, 1, 1, 4, 2, 2, 2, 7},
    {1, 64, 128, 1, 0, 3, 1, 2, 2, 1},
    {3, 128, 128, 1, 0, 2, 2, 2, 2, 3},
    {5, 128, 128, 1, 0, 1, 2, 2, 2, 5},
    {3, 16, 96, 1, 0, -1, 2, 2, 2, 9},
    {5, 96, 32, 3, 1, -1, 2, 2, 1, 5},
    // gradients with respect to the packed 16-channel input (only when an input image requires grad):
    // from cmg.conv1 (K = 128) and from the three refiner conv1 (K = 96); 32 rows, 12 real
    {7, 128, 32, 1, 1, 0, 2, 2, 2, 7},
    {7, 96, 32, 1, 1, -2, 2, 2, 2, 7}};

struct UmmaBwd {
  uint8_t* stages[kNumDgrad];
  float* zero_bias;  // 256 zeros: the dgrad epilogue has no bias
  float* dense;      // packing scratch
};

static size_t dgrad_stage_bytes(const DgradSpec& s) {
  if (s.cg == 2) return (size_t)2 * (s.kpad / 16) * s.ks * s.ks * s.npad * (s.concat ? 48 : 32);
  return (size_t)(s.kpad / 16) * s.ks * s.ks * s.npad * 64;
}

int bwd_pack_weights(wn_handle* h, const float* const* params, cudaStream_t stream) {
  if (!h->bwd) h->bwd = (UmmaBwd*)calloc(1, sizeof(UmmaBwd));
  for (int i = 0; i < kNumDgrad; i++)
    if (!h->bwd->stages[i]) WN_CUDA(cudaMalloc(&h->bwd->stages[i], dgrad_stage_bytes(kDSpecs[i])));
  if (!h->bwd->zero_bias) WN_CUDA(cudaMalloc(&h->bwd->zero_bias, 256 * sizeof(float)));
  if (!h->bwd->dense) WN_CUDA(cudaMalloc(&h->bwd->dense, (size_t)128 * 128 * 49 * sizeof(float)));
  UmmaBwd* u = h->bwd;
  WN_CUDA(cudaMemsetAsync(u->zero_bias, 0, 256 * sizeof(float), stream));
  for (int li = 0; li < kNumDgrad; li++) {
    const DgradSpec& s = kDSpecs[li];
    const int kk = s.ks * s.ks, rows = s.npad * s.nblk;
    WN_CUDA(cudaMemsetAsync(u->dense, 0, (size_t)rows * s.kpad * kk * sizeof(float), stream));
    if (s.conv >= 0) {
      const LayerDesc& d = kCmg[s.conv];
      scatter_weights_T_kernel<<<128, 256, 0, stream>>>(params[2 * s.conv], u->dense, d.cout, d.cin, kk, s.kpad, 0, 0,
                                                        d.cin, 0);
      WN_LAUNCH_CHECK(h);
    } else if (s.conv == -2) {
      for (int r = 0; r < 3; r++) {  // refiner r reads cat[x, input r+1]: rows 0..2 and 3(r+1)..3(r+1)+2
        scatter_weights_T_kernel<<<128, 256, 0, stream>>>(params[2 * (8 + 3 * r)], u->dense, 32, 6, kk, s.kpad, 0, 32 * r,
                                                          3, 3 * (r + 1) - 3);
        WN_LAUNCH_CHECK(h);
      }
    } else {
      for (int r = 0; r < 3; r++) {
        const int conv = 8 + 3 * r + (li == kDR3 ? 2 : 1);
        const int co = li == kDR3 ? 3 : 32;
        scatter_weights_T_kernel<<<128, 256, 0, stream>>>(params[2 * conv], u->dense, co, 32, kk, s.kpad, 32 * r,
                                                          (li == kDR3 ? 3 : 32) * r, 32, 0);
        WN_LAUNCH_CHECK(h);
      }
    }
    if (s.cg == 2)
      pack_stages_cg2_kernel<<<256, 256, 0, stream>>>(u->dense, (__nv_bfloat16*)u->stages[li], s.npad, s.kpad, kk,
                                                      s.concat, s.nblk);
    else
      pack_stages_kernel<<<256, 256, 0, stream>>>(u->dense, (__nv_bfloat16*)u->stages[li], s.npad, s.kpad, kk,
                                                  s.concat, s.nblk);
    WN_LAUNCH_CHECK(h);
  }
  return WN_OK;
}

void bwd_free(wn_handle* h) {
  if (!h->bwd) return;
  for (int i = 0; i < kNumDgrad; i++)
    if (h->bwd->stages[i]) cudaFree(h->bwd->stages[i]);
  if (h->bwd->zero_bias) cudaFree(h->bwd->zero_bias);
  if (h->bwd->dense) cudaFree(h->bwd->dense);
  free(h->bwd);
  h->bwd = nullptr;
}

// ---- training workspace ------------------------------------------------------------------
struct TrainBuffers {
  FwdBuffers f;
  uint4 *ga, *gb, *gra, *grb, *g8, *gr3, *gin_a, *gin_b;
  float* dense;
  float* partial;  // per-CTA partial sums of the weight-gradient GEMM / per-block partial bias sums
};
static constexpr size_t kDenseBytes = (size_t)49 * 128 * 128 * sizeof(float);
// one slot per CTA of a weight-gradient launch (one wave: <= SM count), each TPG * NCI <= 512 accumulator columns
// x 128 rows of fp32
static constexpr size_t kPartialSlotBytes = (size_t)512 * 128 * sizeof(float);
static constexpr int kPartialSlots = 192;
static constexpr size_t kPartialBytes = kPartialSlots * kPartialSlotBytes;
// bytes per pixel: act0 64 | a1..a3 512 each | a4..a7 256 each | r1, r2 384 each | cm 12 | refined 36 |
//                  gradient ping-pong 512 + 512 + 384 + 384 | 16-channel gradients 64 + 64
static constexpr size_t kTrainBytesPerPixel =
    64 + 3 * 512 + 4 * 256 + 2 * 384 + 12 + 36 + 2 * 512 + 2 * 384 + 2 * 64 + 2 * 128;  // + two 32-ch input-gradient buffers
static constexpr long long kTrainMaxPixels = 8ll << 20;

size_t train_workspace_bytes(int n, int h, int w) {
  return (size_t)n * h * w * kTrainBytesPerPixel + kDenseBytes + kPartialBytes + 8192;
}

static void carve(TrainBuffers* t, void* workspace, size_t px) {
  uint8_t* ws = (uint8_t*)(((uintptr_t)workspace + 1023) / 1024 * 1024);
  auto take = [&](size_t bytes) {
    uint8_t* p = ws;
    ws += (bytes + 1023) / 1024 * 1024;
    return p;
  };
  memset(t, 0, sizeof(*t));
  t->f.act0 = (uint4*)take(px * 64);
  for (int l = 1; l <= 3; l++) t->f.a[l] = (uint4*)take(px * 512);
  for (int l = 4; l <= 7; l++) t->f.a[l] = (uint4*)take(px * 256);
  t->f.r[1] = (uint4*)take(px * 384);
  t->f.r[2] = (uint4*)take(px * 384);
  t->f.cm = (float*)take(px * 12);
  t->f.refined = (float*)take(px * 36);
  t->f.exact_flag = (int*)take(256);
  t->ga = (uint4*)take(px * 512);
  t->gb = (uint4*)take(px * 512);
  t->gra = (uint4*)take(px * 384);
  t->grb = (uint4*)take(px * 384);
  t->g8 = (uint4*)take(px * 64);
  t->gr3 = (uint4*)take(px * 64);
  t->gin_a = (uint4*)take(px * 128);
  t->gin_b = (uint4*)take(px * 128);
  t->dense = (float*)take(kDenseBytes);
  t->partial = (float*)take(kPartialBytes);
}

static int check_train_args(int n, int H, int W, size_t bytes) {
  if ((long long)n * H * W > kTrainMaxPixels) {
    set_error("training pass limited to %lld pixels per call (got %lld)", kTrainMaxPixels, (long long)n * H * W);
    return WN_E_UNSUPPORTED;
  }
  // carve() aligns every region to 1 KiB: allow for it
  if (bytes < train_workspace_bytes(n, H, W) + 24 * 1024) {
    set_error("training workspace too small: %zu < %zu", bytes, train_workspace_bytes(n, H, W) + 24 * 1024);
    return WN_E_WORKSPACE;
  }
  return WN_OK;
}

size_t train_workspace_bytes_padded(int n, int h, int w) { return train_workspace_bytes(n, h, w) + 24 * 1024; }

int forward_train(wn_handle* h, const float* const in[4], const int64_t st[4][4], float* out, int n, int H, int W,
                  void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  int rc = check_train_args(n, H, W, workspace_bytes);
  if (rc) return rc;
  TrainBuffers t;
  carve(&t, workspace, (size_t)n * H * W);
  return umma_forward_layers(h, in, st, out, n, H, W, t.f, stream);
}

static int make_plane_tmap(CUtensorMap* tm, void* base, int planes_total, int N, int H, int W, int box_w, int box_h,
                           int box_planes) {
  cuuint64_t dims[5] = {8, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)planes_total, (cuuint64_t)N};
  cuuint64_t strides[4] = {16, (cuuint64_t)W * 16, (cuuint64_t)H * W * 16, (cuuint64_t)planes_total * H * W * 16};
  cuuint32_t box[5] = {8, (cuuint32_t)box_w, (cuuint32_t)box_h, (cuuint32_t)box_planes, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, base, dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with %d (wgrad planes=%d box=%dx%dx%d)", (int)r, planes_total, box_w,
              box_h, box_planes);
    return WN_E_CUDA;
  }
  return WN_OK;
}

// dense[tap][128][NCI] += sum_px g[px][co] * a[px + tap][ci]
template <int KS, int NCI, int TPG>
static int launch_wgrad(wn_handle* h, uint4* gplanes, int co_valid, uint4* aplanes, float* dense, float* partial, int n,
                        int H, int W, cudaStream_t stream) {
  using C = WgradCfg<KS, NCI, TPG>;
  const int co_planes = (co_valid + 7) / 8;
  const int planes_half = (co_valid + 15) / 16 * 2;  // gradient buffers hold a multiple of 16 channels
  CUtensorMap tg, ta;
  int rc = make_plane_tmap(&tg, gplanes, 2 * planes_half, n, H, W, C::TX, C::TY, co_planes);
  if (rc) return rc;
  rc = make_plane_tmap(&ta, aplanes, 2 * C::A_PLANES, n, H, W, C::HALO_W, C::HALO_H, C::A_PLANES);
  if (rc) return rc;
  WgradArgs a;
  a.partial = partial;
  a.N = n; a.H = H; a.W = W;
  a.co_planes = co_planes;
  a.planes_half = planes_half;
  a.co_valid = co_valid;
  a.tiles_x = (W + C::TX - 1) / C::TX;
  a.tiles_y = (H + C::TY - 1) / C::TY;
  const long long tiles = (long long)a.tiles_x * a.tiles_y * n;
  long long splits = h->sm_count / C::NGROUPS;  // one wave: every CTA owns an SM (shared memory footprint)
  if (splits > tiles) splits = tiles;
  if (splits < 1) splits = 1;
  if (splits * C::NGROUPS > kPartialSlots) splits = kPartialSlots / C::NGROUPS;
  static_assert((size_t)TPG * 128 * NCI * sizeof(float) <= kPartialSlotBytes, "partial-sum slot");
  auto kern = wgrad_umma_kernel<KS, NCI, TPG>;
  WN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
  kern<<<dim3(C::NGROUPS, (unsigned)splits), kWgradThreads, C::SMEM_BYTES, stream>>>(tg, ta, a);
  WN_LAUNCH_CHECK(h);
  reduce_wgrad_kernel<<<256, 256, 0, stream>>>(partial, dense, KS * KS, TPG, C::NGROUPS, (int)splits, NCI, co_valid);
  WN_LAUNCH_CHECK(h);
  return WN_OK;
}

static int extract(wn_handle* h, const float* dense, float* dst, int co, int ci, int ks, int nci, int row_off,
                   int split, int base0, int base1, float scale, cudaStream_t stream) {
  extract_wgrad_kernel<<<64, 256, 0, stream>>>(dense, dst, co, ci, ks * ks, nci, row_off, split, base0, base1, scale);
  WN_LAUNCH_CHECK(h);
  return WN_OK;
}

static int bias_grad(wn_handle* h, const uint4* gplanes, int planes_half, int co_valid, float* db, float* partial, int n,
                     int hw, cudaStream_t stream) {
  const int planes = (co_valid + 7) / 8;
  bias_grad_kernel<<<dim3(planes, 64), 256, 0, stream>>>(gplanes, partial, planes_half, n, hw, co_valid);
  WN_LAUNCH_CHECK(h);
  reduce_bias_kernel<<<(co_valid + 127) / 128, 128, 0, stream>>>(partial, db, 64, planes * 8, co_valid);
  WN_LAUNCH_CHECK(h);
  return WN_OK;
}

template <int L>
static int launch_dgrad(wn_handle* h, uint4* g_in, uint4* g_out, int out_channels, const uint4* saved, int n, int H,
                        int W, cudaStream_t stream) {
  constexpr DgradSpec s = kDSpecs[L];
  ConvArgs a;
  memset(&a, 0, sizeof(a));
  a.N = n; a.H = H; a.W = W;
  a.dst0.base = g_out;
  a.dst0.planes_half = out_channels / 8;
  a.split_c = out_channels;
  a.cout = out_channels;
  a.mask_base = saved;  // nullptr: no ReLU in front (network input)
  a.mask_planes_half = out_channels / 8;
  return launch_conv<s.ks, s.kpad, s.npad, s.s, s.as, kEpiDgrad, s.concat, s.nblk, s.tps, s.cg>(
      h, kSlotGate, h->bwd->stages[L], h->bwd->zero_bias, g_in, a, stream);
}

int backward(wn_handle* h, const float* grad_out, float* const* grads, float* const* input_grads, int n, int H,
             int W, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  if (!h->bwd) {
    set_error("backward weights have not been packed");
    return WN_E_STATE;
  }
  int rc = check_train_args(n, H, W, workspace_bytes);
  if (rc) return rc;
  if ((rc = get_encoder())) return rc;
  TrainBuffers t;
  carve(&t, workspace, (size_t)n * H * W);
  const int hw = H * W;
  auto gw = [&](int conv) { return grads[2 * conv]; };
  auto gb = [&](int conv) { return grads[2 * conv + 1]; };

  gate_bwd_kernel<<<dim3((hw + 255) / 256, n), 256, 0, stream>>>(grad_out, t.f.cm, t.f.refined, t.g8, t.gr3, hw);
  WN_LAUNCH_CHECK(h);

  // ---- confidence-map stack: conv8 ... conv1 ---------------------------------------------
  // conv8 (64 -> 3, 3x3): g = g8 (16-channel planes, 3 valid), a = a7
  if ((rc = launch_wgrad<3, 64, 8>(h, t.g8, 3, t.f.a[7], t.dense, t.partial, n, H, W, stream))) return rc;
  if ((rc = extract(h, t.dense, gw(7), 3, 64, 3, 64, 0, 64, 0, 0, 1.f, stream))) return rc;
  if ((rc = bias_grad(h, t.g8, 2, 3, gb(7), t.partial, n, hw, stream))) return rc;
  if ((rc = launch_dgrad<kD8>(h, t.g8, t.ga, 64, t.f.a[7], n, H, W, stream))) return rc;
  // conv7 (64 -> 64, 3x3): g = ga
  if ((rc = launch_wgrad<3, 64, 8>(h, t.ga, 64, t.f.a[6], t.dense, t.partial, n, H, W, stream))) return rc;
  if ((rc = extract(h, t.dense, gw(6), 64, 64, 3, 64, 0, 64, 0, 0, 1.f, stream))) return rc;
  if ((rc = bias_grad(h, t.ga, 8, 64, gb(6), t.partial, n, hw, stream))) return rc;
  if ((rc = launch_dgrad<kD7>(h, t.ga, t.gb, 64, t.f.a[6], n, H, W, stream))) return rc;
  // conv6 (5x5): g = gb
  if ((rc = launch_wgrad<5, 64, 8>(h, t.gb, 64, t.f.a[5], t.dense, t.partial, n, H, W, stream))) return rc;
  if ((rc = extract(h, t.dense, gw(5), 64, 64, 5, 64, 0, 64, 0, 0, 1.f, stream))) return rc;
  if ((rc = bias_grad(h, t.gb, 8, 64, gb(5), t.partial, n, hw, stream))) return rc;
  if ((rc = launch_dgrad<kD6>(h, t.gb, t.ga, 64, t.f.a[5], n, H, W, stream))) return rc;
  // conv5 (7x7): g = ga
  if ((rc = launch_wgrad<7, 64, 8>(h, t.ga, 64, t.f.a[4], t.dense, t.partial, n, H, W, stream))) return rc;
  if ((rc = extract(h, t.dense, gw(4), 64, 64, 7, 64, 0, 64, 0, 0, 1.f, stream))) return rc;
  if ((rc = bias_grad(h, t.ga, 8, 64, gb(4), t.partial, n, hw, stream))) return rc;
  if ((rc = launch_dgrad<kD5>(h, t.ga, t.gb, 64, t.f.a[4], n, H, W, stream))) return rc;
  // conv4 (128 -> 64, 1x1): g = gb (64), a = a3 (128)
  if ((rc = launch_wgrad<1, 128, 1>(h, t.gb, 64, t.f.a[3], t.dense, t.partial, n, H, W, stream))) return rc;
  if ((rc = extract(h, t.dense, gw(3), 64, 128, 1, 128, 0, 128, 0, 0, 1.f, stream))) return rc;
  if ((rc = bias_grad(h, t.gb, 8, 64, gb(3), t.partial, n, hw, stream))) return rc;
  if ((rc = launch_dgrad<kD4>(h, t.gb, t.ga, 128, t.f.a[3], n, H, W, stream))) return rc;
  // conv3 (128 -> 128, 3x3): g = ga
  if ((rc = launch_wgrad<3, 128, 4>(h, t.ga, 128, t.f.a[2], t.dense, t.partial, n, H, W, stream))) return rc;
  if ((rc = extract(h, t.dense, gw(2), 128, 128, 3, 128, 0, 128, 0, 0, 1.f, stream))) return rc;
  if ((rc = bias_grad(h, t.ga, 16, 128, gb(2), t.partial, n, hw, stream))) return rc;
  if ((rc = launch_dgrad<kD3>(h, t.ga, t.gb, 128, t.f.a[2], n, H, W, stream))) return rc;
  // conv2 (5x5): g = gb
  if ((rc = launch_wgrad<5, 128, 4>(h, t.gb, 128, t.f.a[1], t.dense, t.partial, n, H, W, stream))) return rc;
  if ((rc = extract(h, t.dense, gw(1), 128, 128, 5, 128, 0, 128, 0, 0, 1.f, stream))) return rc;
  if ((rc = bias_grad(h, t.gb, 16, 128, gb(1), t.partial, n, hw, stream))) return rc;
  if ((rc = launch_dgrad<kD2>(h, t.gb, t.ga, 128, t.f.a[1], n, H, W, stream))) return rc;
  // conv1 (12 -> 128, 7x7): g = ga, a = act0 (holds v*255 -> scale the gradient back)
  if ((rc = launch_wgrad<7, 16, 32>(h, t.ga, 128, t.f.act0, t.dense, t.partial, n, H, W, stream))) return rc;
  if ((rc = extract(h, t.dense, gw(0), 128, 12, 7, 16, 0, 12, 0, 0, 1.f / 255.f, stream))) return rc;
  if ((rc = bias_grad(h, t.ga, 16, 128, gb(0), t.partial, n, hw, stream))) return rc;
  if (input_grads) {  // d/d(packed input) from cmg.conv1: ga (128) -> g8 region reused as a 32-channel buffer
    if ((rc = launch_dgrad<kD1>(h, t.ga, t.gin_a, 32, nullptr, n, H, W, stream))) return rc;
  }

  // ---- refiners: conv3, conv2, conv1 (three side by side) ---------------------------------
  if ((rc = launch_wgrad<3, 96, 5>(h, t.gr3, 9, t.f.r[2], t.dense, t.partial, n, H, W, stream))) return rc;
  for (int r = 0; r < 3; r++) {
    if ((rc = extract(h, t.dense, gw(8 + 3 * r + 2), 3, 32, 3, 96, 3 * r, 32, 32 * r, 0, 1.f, stream))) return rc;
  }
  {
    // the nine bias gradients sit in one 16-channel buffer: reduce once, then split per refiner
    float* tmp = t.dense + (size_t)9 * 128 * 96;
    if ((rc = bias_grad(h, t.gr3, 2, 9, tmp, t.partial, n, hw, stream))) return rc;
    for (int r = 0; r < 3; r++)
      WN_CUDA(cudaMemcpyAsync(gb(8 + 3 * r + 2), tmp + 3 * r, 3 * sizeof(float), cudaMemcpyDeviceToDevice, stream));
  }
  if ((rc = launch_dgrad<kDR3>(h, t.gr3, t.gra, 96, t.f.r[2], n, H, W, stream))) return rc;
  if ((rc = launch_wgrad<5, 96, 5>(h, t.gra, 96, t.f.r[1], t.dense, t.partial, n, H, W, stream))) return rc;
  {
    float* tmp = t.dense + (size_t)25 * 128 * 96;
    if ((rc = bias_grad(h, t.gra, 12, 96, tmp, t.partial, n, hw, stream))) return rc;
    for (int r = 0; r < 3; r++) {
      if ((rc = extract(h, t.dense, gw(8 + 3 * r + 1), 32, 32, 5, 96, 32 * r, 32, 32 * r, 0, 1.f, stream))) return rc;
      WN_CUDA(cudaMemcpyAsync(gb(8 + 3 * r + 1), tmp + 32 * r, 32 * sizeof(float), cudaMemcpyDeviceToDevice, stream));
    }
  }
  if ((rc = launch_dgrad<kDR2>(h, t.gra, t.grb, 96, t.f.r[1], n, H, W, stream))) return rc;
  if ((rc = launch_wgrad<7, 16, 32>(h, t.grb, 96, t.f.act0, t.dense, t.partial, n, H, W, stream))) return rc;
  {
    float* tmp = t.dense + (size_t)49 * 128 * 16;
    if ((rc = bias_grad(h, t.grb, 12, 96, tmp, t.partial, n, hw, stream))) return rc;
    for (int r = 0; r < 3; r++) {
      // refiner r reads cat[x, input r+1]: channels 0..2 and 3(r+1)..3(r+1)+2 of the packed input
      if ((rc = extract(h, t.dense, gw(8 + 3 * r), 32, 6, 7, 16, 32 * r, 3, 0, 3 * (r + 1), 1.f / 255.f, stream))) return rc;
      WN_CUDA(cudaMemcpyAsync(gb(8 + 3 * r), tmp + 32 * r, 32 * sizeof(float), cudaMemcpyDeviceToDevice, stream));
    }
  }
  if (input_grads) {
    if ((rc = launch_dgrad<kDR1>(h, t.grb, t.gin_b, 32, nullptr, n, H, W, stream))) return rc;
    InputGrads ig;
    for (int i = 0; i < 4; i++) ig.p[i] = input_grads[i];
    input_grads_kernel<<<dim3((hw + 255) / 256, n), 256, 0, stream>>>(t.gin_a, t.gin_b, ig, hw);
    WN_LAUNCH_CHECK(h);
  }
  return WN_OK;
}

}  // namespace wn
