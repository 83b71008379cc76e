// Shared declarations for the waternet_b200 CUDA library (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/waternet_b200.h"

namespace wn {

void set_error(const char* fmt, ...);

#define WN_CUDA(call)                                                                   \
  do {                                                                                  \
    cudaError_t err__ = (call);                                                         \
    if (err__ != cudaSuccess) {                                                         \
      wn::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(err__)); \
      return WN_E_CUDA;                                                                 \
    }                                                                                   \
  } while (0)

#define WN_LAUNCH_CHECK(h)   \
  do {                       \
    (h)->launches++;         \
    WN_CUDA(cudaGetLastError()); \
  } while (0)

// ---- constant tables (OpenCV 8-bit Lab, gamma 0.7, u/255) -------------------
struct Tables {
  uint16_t gtab[256];    // sRGB decode, scaled 255*8
  uint16_t ctab[3072];   // Lab f(t), scaled 1<<15
  int16_t ytab[256];     // L -> Y, scaled 1<<14
  int16_t fytab[256];    // L -> f(Y), scaled 1<<14
  uint8_t igtab[4096];   // linear -> sRGB 8 bit
  uint8_t gamma[256];    // data.py:61-65 as a LUT
  float div255[256];     // float(u)/255.f
};

void build_tables_host(Tables* t);

// ---- network description (net.py:12-42, 62-70) ------------------------------
struct LayerDesc {
  int cin, cout, ks;
};
static const LayerDesc kCmg[8] = {{12, 128, 7}, {128, 128, 5}, {128, 128, 3}, {128, 64, 1},
                                  {64, 64, 7},  {64, 64, 5},   {64, 64, 3},   {64, 3, 3}};
static const LayerDesc kRef[3] = {{6, 32, 7}, {32, 32, 5}, {32, 3, 3}};
constexpr int kNumConvs = 17;  // 8 + 3*3, in state-dict order

struct SimtLayer {
  int cin, cout, cout_pad, ks;
  float* w;     // [cin][ks*ks][cout_pad]
  float* bias;  // [cout_pad]
};

struct UmmaWeights;  // conv_umma.cu
struct UmmaBwd;      // conv_bwd.cu

// Optional per-kernel timing with CUDA events on the launching stream (bench.py's roofline leg).
enum TimingSlot {
  kSlotConv0 = 0,  // 0..16: the 17 convolutions in state-dict order (fused kernels use their first layer)
  kSlotPack = 17,  // input concat / operand packing
  kSlotGate = 18,  // sigmoid-gated weighted sum
  kSlotStats = 19,
  kSlotLuts = 20,
  kSlotApply = 21,
  kSlotPost = 22,
  kNumSlots = 23
};
// which part of WaterNet.forward a forward call evaluates (the reference's sub-modules are callable: net.py:45-56, :75-80)
enum FwdStack { kStackAll = 0, kStackCmg = 1, kStackRefiners = 2 };
struct Timing {
  static constexpr int kMax = 8192;
  bool on;
  int used, created;
  cudaEvent_t a[kMax], b[kMax];
  int slot[kMax];
};

}  // namespace wn

struct wn_handle {
  int device;
  uint64_t launches;
  wn::Tables* d_tables;
  bool packed;
  wn::SimtLayer simt[wn::kNumConvs];
  wn::UmmaWeights* umma;
  int sm_count;
  wn::Timing* timing;
  wn::UmmaBwd* bwd;
  int dbg_flags;  // unfused / plain forms of the tensor-core forward (wn_debug_set_flags); 0 in normal use
  long long chunk_pixels;  // cap on pixels per pass of the tensor-core forward (0 = default, wn_set_chunk_pixels)
};

namespace wn {

// Scope guard: records an event pair around the launches issued while it is alive.
struct TimedScope {
  Timing* t;
  int idx;
  cudaStream_t stream;
  TimedScope(wn_handle* h, int slot, cudaStream_t s) : t(h->timing), idx(-1), stream(s) {
    if (!t || !t->on || t->used >= Timing::kMax) return;
    idx = t->used;
    if (idx >= t->created) {
      if (cudaEventCreate(&t->a[idx]) != cudaSuccess || cudaEventCreate(&t->b[idx]) != cudaSuccess) {
        idx = -1;
        return;
      }
      t->created = idx + 1;
    }
    t->used++;
    t->slot[idx] = slot;
    cudaEventRecord(t->a[idx], stream);
  }
  ~TimedScope() {
    if (idx >= 0) cudaEventRecord(t->b[idx], stream);
  }
};

// K-packed first-layer planes (umma_conv.cuh, UmmaCfg KP): rows of W + 1 columns, column x + 1 = pixel x.  `o` points at
// the pixel's own column in plane 0; plane 1 (one `plane` further) holds per column [c8..11 @ x | c8..11 @ x + 1]: the
// pixel writes its c8..11 into the first half of its own column and the second half of the column to its left; the
// image's first / last pixel also write the zero halves and the zero column that padding needs.
#ifdef __CUDACC__
__device__ __forceinline__ void store_kp_pixel(uint4* o, size_t plane, int x, int W, uint4 c0_7, uint2 c8_11) {
  o[0] = c0_7;
  uint2* p1 = reinterpret_cast<uint2*>(o + plane);
  p1[0] = c8_11;        // first half of column x + 1
  p1[-1] = c8_11;       // second half of column x
  if (x == 0) {
    o[-1] = make_uint4(0u, 0u, 0u, 0u);   // plane 0, column 0 = the pixel left of the image
    p1[-2] = make_uint2(0u, 0u);          // plane 1, column 0, first half = c8..11 of that pixel
  }
  if (x == W - 1) p1[1] = make_uint2(0u, 0u);   // second half of the last column = c8..11 of the pixel right of the image
}
#endif

// preprocess.cu
size_t preprocess_workspace_bytes(int n, int h, int w);
int preprocess_u8(wn_handle* h, const uint8_t* rgb, int n, int height, int width, float* x,
                  float* wb, float* he, float* gc, uint8_t* wb_u8, uint8_t* he_u8, uint8_t* gc_u8,
                  void* workspace, size_t workspace_bytes, cudaStream_t stream);
int postprocess_u8(wn_handle* h, const float* out_nchw, uint8_t* out_nhwc, int n, int height,
                   int width, cudaStream_t stream);
size_t white_balance_gray_workspace_bytes(int n, int h, int w);
int white_balance_gray_u8(wn_handle* h, const uint8_t* gray, uint8_t* out, int n, int height, int width,
                          void* workspace, size_t workspace_bytes, cudaStream_t stream);
int resize_u8(wn_handle* h, const uint8_t* const* src, const int* src_h, const int* src_w, int n, uint8_t* dst,
              int dst_h, int dst_w, int swap_rb, cudaStream_t stream);
// transform + cat[x, wb, he, gc] straight into the first layer's operand planes: planes[n][2][H*W] of 16 B
// (8 bf16 levels 0..255: plane 0 = x.rgb wb.rgb he.rg, plane 1 = he.b gc.rgb 0 0 0 0)
// kp != 0: the K-packed layout (planes[n][2][H][W + 1], see store_kp_pixel)
int preprocess_u8_planes(wn_handle* h, const uint8_t* rgb, int n, int height, int width, uint4* planes,
                         void* workspace, size_t workspace_bytes, cudaStream_t stream, int kp = 0);

// conv_simt.cu
int simt_pack_weights(wn_handle* h, const float* const* params, cudaStream_t stream);
void simt_free(wn_handle* h);
size_t simt_forward_workspace_bytes(int n, int h, int w);
// stack (FwdStack): kStackCmg -> out = the three confidence maps; kStackRefiners -> out = refiner `which`'s image
int simt_forward(wn_handle* h, const float* const in[4], const int64_t in_strides[4][4], float* out,
                 int n, int height, int width, void* workspace, size_t workspace_bytes,
                 cudaStream_t stream, int stack = 0, int which = 0);

int simt_debug_layer(wn_handle* h, const float* const in[4], const int64_t in_strides[4][4], int n,
                     int height, int width, int layer, float* dst, void* workspace,
                     size_t workspace_bytes, cudaStream_t stream);

// conv_umma.cu
struct FwdBuffers {
  uint4* act0;    // packed input, 16 channels (bf16 hi/lo planes of v*255)
  uint4* a[8];    // a[l] = output of cmg.conv<l>, l = 1..7 (planes)
  uint4* r[3];    // r[1], r[2] = refiner conv1 / conv2 outputs, three refiners side by side (96 channels)
  float* cm;      // sigmoid confidence maps, fp32 [n][3][H][W]
  float* refined; // optional: refined images after ReLU, fp32 [n][9][H][W]
  int* exact_flag;
};
// Peer copies of the uint8 output (multi-GPU all-gather fused into the kernel that produces the output: plain stores
// to addresses mapped from the other ranks' buffers, wn_enhance_u8_peers)
struct PeerOut {
  uint8_t* p[WN_MAX_PEERS];
  int n;
};
struct FwdOpts {
  int scheme = 0;              // 1 = fp8 correction passes (WN_MODE_BF16_FP8)
  int dbg_layer = -1;          // wn_debug_forward_layer: stop after this layer and decode it into dbg_dst
  float* dbg_dst = nullptr;
  bool packed = false;         // act0 already holds the 16-channel operand planes of this batch
  bool hi_only = false;        // ... as exact 8-bit levels, hi planes only (written by the preprocess kernel)
  bool kpack = false;          // act0 is in the K-packed first-layer layout (inference; UmmaCfg KP)
  const int* run_if = nullptr; // every launch is conditional on *run_if != 0 (ConvArgs::run_if)
  uint8_t* out_u8 = nullptr;   // the last launch also writes ten2arr(out) as uint8 NHWC
  PeerOut peers = {};          // ... and the same bytes to every peer address (offsets as out_u8)
  int stack = kStackAll;       // kStackCmg: stop after the confidence maps; kStackRefiners: refiners only
};
int umma_forward_layers(wn_handle* h, const float* const in[4], const int64_t st[4][4], float* out, int n,
                        int height, int width, const FwdBuffers& b, cudaStream_t stream,
                        const FwdOpts& opts = FwdOpts());
int umma_debug_layer(wn_handle* h, const float* const in[4], const int64_t in_strides[4][4], int n,
                     int height, int width, int layer, float* dst, void* workspace,
                     size_t workspace_bytes, cudaStream_t stream, int scheme = 0);
int umma_pack_weights(wn_handle* h, const float* const* params, cudaStream_t stream);
void umma_free(wn_handle* h);
size_t umma_forward_workspace_bytes(int n, int h, int w);
int umma_chunk_images(const wn_handle* h, int n, int height, int width);
// stack = kStackCmg: out receives the three confidence maps; kStackRefiners: `refined` receives the three
// refined images as [n][9][H][W] and out is unused
int umma_forward(wn_handle* h, const float* const in[4], const int64_t in_strides[4][4], float* out,
                 int n, int height, int width, void* workspace, size_t workspace_bytes,
                 cudaStream_t stream, int scheme = 0, int stack = kStackAll, float* refined = nullptr);
size_t umma_enhance_workspace_bytes(int n, int h, int w);
int mirror_u8(wn_handle* h, const uint8_t* src, const PeerOut& peers, size_t bytes, const int* run_if, cudaStream_t stream);
int umma_enhance_u8(wn_handle* h, const uint8_t* rgb, uint8_t* out_u8, float* out_f32, int n, int height,
                    int width, void* workspace, size_t workspace_bytes, cudaStream_t stream, int scheme,
                    const PeerOut& peers = PeerOut());
int umma_f8_overflowed(const wn_handle* h);

// conv_bwd.cu
int bwd_pack_weights(wn_handle* h, const float* const* params, cudaStream_t stream);
void bwd_free(wn_handle* h);
size_t train_workspace_bytes_padded(int n, int h, int w);
int forward_train(wn_handle* h, const float* const in[4], const int64_t in_strides[4][4], float* out, int n,
                  int height, int width, void* workspace, size_t workspace_bytes, cudaStream_t stream);
int backward(wn_handle* h, const float* grad_out, float* const* grads, float* const* input_grads, int n,
             int height, int width, void* workspace, size_t workspace_bytes, cudaStream_t stream);

}  // namespace wn
