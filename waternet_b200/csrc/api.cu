// C ABI of libwaternet_b200.so (see include/waternet_b200.h for the contract).
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace wn {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static int resolve_mode(int mode) {
  if (mode == WN_MODE_DEFAULT) return WN_MODE_BF16_FP8;
  return mode;
}

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) ok = false;
    if (ok && prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

}  // namespace wn

using namespace wn;

extern "C" {

int wn_abi_version(void) { return WN_ABI_VERSION; }

const char* wn_last_error(void) { return g_err; }

int wn_build_tables_host(uint16_t* gtab, uint16_t* ctab, int16_t* ytab, int16_t* fytab,
                         uint8_t* igtab, uint8_t* gamma, float* div255) {
  if (!gtab || !ctab || !ytab || !fytab || !igtab || !gamma || !div255) {
    set_error("wn_build_tables_host: null output");
    return WN_E_INVALID;
  }
  Tables* t = (Tables*)malloc(sizeof(Tables));
  build_tables_host(t);
  memcpy(gtab, t->gtab, sizeof(t->gtab));
  memcpy(ctab, t->ctab, sizeof(t->ctab));
  memcpy(ytab, t->ytab, sizeof(t->ytab));
  memcpy(fytab, t->fytab, sizeof(t->fytab));
  memcpy(igtab, t->igtab, sizeof(t->igtab));
  memcpy(gamma, t->gamma, sizeof(t->gamma));
  memcpy(div255, t->div255, sizeof(t->div255));
  free(t);
  return WN_OK;
}

int wn_create(int device, wn_handle** out) {
  if (!out) {
    set_error("wn_create: out is NULL");
    return WN_E_INVALID;
  }
  *out = nullptr;
  int count = 0;
  WN_CUDA(cudaGetDeviceCount(&count));
  if (device < 0 || device >= count) {
    set_error("wn_create: device %d out of range (%d devices)", device, count);
    return WN_E_INVALID;
  }
  DeviceGuard guard(device);
  cudaDeviceProp prop;
  WN_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_error("wn_create: device %d is sm_%d%d; this library is built for sm_100a only", device,
              prop.major, prop.minor);
    return WN_E_UNSUPPORTED;
  }
  wn_handle* h = (wn_handle*)calloc(1, sizeof(wn_handle));
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  Tables* t = (Tables*)malloc(sizeof(Tables));
  build_tables_host(t);
  cudaError_t e = cudaMalloc(&h->d_tables, sizeof(Tables));
  if (e == cudaSuccess) e = cudaMemcpy(h->d_tables, t, sizeof(Tables), cudaMemcpyHostToDevice);
  free(t);
  if (e != cudaSuccess) {
    set_error("wn_create: %s", cudaGetErrorString(e));
    free(h);
    return WN_E_CUDA;
  }
  *out = h;
  return WN_OK;
}

void wn_destroy(wn_handle* h) {
  if (!h) return;
  DeviceGuard guard(h->device);
  simt_free(h);
  umma_free(h);
  bwd_free(h);
  if (h->d_tables) cudaFree(h->d_tables);
  if (h->timing) {
    for (int i = 0; i < h->timing->created; i++) {
      cudaEventDestroy(h->timing->a[i]);
      cudaEventDestroy(h->timing->b[i]);
    }
    free(h->timing);
  }
  free(h);
}

int wn_pack_weights(wn_handle* h, const float* const* params, void* stream) {
  if (!h || !params) {
    set_error("wn_pack_weights: null argument");
    return WN_E_INVALID;
  }
  for (int i = 0; i < WN_NUM_PARAMS; i++)
    if (!params[i]) {
      set_error("wn_pack_weights: params[%d] is NULL", i);
      return WN_E_INVALID;
    }
  DeviceGuard guard(h->device);
  int rc = simt_pack_weights(h, params, (cudaStream_t)stream);
  if (rc) return rc;
  rc = umma_pack_weights(h, params, (cudaStream_t)stream);
  if (rc) return rc;
  rc = bwd_pack_weights(h, params, (cudaStream_t)stream);
  if (rc) return rc;
  h->packed = true;
  return WN_OK;
}

size_t wn_forward_workspace_bytes(int n, int h, int w, int mode) {
  if (n <= 0 || h <= 0 || w <= 0) return 0;
  switch (resolve_mode(mode)) {
    case WN_MODE_FP32_SIMT: return simt_forward_workspace_bytes(n, h, w);
    case WN_MODE_BF16X3:
    case WN_MODE_BF16_FP8: return umma_forward_workspace_bytes(n, h, w);
  }
  return 0;
}

int wn_forward(wn_handle* h, const float* x, const float* wb, const float* he, const float* gc,
               const int64_t in_strides[4][4], float* out, int n, int height, int width, int mode,
               void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !x || !wb || !he || !gc || !in_strides || !out || !workspace) {
    set_error("wn_forward: null argument");
    return WN_E_INVALID;
  }
  if (n <= 0 || height <= 0 || width <= 0) {
    set_error("wn_forward: bad shape n=%d h=%d w=%d", n, height, width);
    return WN_E_INVALID;
  }
  if (!h->packed) {
    set_error("wn_forward: wn_pack_weights has not been called");
    return WN_E_STATE;
  }
  DeviceGuard guard(h->device);
  const float* in[4] = {x, wb, he, gc};
  switch (resolve_mode(mode)) {
    case WN_MODE_FP32_SIMT:
      return simt_forward(h, in, in_strides, out, n, height, width, workspace, workspace_bytes,
                          (cudaStream_t)stream);
    case WN_MODE_BF16X3:
      return umma_forward(h, in, in_strides, out, n, height, width, workspace, workspace_bytes,
                          (cudaStream_t)stream, 0);
    case WN_MODE_BF16_FP8:
      return umma_forward(h, in, in_strides, out, n, height, width, workspace, workspace_bytes,
                          (cudaStream_t)stream, 1);
  }
  set_error("wn_forward: unknown mode %d", mode);
  return WN_E_INVALID;
}

size_t wn_preprocess_workspace_bytes(int n, int h, int w) {
  if (n <= 0 || h <= 0 || w <= 0) return 0;
  return preprocess_workspace_bytes(n, h, w);
}

int wn_preprocess_u8(wn_handle* h, const uint8_t* rgb, int n, int height, int width, float* x,
                     float* wb, float* he, float* gc, uint8_t* wb_u8, uint8_t* he_u8,
                     uint8_t* gc_u8, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !rgb || !workspace) {
    set_error("wn_preprocess_u8: null argument");
    return WN_E_INVALID;
  }
  if (n <= 0 || height <= 0 || width <= 0) {
    set_error("wn_preprocess_u8: bad shape n=%d h=%d w=%d", n, height, width);
    return WN_E_INVALID;
  }
  DeviceGuard guard(h->device);
  return preprocess_u8(h, rgb, n, height, width, x, wb, he, gc, wb_u8, he_u8, gc_u8, workspace,
                       workspace_bytes, (cudaStream_t)stream);
}

int wn_postprocess_u8(wn_handle* h, const float* out_nchw, uint8_t* out_nhwc, int n, int height,
                      int width, void* stream) {
  if (!h || !out_nchw || !out_nhwc || n <= 0 || height <= 0 || width <= 0) {
    set_error("wn_postprocess_u8: bad argument");
    return WN_E_INVALID;
  }
  DeviceGuard guard(h->device);
  return postprocess_u8(h, out_nchw, out_nhwc, n, height, width, (cudaStream_t)stream);
}

size_t wn_white_balance_gray_workspace_bytes(int n, int h, int w) {
  if (n <= 0 || h <= 0 || w <= 0) return 0;
  return white_balance_gray_workspace_bytes(n, h, w);
}

int wn_white_balance_gray_u8(wn_handle* h, const uint8_t* gray, uint8_t* out, int n, int height, int width,
                             void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !gray || !out || !workspace || n <= 0 || height <= 0 || width <= 0) {
    set_error("wn_white_balance_gray_u8: bad argument");
    return WN_E_INVALID;
  }
  if ((size_t)height * width > (size_t)0x7fffffff / 3 || n > 65535) {
    set_error("image too large: n=%d h=%d w=%d", n, height, width);
    return WN_E_UNSUPPORTED;
  }
  DeviceGuard guard(h->device);
  return white_balance_gray_u8(h, gray, out, n, height, width, workspace, workspace_bytes, (cudaStream_t)stream);
}

int wn_resize_u8(wn_handle* h, const uint8_t* const* src_dev, const int* src_h, const int* src_w, int n,
                 uint8_t* dst_nhwc, int dst_h, int dst_w, int swap_rb, void* stream) {
  if (!h || !src_dev || !src_h || !src_w || !dst_nhwc || n <= 0 || dst_h <= 0 || dst_w <= 0) {
    set_error("wn_resize_u8: bad argument");
    return WN_E_INVALID;
  }
  DeviceGuard guard(h->device);
  return resize_u8(h, src_dev, src_h, src_w, n, dst_nhwc, dst_h, dst_w, swap_rb, (cudaStream_t)stream);
}

static size_t align256(size_t v) { return (v + 255) / 256 * 256; }

// fp32 CUDA-core mode: the API tensors are materialised (preprocess -> 4 fp32 tensors -> forward -> fp32 -> ten2arr)
static size_t enhance_simt_workspace_bytes(int n, int h, int w) {
  size_t tens = align256((size_t)n * 3 * h * w * sizeof(float));
  return 5 * tens + align256(preprocess_workspace_bytes(n, h, w)) +
         align256(simt_forward_workspace_bytes(n, h, w)) + 256;
}

size_t wn_enhance_workspace_bytes(int n, int h, int w, int mode) {
  if (n <= 0 || h <= 0 || w <= 0) return 0;
  if (resolve_mode(mode) == WN_MODE_FP32_SIMT) return enhance_simt_workspace_bytes(n, h, w);
  return umma_enhance_workspace_bytes(n, h, w);
}

int wn_enhance_u8(wn_handle* h, const uint8_t* rgb, uint8_t* out_nhwc, float* out_f32_or_null,
                  int n, int height, int width, int mode, void* workspace, size_t workspace_bytes,
                  void* stream) {
  return wn_enhance_u8_peers(h, rgb, out_nhwc, out_f32_or_null, nullptr, 0, n, height, width, mode, workspace,
                             workspace_bytes, stream);
}

int wn_enhance_u8_peers(wn_handle* h, const uint8_t* rgb, uint8_t* out_nhwc, float* out_f32_or_null,
                        uint8_t* const* peer_out, int n_peers, int n, int height, int width, int mode,
                        void* workspace, size_t workspace_bytes, void* stream) {
  PeerOut peers = {};
  if (n_peers < 0 || n_peers > WN_MAX_PEERS || (n_peers > 0 && !peer_out)) {
    set_error("wn_enhance_u8_peers: 0..%d peer addresses", WN_MAX_PEERS);
    return WN_E_INVALID;
  }
  for (int k = 0; k < n_peers; k++) {
    if (!peer_out[k]) {
      set_error("wn_enhance_u8_peers: peer address %d is null", k);
      return WN_E_INVALID;
    }
    peers.p[k] = peer_out[k];
  }
  peers.n = n_peers;
  if (!h || !rgb || !out_nhwc || !workspace) {
    set_error("wn_enhance_u8: null argument");
    return WN_E_INVALID;
  }
  if (n <= 0 || height <= 0 || width <= 0) {
    set_error("wn_enhance_u8: bad shape n=%d h=%d w=%d", n, height, width);
    return WN_E_INVALID;
  }
  if (!h->packed) {
    set_error("wn_enhance_u8: wn_pack_weights has not been called");
    return WN_E_STATE;
  }
  if (workspace_bytes < wn_enhance_workspace_bytes(n, height, width, mode)) {
    set_error("wn_enhance_u8: workspace too small");
    return WN_E_WORKSPACE;
  }
  if ((size_t)height * width > (size_t)0x7fffffff / 3 || n > 65535) {
    set_error("image too large: n=%d h=%d w=%d", n, height, width);
    return WN_E_UNSUPPORTED;
  }
  DeviceGuard guard(h->device);
  if (resolve_mode(mode) != WN_MODE_FP32_SIMT)  // tensor-core modes: folded path, nothing fp32 is materialised
    return umma_enhance_u8(h, rgb, out_nhwc, out_f32_or_null, n, height, width, workspace, workspace_bytes,
                           (cudaStream_t)stream, resolve_mode(mode) == WN_MODE_BF16_FP8 ? 1 : 0, peers);
  uint8_t* ws = (uint8_t*)(((uintptr_t)workspace + 255) / 256 * 256);
  const size_t tens = align256((size_t)n * 3 * height * width * sizeof(float));
  float* t[5];
  for (int i = 0; i < 5; i++) {
    t[i] = (float*)ws;
    ws += tens;
  }
  void* pre_ws = ws;
  size_t pre_b = align256(preprocess_workspace_bytes(n, height, width));
  ws += pre_b;
  void* fwd_ws = ws;
  size_t fwd_b = align256(simt_forward_workspace_bytes(n, height, width));
  int rc = wn_preprocess_u8(h, rgb, n, height, width, t[0], t[1], t[2], t[3], nullptr, nullptr,
                            nullptr, pre_ws, pre_b, stream);
  if (rc) return rc;
  const int64_t hw = (int64_t)height * width;
  const int64_t st[4][4] = {{3 * hw, hw, width, 1}, {3 * hw, hw, width, 1}, {3 * hw, hw, width, 1},
                            {3 * hw, hw, width, 1}};
  float* outf = out_f32_or_null ? out_f32_or_null : t[4];
  rc = wn_forward(h, t[0], t[1], t[2], t[3], st, outf, n, height, width, mode, fwd_ws, fwd_b, stream);
  if (rc) return rc;
  rc = wn_postprocess_u8(h, outf, out_nhwc, n, height, width, stream);
  if (rc) return rc;
  return mirror_u8(h, out_nhwc, peers, (size_t)n * height * width * 3, nullptr, (cudaStream_t)stream);
}

// ---- the reference's callable sub-modules (net.py:45-56 ConfidenceMapGenerator.forward, :75-80 Refiner.forward)
size_t wn_submodule_workspace_bytes(int n, int h, int w, int mode) {
  if (n <= 0 || h <= 0 || w <= 0) return 0;
  if (resolve_mode(mode) == WN_MODE_FP32_SIMT) return simt_forward_workspace_bytes(n, h, w);
  // + the three refined images side by side (the refiners run as one block-diagonal stack)
  return align256(umma_forward_workspace_bytes(n, h, w)) + align256((size_t)n * 9 * h * w * sizeof(float)) + 256;
}

int wn_confidence_maps(wn_handle* h, const float* x, const float* wb, const float* he, const float* gc,
                       const int64_t in_strides[4][4], float* out_maps, int n, int height, int width, int mode,
                       void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !x || !wb || !he || !gc || !in_strides || !out_maps || !workspace || n <= 0 || height <= 0 || width <= 0) {
    set_error("wn_confidence_maps: bad argument");
    return WN_E_INVALID;
  }
  if (!h->packed) {
    set_error("wn_confidence_maps: wn_pack_weights has not been called");
    return WN_E_STATE;
  }
  if (workspace_bytes < wn_submodule_workspace_bytes(n, height, width, mode)) {
    set_error("wn_confidence_maps: workspace too small");
    return WN_E_WORKSPACE;
  }
  DeviceGuard guard(h->device);
  const float* in[4] = {x, wb, he, gc};
  const int m = resolve_mode(mode);
  if (m == WN_MODE_FP32_SIMT)
    return simt_forward(h, in, in_strides, out_maps, n, height, width, workspace, workspace_bytes,
                        (cudaStream_t)stream, kStackCmg, 0);
  if (m != WN_MODE_BF16X3 && m != WN_MODE_BF16_FP8) {
    set_error("wn_confidence_maps: unknown mode %d", mode);
    return WN_E_INVALID;
  }
  return umma_forward(h, in, in_strides, out_maps, n, height, width, workspace, workspace_bytes,
                      (cudaStream_t)stream, m == WN_MODE_BF16_FP8 ? 1 : 0, kStackCmg, nullptr);
}

int wn_refine(wn_handle* h, int which, const float* x, const float* xbar, const int64_t in_strides[2][4],
              float* out, int n, int height, int width, int mode, void* workspace, size_t workspace_bytes,
              void* stream) {
  if (!h || !x || !xbar || !in_strides || !out || !workspace || n <= 0 || height <= 0 || width <= 0 || which < 0 ||
      which > 2) {
    set_error("wn_refine: bad argument");
    return WN_E_INVALID;
  }
  if (!h->packed) {
    set_error("wn_refine: wn_pack_weights has not been called");
    return WN_E_STATE;
  }
  if (workspace_bytes < wn_submodule_workspace_bytes(n, height, width, mode)) {
    set_error("wn_refine: workspace too small");
    return WN_E_WORKSPACE;
  }
  DeviceGuard guard(h->device);
  // refiner r sees cat[x, input r+1] (net.py:101-103): hand xbar to every slot, keep refiner `which`
  const float* in[4] = {x, xbar, xbar, xbar};
  int64_t st[4][4];
  for (int t = 0; t < 4; t++)
    for (int k = 0; k < 4; k++) st[t][k] = in_strides[t == 0 ? 0 : 1][k];
  const int m = resolve_mode(mode);
  if (m == WN_MODE_FP32_SIMT)
    return simt_forward(h, in, st, out, n, height, width, workspace, workspace_bytes, (cudaStream_t)stream,
                        kStackRefiners, which);
  if (m != WN_MODE_BF16X3 && m != WN_MODE_BF16_FP8) {
    set_error("wn_refine: unknown mode %d", mode);
    return WN_E_INVALID;
  }
  uint8_t* ws = (uint8_t*)(((uintptr_t)workspace + 255) / 256 * 256);
  const size_t fwd_b = align256(umma_forward_workspace_bytes(n, height, width));
  float* refined = (float*)(ws + fwd_b);
  int rc = umma_forward(h, in, st, nullptr, n, height, width, ws, fwd_b, (cudaStream_t)stream,
                        m == WN_MODE_BF16_FP8 ? 1 : 0, kStackRefiners, refined);
  if (rc) return rc;
  const size_t img = (size_t)3 * height * width * sizeof(float);
  WN_CUDA(cudaMemcpy2DAsync(out, img, refined + (size_t)which * 3 * height * width, 3 * img, img, n,
                            cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return WN_OK;
}

int wn_set_chunk_pixels(wn_handle* h, long long max_pixels) {
  if (!h || max_pixels < 0) {
    set_error("wn_set_chunk_pixels: bad argument");
    return WN_E_INVALID;
  }
  h->chunk_pixels = max_pixels;
  return WN_OK;
}

int wn_forward_chunk_images(const wn_handle* h, int n, int height, int width) {
  if (!h || n <= 0 || height <= 0 || width <= 0) return 0;
  return umma_chunk_images(h, n, height, width);
}

int wn_f8_overflowed(const wn_handle* h) { return h ? umma_f8_overflowed(h) : 0; }

uint64_t wn_launch_count(const wn_handle* h) { return h ? h->launches : 0; }

int wn_debug_set_flags(wn_handle* h, int flags) {
  if (!h) {
    set_error("wn_debug_set_flags: null handle");
    return WN_E_INVALID;
  }
  if (flags & ~(256 | 512 | 1024 | 2048)) {
    set_error("wn_debug_set_flags: unknown flag bits 0x%x", flags & ~(256 | 512 | 1024 | 2048));
    return WN_E_INVALID;
  }
  h->dbg_flags = flags;
  return WN_OK;
}

size_t wn_train_workspace_bytes(int n, int h, int w) {
  if (n <= 0 || h <= 0 || w <= 0) return 0;
  return train_workspace_bytes_padded(n, h, w);
}

int wn_forward_train(wn_handle* h, const float* x, const float* wb, const float* he, const float* gc,
                     const int64_t in_strides[4][4], float* out, int n, int height, int width,
                     void* train_workspace, size_t workspace_bytes, void* stream) {
  if (!h || !x || !wb || !he || !gc || !in_strides || !out || !train_workspace || n <= 0 || height <= 0 ||
      width <= 0) {
    set_error("wn_forward_train: bad argument");
    return WN_E_INVALID;
  }
  if (!h->packed) {
    set_error("wn_forward_train: wn_pack_weights has not been called");
    return WN_E_STATE;
  }
  DeviceGuard guard(h->device);
  const float* in[4] = {x, wb, he, gc};
  return forward_train(h, in, in_strides, out, n, height, width, train_workspace, workspace_bytes,
                       (cudaStream_t)stream);
}

int wn_backward(wn_handle* h, const float* grad_out, float* const* grads, float* const* input_grads, int n,
                int height, int width, void* train_workspace, size_t workspace_bytes, void* stream) {
  if (!h || !grad_out || !grads || !train_workspace || n <= 0 || height <= 0 || width <= 0) {
    set_error("wn_backward: bad argument");
    return WN_E_INVALID;
  }
  for (int i = 0; i < WN_NUM_PARAMS; i++)
    if (!grads[i]) {
      set_error("wn_backward: grads[%d] is NULL", i);
      return WN_E_INVALID;
    }
  if (!h->packed) {
    set_error("wn_backward: wn_pack_weights has not been called");
    return WN_E_STATE;
  }
  if (input_grads)
    for (int i = 0; i < 4; i++)
      if (!input_grads[i]) {
        set_error("wn_backward: input_grads[%d] is NULL", i);
        return WN_E_INVALID;
      }
  DeviceGuard guard(h->device);
  return backward(h, grad_out, grads, input_grads, n, height, width, train_workspace, workspace_bytes,
                  (cudaStream_t)stream);
}

int wn_debug_forward_layer(wn_handle* h, const float* x, const float* wb, const float* he,
                           const float* gc, const int64_t in_strides[4][4], int n, int height,
                           int width, int mode, int layer, float* dst, void* workspace,
                           size_t workspace_bytes, void* stream) {
  if (!h || !x || !wb || !he || !gc || !in_strides || !dst || !workspace || layer < 0 || layer > 9) {
    set_error("wn_debug_forward_layer: bad argument");
    return WN_E_INVALID;
  }
  if (!h->packed) {
    set_error("wn_debug_forward_layer: wn_pack_weights has not been called");
    return WN_E_STATE;
  }
  DeviceGuard guard(h->device);
  const float* in[4] = {x, wb, he, gc};
  if (resolve_mode(mode) == WN_MODE_FP32_SIMT)
    return simt_debug_layer(h, in, in_strides, n, height, width, layer, dst, workspace, workspace_bytes,
                            (cudaStream_t)stream);
  return umma_debug_layer(h, in, in_strides, n, height, width, layer, dst, workspace, workspace_bytes,
                          (cudaStream_t)stream, resolve_mode(mode) == WN_MODE_BF16_FP8 ? 1 : 0);
}

int wn_enable_timing(wn_handle* h, int on) {
  if (!h) {
    set_error("wn_enable_timing: null handle");
    return WN_E_INVALID;
  }
  if (!h->timing) h->timing = (Timing*)calloc(1, sizeof(Timing));
  h->timing->on = on != 0;
  h->timing->used = 0;
  return WN_OK;
}

int wn_read_timings(wn_handle* h, float* ms, int* count) {
  if (!h || !ms || !count) {
    set_error("wn_read_timings: null argument");
    return WN_E_INVALID;
  }
  if (!h->timing) return WN_OK;
  DeviceGuard guard(h->device);
  Timing* t = h->timing;
  for (int i = 0; i < t->used; i++) {
    float e = 0.f;
    WN_CUDA(cudaEventElapsedTime(&e, t->a[i], t->b[i]));
    ms[t->slot[i]] += e;
    count[t->slot[i]] += 1;
  }
  t->used = 0;
  return WN_OK;
}

}  // extern "C"
