/*
 * waternet_b200 -- C ABI of the B200-native WaterNet hot path.
 *
 * The reference (tnwei/waternet @ 2091896) is pure Python; it has no FFI.  The
 * boundary it exposes for this path is its Python API, and every entry point
 * below is what a binding for one of those calls would bind (file:line are
 * relative to the reference checkout):
 *
 *   wn_preprocess_u8      waternet/data.py:81-90   transform(rgb) -> wb, gc, he
 *                         + hubconf.py:8-21        arr2ten_noeinops (x/255, HWC->1CHW)
 *                         + hubconf.py:85-91       preprocess(rgb) -> rgb, wb, he, gc tensors
 *   wn_pack_weights       waternet/net.py:12-42,62-70,94-97  the 34-tensor state dict
 *                         (hubconf.py:83 / inference.py:111-120 load_state_dict)
 *   wn_forward            waternet/net.py:99-108   WaterNet.forward(x, wb, ce, gc)
 *   wn_confidence_maps    waternet/net.py:45-56    ConfidenceMapGenerator.forward(x, wb, ce, gc)
 *   wn_refine             waternet/net.py:75-80    Refiner.forward(x, xbar)
 *   wn_resize_u8          waternet/training_utils.py:94-107  cv2.resize + BGR2RGB of the dataset items
 *   wn_postprocess_u8     hubconf.py:24-34         ten2arr_noeinops (clip, *255, truncate, NCHW->NHWC)
 *   wn_enhance_u8         hubconf.py:85-94 + net.py:99-108: preprocess -> model -> postprocess
 *                         (the per-frame body of inference.py:261-323)
 *   wn_forward_train /    train.py:108 `out = model(...)` and train.py:130-131 `loss.backward()`
 *   wn_backward           (autograd through net.py:99-108)
 *
 * Conventions: every data pointer is a DEVICE pointer on the handle's device
 * unless its name ends in _host; the caller owns every buffer (the handle only
 * owns its packed weights and constant tables); every call is asynchronous on
 * `stream` (a cudaStream_t passed as void*); return 0 on success, a negative
 * WN_E_* code otherwise with a message available from wn_last_error() (thread
 * local).  A handle may be used from one thread at a time.
 */
#ifndef WATERNET_B200_H_
#define WATERNET_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WN_ABI_VERSION 3

#define WN_OK 0
#define WN_E_INVALID (-1)   /* bad argument (NULL pointer, non-positive size, unknown mode) */
#define WN_E_CUDA (-2)      /* a CUDA call failed; wn_last_error() has cudaGetErrorString */
#define WN_E_STATE (-3)     /* call order: forward before wn_pack_weights, etc. */
#define WN_E_WORKSPACE (-4) /* workspace smaller than wn_*_workspace_bytes() */
#define WN_E_UNSUPPORTED (-5)

/* Arithmetic used for the 17 convolutions of wn_forward. */
#define WN_MODE_FP32_SIMT 0 /* fp32 FMA on CUDA cores (bit-for-bit independent of tensor cores) */
#define WN_MODE_BF16X3 1    /* tcgen05 tensor cores, 3-term bf16 split operands, fp32 accumulate */
#define WN_MODE_BF16_FP8 2  /* same, the two correction terms of the tensor-bound layers as one fp8 MMA */
#define WN_MODE_DEFAULT (-1) /* the library's fastest mode that meets the 1e-3 parity bar: WN_MODE_BF16_FP8 */

#define WN_NUM_PARAMS 34

typedef struct wn_handle wn_handle;

int wn_abi_version(void);
const char* wn_last_error(void);

/* One handle per device.  Builds the constant tables (sRGB / Lab / gamma). */
int wn_create(int device, wn_handle** out);
void wn_destroy(wn_handle* h);

/*
 * Host-only: fill the constant tables the preprocess kernels use, so that they
 * can be checked on a machine without a GPU.  Sizes: gtab[256], ctab[3072],
 * ytab[256], fytab[256], igtab[4096], gamma[256], div255[256].
 */
int wn_build_tables_host(uint16_t* gtab, uint16_t* ctab, int16_t* ytab, int16_t* fytab,
                         uint8_t* igtab, uint8_t* gamma, float* div255);

/*
 * params: WN_NUM_PARAMS device pointers to contiguous fp32 tensors in the order of
 * WaterNet().state_dict(): cmg.conv1.weight, cmg.conv1.bias, ... cmg.conv8.bias,
 * wb_refiner.conv1.weight ... gc_refiner.conv3.bias; weights are OIHW.
 * Re-packs them into the kernels' layouts (device side, asynchronous).
 */
int wn_pack_weights(wn_handle* h, const float* const* params, void* stream);

/*
 * WaterNet.forward.  x/wb/he/gc: fp32 (N,3,H,W) with arbitrary element strides
 * in_strides[i] = {sN, sC, sH, sW} (contiguous NCHW and the channels_last strides
 * arr2ten produces are both accepted).  out: fp32 contiguous NCHW (N,3,H,W).
 */
size_t wn_forward_workspace_bytes(int n, int h, int w, int mode);
int wn_forward(wn_handle* h, const float* x, const float* wb, const float* he, const float* gc,
               const int64_t in_strides[4][4], float* out, int n, int height, int width, int mode,
               void* workspace, size_t workspace_bytes, void* stream);

/*
 * transform + arr2ten.  rgb: uint8 NHWC (N,H,W,3).  Any output pointer may be
 * NULL.  fp32 outputs are contiguous NCHW (N,3,H,W) in [0,1] (u/255, true
 * division); *_u8 outputs are NHWC like the reference's numpy arrays.
 * Statistics (white balance quantiles, CLAHE tiles) are per image.
 */
size_t wn_preprocess_workspace_bytes(int n, int h, int w);
int wn_preprocess_u8(wn_handle* h, const uint8_t* rgb, int n, int height, int width, float* x,
                     float* wb, float* he, float* gc, uint8_t* wb_u8, uint8_t* he_u8,
                     uint8_t* gc_u8, void* workspace, size_t workspace_bytes, void* stream);

/*
 * The grayscale branch of white_balance_transform (waternet/data.py:30-36: saturation levels 0.001 / 0.005):
 * gray / out are uint8 (N,H,W).  No caller in the reference uses it; provided for completeness of data.py.
 */
size_t wn_white_balance_gray_workspace_bytes(int n, int h, int w);
int wn_white_balance_gray_u8(wn_handle* h, const uint8_t* gray, uint8_t* out, int n, int height, int width,
                             void* workspace, size_t workspace_bytes, void* stream);

/*
 * Batched cv2.resize(img, (dst_w, dst_h)) of 8-bit 3-channel images, default INTER_LINEAR, as the training
 * dataset applies it per item (waternet/training_utils.py:94-103) -- bit-exact OpenCV arithmetic.  src_dev,
 * src_h, src_w are HOST arrays of n entries: device pointers to HWC uint8 images and their sizes.  dst_nhwc:
 * (n, dst_h, dst_w, 3).  swap_rb != 0 also applies the BGR<->RGB swap that follows the resize
 * (training_utils.py:106-107).
 */
int wn_resize_u8(wn_handle* h, const uint8_t* const* src_dev, const int* src_h, const int* src_w, int n,
                 uint8_t* dst_nhwc, int dst_h, int dst_w, int swap_rb, void* stream);

/* ten2arr: fp32 NCHW (N,3,H,W) -> uint8 NHWC, clip to [0,1], *255, truncate. */
int wn_postprocess_u8(wn_handle* h, const float* out_nchw, uint8_t* out_nhwc, int n, int height,
                      int width, void* stream);

/*
 * The reference's callable sub-modules, evaluated with the weights of the packed state dict.
 * wn_confidence_maps: the three sigmoid maps as one fp32 contiguous (N,3,H,W) tensor (channel r = the map
 * net.py:55 returns as out<r+1>).  wn_refine: refiner `which` (0 = wb_refiner, 1 = ce_refiner, 2 = gc_refiner)
 * applied to cat[x, xbar]; in_strides[0] / [1] are the element strides of x / xbar; out fp32 contiguous
 * (N,3,H,W).  Both take the workspace of wn_submodule_workspace_bytes.
 */
size_t wn_submodule_workspace_bytes(int n, int h, int w, int mode);
int wn_confidence_maps(wn_handle* h, const float* x, const float* wb, const float* he, const float* gc,
                       const int64_t in_strides[4][4], float* out_maps, int n, int height, int width, int mode,
                       void* workspace, size_t workspace_bytes, void* stream);
int wn_refine(wn_handle* h, int which, const float* x, const float* xbar, const int64_t in_strides[2][4],
              float* out, int n, int height, int width, int mode, void* workspace, size_t workspace_bytes,
              void* stream);

/*
 * preprocess -> forward -> postprocess without leaving the device.  In the tensor-core modes nothing fp32 is
 * materialised: the per-pixel preprocess kernel writes the first layer's operand planes (8-bit levels, the /255
 * of arr2ten is folded into the first layer's weights) and the last launch's epilogue writes the uint8 image
 * (and the fp32 output too when out_f32_or_null is given).
 */
size_t wn_enhance_workspace_bytes(int n, int h, int w, int mode);
int wn_enhance_u8(wn_handle* h, const uint8_t* rgb, uint8_t* out_nhwc, float* out_f32_or_null,
                  int n, int height, int width, int mode, void* workspace, size_t workspace_bytes,
                  void* stream);

/*
 * wn_enhance_u8 with the all-gather of the output fused into the kernel that produces it (SURVEY 8e: the one
 * exchange of the sharded path): the launch that writes out_nhwc stores the same bytes to peer_out[0..n_peers) --
 * addresses inside the other ranks' buffers, mapped with wn_peer_open (NVLink stores), each the start of where THIS
 * batch belongs there.  Any alignment works; 4-byte aligned rows leave as whole 96-byte segments (16-byte aligned
 * buffers as 16-byte copies in the copy-kernel forms), anything else byte by byte.  In the default mode that launch is
 * the HBM-bound gather/gate kernel at the end of every pass, so the exchange of a pass rides on a kernel that
 * leaves the tensor cores and most of the power budget idle; the other modes (and the range guard's re-run)
 * finish with a copy kernel.  Completion at the peers is the caller's business (wn_stream_write_value32 +
 * wn_memcpy_async of the flag word + wn_stream_wait_value32, see below).
 */
#define WN_MAX_PEERS 15
int wn_enhance_u8_peers(wn_handle* h, const uint8_t* rgb, uint8_t* out_nhwc, float* out_f32_or_null,
                        uint8_t* const* peer_out, int n_peers, int n, int height, int width, int mode,
                        void* workspace, size_t workspace_bytes, void* stream);

/*
 * Training step (reference train.py:100-133: out = model(...); loss.backward()).
 * wn_forward_train is wn_forward (tensor-core mode) that additionally keeps every activation in
 * `train_workspace`; wn_backward consumes that workspace and d(loss)/d(out) (fp32 contiguous NCHW)
 * and OVERWRITES the 34 gradient tensors `grads` (device pointers, same order, shapes and layout as
 * `params` of wn_pack_weights).  input_grads is NULL or four device pointers to fp32 contiguous
 * (N,3,H,W) tensors that receive d(loss)/d(x), d/d(wb), d/d(he), d/d(gc).
 * The workspace must stay untouched between the two calls; n*h*w <= 8 Mi pixels per call.
 */
size_t wn_train_workspace_bytes(int n, int h, int w);
int wn_forward_train(wn_handle* h, const float* x, const float* wb, const float* he, const float* gc,
                     const int64_t in_strides[4][4], float* out, int n, int height, int width,
                     void* train_workspace, size_t workspace_bytes, void* stream);
int wn_backward(wn_handle* h, const float* grad_out, float* const* grads, float* const* input_grads, int n,
                int height, int width, void* train_workspace, size_t workspace_bytes, void* stream);

/*
 * Per-kernel device timing (measurement aid for bench.py, off by default).  When on, every
 * kernel group is bracketed by a cudaEvent pair on the launching stream.  wn_read_timings
 * must be called after the stream has been synchronised; it adds the elapsed milliseconds and
 * the number of bracketed launches per slot into ms[] / count[] (WN_NUM_TIMING_SLOTS entries:
 * 0..16 the convolutions in state-dict order, 17 operand packing, 18 gated sum, 19 preprocess
 * statistics, 20 LUT build, 21 per-pixel apply, 22 postprocess) and clears the record.
 */
#define WN_NUM_TIMING_SLOTS 23
int wn_enable_timing(wn_handle* h, int on);
int wn_read_timings(wn_handle* h, float* ms, int* count);

/*
 * Test aid: run wn_forward's layer chain in `mode` up to an intermediate activation and return it
 * as contiguous fp32 NCHW.  layer: 0..6 = output of cmg.conv1..conv7 (after ReLU), 7 = the three
 * sigmoid confidence maps, 8 = the three refiners' conv1 outputs concatenated (96 channels),
 * 9 = their conv2 outputs (96 channels).  dst must hold n*C*h*w floats.  Workspace as wn_forward.
 */
int wn_debug_forward_layer(wn_handle* h, const float* x, const float* wb, const float* he,
                           const float* gc, const int64_t in_strides[4][4], int n, int height,
                           int width, int mode, int layer, float* dst, void* workspace,
                           size_t workspace_bytes, void* stream);

/*
 * Select the unfused / plain forms of the tensor-core forward, which compute the same network and serve as
 * references: 256 = cmg.conv3 and conv4 as two launches (instead of conv4 as conv3's fused tail layer),
 * 512 = cmg.conv7 and conv8 as two launches (instead of conv8 tap-stacked behind conv7 + gather), 1024 = the
 * refiners' conv2 and conv3 + gate as two launches (instead of conv3 tap-stacked behind conv2 + gather/gate),
 * 2048 = the plain 49-tap first layer (instead of the K-packed one).  0 restores the default forms.  Any other
 * bit: WN_E_INVALID, flags unchanged.
 */
int wn_debug_set_flags(wn_handle* h, int flags);

/* Number of kernels the library has launched on this handle since creation. */
uint64_t wn_launch_count(const wn_handle* h);

/*
 * The tensor-core forward processes a batch in passes of at most 8 Mi pixels (workspace ~1.9 KB per pixel);
 * wn_forward_chunk_images returns the number of images per pass for a batch of n (callers that pipeline
 * host<->device copies or a collective against the passes split their batch at this granularity).
 * wn_set_chunk_pixels lowers the cap (0 restores the default); it never raises the workspace need.
 */
int wn_forward_chunk_images(const wn_handle* h, int n, int height, int width);
int wn_set_chunk_pixels(wn_handle* h, long long max_pixels);

/*
 * WN_MODE_BF16_FP8 keeps the correction terms of an activation in e4m3 (|v| <= 448).  A forward pass that
 * produces a larger activation -- far outside what the reference's [0,1] images and trained weights give --
 * raises a sticky device flag, and the batch that raised it is recomputed by the WN_MODE_BF16X3 kernels
 * WITHIN THE SAME CALL (the re-run is enqueued behind every pass, its launches return at once while the flag
 * is down).  The flag reaches the host with the completion of that call; from then on the handle goes
 * straight to the WN_MODE_BF16X3 kernels until wn_pack_weights is called again.  Returns the host-side value
 * of the flag (0/1).
 */
int wn_f8_overflowed(const wn_handle* h);

/*
 * Multi-GPU exchange without a kernel and without touching the peer device's contexts (SURVEY 8e; the all-gather
 * of the output batch, waternet_b200/dist.py PeerGather).  Two things a collective library does cost this path
 * time, measured at N=2 (tools/probe_gather.py): (1) the convolution kernels are persistent and own every SM's shared
 * memory, so a collective's kernel beside them takes an SM at a kernel boundary and stalls that SM's CTA pair while
 * it waits for the peer; (2) work submitted to a context this process holds ON THE PEER GPU -- which is what a
 * framework-level cross-device copy does to order itself against the destination's streams -- makes the peer GPU
 * time-slice away from its owner process, ~0.4 ms per switch with these kernels resident.  Hence this plumbing;
 * every call acts on the calling thread's current device, none launches a kernel:
 *
 *   wn_peer_alloc   cudaMalloc + zero fill + cudaIpcGetMemHandle: a buffer other ranks may map; handle_out
 *                   receives WN_PEER_HANDLE_BYTES bytes to send to them (any transport).
 *   wn_peer_open    cudaIpcOpenMemHandle in the CURRENT device's context (peer access enabled lazily): the
 *                   returned pointer is valid for copies issued on this device's streams.  wn_peer_close unmaps.
 *   wn_memcpy_async cudaMemcpyAsync(cudaMemcpyDefault): with a wn_peer_open'ed destination it is a copy-engine
 *                   push over NVLink, ordered on `stream`, issued entirely from this device.
 *   wn_stream_write_value32 / wn_stream_wait_value32
 *                   the driver's stream memory operations (cuStreamWriteValue32 / cuStreamWaitValue32, executed by
 *                   the stream's front end): store `value` to the 4-byte aligned device address when the stream
 *                   reaches it / hold the stream until (int32)(*addr - value) >= 0.  A peer's copy engine may be
 *                   the writer of a waited-on address.
 */
#define WN_PEER_HANDLE_BYTES 64
int wn_peer_alloc(size_t bytes, void** ptr, unsigned char* handle_out);
int wn_peer_open(const unsigned char* handle, void** ptr);
int wn_peer_close(void* ptr);
int wn_peer_free(void* ptr);
int wn_memcpy_async(void* dst, const void* src, size_t bytes, void* stream);
int wn_stream_write_value32(void* stream, void* addr, uint32_t value);
int wn_stream_wait_value32(void* stream, void* addr, uint32_t value);

#ifdef __cplusplus
}
#endif
#endif /* WATERNET_B200_H_ */
