"""Per-device engine: owns the C-ABI handle, packed weights and workspaces.

torch is plumbing here (device memory, streams); all arithmetic happens in
libwaternet_b200.so.
"""
from __future__ import annotations

import ctypes
import os
import threading
from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib

_engines: Dict[int, "Engine"] = {}
_engines_lock = threading.Lock()
# scratch buffers are shared by every engine of a device (all work is stream-ordered on the caller's stream)
_ws_pool: Dict[int, Dict[str, torch.Tensor]] = {}


def _require_cuda(device=None) -> torch.device:
    if not torch.cuda.is_available():
        raise _lib.WaterNetLibraryError(
            "waternet_b200 needs a CUDA device (B200, sm_100a); none is visible and there is no CPU fallback")
    dev = torch.device("cuda" if device is None else device)
    if dev.type != "cuda":
        raise _lib.WaterNetLibraryError(f"waternet_b200 runs on CUDA devices only, got {dev}")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev


def get_engine(device=None) -> "Engine":
    """The device's shared engine: preprocess / postprocess and callers that pack weights themselves."""
    dev = _require_cuda(device)
    with _engines_lock:
        eng = _engines.get(dev.index)
        if eng is None:
            eng = Engine(dev)
            _engines[dev.index] = eng
        return eng


def new_engine(device=None) -> "Engine":
    """A private engine (its own C-ABI handle, i.e. its own packed-weight slot) for one model on one device.

    Every ``WaterNet`` / ``ConfidenceMapGenerator`` / ``Refiner`` instance owns one per device, so two models on
    a device never evict -- or silently run with -- each other's packed weights.
    """
    return Engine(_require_cuda(device))


def _stream_ptr(device: torch.device) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class Engine:
    def __init__(self, device: torch.device):
        self.lib = _lib.load()
        self.device = device
        handle = ctypes.c_void_p()
        _lib.check(self.lib.wn_create(device.index, ctypes.byref(handle)), "wn_create")
        self.handle = handle
        # unfused / plain forms of the tensor-core forward (wn_debug_set_flags), for same-box A/B runs
        flags = int(os.environ.get("WATERNET_B200_DEBUG_FLAGS", "0"), 0)
        if flags:
            _lib.check(self.lib.wn_debug_set_flags(handle, flags), "wn_debug_set_flags")
        self._ws = _ws_pool.setdefault(device.index, {})
        self._weights_key = None
        self._weights_keepalive = None

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.wn_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    # ---- plumbing ----------------------------------------------------------
    def _workspace(self, tag: str, nbytes: int) -> torch.Tensor:
        buf = self._ws.get(tag)
        if buf is None or buf.numel() < nbytes:
            self._ws[tag] = None
            buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=self.device)
            self._ws[tag] = buf
        return buf

    def release_workspaces(self) -> None:
        self._ws.clear()

    def chunk_images(self, n: int, h: int, w: int) -> int:
        """Images per pass of the tensor-core forward for a batch of ``n`` (wn_forward_chunk_images)."""
        return max(1, int(self.lib.wn_forward_chunk_images(self.handle, n, h, w)))

    def set_chunk_pixels(self, max_pixels: int) -> None:
        """Lower the per-pass pixel cap (0 = default 8 Mi); tests force the multi-pass path with it."""
        _lib.check(self.lib.wn_set_chunk_pixels(self.handle, int(max_pixels)), "wn_set_chunk_pixels")

    def set_debug_flags(self, flags: int) -> None:
        """wn_debug_set_flags: 256 / 512 / 1024 run conv3+conv4 / conv7+conv8 / the refiners' conv2+conv3 unfused,
        2048 the plain first layer: the same network, used as references; any other bit raises."""
        _lib.check(self.lib.wn_debug_set_flags(self.handle, int(flags)), "wn_debug_set_flags")

    def f8_overflowed(self) -> bool:
        """True once the fp8-correction mode saw an activation beyond the e4m3 range.  The batch that did was
        recomputed by the bf16x3 kernels within the same call; from then on the handle uses those kernels
        directly until new weights are packed (wn_f8_overflowed).  Valid after the stream has been synchronised."""
        return bool(self.lib.wn_f8_overflowed(self.handle))

    @property
    def launch_count(self) -> int:
        return int(self.lib.wn_launch_count(self.handle))

    def enable_timing(self, on: bool = True) -> None:
        _lib.check(self.lib.wn_enable_timing(self.handle, 1 if on else 0), "wn_enable_timing")

    def read_timings(self):
        """(ms[slot], count[slot]) accumulated since the last read; synchronises the device first."""
        torch.cuda.synchronize(self.device)
        ms = (ctypes.c_float * _lib.NUM_TIMING_SLOTS)()
        cnt = (ctypes.c_int * _lib.NUM_TIMING_SLOTS)()
        _lib.check(self.lib.wn_read_timings(self.handle, ms, cnt), "wn_read_timings")
        return list(ms), list(cnt)

    # ---- weights -------------------------------------------------------------
    def pack_weights(self, params: Sequence[torch.Tensor], key=None) -> None:
        """params: the 34 tensors in state-dict order (net.py:12-42,62-70,94-97)."""
        if len(params) != _lib.NUM_PARAMS:
            raise ValueError(f"expected {_lib.NUM_PARAMS} parameter tensors, got {len(params)}")
        if key is not None and key == self._weights_key:
            return
        staged = [p.detach().to(device=self.device, dtype=torch.float32).contiguous() for p in params]
        arr = (ctypes.c_void_p * _lib.NUM_PARAMS)(*[t.data_ptr() for t in staged])
        with torch.cuda.device(self.device):
            _lib.check(self.lib.wn_pack_weights(self.handle, arr, _stream_ptr(self.device)), "wn_pack_weights")
        self._weights_keepalive = staged  # until the async pack kernels have consumed them
        self._weights_key = key

    # ---- forward -------------------------------------------------------------
    def forward(self, x, wb, he, gc, mode: int = _lib.MODE_DEFAULT, out: Optional[torch.Tensor] = None):
        """WaterNet.forward (net.py:99-108) on (N,3,H,W) fp32 CUDA tensors of any strides."""
        ins = self._check_inputs((x, wb, he, gc))
        n, _, h, w = ins[0].shape
        if out is None:
            out = torch.empty((n, 3, h, w), dtype=torch.float32, device=self.device)
        if n == 0 or h == 0 or w == 0:  # empty batch: nothing to launch (torch's convs return empty too)
            return out
        strides = (ctypes.c_int64 * 16)(*[s for t in ins for s in t.stride()])
        nbytes = self.lib.wn_forward_workspace_bytes(n, h, w, mode)
        ws = self._workspace("forward", nbytes)
        with torch.cuda.device(self.device):
            rc = self.lib.wn_forward(self.handle, ins[0].data_ptr(), ins[1].data_ptr(), ins[2].data_ptr(),
                                     ins[3].data_ptr(), strides, out.data_ptr(), n, h, w, mode,
                                     ws.data_ptr(), ws.numel(), _stream_ptr(self.device))
        _lib.check(rc, "wn_forward")
        return out

    def _check_inputs(self, tensors):
        ins = []
        for t in tensors:
            if t.device != self.device:
                raise ValueError(f"input on {t.device}, engine on {self.device}")
            if t.dim() != 4 or t.shape[1] != 3:
                raise ValueError(f"expected (N,3,H,W) inputs, got {tuple(t.shape)}")
            ins.append(t.detach() if t.dtype == torch.float32 else t.detach().float())
        for t in ins[1:]:
            if t.shape != ins[0].shape:
                raise ValueError("the inputs must have the same shape")
        return ins

    def confidence_maps(self, x, wb, he, gc, mode: int = _lib.MODE_DEFAULT) -> torch.Tensor:
        """ConfidenceMapGenerator.forward (net.py:45-56): the three sigmoid maps as one (N,3,H,W) tensor."""
        ins = self._check_inputs((x, wb, he, gc))
        n, _, h, w = ins[0].shape
        out = torch.empty((n, 3, h, w), dtype=torch.float32, device=self.device)
        if out.numel() == 0:
            return out
        strides = (ctypes.c_int64 * 16)(*[s for t in ins for s in t.stride()])
        ws = self._workspace("forward", self.lib.wn_submodule_workspace_bytes(n, h, w, mode))
        with torch.cuda.device(self.device):
            rc = self.lib.wn_confidence_maps(self.handle, ins[0].data_ptr(), ins[1].data_ptr(), ins[2].data_ptr(),
                                             ins[3].data_ptr(), strides, out.data_ptr(), n, h, w, mode,
                                             ws.data_ptr(), ws.numel(), _stream_ptr(self.device))
        _lib.check(rc, "wn_confidence_maps")
        return out

    def refine(self, which: int, x, xbar, mode: int = _lib.MODE_DEFAULT) -> torch.Tensor:
        """Refiner.forward (net.py:75-80) of refiner ``which`` (0 wb, 1 ce, 2 gc) of the packed state dict."""
        ins = self._check_inputs((x, xbar))
        n, _, h, w = ins[0].shape
        out = torch.empty((n, 3, h, w), dtype=torch.float32, device=self.device)
        if out.numel() == 0:
            return out
        strides = (ctypes.c_int64 * 8)(*[s for t in ins for s in t.stride()])
        ws = self._workspace("forward", self.lib.wn_submodule_workspace_bytes(n, h, w, mode))
        with torch.cuda.device(self.device):
            rc = self.lib.wn_refine(self.handle, int(which), ins[0].data_ptr(), ins[1].data_ptr(), strides,
                                    out.data_ptr(), n, h, w, mode, ws.data_ptr(), ws.numel(),
                                    _stream_ptr(self.device))
        _lib.check(rc, "wn_refine")
        return out

    LAYER_CHANNELS = (128, 128, 128, 64, 64, 64, 64, 3, 96, 96)

    def debug_layer(self, x, wb, he, gc, layer: int, mode: int) -> torch.Tensor:
        """Test aid (wn_debug_forward_layer): an intermediate activation as fp32 (N,C,H,W)."""
        ins = [t.detach().float() for t in (x, wb, he, gc)]
        n, _, h, w = ins[0].shape
        dst = torch.empty((n, self.LAYER_CHANNELS[layer], h, w), dtype=torch.float32, device=self.device)
        strides = (ctypes.c_int64 * 16)(*[s for t in ins for s in t.stride()])
        ws = self._workspace("forward", self.lib.wn_forward_workspace_bytes(n, h, w, mode))
        with torch.cuda.device(self.device):
            rc = self.lib.wn_debug_forward_layer(self.handle, ins[0].data_ptr(), ins[1].data_ptr(), ins[2].data_ptr(),
                                                 ins[3].data_ptr(), strides, n, h, w, mode, layer, dst.data_ptr(),
                                                 ws.data_ptr(), ws.numel(), _stream_ptr(self.device))
        _lib.check(rc, "wn_debug_forward_layer")
        return dst

    # ---- training step (wn_forward_train / wn_backward) ---------------------------------------
    TRAIN_MAX_PIXELS = 8 << 20

    def forward_train(self, x, wb, he, gc):
        """Tensor-core forward that keeps every activation.  Returns (out, saved workspaces).

        wn_forward_train takes at most TRAIN_MAX_PIXELS per call; a larger batch runs as several calls over slices
        of the batch, each with its own workspace (~5.6 KB per pixel in total, like the reference's autograd graph)."""
        ins = self._check_inputs((x, wb, he, gc))
        n, _, h, w = ins[0].shape
        out = torch.empty((n, 3, h, w), dtype=torch.float32, device=self.device)
        if out.numel() == 0:
            return out, None
        if h * w > self.TRAIN_MAX_PIXELS:
            raise _lib.WaterNetLibraryError(
                f"a forward pass that keeps its activations for autograd holds ~5.6 KB per pixel: one {h}x{w} image "
                f"exceeds the {self.TRAIN_MAX_PIXELS >> 20} Mi-pixel limit of wn_forward_train.  For inference wrap the "
                "call in torch.no_grad()")
        per = max(1, self.TRAIN_MAX_PIXELS // (h * w))
        saved = []
        for a in range(0, n, per):
            b = min(n, a + per)
            part = [t[a:b] for t in ins]
            strides = (ctypes.c_int64 * 16)(*[s for t in part for s in t.stride()])
            ws = torch.empty(self.lib.wn_train_workspace_bytes(b - a, h, w), dtype=torch.uint8, device=self.device)
            with torch.cuda.device(self.device):
                rc = self.lib.wn_forward_train(self.handle, part[0].data_ptr(), part[1].data_ptr(), part[2].data_ptr(),
                                               part[3].data_ptr(), strides, out[a:b].data_ptr(), b - a, h, w,
                                               ws.data_ptr(), ws.numel(), _stream_ptr(self.device))
            _lib.check(rc, "wn_forward_train")
            saved.append((a, b, ws))
        return out, saved

    def backward(self, grad_out: torch.Tensor, saved, shapes, want_input_grads: bool = False):
        """d(loss)/d(out) + the workspaces of forward_train -> the 34 parameter gradients (state-dict order)
        and, on request, the gradients of the four input images.  Batch slices are processed in order and their
        parameter gradients added in that order (deterministic)."""
        g = grad_out.detach().to(self.device, torch.float32).contiguous()
        n, _, h, w = g.shape
        saved = saved or []
        make = torch.empty if saved else torch.zeros  # an empty batch has zero gradients
        grads = [make(tuple(s), dtype=torch.float32, device=self.device) for s in shapes]
        part = grads if len(saved) <= 1 else [torch.empty_like(t) for t in grads]
        gin = None
        if want_input_grads:
            gin = [torch.empty((n, 3, h, w), dtype=torch.float32, device=self.device) for _ in range(4)]
        for i, (a, b, ws) in enumerate(saved):
            dst = grads if i == 0 else part
            arr = (ctypes.c_void_p * _lib.NUM_PARAMS)(*[t.data_ptr() for t in dst])
            gin_arr = (ctypes.c_void_p * 4)(*[t[a:b].data_ptr() for t in gin]) if want_input_grads else None
            with torch.cuda.device(self.device):
                rc = self.lib.wn_backward(self.handle, g[a:b].data_ptr(), arr, gin_arr, b - a, h, w, ws.data_ptr(),
                                          ws.numel(), _stream_ptr(self.device))
            _lib.check(rc, "wn_backward")
            if i > 0:
                torch._foreach_add_(grads, part)
        return (grads, gin) if want_input_grads else grads

    # ---- preprocess / postprocess ----------------------------------------------
    def preprocess(self, rgb_u8: torch.Tensor, tensors: bool = True, images: bool = False):
        """rgb_u8: uint8 (N,H,W,3) CUDA tensor.  Returns dict with the requested outputs.

        tensors -> 'x','wb','he','gc' fp32 (N,3,H,W); images -> 'wb_u8','he_u8','gc_u8' uint8 NHWC.
        """
        if rgb_u8.dtype != torch.uint8 or rgb_u8.dim() != 4 or rgb_u8.shape[3] != 3:
            raise ValueError(f"expected uint8 (N,H,W,3), got {rgb_u8.dtype} {tuple(rgb_u8.shape)}")
        rgb_u8 = rgb_u8.to(self.device).contiguous()
        n, h, w, _ = rgb_u8.shape
        if n == 0 or h == 0 or w == 0:
            res = {}
            if tensors:
                res.update({k: torch.empty((n, 3, h, w), dtype=torch.float32, device=self.device) for k in ("x", "wb", "he", "gc")})
            if images:
                res.update({k: torch.empty((n, h, w, 3), dtype=torch.uint8, device=self.device) for k in ("wb_u8", "he_u8", "gc_u8")})
            return res
        res = {}
        ptr = {k: None for k in ("x", "wb", "he", "gc", "wb_u8", "he_u8", "gc_u8")}
        if tensors:
            for k in ("x", "wb", "he", "gc"):
                res[k] = torch.empty((n, 3, h, w), dtype=torch.float32, device=self.device)
                ptr[k] = res[k].data_ptr()
        if images:
            for k in ("wb_u8", "he_u8", "gc_u8"):
                res[k] = torch.empty((n, h, w, 3), dtype=torch.uint8, device=self.device)
                ptr[k] = res[k].data_ptr()
        ws = self._workspace("preprocess", self.lib.wn_preprocess_workspace_bytes(n, h, w))
        with torch.cuda.device(self.device):
            rc = self.lib.wn_preprocess_u8(self.handle, rgb_u8.data_ptr(), n, h, w, ptr["x"], ptr["wb"], ptr["he"],
                                           ptr["gc"], ptr["wb_u8"], ptr["he_u8"], ptr["gc_u8"],
                                           ws.data_ptr(), ws.numel(), _stream_ptr(self.device))
        _lib.check(rc, "wn_preprocess_u8")
        return res

    def white_balance_gray(self, gray_u8: torch.Tensor) -> torch.Tensor:
        """Grayscale branch of ``white_balance_transform`` (data.py:30-36) on uint8 (N,H,W) CUDA tensors."""
        if gray_u8.dtype != torch.uint8 or gray_u8.dim() != 3:
            raise ValueError(f"expected uint8 (N,H,W), got {gray_u8.dtype} {tuple(gray_u8.shape)}")
        g = gray_u8.to(self.device).contiguous()
        out = torch.empty_like(g)
        if g.numel() == 0:
            return out
        n, h, w = g.shape
        ws = self._workspace("preprocess", self.lib.wn_white_balance_gray_workspace_bytes(n, h, w))
        with torch.cuda.device(self.device):
            rc = self.lib.wn_white_balance_gray_u8(self.handle, g.data_ptr(), out.data_ptr(), n, h, w, ws.data_ptr(),
                                                   ws.numel(), _stream_ptr(self.device))
        _lib.check(rc, "wn_white_balance_gray_u8")
        return out

    def resize_batch(self, images, dst_h: int, dst_w: int, swap_rb: bool = False) -> torch.Tensor:
        """Batched ``cv2.resize(img, (dst_w, dst_h))`` (+ optional BGR<->RGB swap) of differently sized uint8 HWC
        images (numpy arrays or CUDA tensors) into one uint8 (N, dst_h, dst_w, 3) CUDA tensor -- bit-exact
        OpenCV INTER_LINEAR arithmetic on the device (wn_resize_u8; training_utils.py:94-107)."""
        devs = []
        for im in images:
            t = torch.from_numpy(np.ascontiguousarray(im)) if isinstance(im, np.ndarray) else im
            if t.dtype != torch.uint8 or t.dim() != 3 or t.shape[2] != 3:
                raise ValueError(f"expected uint8 HWC images, got {t.dtype} {tuple(t.shape)}")
            devs.append(t.to(self.device, non_blocking=True).contiguous())
        n = len(devs)
        out = torch.empty((n, dst_h, dst_w, 3), dtype=torch.uint8, device=self.device)
        if n == 0 or out.numel() == 0:
            return out
        ptrs = (ctypes.c_void_p * n)(*[t.data_ptr() for t in devs])
        hs = (ctypes.c_int * n)(*[t.shape[0] for t in devs])
        ws = (ctypes.c_int * n)(*[t.shape[1] for t in devs])
        with torch.cuda.device(self.device):
            rc = self.lib.wn_resize_u8(self.handle, ptrs, hs, ws, n, out.data_ptr(), dst_h, dst_w, 1 if swap_rb else 0,
                                       _stream_ptr(self.device))
        _lib.check(rc, "wn_resize_u8")
        for t in devs:  # the kernel reads them on the current stream after this call returns
            t.record_stream(torch.cuda.current_stream(self.device))
        return out

    def postprocess(self, out: torch.Tensor) -> torch.Tensor:
        """ten2arr on the device: fp32 (N,3,H,W) -> uint8 (N,H,W,3) CUDA tensor."""
        out = out.detach().to(self.device, torch.float32).contiguous()
        n, c, h, w = out.shape
        if c != 3:
            raise ValueError("expected (N,3,H,W)")
        res = torch.empty((n, h, w, 3), dtype=torch.uint8, device=self.device)
        if res.numel() == 0:
            return res
        with torch.cuda.device(self.device):
            rc = self.lib.wn_postprocess_u8(self.handle, out.data_ptr(), res.data_ptr(), n, h, w,
                                            _stream_ptr(self.device))
        _lib.check(rc, "wn_postprocess_u8")
        return res

    def enhance(self, rgb_u8: torch.Tensor, mode: int = _lib.MODE_DEFAULT, out_u8: Optional[torch.Tensor] = None,
                out_f32: Optional[torch.Tensor] = None, peer_out=()) -> torch.Tensor:
        """preprocess -> forward -> postprocess on uint8 (N,H,W,3) CUDA input; returns uint8 NHWC.

        ``peer_out``: device addresses (ints) inside other ranks' buffers (``dist.PeerGather.peer_addresses``) that
        receive the same bytes as ``out_u8`` from the kernel that writes it (wn_enhance_u8_peers)."""
        if rgb_u8.dtype != torch.uint8 or rgb_u8.dim() != 4 or rgb_u8.shape[3] != 3:
            raise ValueError(f"expected uint8 (N,H,W,3), got {rgb_u8.dtype} {tuple(rgb_u8.shape)}")
        rgb_u8 = rgb_u8.to(self.device).contiguous()
        n, h, w, _ = rgb_u8.shape
        if out_u8 is None:
            out_u8 = torch.empty((n, h, w, 3), dtype=torch.uint8, device=self.device)
        elif (out_u8.dtype != torch.uint8 or tuple(out_u8.shape) != (n, h, w, 3) or not out_u8.is_contiguous()
              or out_u8.device != rgb_u8.device):
            raise ValueError(f"out_u8 must be a contiguous uint8 {(n, h, w, 3)} tensor on {rgb_u8.device}, got "
                             f"{out_u8.dtype} {tuple(out_u8.shape)} strides {out_u8.stride()} on {out_u8.device}")
        if out_f32 is not None and (out_f32.dtype != torch.float32 or tuple(out_f32.shape) != (n, 3, h, w)
                                    or not out_f32.is_contiguous() or out_f32.device != rgb_u8.device):
            raise ValueError(f"out_f32 must be a contiguous float32 {(n, 3, h, w)} tensor on {rgb_u8.device}")
        if out_u8.numel() == 0:
            return out_u8
        ws = self._workspace("enhance", self.lib.wn_enhance_workspace_bytes(n, h, w, mode))
        peers = (ctypes.c_void_p * max(1, len(peer_out)))(*peer_out)
        with torch.cuda.device(self.device):
            rc = self.lib.wn_enhance_u8_peers(self.handle, rgb_u8.data_ptr(), out_u8.data_ptr(),
                                              None if out_f32 is None else out_f32.data_ptr(), peers, len(peer_out),
                                              n, h, w, mode, ws.data_ptr(), ws.numel(), _stream_ptr(self.device))
        _lib.check(rc, "wn_enhance_u8_peers")
        return out_u8
