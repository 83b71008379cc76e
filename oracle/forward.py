"""torch restatement of the reference network forward and its gradients (TEST INFRASTRUCTURE ONLY).

Follows ``/root/reference/waternet/net.py``: ``ConfidenceMapGenerator.forward``
(``net.py:45-56``), ``Refiner.forward`` (``net.py:75-80``) and
``WaterNet.forward`` (``net.py:99-108``) as one functional evaluation over a
plain ``{key: tensor}`` state dict with the reference's 34 keys.  Floating-point
kernel => a torch reference is kept (fp32 = what the reference computes on CPU;
fp64 = ground truth used to judge both implementations).
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

# (name, in_channels, out_channels, kernel) -- net.py:12-42
CMG_LAYERS = [
    ("conv1", 12, 128, 7),
    ("conv2", 128, 128, 5),
    ("conv3", 128, 128, 3),
    ("conv4", 128, 64, 1),
    ("conv5", 64, 64, 7),
    ("conv6", 64, 64, 5),
    ("conv7", 64, 64, 3),
    ("conv8", 64, 3, 3),
]
# net.py:62-70
REFINER_LAYERS = [("conv1", 6, 32, 7), ("conv2", 32, 32, 5), ("conv3", 32, 3, 3)]
REFINERS = ["wb_refiner", "ce_refiner", "gc_refiner"]  # net.py:95-97


def state_dict_spec():
    """[(key, shape)] in the order ``WaterNet().state_dict()`` lists them."""
    spec = []
    for name, cin, cout, k in CMG_LAYERS:
        spec.append((f"cmg.{name}.weight", (cout, cin, k, k)))
        spec.append((f"cmg.{name}.bias", (cout,)))
    for ref in REFINERS:
        for name, cin, cout, k in REFINER_LAYERS:
            spec.append((f"{ref}.{name}.weight", (cout, cin, k, k)))
            spec.append((f"{ref}.{name}.bias", (cout,)))
    return spec


def synthetic_state_dict(seed: int = 0, gain: float = 1.0):
    """Deterministic stand-in weights (no pretrained checkpoint offline).

    U(-b, b) with b = gain / sqrt(fan_in) for weights and biases -- the bound
    torch's default Conv2d init uses -- drawn from numpy's PCG64 so the values do
    not depend on the torch version.  ``gain=3`` gives O(1) outputs that stress
    precision (SURVEY.md section 8d).
    """
    rng = np.random.default_rng(seed)
    sd = {}
    for key, shape in state_dict_spec():
        if key.endswith("weight"):
            fan_in = shape[1] * shape[2] * shape[3]
            bound = gain / np.sqrt(fan_in)
            last_bound = 1.0 / np.sqrt(fan_in)
        else:
            bound = last_bound
        sd[key] = torch.from_numpy(rng.uniform(-bound, bound, size=shape).astype(np.float32))
    return sd


def _conv(sd, prefix, x, k, preacts=None):
    w = sd[prefix + ".weight"].to(x.dtype)
    b = sd[prefix + ".bias"].to(x.dtype)
    z = F.conv2d(x, w, b, stride=1, padding=k // 2)  # padding="same", odd kernels
    if preacts is not None:
        preacts[prefix] = z.detach()
    return z


def confidence_maps(sd, x, wb, ce, gc, preacts=None):
    """net.py:45-56 -- returns the (N,3,H,W) sigmoid maps (wb, ce, gc order)."""
    out = torch.cat([x, wb, ce, gc], dim=1)
    for name, _, _, k in CMG_LAYERS[:-1]:
        out = F.relu(_conv(sd, f"cmg.{name}", out, k, preacts))
    return torch.sigmoid(_conv(sd, "cmg.conv8", out, 3, preacts))


def refine(sd, which, x, xbar, preacts=None):
    """net.py:75-80 -- three conv+ReLU (the last conv is followed by ReLU too)."""
    out = torch.cat([x, xbar], dim=1)
    for name, _, _, k in REFINER_LAYERS:
        out = F.relu(_conv(sd, f"{which}.{name}", out, k, preacts))
    return out


def _waternet(sd, x, wb, ce, gc, preacts=None):
    cm = confidence_maps(sd, x, wb, ce, gc, preacts)
    r_wb = refine(sd, "wb_refiner", x, wb, preacts)
    r_ce = refine(sd, "ce_refiner", x, ce, preacts)
    r_gc = refine(sd, "gc_refiner", x, gc, preacts)
    return r_wb * cm[:, 0:1] + r_ce * cm[:, 1:2] + r_gc * cm[:, 2:3], cm, (r_wb, r_ce, r_gc)


def waternet_forward(sd, x, wb, ce, gc, dtype=torch.float32, return_parts=False):
    """net.py:99-108.  Inputs (N,3,H,W) in the order (raw, wb, he, gc)."""
    with torch.no_grad():
        x, wb, ce, gc = (t.detach().to("cpu", dtype).contiguous() for t in (x, wb, ce, gc))
        out, cm, parts = _waternet(sd, x, wb, ce, gc)
    if return_parts:
        return out, cm, parts
    return out


def waternet_grads(sd, ins, grad_out, dtype=torch.float64, device=None, return_preacts=False):
    """Ground truth for the backward pass: ``out.backward(grad_out)`` through the functional graph above.

    ``ins`` = (x, wb, he, gc), (N,3,H,W) each; ``grad_out`` = d(loss)/d(out), (N,3,H,W).  Runs on ``device``
    (default: the device of ``grad_out``) in ``dtype``.  Returns ``(out, grads, input_grads)``: the output, a
    ``{key: gradient}`` dict of the 34 state-dict tensors and the four input-image gradients; with
    ``return_preacts`` also ``{layer: pre-activation}`` of the 16 ReLU layers and of ``cmg.conv8`` (the
    sigmoid's input).

    On CUDA the convolutions are torch's own im2col + GEMM ones, not cuDNN: every value is then a plain sum of
    products, so a gradient that is zero by structure (a dead channel, a pixel outside the receptive field of
    the loss) is exactly zero, as on the CPU.  An FFT or Winograd algorithm would leave rounding noise there.
    Float64 on CUDA involves no TF32.
    """
    dev = torch.device(device) if device is not None else grad_out.device
    params = {k: v.detach().to(dev, dtype).clone().requires_grad_(True) for k, v in sd.items()}
    leaves = [t.detach().to(dev, dtype).contiguous().requires_grad_(True) for t in ins]
    preacts = {} if return_preacts else None
    with torch.backends.cudnn.flags(enabled=False):
        with torch.enable_grad():
            out = _waternet(params, *leaves, preacts)[0]
            out.backward(grad_out.detach().to(dev, dtype))
    grads = {k: v.grad for k, v in params.items()}
    res = (out.detach(), grads, [t.grad for t in leaves])
    return res + (preacts,) if return_preacts else res


# the layers followed by a ReLU (all but cmg.conv8, which feeds the sigmoid)
RELU_LAYERS = [f"cmg.{name}" for name, *_ in CMG_LAYERS[:-1]] + [f"{r}.{name}" for r in REFINERS for name, *_ in REFINER_LAYERS]


def margin_state_dict(half_dead: bool = False, seed: int = 7, gain: float = 0.2):
    """Weights whose ReLUs all sit far from their kink, so that a gradient has no ReLU-flip excuse for an error.

    Small weights (``synthetic_state_dict(seed, gain)``) and every ReLU layer's bias at +2: all channels active.
    With ``half_dead`` the odd output channels get -2 instead: those channels are zero everywhere, and so is every
    gradient entry of their rows (the layer's own weights and bias) and columns (the next layer's weights).
    ``cmg.conv8.bias`` (the sigmoid's) keeps its value.  :func:`relu_margins` measures what a given input gets.
    """
    sd = synthetic_state_dict(seed, gain)
    for layer in RELU_LAYERS:
        b = torch.full_like(sd[layer + ".bias"], 2.0)
        if half_dead:
            b[1::2] = -2.0
        sd[layer + ".bias"] = b
    return sd


def relu_margins(preacts):
    """(min |z| over every ReLU pre-activation, {layer: bool mask of dead channels}, {layer: bool mask of
    channels whose sign changes somewhere}) from ``waternet_grads(..., return_preacts=True)``."""
    smallest = min(float(preacts[layer].abs().min()) for layer in RELU_LAYERS)
    dead, mixed = {}, {}
    for layer in RELU_LAYERS:
        z = preacts[layer]
        dead[layer] = (z.amax(dim=(0, 2, 3)) < 0).cpu()
        mixed[layer] = ~(dead[layer] | (z.amin(dim=(0, 2, 3)) > 0).cpu())
    return smallest, dead, mixed


def synthetic_image(seed: int, h: int, w: int, kind: str = "noise") -> np.ndarray:
    """SURVEY.md section 8d inputs: uniform noise, or a smooth blue-green cast."""
    rng = np.random.default_rng(seed)
    if kind == "noise":
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    base = rng.random((h // 8 + 3, w // 8 + 3, 3))
    ys = np.linspace(0, base.shape[0] - 1.001, h)
    xs = np.linspace(0, base.shape[1] - 1.001, w)
    y0 = ys.astype(int)
    x0 = xs.astype(int)
    fy = (ys - y0)[:, None, None]
    fx = (xs - x0)[None, :, None]
    img = (
        base[y0][:, x0] * (1 - fy) * (1 - fx)
        + base[y0][:, x0 + 1] * (1 - fy) * fx
        + base[y0 + 1][:, x0] * fy * (1 - fx)
        + base[y0 + 1][:, x0 + 1] * fy * fx
    )
    img = (img - img.min()) / (img.max() - img.min())
    return (img * np.array([90.0, 200.0, 230.0])).astype(np.uint8)
