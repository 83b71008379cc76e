"""Pin the CPU oracle: outputs of the unmodified reference stored under tests/golden, and cv2 where importable."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, golden_files, load_golden
from oracle import forward as ofw
from oracle import preprocess as opre

with open(os.path.join(GOLDEN, "reference_digests.json")) as _f:
    REFERENCE_DIGESTS = json.load(_f)


def _sha256(arr):
    return hashlib.sha256(np.ascontiguousarray(arr).tobytes()).hexdigest()


@pytest.mark.parametrize("path", golden_files("preprocess"), ids=os.path.basename)
def test_preprocess_matches_golden(path):
    g = load_golden(path)
    wb, gc, he = opre.transform(g["rgb"])
    assert np.array_equal(wb, g["wb"])
    assert np.array_equal(gc, g["gc"])
    assert np.array_equal(he, g["he"])


@pytest.mark.parametrize("path", golden_files("forward"), ids=os.path.basename)
def test_forward_matches_golden(path):
    g = load_golden(path)
    sd = ofw.synthetic_state_dict(int(g["weight_seed"]), float(g["gain"]))
    ins = [[], [], [], []]
    for rgb in g["rgb"]:
        wb, gc, he = opre.transform(rgb)
        for slot, arr in zip(ins, (rgb, wb, he, gc)):
            slot.append(torch.from_numpy(opre.arr2ten(arr).copy()))
    x, wb, he, gc = (torch.cat(s) for s in ins)
    out = ofw.waternet_forward(sd, x, wb, he, gc).numpy()
    ref = g["out"]
    # same arithmetic (oneDNN fp32 conv) => agreement far inside the 1e-3 bar
    assert np.max(np.abs(out - ref)) <= 1e-5 * np.max(np.abs(ref))
    assert np.array_equal(opre.ten2arr(ref), g["post"])
    # fp64 ground truth agrees with the fp32 reference output
    out64 = ofw.waternet_forward(sd, x, wb, he, gc, dtype=torch.float64).numpy()
    assert np.max(np.abs(out64 - ref)) <= 1e-5 * np.max(np.abs(ref))


def test_state_dict_spec_matches_reference_keys():
    spec = ofw.state_dict_spec()
    assert len(spec) == 34
    assert sum(int(np.prod(s)) for _, s in spec) == 1_090_668
    assert spec[0] == ("cmg.conv1.weight", (128, 12, 7, 7))
    assert spec[-1] == ("gc_refiner.conv3.bias", (3,))


def test_arr2ten_ten2arr_contract():
    rgb = ofw.synthetic_image(3, 9, 7, "noise")
    ten = opre.arr2ten(rgb)
    assert ten.shape == (1, 3, 9, 7) and ten.dtype == np.float32
    assert np.array_equal(ten[0, 1], rgb[..., 1].astype(np.float32) / np.float32(255))
    assert np.array_equal(opre.ten2arr(ten), rgb[None])  # u/255*255 truncates back to u
    weird = np.array([[[[-0.5, 0.9999, 1.7, 0.5]]]], dtype=np.float32)
    assert opre.ten2arr(weird).reshape(-1).tolist() == [0, 254, 255, 127]


# ---- the reference's outputs on more shapes: SHA-256 digests written by tests/golden/make_golden.py ----


@pytest.mark.parametrize("shape", [(112, 112), (113, 117), (112, 117), (115, 112), (48, 200), (270, 480)])
@pytest.mark.parametrize("kind", ["noise", "smooth"])
def test_preprocess_matches_live_reference(shape, kind):
    """transform() bit for bit against the reference's wb / gc / he of the same seeded frame."""
    want = REFERENCE_DIGESTS["preprocess"][f"{shape[0]}x{shape[1]}_{kind}"]
    rgb = ofw.synthetic_image(want["seed"], shape[0], shape[1], kind)
    for name, got in zip(("wb", "gc", "he"), opre.transform(rgb)):
        assert got.dtype == np.uint8 and got.shape == rgb.shape, name
        assert _sha256(got) == want[name], f"{name} differs from the reference's"


def test_lab_conversions_match_cv2_on_a_colour_lattice():
    cv2 = pytest.importorskip("cv2")
    # every 3rd level of each channel plus the extremes: 86^3 colours (exhaustive 2^24 verified offline)
    lv = np.unique(np.concatenate([np.arange(0, 256, 3), [254, 255]])).astype(np.uint8)
    cols = np.stack(np.meshgrid(lv, lv, lv, indexing="ij"), -1).reshape(1, -1, 3)
    assert np.array_equal(opre.rgb2lab_u8(cols), cv2.cvtColor(cols, cv2.COLOR_RGB2LAB))
    assert np.array_equal(opre.lab2rgb_u8(cols), cv2.cvtColor(cols, cv2.COLOR_LAB2RGB))


@pytest.mark.parametrize("shape", [(8, 8), (16, 9), (7, 5), (64, 64), (65, 64), (100, 37)])
def test_clahe_matches_cv2(shape):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    for clip in (0.1, 2.0, 40.0):
        plane = rng.integers(0, 256, shape, dtype=np.uint8)
        want = cv2.createCLAHE(clipLimit=clip, tileGridSize=(8, 8)).apply(plane)
        assert np.array_equal(opre.clahe_apply(plane, clip, 8), want)


def test_resize_restatement_matches_cv2():
    """oracle.preprocess.resize_linear_u8 == cv2.resize(img, (w, h)) (default INTER_LINEAR) bit for bit: the
    training dataset's resize (training_utils.py:94-103) is third-party arithmetic like CLAHE."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(3)
    cases = [(300, 400, 112, 112), (224, 224, 112, 112), (112, 112, 112, 112), (57, 91, 112, 112), (113, 225, 112, 112),
             (641, 480, 320, 240), (1, 1, 8, 8), (2, 3, 112, 112), (700, 900, 256, 256), (225, 224, 112, 112)]
    for sh, sw, dh, dw in cases:
        src = rng.integers(0, 256, (sh, sw, 3), dtype=np.uint8)
        assert np.array_equal(opre.resize_linear_u8(src, (dw, dh)), cv2.resize(src, (dw, dh))), (sh, sw, dh, dw)


def test_grayscale_white_balance_matches_live_reference():
    """The 2-D branch of white_balance_transform (data.py:30-36), including its uint8 truncation of the quantiles,
    bit for bit against the reference's output on the same inputs."""
    want = iter(REFERENCE_DIGESTS["white_balance_gray"])
    rng = np.random.default_rng(0)
    for shape in [(40, 56), (7, 9), (33, 17), (112, 112)]:
        for k in range(2):
            g = rng.integers(0, 256, shape, dtype=np.uint8) if k == 0 else (rng.random(shape) * 90 + 40).astype(np.uint8)
            ref = next(want)
            assert (tuple(ref["shape"]), ref["kind"]) == (shape, k)
            got = opre.white_balance_transform(g)
            assert got.dtype == np.uint8 and got.shape == shape
            assert _sha256(got) == ref["sha256"], (shape, k)
    assert next(want, None) is None


# ---- the float64 gradient oracle (waternet_grads): the ground truth of the native backward tests ----


def test_fp64_gradients_match_autograd_through_the_module_graph():
    """waternet_grads (the functional graph of oracle.forward) against torch.autograd through WaterNet._graph (the
    nn.Conv2d modules of waternet_b200.net) in float64: two formulations of the same network, stress weights, a
    ragged shape, float inputs, an arbitrary d(loss)/d(out)."""
    from waternet_b200.net import WaterNet
    sd = ofw.synthetic_state_dict(5, 3.0)
    gen = torch.Generator().manual_seed(11)
    ins = [torch.rand(2, 3, 13, 19, generator=gen) for _ in range(4)]
    g_out = torch.randn(2, 3, 13, 19, generator=gen, dtype=torch.float64)
    out, grads, in_grads = ofw.waternet_grads(sd, ins, g_out)
    m = WaterNet()
    m.load_state_dict(sd, strict=True)
    m = m.double()
    leaves = [t.double().requires_grad_(True) for t in ins]
    want_out = m._graph(*leaves)
    want_out.backward(g_out)

    def rel(a, b):
        return ((a - b).norm() / b.norm()).item()

    assert rel(out, want_out.detach()) < 1e-12
    named = dict(m.named_parameters())
    assert sorted(grads) == sorted(named) and len(grads) == 34
    for key, g in grads.items():
        assert g.dtype == torch.float64 and g.shape == named[key].shape
        assert rel(g, named[key].grad) < 1e-12, key
    for g, t in zip(in_grads, leaves):
        assert rel(g, t.grad) < 1e-12


def test_fp64_input_gradient_support_is_the_receptive_field():
    """d(loss)/d(out) nonzero at one pixel: the input gradients are exactly zero beyond Chebyshev distance 13 of it
    (the confidence-map stack's radius, 3+2+1+0+3+2+1+1; the refiners' is 6) and nonzero at distance 13.  The GPU
    tile-probe test relies on both."""
    sd = ofw.margin_state_dict()      # every ReLU active: the support is not cut short by a dead unit
    h, w, py, px = 48, 64, 20, 30
    ins = [torch.rand(1, 3, h, w, generator=torch.Generator().manual_seed(i)) for i in range(4)]
    g_out = torch.zeros(1, 3, h, w, dtype=torch.float64)
    g_out[0, :, py, px] = torch.tensor([0.7, -1.3, 0.4], dtype=torch.float64)
    _, _, in_grads = ofw.waternet_grads(sd, ins, g_out)
    for g in in_grads:
        rows, cols = torch.nonzero(g[0].abs().amax(0), as_tuple=True)
        assert (int(rows.min()), int(rows.max())) == (py - 13, py + 13)
        assert (int(cols.min()), int(cols.max())) == (px - 13, px + 13)


@pytest.mark.parametrize("half_dead", [False, True], ids=["all_active", "half_dead"])
def test_margin_weight_sets_keep_every_relu_away_from_zero(half_dead):
    """The weight sets of the strict native-backward tests: every ReLU pre-activation at least 1 away from zero
    (measured: 1.26 all active, 1.50 half dead), every channel of one sign over the whole input, and 25-75 % dead
    channels per ReLU layer in the half-dead set (none in the other)."""
    sd = ofw.margin_state_dict(half_dead)
    rgbs = [ofw.synthetic_image(90 + i, 48, 64, "smooth") for i in range(4)]
    ins = [torch.from_numpy(opre.arr2ten(a).copy()) for a in rgbs]
    g_out = torch.randn(1, 3, 48, 64, generator=torch.Generator().manual_seed(0), dtype=torch.float64)
    *_, pre = ofw.waternet_grads(sd, ins, g_out, return_preacts=True)
    assert sorted(pre) == sorted(ofw.RELU_LAYERS + ["cmg.conv8"]) and len(ofw.RELU_LAYERS) == 16
    smallest, dead, mixed = ofw.relu_margins(pre)
    assert smallest >= 1.0
    for layer in ofw.RELU_LAYERS:
        assert not mixed[layer].any(), layer
        frac = dead[layer].float().mean().item()
        if half_dead:
            assert 0.25 <= frac <= 0.75, (layer, frac)
            assert torch.equal(dead[layer], torch.arange(len(dead[layer])) % 2 == 1), layer
        else:
            assert frac == 0.0, layer
