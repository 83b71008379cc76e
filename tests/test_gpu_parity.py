"""Parity of the CUDA path (through the C ABI) against the CPU oracle and the golden fixtures."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, golden_files, load_golden
from oracle import forward as ofw
from oracle import preprocess as opre

pytestmark = pytest.mark.gpu

REL_TOL = 1e-3  # north_star: "within 1e-3 relative fp32"; metric of SURVEY.md section 8d


@pytest.fixture(scope="module")
def eng():
    from waternet_b200.engine import get_engine
    return get_engine("cuda:0")


def _assert_close(out, ref, tol=REL_TOL):
    out = np.asarray(out, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    scale = np.max(np.abs(ref))
    err = np.max(np.abs(out - ref))
    assert err <= tol * scale, f"max|d|={err:.3e} > {tol}*max|ref|={tol * scale:.3e}"
    assert np.allclose(out, ref, rtol=tol, atol=tol * scale)
    return err / scale


def _inputs_from_rgb(rgbs):
    ins = [[], [], [], []]
    for rgb in rgbs:
        wb, gc, he = opre.transform(rgb)
        for slot, arr in zip(ins, (rgb, wb, he, gc)):
            slot.append(torch.from_numpy(opre.arr2ten(arr).copy()))
    return [torch.cat(s) for s in ins]


# ------------------------------------------------------------------ preprocess (bit exact)
@pytest.mark.parametrize("path", golden_files("preprocess"), ids=os.path.basename)
def test_preprocess_bit_exact_vs_golden(eng, path):
    g = load_golden(path)
    res = eng.preprocess(torch.from_numpy(g["rgb"][None]).cuda(), tensors=True, images=True)
    for key, name in (("wb", "wb_u8"), ("he", "he_u8"), ("gc", "gc_u8")):
        got = res[name][0].cpu().numpy()
        assert np.array_equal(got, g[key]), f"{name}: {(got != g[key]).sum()} bytes differ"
    for key, arr in (("x", g["rgb"]), ("wb", g["wb"]), ("he", g["he"]), ("gc", g["gc"])):
        assert np.array_equal(res[key].cpu().numpy(), opre.arr2ten(arr)), key


@pytest.mark.parametrize("shape", [(112, 112), (113, 117), (112, 117), (115, 112), (9, 11), (16, 9), (8, 8), (7, 5),
                                   (3, 4), (64, 512), (270, 480), (1080, 1920)])
@pytest.mark.parametrize("kind", ["noise", "smooth"])
def test_preprocess_bit_exact_vs_oracle(eng, shape, kind):
    rgb = ofw.synthetic_image(7 + shape[0], shape[0], shape[1], kind)
    wb, gc, he = opre.transform(rgb)
    res = eng.preprocess(torch.from_numpy(rgb[None]).cuda(), tensors=False, images=True)
    assert np.array_equal(res["wb_u8"][0].cpu().numpy(), wb)
    assert np.array_equal(res["gc_u8"][0].cpu().numpy(), gc)
    assert np.array_equal(res["he_u8"][0].cpu().numpy(), he)


def test_preprocess_batch_is_per_image(eng):
    imgs = np.stack([ofw.synthetic_image(s, 96, 160, k) for s, k in [(1, "noise"), (2, "smooth"), (3, "smooth")]])
    res = eng.preprocess(torch.from_numpy(imgs).cuda(), tensors=False, images=True)
    for i, rgb in enumerate(imgs):
        wb, gc, he = opre.transform(rgb)
        assert np.array_equal(res["wb_u8"][i].cpu().numpy(), wb)
        assert np.array_equal(res["he_u8"][i].cpu().numpy(), he)
        assert np.array_equal(res["gc_u8"][i].cpu().numpy(), gc)


def test_preprocess_degenerate_channel_does_not_crash(eng):
    # reference behaviour is undefined here (SURVEY appendix B.7); only require that nothing faults
    rgb = ofw.synthetic_image(0, 32, 32, "noise")
    rgb[..., 0] = 0
    rgb[..., 1] = 77
    res = eng.preprocess(torch.from_numpy(rgb[None]).cuda(), tensors=False, images=True)
    torch.cuda.synchronize()
    assert np.array_equal(res["gc_u8"][0].cpu().numpy(), opre.gamma_correction(rgb))


def test_postprocess_matches_ten2arr(eng):
    rng = np.random.default_rng(0)
    t = rng.uniform(-0.2, 1.3, (2, 3, 37, 53)).astype(np.float32)
    t[0, 0, 0, :4] = [0.0, 1.0, 0.99999994, 254.5 / 255]
    got = eng.postprocess(torch.from_numpy(t).cuda()).cpu().numpy()
    assert np.array_equal(got, opre.ten2arr(t))


# ------------------------------------------------------------------ forward
# "default" = the library's fastest mode inside the 1e-3 bar: bf16 tensor-core products with the two
# correction terms of the heavy layers as one fp8 MMA ("bf16_fp8"); "bf16x3" = all three terms in bf16
MODES = ["fp32", "bf16x3", "bf16_fp8"]


def _assert_u8_close(got, want, share=0.01):
    """uint8 images of two evaluations that differ by rounding: a truncating cast flips a level where the value sits
    on a boundary -- one level at most, on a small share of the bytes."""
    diff = np.abs(np.asarray(got).astype(int) - np.asarray(want).astype(int))
    assert diff.max() <= 1 and (diff != 0).mean() < share, (diff.max(), (diff != 0).mean())


def _model(seed, gain, precision):
    from waternet_b200.net import WaterNet
    m = WaterNet(precision=precision)
    m.load_state_dict(ofw.synthetic_state_dict(seed, gain), strict=True)
    return m.cuda().eval()


@pytest.mark.parametrize("precision", MODES)
@pytest.mark.parametrize("path", golden_files("forward"), ids=os.path.basename)
def test_forward_vs_golden(path, precision):
    g = load_golden(path)
    m = _model(int(g["weight_seed"]), float(g["gain"]), precision)
    x, wb, he, gc = [t.cuda() for t in _inputs_from_rgb(g["rgb"])]
    with torch.no_grad():
        out = m(x, wb, he, gc)
    assert out.shape == g["out"].shape and out.dtype == torch.float32 and out.is_contiguous()
    rel = _assert_close(out.cpu().numpy(), g["out"])
    print(f"{os.path.basename(path)} {precision}: max rel err {rel:.2e}")


@pytest.mark.parametrize("precision", MODES)
@pytest.mark.parametrize("shape", [(1, 16, 16), (2, 33, 47), (1, 8, 200), (3, 64, 40), (1, 130, 70), (1, 1, 1), (2, 3, 5),
                                   (1, 1, 40), (1, 17, 2)])
def test_forward_vs_oracle_ragged_shapes(precision, shape):
    n, h, w = shape
    torch.manual_seed(h * w)
    ins = [torch.rand(n, 3, h, w) for _ in range(4)]
    sd = ofw.synthetic_state_dict(3, 3.0)
    m = _model(3, 3.0, precision)
    with torch.no_grad():
        out = m(*[t.cuda() for t in ins]).cpu().numpy()
    ref64 = ofw.waternet_forward(sd, *ins, dtype=torch.float64).numpy()
    _assert_close(out, ref64)


@pytest.mark.parametrize("precision", MODES)
def test_forward_accepts_channels_last_strides(precision):
    # what arr2ten produces: shape (1,3,H,W), strides (3HW, 1, 3W, 3) (hubconf.py:18-20)
    rgb = ofw.synthetic_image(5, 40, 56, "smooth")
    wb, gc, he = opre.transform(rgb)
    strided = [(torch.from_numpy(a.copy()).cuda().float() / 255).permute(2, 0, 1).unsqueeze(0) for a in (rgb, wb, he, gc)]
    assert strided[0].stride()[1:] == (1, 56 * 3, 3)  # channels_last view, as hubconf.py:18-20 produces
    m = _model(0, 1.0, precision)
    with torch.no_grad():
        a = m(*strided)
        b = m(*[t.contiguous() for t in strided])
    assert torch.equal(a, b)


@pytest.mark.parametrize("precision", MODES)
def test_first_layer_fast_path_equals_general_path(precision):
    """8-bit image levels take the 2-pass first layer; a perturbed copy takes the general 3-pass one."""
    rgb = ofw.synthetic_image(8, 48, 64, "smooth")
    sd = ofw.synthetic_state_dict(4, 3.0)
    ins = _inputs_from_rgb([rgb])
    m = _model(4, 3.0, precision)
    with torch.no_grad():
        exact = m(*[t.cuda() for t in ins]).cpu().numpy()
        bumped = [t.clone() for t in ins]
        bumped[0][0, 0, 0, 0] += 1e-3  # one non-level value disables the fast path for the whole batch
        general = m(*[t.cuda() for t in bumped]).cpu().numpy()
    _assert_close(exact, ofw.waternet_forward(sd, *ins, dtype=torch.float64).numpy())
    _assert_close(general, ofw.waternet_forward(sd, *bumped, dtype=torch.float64).numpy())


@pytest.mark.parametrize("precision", MODES)
def test_forward_batch_independent(precision):
    torch.manual_seed(0)
    ins = [torch.rand(3, 3, 48, 80).cuda() for _ in range(4)]
    m = _model(2, 1.0, precision)
    with torch.no_grad():
        full = m(*ins)
        one = m(*[t[1:2] for t in ins])
    assert torch.equal(full[1:2], one)


def test_tensor_core_path_matches_fp32_path_at_1080p():
    """Full-size check the CPU oracle is too slow for: the two independent CUDA paths agree."""
    rgb = ofw.synthetic_image(42, 1080, 1920, "smooth")
    from waternet_b200.engine import get_engine
    eng = get_engine("cuda:0")
    r = eng.preprocess(torch.from_numpy(rgb[None]).cuda())
    ins = [r[k] for k in ("x", "wb", "he", "gc")]
    with torch.no_grad():
        a = _model(0, 3.0, "fp32")(*ins).cpu().numpy()
        b = _model(0, 3.0, "bf16x3")(*ins).cpu().numpy()
        c = _model(0, 3.0, "default")(*ins).cpu().numpy()
    assert _assert_close(b, a) < 1e-4          # three bf16 terms: ~3e-5
    err = _assert_close(c, a)                  # fp8 corrections: inside the 1e-3 bar with margin
    print(f"1080p, stress weights: bf16x3 vs fp32 {np.max(np.abs(b - a)) / np.max(np.abs(a)):.2e}, default {err:.2e}")
    assert err < 8e-4


@pytest.mark.parametrize("precision", MODES)
def test_translation_equivariance_at_full_width(precision):
    """Size-independent property: away from the borders a shifted input gives the shifted output."""
    torch.manual_seed(1)
    h, w, dy, dx = 200, 1920, 5, 16
    base = [torch.rand(1, 3, h + dy, w + dx).cuda() for _ in range(4)]
    m = _model(1, 1.0, precision)
    with torch.no_grad():
        a = m(*[t[:, :, :h, :w].contiguous() for t in base])
        b = m(*[t[:, :, dy:, dx:].contiguous() for t in base])
    halo = 14  # receptive field 27x27
    ia = a[:, :, halo + dy:h - halo, halo + dx:w - halo]
    ib = b[:, :, halo:h - halo - dy, halo:w - halo - dx]
    _assert_close(ib.cpu().numpy(), ia.cpu().numpy(), tol=1e-4)


# ------------------------------------------------------------------ end to end + API
@pytest.mark.parametrize("precision", MODES)
def test_enhance_u8_end_to_end(eng, precision):
    from waternet_b200 import _lib
    rgbs = np.stack([ofw.synthetic_image(20 + i, 72, 104, k) for i, k in enumerate(["noise", "smooth"])])
    sd = ofw.synthetic_state_dict(0, 3.0)
    m = _model(0, 3.0, precision)
    eng.pack_weights(m._ordered_params())
    mode = {"fp32": _lib.MODE_FP32_SIMT, "bf16x3": _lib.MODE_BF16X3, "bf16_fp8": _lib.MODE_BF16_FP8}[precision]
    got = eng.enhance(torch.from_numpy(rgbs).cuda(), mode=mode).cpu().numpy()
    ref = opre.ten2arr(ofw.waternet_forward(sd, *_inputs_from_rgb(rgbs)).numpy())
    diff = np.abs(got.astype(int) - ref.astype(int))
    assert diff.max() <= 1, "truncating cast may flip one level at most"
    # a value within the forward error of a level boundary truncates to the neighbouring level: the share of
    # such pixels is ~255 x the mean error (3e-5-class modes: < 1 %; fp8 corrections, ~10x the error: < 10 %)
    assert (diff != 0).mean() < (0.10 if precision == "bf16_fp8" else 0.01)


def test_hub_api_roundtrip():
    from waternet_b200.hub import waternet
    preprocess, postprocess, model = waternet(pretrained=False, device="cuda:0")
    model.load_state_dict(ofw.synthetic_state_dict(0, 3.0))
    model.eval()
    rgb = ofw.synthetic_image(9, 48, 64, "smooth")
    rgb_t, wb_t, he_t, gc_t = preprocess(rgb)
    assert rgb_t.shape == (1, 3, 48, 64) and rgb_t.dtype == torch.float32 and rgb_t.is_cuda
    wb, gc, he = opre.transform(rgb)
    assert np.array_equal(he_t.cpu().numpy(), opre.arr2ten(he))
    assert np.array_equal(gc_t.cpu().numpy(), opre.arr2ten(gc))
    with torch.no_grad():
        out = model(rgb_t, wb_t, he_t, gc_t)
    arr = postprocess(out)
    assert arr.shape == (1, 48, 64, 3) and arr.dtype == np.uint8
    ref = opre.ten2arr(ofw.waternet_forward(ofw.synthetic_state_dict(0, 3.0), rgb_t, wb_t, he_t, gc_t).numpy())
    assert np.abs(arr.astype(int) - ref.astype(int)).max() <= 1


def test_data_module_numpy_api():
    from waternet_b200 import data
    rgb = ofw.synthetic_image(11, 50, 70, "noise")
    wb, gc, he = data.transform(rgb)
    rwb, rgc, rhe = opre.transform(rgb)
    assert np.array_equal(wb, rwb) and np.array_equal(gc, rgc) and np.array_equal(he, rhe)
    assert np.array_equal(data.histeq(rgb), rhe)
    assert np.array_equal(data.white_balance_transform(rgb), rwb)
    assert np.array_equal(data.gamma_correction(rgb), rgc)


def test_cpu_tensors_fail_loudly():
    from waternet_b200 import WaterNetLibraryError
    from waternet_b200.net import WaterNet
    m = WaterNet()
    t = torch.rand(1, 3, 16, 16)
    with pytest.raises(WaterNetLibraryError):
        with torch.no_grad():
            m(t, t, t, t)


def test_training_step_gradients_match_torch_graph():
    """fp32 CUDA-core mode only: forward values from the SIMT kernels, gradients by re-evaluating the torch graph
    (the tensor-core modes use the native wn_forward_train / wn_backward pair, tested below)."""
    import copy
    torch.manual_seed(0)
    m = _model(0, 1.0, "fp32").train()
    ins = [torch.rand(2, 3, 24, 24).cuda() for _ in range(4)]
    target = torch.rand(2, 3, 24, 24).cuda()
    out = m(*ins)
    assert out.requires_grad
    torch.nn.functional.mse_loss(out, target).backward()
    g1 = m.cmg.conv1.weight.grad.clone()
    g1r = m.gc_refiner.conv3.bias.grad.clone()
    # ground truth: the same network evaluated in float64 by autograd (no TF32, no cuDNN heuristics)
    m64 = copy.deepcopy(m).double()
    m64.zero_grad()
    out64 = m64._graph(*[t.double() for t in ins])
    torch.nn.functional.mse_loss(out64, target.double()).backward()
    assert torch.allclose(out.double(), out64, rtol=1e-4, atol=1e-6)
    # the backward pass re-evaluates the graph with torch's fp32 convolutions (TF32 on by default,
    # like the reference on a GPU: SURVEY appendix B.8), hence the looser gradient tolerance
    def rel(a, b):
        return ((a.double() - b).norm() / b.norm()).item()
    assert rel(g1, m64.cmg.conv1.weight.grad) < 2e-2
    assert rel(g1r, m64.gc_refiner.conv3.bias.grad) < 2e-2


def _mse_grad(out, target):
    """d mse_loss(out, target) / d out: what loss.backward() hands the model, given to the float64 oracle too."""
    return 2.0 * (out.detach() - target) / out.numel()


# the 16 x 112^2 training batch (BASELINE configs[4]) and a ragged shape run the float64 oracle on the GPU
@pytest.mark.parametrize("shape", [(2, 24, 24), (1, 37, 53), (3, 16, 40), (16, 112, 112), (3, 203, 157)])
def test_native_backward_matches_fp64_autograd(shape):
    """wn_forward_train + wn_backward: all 34 parameter gradients against float64 autograd."""
    n, h, w = shape
    torch.manual_seed(h)
    sd = ofw.synthetic_state_dict(5, 3.0)
    m = _model(5, 3.0, "default").train()
    rgbs = [ofw.synthetic_image(30 + i, h, w, "smooth") for i in range(n)]
    ins = _inputs_from_rgb(rgbs)
    target = torch.rand(n, 3, h, w)
    out = m(*[t.cuda() for t in ins])
    assert out.grad_fn is not None
    g_out = _mse_grad(out, target.cuda())
    out.backward(g_out)
    dev = "cuda" if n * h * w > 10_000 else "cpu"
    ref_out, ref, _ = ofw.waternet_grads(sd, ins, g_out, device=dev)
    _assert_close(out.detach().cpu().numpy(), ref_out.cpu().numpy())
    worst = 0.0
    for (name, p) in m.named_parameters():
        g, r = p.grad.double().to(dev), ref[name]
        rel = ((g - r).norm() / r.norm().clamp_min(1e-30)).item()
        worst = max(worst, rel)
        assert rel < 2e-3, f"{name}: relative gradient error {rel:.2e}"
    print(f"{n}x{h}x{w}: worst relative gradient error {worst:.2e}")


def test_training_forward_runs_a_large_batch_as_slices(monkeypatch):
    """A grad-enabled call beyond wn_forward_train's pixel limit (the reference's hub example calls the model
    without no_grad) runs as several calls over slices of the batch: same output, same gradients (parameter
    gradients added slice by slice), for parameters and input images."""
    from waternet_b200.engine import Engine
    n, h, w = 5, 24, 40
    ins = [t.cuda() for t in _inputs_from_rgb([ofw.synthetic_image(70 + i, h, w, "smooth") for i in range(n)])]
    target = torch.rand(n, 3, h, w, generator=torch.Generator().manual_seed(4)).cuda()

    def run():
        m = _model(5, 3.0, "default").train()
        cu = [t.clone().requires_grad_(i == 1) for i, t in enumerate(ins)]
        out = m(*cu)
        torch.nn.functional.mse_loss(out, target).backward()
        return out.detach(), [p.grad.clone() for p in m.parameters()], cu[1].grad.clone()

    out1, g1, gi1 = run()
    monkeypatch.setattr(Engine, "TRAIN_MAX_PIXELS", 2 * h * w)   # 5 images -> slices of 2, 2, 1
    out2, g2, gi2 = run()
    assert torch.equal(out1, out2) and torch.equal(gi1, gi2)     # per-image quantities: bitwise
    for a, b in zip(g1, g2):                                      # sums over the batch: another order of additions
        assert ((a - b).norm() / a.norm().clamp_min(1e-30)).item() < 1e-5
    monkeypatch.setattr(Engine, "TRAIN_MAX_PIXELS", h * w - 1)
    with pytest.raises(Exception):
        run()


def _input_grad_case(sd, needs, n=2, h=29, w=43):
    from waternet_b200.net import WaterNet
    m = WaterNet(precision="default")
    m.load_state_dict(sd, strict=True)
    m = m.cuda().train()
    ins = _inputs_from_rgb([ofw.synthetic_image(60 + i, h, w, "smooth") for i in range(n)])
    target = torch.rand(n, 3, h, w, generator=torch.Generator().manual_seed(3))
    cu = [t.cuda().requires_grad_(need) for t, need in zip(ins, needs)]
    out = m(*cu)
    g_out = _mse_grad(out, target.cuda())
    out.backward(g_out)
    ref_out, ref, ref_in = ofw.waternet_grads(sd, ins, g_out.cpu())
    _assert_close(out.detach().cpu().numpy(), ref_out.numpy())
    rels = []
    for t, need, r in zip(cu, needs, ref_in):
        if not need:
            assert t.grad is None
            continue
        assert t.grad.shape == r.shape
        rels.append(((t.grad.double().cpu() - r).norm() / r.norm()).item())
    prels = {name: ((p.grad.double().cpu() - ref[name]).norm() / ref[name].norm().clamp_min(1e-30)).item()
             for name, p in m.named_parameters()}
    return rels, prels


@pytest.mark.parametrize("needs", [(True, True, True, True), (False, True, False, False)])
def test_native_input_image_gradients_smooth_network(needs):
    """wn_backward's optional input_grads against float64 autograd on a network whose ReLUs are all
    active (small weights, bias 2): the gradient is a smooth function of the activations there, so
    the kernels must agree to bf16x3 accuracy."""
    rels, prels = _input_grad_case(ofw.margin_state_dict(), needs)
    assert max(rels) < 2e-4, rels
    assert max(prels.values()) < 2e-4, max(prels.items(), key=lambda kv: kv[1])


def test_native_input_image_gradients_general_network():
    """Same with the usual stress weights.  A ReLU whose pre-activation is within the forward error of
    zero passes the gradient in one arithmetic and blocks it in the other -- a full-size difference in
    a ~1e-5 fraction of the elements, i.e. ~sqrt(1e-5) in the L2 norm -- so the bar against float64 is
    looser here (fp32 cuDNN autograd shows the same effect at its own, smaller forward error)."""
    rels, prels = _input_grad_case(ofw.synthetic_state_dict(7, 3.0), (True, True, True, True))
    assert max(rels) < 2e-2, rels
    assert max(prels.values()) < 2e-2, max(prels.items(), key=lambda kv: kv[1])


# ------------------------------------------------------------------ backward at the training shapes
# BASELINE configs[4] (16 x 112^2), the larger batch of tools/bench_train.py (4 x 512^2) and a ragged shape whose
# every kernel ends on partial tiles (203 is no multiple of 4 or 8, 157 none of 16), against float64 on the GPU.
# The networks' ReLUs all sit at least 1 away from their kink (oracle.forward.margin_state_dict, re-measured on each
# case's own inputs), so no pre-activation can flip between the two arithmetics: the bars are those of the smooth
# small-shape test (except the weight gradients at 4 x 512^2, see _weight_grad_rel_l2_bar).
BWD_SHAPES = [(16, 112, 112), (4, 512, 512), (3, 203, 157)]
BWD_REL_L2 = 2e-4    # relative L2 error of a gradient tensor (test_native_input_image_gradients_smooth_network)
BWD_MAX_ABS = 1e-3   # max |g - r| over max |r|, per tensor


def _weight_grad_rel_l2_bar(n, h, w):
    """The weight-gradient bar grows past 16 x 112^2.  Each CTA of a weight-gradient launch adds all its tiles into
    one fp32 tensor-memory accumulator, and the error of that sum grows with the number of tiles per CTA.  It is
    almost all a uniform scale error of the tensor (the sign varies with the data).  Worst tensor on one B200, at
    1000 W, cmg.conv2 / conv5 and the refiners' conv2: <= 4.3e-5 at 16 x 112^2, where the longest CTA adds ~150
    tiles.  At 1, 2 and 4 x 512^2 it is 5.7e-5, 1.9e-4 and 5.2e-4 over two seed sets; at 4 x 512^2 the longest
    CTA adds ~780 tiles.  Half the 2e-3 bar of test_native_backward_matches_fp64_autograd."""
    return BWD_REL_L2 if n * h * w <= 16 * 112 * 112 else 1e-3


def _shape_id(shape):
    return "x".join(map(str, shape))


def _level_images(seed, n, h, w):
    """Four (N,3,H,W) batches of 8-bit levels (u / 255, as arr2ten makes them) from independent smooth images: the
    training first layer's 2-pass form (hi planes only)."""
    return [torch.cat([torch.from_numpy(opre.arr2ten(ofw.synthetic_image(seed + 4 * i + j, h, w, "smooth")).copy())
                       for i in range(n)]) for j in range(4)]


def _float_images(seed, n, h, w):
    """Four (N,3,H,W) batches of arbitrary floats in [0, 1): the training first layer's 3-pass form (hi + lo
    planes), and the g_hi x a_lo term of the first layers' weight gradients."""
    gen = torch.Generator().manual_seed(seed)
    return [torch.rand(n, 3, h, w, generator=gen) for _ in range(4)]


def _probe_grad(n, h, w, seed, tiles=50):
    """d(loss)/d(out), seeded random values at ~100 pixels and zero elsewhere: the first and last pixel of the batch,
    the four corners of every image, one pixel inside the bottom-right 16 x 4 tile (partial on a ragged shape) and
    one pixel in each of ``tiles`` random 16 x 4 tiles.  Each probed tile then carries a ~1 % share of every weight
    gradient: a tile that a weight-gradient launch loses, counts twice or misplaces moves it by about that much."""
    rng = np.random.default_rng(seed)
    pts = {(0, 0, 0), (n - 1, h - 1, w - 1)}
    for i in range(n):
        pts |= {(i, 0, 0), (i, 0, w - 1), (i, h - 1, 0), (i, h - 1, w - 1)}
    y0, x0 = (h - 1) // 4 * 4, (w - 1) // 16 * 16
    pts.add((n - 1, (y0 + h - 1) // 2, (x0 + w - 1) // 2))
    ty, tx = -(-h // 4), -(-w // 16)
    for t in rng.choice(n * ty * tx, size=tiles, replace=False):
        i, rem = divmod(int(t), ty * tx)
        a, b = divmod(rem, tx)
        pts.add((i, min(h - 1, 4 * a + int(rng.integers(4))), min(w - 1, 16 * b + int(rng.integers(16)))))
    g = torch.zeros(n, 3, h, w)
    for i, y, x in sorted(pts):
        g[i, :, y, x] = torch.from_numpy(rng.standard_normal(3).astype(np.float32))
    return g


def _native_backward(sd, ins, g_out):
    """out.backward(g_out) through wn_forward_train / wn_backward, with every input image requiring grad."""
    from waternet_b200.net import WaterNet
    m = WaterNet(precision="default")
    m.load_state_dict(sd, strict=True)
    m = m.cuda().train()
    cu = [t.cuda().requires_grad_(True) for t in ins]
    out = m(*cu)
    assert out.grad_fn is not None
    out.backward(g_out)
    grads = {name: p.grad for name, p in m.named_parameters()}
    in_grads = [t.grad for t in cu]
    m.engine().release_workspaces()
    return out.detach(), grads, in_grads


def _grad_error(got, ref):
    """(relative L2, max |got - ref| / max |ref|) of one gradient tensor against its float64 value."""
    d = got.double() - ref
    scale = ref.abs().max().item()
    if scale == 0:
        return (0.0, 0.0) if not got.any() else (float("inf"), float("inf"))
    return (d.norm() / ref.norm()).item(), d.abs().max().item() / scale


def _layer_input(layer):
    """The ReLU layer whose output ``layer`` reads (None: it reads the input images)."""
    stack, conv = layer.rsplit(".", 1)
    k = int(conv[4:])
    return None if k == 1 else f"{stack}.conv{k - 1}"


def _check_backward(sd, ins, g_out, label, half_dead=False):
    """Native forward + backward against float64 (the oracle on the GPU): output, 34 parameter gradients and four
    input gradients within the strict bars; the networks' ReLU margins re-measured on these inputs.  With
    ``half_dead``: every gradient entry that is zero by structure (rows of dead output channels, columns of dead
    input channels) is exactly zero.  With a sparse ``g_out``: the input gradients are exactly zero beyond the
    receptive-field radius 13 of every nonzero pixel (test_oracle.py shows the float64 support is that box)."""
    import time
    n, _, h, w = g_out.shape
    g_out = g_out.cuda()
    out, grads, in_grads = _native_backward(sd, ins, g_out)
    t0 = time.perf_counter()
    ref_out, ref, ref_in, pre = ofw.waternet_grads(sd, ins, g_out, device="cuda", return_preacts=True)
    torch.cuda.synchronize()
    t_ref = time.perf_counter() - t0
    smallest, dead, mixed = ofw.relu_margins(pre)
    del pre
    assert smallest >= 1.0, f"a ReLU pre-activation {smallest:.3f} from zero: the strict bars do not apply"
    for layer in ofw.RELU_LAYERS:
        assert not mixed[layer].any(), layer
        frac = dead[layer].float().mean().item()
        assert (0.25 <= frac <= 0.75) if half_dead else frac == 0.0, (layer, frac)

    rel_out = _assert_close(out.cpu().numpy(), ref_out.cpu().numpy())
    assert rel_out < 1e-4, f"forward: max rel err {rel_out:.2e}"
    worst = {}
    for name, g in grads.items():
        worst[name] = _grad_error(g, ref[name])
    zeros = 0
    if half_dead:
        for layer in ofw.RELU_LAYERS + ["cmg.conv8"]:
            cout, cin = ref[layer + ".weight"].shape[:2]
            src = _layer_input(layer)
            rows = dead.get(layer, torch.zeros(cout, dtype=torch.bool)).to(g_out.device)
            cols = (dead[src] if src else torch.zeros(cin, dtype=torch.bool)).to(g_out.device)
            structural = {layer + ".weight": rows[:, None, None, None] | cols[None, :, None, None], layer + ".bias": rows}
            for name, mask in structural.items():
                r, g = ref[name], grads[name]
                assert not r[mask.expand_as(r)].any(), f"{name}: the float64 gradient is not zero by structure"
                exact = r == 0
                assert not g[exact].any(), f"{name}: {int((g[exact] != 0).sum())} entries nonzero where float64 is 0"
                zeros += int(exact.sum())
    in_worst = []
    outside = 0
    support = torch.nn.functional.max_pool2d((g_out != 0).any(1, keepdim=True).float(), 27, stride=1, padding=13) > 0
    sparse = not bool(support.all())
    for k, (g, r) in enumerate(zip(in_grads, ref_in)):
        assert g.shape == r.shape
        if sparse:
            off = ~support.expand_as(r)
            assert not r[off].any(), "float64 input gradient outside the receptive field of the probes"
            assert not g[off].any(), f"input {k}: {int((g[off] != 0).sum())} nonzero values outside the probes' support"
            outside += int(off.sum())
        in_worst.append(_grad_error(g, r))
    name_l2 = max(worst, key=lambda k: worst[k][0])
    name_mx = max(worst, key=lambda k: worst[k][1])
    print(f"{label}: forward {rel_out:.2e}; parameters rel-L2 {worst[name_l2][0]:.2e} ({name_l2}), max-abs "
          f"{worst[name_mx][1]:.2e} ({name_mx}); inputs rel-L2 {max(e[0] for e in in_worst):.2e}, max-abs "
          f"{max(e[1] for e in in_worst):.2e}; ReLU margin {smallest:.2f}; exact zeros {zeros} parameter entries, "
          f"{outside} input values; float64 reference {t_ref:.1f} s")
    bar = _weight_grad_rel_l2_bar(n, h, w)
    for name, (rel, mx) in worst.items():
        assert rel < bar and mx <= BWD_MAX_ABS, f"{name}: rel-L2 {rel:.2e}, max-abs {mx:.2e}"
    for k, (rel, mx) in enumerate(in_worst):
        assert rel < BWD_REL_L2 and mx <= BWD_MAX_ABS, f"input {k}: rel-L2 {rel:.2e}, max-abs {mx:.2e}"
    del ref, ref_in, ref_out, grads, in_grads
    torch.cuda.empty_cache()


@pytest.mark.parametrize("inputs", ["levels", "floats"])
@pytest.mark.parametrize("shape", BWD_SHAPES, ids=_shape_id)
def test_native_backward_at_training_shapes_smooth_network(shape, inputs):
    """Every ReLU active: the gradients are smooth functions of the activations, and the weight-gradient launches
    accumulate up to ~150 tiles per CTA (16 x 112^2) or more (4 x 512^2).  Float inputs take the 3-pass first layer."""
    n, h, w = shape
    ins = (_level_images if inputs == "levels" else _float_images)(1000 + h, n, h, w)
    g_out = torch.randn(n, 3, h, w, generator=torch.Generator().manual_seed(w))
    _check_backward(ofw.margin_state_dict(), ins, g_out, f"smooth {_shape_id(shape)} {inputs}")


@pytest.mark.parametrize("shape", BWD_SHAPES, ids=_shape_id)
def test_native_backward_at_training_shapes_half_dead_network(shape):
    """Half of every ReLU layer's channels dead, with margin: the ReLU' masks of the data-gradient epilogues and of
    gate_bwd_kernel, and the row / column mapping of the weight-gradient extraction, leave exact zeros exactly
    where float64 has them."""
    n, h, w = shape
    g_out = torch.randn(n, 3, h, w, generator=torch.Generator().manual_seed(h))
    _check_backward(ofw.margin_state_dict(half_dead=True), _level_images(2000 + h, n, h, w), g_out,
                    f"half-dead {_shape_id(shape)}", half_dead=True)


@pytest.mark.parametrize("network", ["smooth", "half_dead"])
@pytest.mark.parametrize("shape", [(16, 112, 112), (3, 203, 157)], ids=_shape_id)
def test_native_backward_tile_probe(shape, network):
    """A sparse d(loss)/d(out) (_probe_grad): per-tensor bars that a lost, doubled or misplaced tile of a
    weight-gradient launch fails, and input gradients exactly zero outside the probes' receptive fields (no stray
    writes, no reads of the uninitialised training workspace)."""
    n, h, w = shape
    half_dead = network == "half_dead"
    _check_backward(ofw.margin_state_dict(half_dead=half_dead), _level_images(3000 + h, n, h, w),
                    _probe_grad(n, h, w, seed=h), f"tile probe, {network} {_shape_id(shape)}", half_dead=half_dead)


def test_native_training_steps_track_the_torch_graph():
    """A few Adam steps with native gradients follow the same loss curve as pure torch autograd."""
    import copy
    torch.manual_seed(0)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    base = _model(6, 1.0, "default").train()
    twin = copy.deepcopy(base)
    ins = [t.cuda() for t in _inputs_from_rgb([ofw.synthetic_image(40 + i, 32, 32, "smooth") for i in range(4)])]
    target = torch.rand(4, 3, 32, 32).cuda()
    opt_a = torch.optim.Adam(base.parameters(), lr=1e-3)
    opt_b = torch.optim.Adam(twin.parameters(), lr=1e-3)
    la, lb = [], []
    for _ in range(5):
        opt_a.zero_grad()
        loss = torch.nn.functional.mse_loss(base(*ins), target)
        loss.backward()
        opt_a.step()
        la.append(loss.item())
        opt_b.zero_grad()
        loss = torch.nn.functional.mse_loss(twin._graph(*ins), target)
        loss.backward()
        opt_b.step()
        lb.append(loss.item())
    assert la[-1] < la[0]
    assert np.allclose(la, lb, rtol=2e-3), (la, lb)


def test_gpu_batch_loader_matches_per_item_path():
    """GpuBatchLoader (one batched preprocess on the device) == the reference-style per-item dictionary."""
    from waternet_b200.training_utils import GpuBatchLoader, SyntheticUIEB
    ds = SyntheticUIEB(length=10, im_height=48, im_width=64, seed=3)
    subset = torch.utils.data.Subset(ds, [7, 2, 5, 0, 9])
    loader = GpuBatchLoader(subset, batch_size=2, device="cuda:0", augment=False)
    assert len(loader) == 3
    seen = 0
    for b, batch in enumerate(loader):
        for j in range(batch["raw"].shape[0]):
            raw, ref = ds.pair(subset.indices[b * 2 + j])
            wb, gc, he = opre.transform(raw)
            for key, arr in (("raw", raw), ("wb", wb), ("gc", gc), ("he", he), ("ref", ref)):
                assert np.array_equal(batch[key][j].cpu().numpy(), opre.arr2ten(arr)[0]), key
            seen += 1
    assert seen == 5
    # augmentation: raw and ref receive the same flips / rotations, values only permuted
    aug = GpuBatchLoader(ds, batch_size=4, device="cuda:0", augment=True, seed=0)
    batch = next(iter(aug))
    assert batch["raw"].shape == (4, 3, 48, 64) and batch["ref"].shape == (4, 3, 48, 64)
    for j in range(4):
        raw, ref = ds.pair(j)
        assert np.array_equal(np.sort((batch["raw"][j].cpu().numpy() * 255).round().astype(np.uint8).ravel()), np.sort(raw.ravel()))
        assert np.array_equal(np.sort((batch["ref"][j].cpu().numpy() * 255).round().astype(np.uint8).ravel()), np.sort(ref.ravel()))


def test_enhancer_cuda_graph_replay_equals_direct_launches():
    """Small frames replay a captured CUDA graph; results must be identical to plain launches."""
    from waternet_b200.api import Enhancer
    m = _model(0, 3.0, "default")
    direct = Enhancer(m, cuda_graph=False)
    graphed = Enhancer(m, cuda_graph=True)
    frames = [ofw.synthetic_image(60 + i, 72, 96, "smooth") for i in range(4)]
    for f in frames:  # first call captures, later calls replay with new input contents
        assert np.array_equal(graphed(f), direct(f))
    assert any(slot.graph is not None for slot in graphed._slots)
    batch = np.stack(frames[:2])
    assert np.array_equal(graphed(batch), direct(batch))  # new shape -> new capture
    assert np.array_equal(graphed(batch[::-1].copy()), direct(batch[::-1].copy()))


def test_empty_batch_is_a_no_op(eng):
    m = _model(0, 1.0, "default")
    empty = [torch.empty(0, 3, 32, 48).cuda() for _ in range(4)]
    with torch.no_grad():
        assert m(*empty).shape == (0, 3, 32, 48)
    assert eng.enhance(torch.empty(0, 32, 48, 3, dtype=torch.uint8).cuda()).shape == (0, 32, 48, 3)
    res = eng.preprocess(torch.empty(0, 32, 48, 3, dtype=torch.uint8).cuda(), tensors=True, images=True)
    assert res["x"].shape == (0, 3, 32, 48) and res["he_u8"].shape == (0, 32, 48, 3)
    assert eng.postprocess(torch.empty(0, 3, 8, 8).cuda()).shape == (0, 8, 8, 3)


def test_single_4k_frame_tensor_cores_vs_fp32_path():
    """Largest single-image case exercised: 3840x2160 (one image per pass, ~16 GB of workspace)."""
    from waternet_b200.engine import get_engine
    eng = get_engine("cuda:0")
    rgb = ofw.synthetic_image(77, 2160, 3840, "smooth")
    r = eng.preprocess(torch.from_numpy(rgb[None]).cuda())
    ins = [r[k] for k in ("x", "wb", "he", "gc")]
    with torch.no_grad():
        a = _model(0, 3.0, "fp32")(*ins).cpu().numpy()
        b = _model(0, 3.0, "bf16x3")(*ins).cpu().numpy()
        c = _model(0, 3.0, "default")(*ins).cpu().numpy()
    _assert_close(b, a)
    _assert_close(c, a)
    eng.release_workspaces()


# ------------------------------------------------------------------ headline-configuration code paths
TC_MODES = ["bf16x3", "bf16_fp8"]


@pytest.mark.parametrize("precision", TC_MODES)
def test_multi_pass_batch_equals_per_image_and_oracle(precision):
    """The 16 x 1080p bench batch runs as 4 passes of 4 images (8 Mi-pixel cap) with per-pass pointer offsets.
    Force that path on a small batch (wn_set_chunk_pixels): 5 images, 2 per pass -> passes of 2, 2, 1."""
    n, h, w = 5, 64, 96
    rgbs = [ofw.synthetic_image(200 + i, h, w, "smooth" if i % 2 else "noise") for i in range(n)]
    ins = _inputs_from_rgb(rgbs)
    sd = ofw.synthetic_state_dict(2, 3.0)
    m = _model(2, 3.0, precision)
    cu = [t.cuda() for t in ins]
    eng = m.engine()
    with torch.no_grad():
        one_pass = m(*cu)
        eng.set_chunk_pixels(2 * h * w)
        try:
            assert eng.chunk_images(n, h, w) == 2
            chunked = m(*cu)
            singles = torch.cat([m(*[t[i:i + 1] for t in cu]) for i in range(n)])
            maps = torch.cat(m.cmg(*cu), 1)
            refined = m.gc_refiner(cu[0], cu[3])
            u8 = eng.enhance(torch.from_numpy(np.stack(rgbs)).cuda(), mode=m._mode())
            f32 = torch.empty(n, 3, h, w, device="cuda")
            eng.enhance(torch.from_numpy(np.stack(rgbs)).cuda(), mode=m._mode(), out_f32=f32)
        finally:
            eng.set_chunk_pixels(0)
        maps_one = torch.cat(m.cmg(*cu), 1)
    assert torch.equal(chunked, one_pass), "pass boundaries changed the result"
    assert torch.equal(chunked, singles), "image i of a batch differs from image i alone"
    assert torch.equal(maps, maps_one)
    assert torch.equal(f32, chunked), "the folded uint8 path computes a different forward"
    ref, cm_ref, parts = ofw.waternet_forward(sd, *ins, return_parts=True)
    _assert_close(chunked.cpu().numpy(), ref.numpy())
    _assert_close(maps.cpu().numpy(), cm_ref.numpy())
    _assert_close(refined.cpu().numpy(), parts[2].numpy())
    _assert_close(f32.cpu().numpy(), ref.numpy())
    assert np.array_equal(u8.cpu().numpy(), opre.ten2arr(f32.cpu().numpy())), "uint8 epilogue != ten2arr(fp32 output)"


@pytest.mark.parametrize("precision", TC_MODES)
def test_full_size_1080p_frame_vs_cpu_oracle(precision):
    """One 1920x1080 frame against the fp32 CPU oracle (what the reference computes on CPU; ~20 s of host time),
    stress weights.  Also the uint8 end-to-end result against ten2arr of the oracle output."""
    rgb = ofw.synthetic_image(42, 1080, 1920, "smooth")
    sd = ofw.synthetic_state_dict(0, 3.0)
    ins = _inputs_from_rgb([rgb])
    torch.set_num_threads(os.cpu_count() or 1)
    ref = ofw.waternet_forward(sd, *ins).numpy()
    m = _model(0, 3.0, precision)
    eng = m.engine()
    with torch.no_grad():
        out = m(*[t.cuda() for t in ins]).cpu().numpy()
    rel = _assert_close(out, ref)
    print(f"1080p vs CPU oracle, {precision}: max rel err {rel:.2e}")
    assert rel < (6e-4 if precision == "bf16_fp8" else 1e-4)
    got = eng.enhance(torch.from_numpy(rgb[None]).cuda(), mode=m._mode()).cpu().numpy()
    diff = np.abs(got.astype(int) - opre.ten2arr(ref).astype(int))
    assert diff.max() <= 1 and (diff != 0).mean() < (0.10 if precision == "bf16_fp8" else 0.01)
    eng.release_workspaces()


@pytest.mark.parametrize("precision", MODES)
def test_submodules_match_oracle(precision):
    """ConfidenceMapGenerator.forward / Refiner.forward (net.py:45-56, :75-80) on the kernels: as children of a
    WaterNet (parent's packed state dict) and free-standing (own tensors, zeros elsewhere)."""
    from waternet_b200.net import ConfidenceMapGenerator, Refiner
    sd = ofw.synthetic_state_dict(9, 3.0)
    m = _model(9, 3.0, precision)
    ins = _inputs_from_rgb([ofw.synthetic_image(70 + i, 40, 56, "smooth") for i in range(2)])
    cu = [t.cuda() for t in ins]
    _, cm_ref, parts = ofw.waternet_forward(sd, *ins, dtype=torch.float64, return_parts=True)
    with torch.no_grad():
        maps = m.cmg(*cu)
        assert len(maps) == 3 and maps[1].shape == (2, 1, 40, 56)
        _assert_close(torch.cat(maps, 1).cpu().numpy(), cm_ref.numpy())
        for r, (mod, other) in enumerate(zip((m.wb_refiner, m.ce_refiner, m.gc_refiner), cu[1:])):
            _assert_close(mod(cu[0], other).cpu().numpy(), parts[r].numpy())
        cmg = ConfidenceMapGenerator()
        cmg.load_state_dict({k[4:]: v for k, v in sd.items() if k.startswith("cmg.")})
        cmg.precision = precision
        _assert_close(torch.cat(cmg.cuda()(*cu), 1).cpu().numpy(), cm_ref.numpy())
        ref = Refiner()
        ref.load_state_dict({k[len("ce_refiner."):]: v for k, v in sd.items() if k.startswith("ce_refiner.")})
        ref.precision = precision
        _assert_close(ref.cuda()(cu[0], cu[2]).cpu().numpy(), parts[1].numpy())
        # the full model is unaffected by the sub-module calls in between (separate packed-weight slots)
        _assert_close(m(*cu).cpu().numpy(), ofw.waternet_forward(sd, *ins, dtype=torch.float64).numpy())


def test_two_models_on_one_device_do_not_share_packed_weights():
    """Advisor finding: an Enhancer must never run with another model's weights."""
    from waternet_b200.api import Enhancer
    rgb = ofw.synthetic_image(3, 48, 64, "smooth")
    ma, mb = _model(0, 3.0, "bf16x3"), _model(1, 3.0, "bf16x3")
    ea, eb = Enhancer(ma, cuda_graph=False), Enhancer(mb, cuda_graph=False)
    a0, b0 = ea(rgb), eb(rgb)
    assert not np.array_equal(a0, b0)
    with torch.no_grad():
        mb(*[t.cuda() for t in _inputs_from_rgb([rgb])])   # other model's forward in between
    assert np.array_equal(ea(rgb), a0) and np.array_equal(eb(rgb), b0)
    # parameter updates are picked up: through autograd-visible ops automatically, through .data after invalidation
    with torch.no_grad():
        ma.cmg.conv8.bias.add_(1.0)
    a1 = ea(rgb)
    assert not np.array_equal(a1, a0)
    ma.cmg.conv8.bias.data.sub_(1.0)
    ma.invalidate_packed_weights()
    assert np.array_equal(ea(rgb), a0)


def test_enhancer_pipeline_of_in_flight_batches():
    """submit()/wait(): several batches in flight (copy-in, kernels, copy-out on three streams, multi-pass) give
    exactly what one synchronous call per batch gives."""
    from waternet_b200.api import Enhancer
    m = _model(0, 3.0, "default")
    enh = Enhancer(m, cuda_graph=False)
    h, w = 72, 96
    eng = m.engine()
    eng.set_chunk_pixels(2 * h * w)   # 3 images -> passes of 2 + 1
    try:
        batches = [np.stack([ofw.synthetic_image(300 + 10 * b + i, h, w, "smooth") for i in range(3)]) for b in range(5)]
        want = [enh(b) for b in batches]
        pins = [(torch.from_numpy(b).pin_memory(), torch.empty(b.shape, dtype=torch.uint8).pin_memory()) for b in batches]
        seen = []
        tickets = [enh.submit(pi, po, on_pass=lambda t, a, b: seen.append((a, b))) for pi, po in pins[:2]]
        for i in range(2, 5):
            enh.wait(tickets[i - 2])
            tickets.append(enh.submit(*pins[i]))
        for t in tickets:
            enh.wait(t)
    finally:
        eng.set_chunk_pixels(0)
    for (_, po), ref in zip(pins, want):
        assert np.array_equal(po.numpy(), ref)
    assert seen == [(0, 2), (2, 3), (0, 2), (2, 3)]


# ------------------------------------------------------------------ e4m3 range guard of the default mode
def _scaled_refiner_sd(gain):
    """Stress weights whose wb_refiner.conv1 is scaled so that its activations leave the e4m3 range (448): that
    layer feeds the refiners' conv2, whose fp8 correction pass would saturate."""
    sd = ofw.synthetic_state_dict(0, 3.0)
    sd["wb_refiner.conv1.weight"] = sd["wb_refiner.conv1.weight"] * gain
    sd["wb_refiner.conv2.weight"] = sd["wb_refiner.conv2.weight"] / gain   # keep the output O(1)
    return sd


def test_fp8_mode_recomputes_in_call_when_activations_leave_the_e4m3_range():
    from waternet_b200.net import WaterNet
    sd = _scaled_refiner_sd(400.0)
    rgbs = [ofw.synthetic_image(5 + i, 40, 56, "smooth") for i in range(3)]
    ins = _inputs_from_rgb(rgbs)
    cu = [t.cuda() for t in ins]
    ref = ofw.waternet_forward(sd, *ins, dtype=torch.float64).numpy()
    m = WaterNet(precision="default")
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval()
    eng = m.engine()
    torch.cuda.synchronize()
    assert not eng.f8_overflowed()
    with torch.no_grad():
        first = m(*cu).cpu().numpy()          # the call that trips the guard is already the bf16x3 result
        assert eng.f8_overflowed()
        second = m(*cu).cpu().numpy()         # later calls go straight to the bf16x3 kernels
        mb = WaterNet(precision="bf16x3")
        mb.load_state_dict(sd, strict=True)
        plain = mb.cuda().eval()(*cu).cpu().numpy()
    assert np.array_equal(first, plain) and np.array_equal(second, plain)
    assert _assert_close(first, ref) < 2e-4
    # the folded uint8 path takes the same detour
    m2 = WaterNet(precision="default")
    m2.load_state_dict(sd, strict=True)
    m2 = m2.cuda().eval()
    e2 = m2.engine()
    got = e2.enhance(torch.from_numpy(np.stack(rgbs)).cuda(), mode=m2._mode()).cpu().numpy()
    assert e2.f8_overflowed()
    assert np.array_equal(got, opre.ten2arr(plain))
    # new weights: the flag is cleared and the fp8 corrections are back
    m.load_state_dict(ofw.synthetic_state_dict(0, 3.0))
    with torch.no_grad():
        m(*cu)
    torch.cuda.synchronize()
    assert not eng.f8_overflowed()


def _trained_state_dict():
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "trained_synthetic_400ep.npz")
    if not os.path.exists(path):
        pytest.skip("trained checkpoint fixture not present")
    with np.load(path) as z:
        return {k: torch.from_numpy(z[k]) for k, _ in ofw.state_dict_spec()}


@pytest.mark.parametrize("weights", ["default_init", "stress_gain3", "trained_400ep"])
def test_default_mode_margin_on_every_weight_set(weights):
    """The default (fp8-correction) mode stays below 6e-4 of the fp32 CPU result -- and never trips the range
    guard -- on default-init weights, the x3 stress set and the checkpoint of the 400-epoch synthetic training
    run (tests/golden/trained_synthetic_400ep.npz, produced by tools/gpu_train400.sh)."""
    sd = {"default_init": lambda: ofw.synthetic_state_dict(0, 1.0), "stress_gain3": lambda: ofw.synthetic_state_dict(0, 3.0),
          "trained_400ep": _trained_state_dict}[weights]()
    from waternet_b200.net import WaterNet
    rgbs = [ofw.synthetic_image(80 + i, 112, 112, "smooth" if i else "noise") for i in range(4)]
    ins = _inputs_from_rgb(rgbs)
    ref = ofw.waternet_forward(sd, *ins).numpy()
    m = WaterNet(precision="default")
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval()
    with torch.no_grad():
        out = m(*[t.cuda() for t in ins]).cpu().numpy()
    assert not m.engine().f8_overflowed()
    rel = _assert_close(out, ref)
    # the folded uint8 path (wn_enhance_u8: the preprocess kernel writes the first layer's level planes)
    frames = torch.from_numpy(np.ascontiguousarray(np.stack(rgbs))).cuda()
    f32 = torch.empty(len(rgbs), 3, 112, 112, device="cuda")
    u8 = m.engine().enhance(frames, mode=m._mode(), out_f32=f32)
    assert not m.engine().f8_overflowed()
    rel_folded = _assert_close(f32.cpu().numpy(), ref)
    print(f"default mode, {weights}: max rel err {rel:.2e} (tensor inputs), {rel_folded:.2e} (folded uint8 path)")
    assert rel < 6e-4 and rel_folded < 6e-4
    _assert_u8_close(u8.cpu().numpy(), opre.ten2arr(ref), share=0.10)


# ------------------------------------------------------------------ output stores fused with the exchange (SURVEY 8e)
@pytest.mark.parametrize("precision", MODES)
def test_peer_out_addresses_receive_the_bytes_of_the_output(precision):
    """wn_enhance_u8_peers: every 'peer' address (here: other buffers of the same GPU, no IPC needed) ends up with
    exactly the uint8 output, whichever launch writes it -- the gather/gate kernel (default mode: whole segments,
    ragged rows, destinations of any alignment), the copy kernel behind the bf16x3 / fp32 chains -- and on multi-pass
    batches.  (In a PeerGather block rank r's slot starts r * B * H * W * 3 bytes in: odd shapes misalign it.)"""
    m = _model(0, 3.0, precision)
    eng = m.engine()
    for (n, h, w), cap in (((3, 64, 96), 2 * 64 * 96), ((2, 33, 47), 0), ((1, 40, 64), 0)):
        frames = torch.from_numpy(np.ascontiguousarray(
            np.stack([ofw.synthetic_image(40 + i, h, w, "smooth") for i in range(n)]))).cuda()
        want = eng.enhance(frames, mode=m._mode()).clone()
        eng.set_chunk_pixels(cap)
        try:
            block = torch.zeros(3 * frames.numel() + 64, dtype=torch.uint8, device="cuda")
            out = torch.zeros_like(frames)
            k = out.data_ptr() % 16    # one peer aligned like the output (the fast stores), one off by a byte
            mirrors = [block[k + 16 + i * (frames.numel() + 17 - frames.numel() % 16):][:frames.numel()] for i in range(2)]
            assert mirrors[0].data_ptr() % 16 == k and mirrors[1].data_ptr() % 16 == (k + 1) % 16
            eng.enhance(frames, mode=m._mode(), out_u8=out, peer_out=[t.data_ptr() for t in mirrors])
            torch.cuda.synchronize()
        finally:
            eng.set_chunk_pixels(0)
        assert torch.equal(out, want)
        for t in mirrors:
            assert torch.equal(t.view(frames.shape), want)
    with pytest.raises(Exception):   # more peers than the ABI takes
        eng.enhance(frames, mode=m._mode(), out_u8=out, peer_out=[mirrors[0].data_ptr()] * 16)
    with pytest.raises(ValueError):  # an output tensor the kernels would fill in the wrong order
        eng.enhance(frames, mode=m._mode(), out_u8=torch.empty((n, w, h, 3), dtype=torch.uint8, device="cuda").permute(0, 2, 1, 3))


def test_peer_out_follows_the_range_guard_rerun():
    from waternet_b200.net import WaterNet
    m = WaterNet(precision="default")
    m.load_state_dict(_scaled_refiner_sd(400.0), strict=True)
    m = m.cuda().eval()
    eng = m.engine()
    frames = torch.from_numpy(np.ascontiguousarray(
        np.stack([ofw.synthetic_image(5 + i, 40, 56, "smooth") for i in range(3)]))).cuda()
    mirror = torch.zeros_like(frames)
    out = eng.enhance(frames, mode=m._mode(), peer_out=[mirror.data_ptr()])   # trips the guard: re-run inside the call
    torch.cuda.synchronize()
    assert eng.f8_overflowed()
    mb = WaterNet(precision="bf16x3")
    mb.load_state_dict(_scaled_refiner_sd(400.0), strict=True)
    mb = mb.cuda().eval()
    want = mb.engine().enhance(frames, mode=mb._mode())
    assert torch.equal(out, want) and torch.equal(mirror, want)


# ------------------------------------------------------------------ 2 ranks on NCCL: sharded == single GPU, bitwise
def _nccl_worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from waternet_b200.api import Enhancer
        from waternet_b200.dist import PassGather, PeerGather
        h, w, per = 64, 96, 3
        frames = np.stack([ofw.synthetic_image(500 + i, h, w, "smooth") for i in range(world * per)])
        m = _model(0, 3.0, "default")
        enh = Enhancer(m, cuda_graph=False)
        full = Enhancer(m, cuda_graph=False)(frames)            # every rank: all images on its own GPU
        m.engine().set_chunk_pixels(2 * h * w)  # 3 local images -> two passes, two exchanges
        local = torch.from_numpy(frames[rank * per:(rank + 1) * per].copy()).pin_memory()
        ok = True
        dev = torch.device("cuda", rank)
        # both exchange forms: NCCL all_gather per pass, and copy-engine pushes into peer memory over CUDA IPC
        for make in (lambda: PassGather(tuple(local.shape), torch.uint8, dev),
                     lambda: PeerGather.create(tuple(local.shape), torch.uint8, dev)):
            gather = make()
            gather.result().zero_()
            torch.cuda.synchronize()
            dist.barrier()                      # nobody pushes into a buffer that is still being cleared
            out = torch.empty_like(local).pin_memory()
            enh.enhance_pinned(local, out, on_pass=gather.on_pass)
            gather.finish()
            torch.cuda.synchronize()
            dist.barrier()
            ok = ok and gather.calls == 2 and np.array_equal(gather.result().cpu().numpy(), full)
            ok = ok and np.array_equal(out.numpy(), full[rank * per:(rank + 1) * per])
            dist.barrier()
            if isinstance(gather, PeerGather):
                kept = gather
        ok = ok and isinstance(gather, PeerGather)   # on one NVSwitch node the IPC path must be available
        if ok:  # third form: the exchange fused into the kernels that write the output (wn_enhance_u8_peers)
            for precision, want in (("default", full), ("bf16x3", None)):
                if want is None:
                    want = Enhancer(m, precision=precision, cuda_graph=False)(frames)
                kept.result().zero_()
                torch.cuda.synchronize()
                dist.barrier()
                out = torch.empty_like(local).pin_memory()
                Enhancer(m, precision=precision, cuda_graph=False).enhance_pinned(local, out, exchange=kept)
                torch.cuda.synchronize()
                dist.barrier()
                ok = ok and np.array_equal(kept.result().cpu().numpy(), want)
                ok = ok and np.array_equal(out.numpy(), want[rank * per:(rank + 1) * per])
                dist.barrier()
            kept.close()
        m.engine().set_chunk_pixels(0)
        ret[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


def test_nccl_sharded_output_equals_single_gpu_bitwise():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    with mp.Manager() as mgr:
        ret = mgr.dict()
        mp.spawn(_nccl_worker, args=(2, port, ret), nprocs=2, join=True)
        assert dict(ret) == {0: True, 1: True}


# ------------------------------------------------------------------ training data path (SURVEY 8f.3 / 8f.4)
def test_batched_resize_matches_cv2_bit_exact(eng):
    """wn_resize_u8 against the oracle's restatement of cv2.resize (and cv2 itself where importable): down-
    and up-scaling, the silent INTER_AREA switch at exactly 2x, equal sizes, 1-pixel sources, BGR->RGB folding."""
    rng = np.random.default_rng(5)
    shapes = [(300, 400), (224, 224), (112, 112), (57, 91), (113, 225), (1, 1), (2, 3), (480, 640), (225, 224)]
    srcs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in shapes]
    for dh, dw in [(112, 112), (96, 160)]:
        got = eng.resize_batch(srcs, dh, dw).cpu().numpy()
        swapped = eng.resize_batch(srcs, dh, dw, swap_rb=True).cpu().numpy()
        for i, src in enumerate(srcs):
            want = opre.resize_linear_u8(src, (dw, dh))
            assert np.array_equal(got[i], want), f"{shapes[i]} -> {(dh, dw)}: {(got[i] != want).sum()} bytes differ"
            assert np.array_equal(swapped[i], want[..., ::-1])
            try:
                import cv2
                assert np.array_equal(got[i], cv2.resize(src, (dw, dh)))
            except ImportError:
                pass
    many = [srcs[i % len(srcs)] for i in range(200)]  # more images than one launch's parameter block holds
    big = eng.resize_batch(many, 64, 64).cpu().numpy()
    assert np.array_equal(big[199], opre.resize_linear_u8(many[199], (64, 64)))


def test_gpu_batch_loader_resizes_files_on_the_device(tmp_path):
    """UIEBDataset (PNG pairs at native sizes) through GpuBatchLoader == the reference-style per-item CPU path."""
    cv2 = pytest.importorskip("cv2")
    from waternet_b200.training_utils import GpuBatchLoader, UIEBDataset, _item
    rng = np.random.default_rng(2)
    (tmp_path / "raw").mkdir()
    (tmp_path / "ref").mkdir()
    for i, (h, w) in enumerate([(150, 200), (224, 224), (131, 117), (300, 180)]):
        for sub in ("raw", "ref"):
            cv2.imwrite(str(tmp_path / sub / f"{i}.png"), rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
    ds = UIEBDataset(tmp_path / "raw", tmp_path / "ref", im_height=112, im_width=112, transform=None)
    loader = GpuBatchLoader(ds, batch_size=3, device="cuda:0", augment=False)
    seen = 0
    for b, batch in enumerate(loader):
        for j in range(batch["raw"].shape[0]):
            # per-item path of the reference (training_utils.py:89-123) without the random flips: cv2.imread,
            # cv2.resize, cvtColor(BGR2RGB), transform, arr2ten
            item = _item(*ds.pair(b * 3 + j))
            for key in ("raw", "wb", "gc", "he", "ref"):
                assert torch.equal(batch[key][j].cpu(), item[key].cpu().reshape(batch[key][j].shape)), key
            seen += 1
    assert seen == 4


def test_metrics_match_hand_computed_values_on_the_device():
    """SSIM / PSNR (torchmetrics functional defaults, train.py:139-144) on CUDA tensors against an independent
    float64 numpy evaluation: 11x11 gaussian (sigma 1.5), reflect padding cropped, k1 0.01, k2 0.03, data range
    = max(range(preds), range(target)); PSNR with data_range 1."""
    from waternet_b200.metrics import psnr, ssim
    rng = np.random.default_rng(0)
    a = rng.random((2, 3, 40, 48)).astype(np.float32)
    b = np.clip(a + 0.1 * rng.standard_normal(a.shape).astype(np.float32), 0, 1)
    g = np.exp(-((np.arange(11) - 5.0) ** 2) / (2 * 1.5 ** 2))
    g /= g.sum()
    k = np.outer(g, g)

    def filt(x):  # valid 11x11 correlation after reflect padding, then the reference crops the padded border
        p = np.pad(x.astype(np.float64), ((0, 0), (0, 0), (5, 5), (5, 5)), mode="reflect")
        out = np.zeros(x.shape, np.float64)
        for dy in range(11):
            for dx in range(11):
                out += k[dy, dx] * p[:, :, dy:dy + x.shape[2], dx:dx + x.shape[3]]
        return out

    dr = max(a.max() - a.min(), b.max() - b.min())
    c1, c2 = (0.01 * dr) ** 2, (0.03 * dr) ** 2
    mu_a, mu_b = filt(a), filt(b)
    va, vb, cab = filt(a * a) - mu_a ** 2, filt(b * b) - mu_b ** 2, filt(a * b) - mu_a * mu_b
    smap = ((2 * mu_a * mu_b + c1) * (2 * cab + c2)) / ((mu_a ** 2 + mu_b ** 2 + c1) * (va + vb + c2))
    want_ssim = smap[..., 5:-5, 5:-5].reshape(2, -1).mean(-1).mean()
    want_psnr = 10 * np.log10(1.0 / np.mean((a.astype(np.float64) - b) ** 2))
    ta, tb = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
    assert abs(ssim(ta, tb).item() - want_ssim) < 2e-5
    assert abs(psnr(ta, tb, 1.0).item() - want_psnr) < 1e-3
    assert abs(ssim(ta, ta).item() - 1.0) < 1e-6


def test_training_loss_curve_matches_the_reference_loop():
    """BASELINE configs[4] in miniature: this repository's loop (native forward/backward kernels, GpuBatchLoader)
    against the curve of the reference's train/eval loops (tests/ref_train_loop.py, train.py:26-152) driving the
    reference's own WaterNet in fp32 with per-item preprocess, stored by tests/golden/make_golden.py -- same synthetic
    pairs, same initial weights, same seeded VGG19, Adam 1e-3, StepLR per minibatch."""
    import json
    from waternet_b200 import training
    from waternet_b200.net import WaterNet
    from waternet_b200.training_utils import GpuBatchLoader, SyntheticUIEB
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda:0")
    with open(os.path.join(GOLDEN, "reference_train_curve.json")) as f:
        curve_r = [(e["train"], e["val"]) for e in json.load(f)]
    assert len(curve_r) == 4
    ours = WaterNet(precision="default")
    ours.load_state_dict(ofw.synthetic_state_dict(11, 1.0), strict=True)
    ours = ours.to(dev).train()
    vgg = training.PerceptualModel(pretrained=False).to(dev).eval()
    ds = SyntheticUIEB(length=80, im_height=64, im_width=64, seed=4)
    train_idx, val_idx = list(range(64)), list(range(64, 80))
    gpu_train = GpuBatchLoader(torch.utils.data.Subset(ds, train_idx), 16, device=dev, augment=False)
    gpu_val = GpuBatchLoader(torch.utils.data.Subset(ds, val_idx), 16, device=dev, augment=False)
    opt_o = torch.optim.Adam(ours.parameters(), lr=1e-3)
    sch_o = torch.optim.lr_scheduler.StepLR(opt_o, step_size=10000, gamma=0.1)
    curve_o = []
    for _ in range(len(curve_r)):
        to = training.train_one_epoch(ours, gpu_train, opt_o, sch_o, vgg, dev)
        vo = training.eval_one_epoch(ours, gpu_val, vgg, dev)
        curve_o.append((to, vo))
    for (tr, vr), (to, vo) in zip(curve_r, curve_o):
        for key in ("loss", "mse", "perceptual_loss", "ssim", "psnr"):
            assert abs(to[key] - tr[key]) <= 2e-2 * abs(tr[key]) + 1e-6, (key, to[key], tr[key])
        for key in ("mse", "ssim", "psnr"):
            assert abs(vo[key] - vr[key]) <= 2e-2 * abs(vr[key]) + 1e-6, (key, vo[key], vr[key])
        # documented deviation: the reference logs "last batch / count" for the validation perceptual loss
        # (train.py:74), this repository logs the mean; with ONE validation batch the two coincide
        assert abs(vo["perceptual_loss"] - vr["perceptual_loss"]) <= 2e-2 * abs(vr["perceptual_loss"]) + 1e-6
    assert curve_r[-1][0]["loss"] < curve_r[0][0]["loss"] and curve_o[-1][0]["loss"] < curve_o[0][0]["loss"]
    print("reference loop losses", [round(t["loss"], 3) for t, _ in curve_r])
    print("this repo's losses   ", [round(t["loss"], 3) for t, _ in curve_o])


def test_fused_tail_layers_equal_separate_launches():
    """Default mode: cmg.conv4 (1x1) runs as the tail GEMM of conv3's kernel (the activation tile goes back into tensor
    memory as the A operand of a second tcgen05.mma, UmmaCfg TN), and cmg.conv8 (3x3, 64 -> 3) as the tap-stacked tail
    of conv7 plus a gather kernel, the refiners' conv3 + gate likewise behind their conv2.  Same arithmetic as the
    separate launches up to the fp32 summation order."""
    from waternet_b200 import _lib
    sd = ofw.synthetic_state_dict(3, 3.0)
    m = _model(3, 3.0, "default")
    eng = m.engine()
    # the last two shapes: many tiles per CTA (a fused launch must not write into the buffer it still reads halos from)
    for n, h, w in [(1, 40, 56), (3, 37, 61), (2, 130, 70), (1, 16, 8), (1, 1, 1), (1, 300, 500), (2, 270, 480)]:
        torch.manual_seed(h)
        ins = [torch.rand(n, 3, h, w) for _ in range(4)]
        cu = [t.cuda() for t in ins]
        res = {}
        with torch.no_grad():
            # 256: conv3 / conv4 as two launches; 512: conv7 / conv8; 1024: refiner conv2 / conv3 + gate; 1792: nothing fused
            for flags in (0, 256, 512, 1024, 1792):
                eng.set_debug_flags(flags)
                try:
                    res[flags] = (m(*cu).cpu().numpy(),
                                  eng.debug_layer(*cu, layer=3, mode=_lib.MODE_BF16_FP8).cpu().numpy(),
                                  eng.debug_layer(*cu, layer=7, mode=_lib.MODE_BF16_FP8).cpu().numpy())
                finally:
                    eng.set_debug_flags(0)
        torch.cuda.synchronize()
        assert not eng.f8_overflowed(), "a garbage tile would trip the range guard and be silently recomputed"
        # the fused and the separate forms add the same products in a different order (~1e-7); where that moves a
        # value across a rounding boundary of the hi + fp8 activation format the fp8-correction scheme's own
        # error (~1e-4) appears between the two -- so the bar between them is that error, the bar against the
        # float64 oracle the parity bar
        ref64 = ofw.waternet_forward(sd, *ins, dtype=torch.float64).numpy()
        for flags in (0, 256, 512, 1024):
            for got, want in zip(res[flags], res[1792]):
                _assert_close(got, want, tol=3e-4)
            _assert_close(res[flags][0], ref64)
    # only the forms above (and 2048, the plain first layer) are selectable
    with pytest.raises(_lib.WaterNetLibraryError, match="unknown flag bits"):
        eng.set_debug_flags(1)


def test_native_backward_is_bit_reproducible():
    """The weight-gradient GEMM merges its per-CTA partial sums in a fixed order (no atomics): two backward passes
    over the same batch give bit-identical gradients -- also at the 16 x 112^2 training batch, where each CTA of a
    weight-gradient launch accumulates up to ~150 tiles."""
    torch.manual_seed(3)
    m = _model(5, 3.0, "default").train()
    for n, h, w in [(3, 61, 83), (16, 112, 112)]:
        ins = [t.cuda() for t in _inputs_from_rgb([ofw.synthetic_image(90 + i, h, w, "smooth") for i in range(n)])]
        target = torch.rand(n, 3, h, w).cuda()
        runs = []
        for _ in range(3):
            m.zero_grad(set_to_none=True)
            torch.nn.functional.mse_loss(m(*ins), target).backward()
            runs.append([p.grad.clone() for p in m.parameters()])
        for other in runs[1:]:
            for a, b in zip(runs[0], other):
                assert torch.equal(a, b), (n, h, w)


def test_white_balance_grayscale_branch(eng):
    """data.py:30-36: the 2-D branch of white_balance_transform (no reference caller uses it; provided for completeness)."""
    from waternet_b200 import data
    rng = np.random.default_rng(4)
    for shape, kind in [((40, 56), 0), ((112, 112), 0), ((7, 9), 0), ((33, 17), 1), ((200, 300), 1)]:
        g = rng.integers(0, 256, shape, dtype=np.uint8) if kind == 0 else (rng.random(shape) * 90 + 40).astype(np.uint8)
        assert np.array_equal(data.white_balance_transform(g), opre.white_balance_transform(g)), shape
    batch = rng.integers(0, 256, (3, 24, 40), dtype=np.uint8)
    got = eng.white_balance_gray(torch.from_numpy(batch).cuda()).cpu().numpy()
    for i in range(3):
        assert np.array_equal(got[i], opre.white_balance_transform(batch[i]))


@pytest.mark.parametrize("precision", TC_MODES)
def test_k_packed_first_layer_equals_plain_layout(precision):
    """Inference runs the 7x7 first layer K-packed (UmmaCfg KP: 40 K steps per tile instead of 49, planes one column
    wider with channels 8-11 of two neighbouring pixels per row); flag 2048 selects the plain 49-tap form.  Same
    products, different summation order -- and different input plane layouts, so the edges matter: widths 1, 2, 7,
    ragged tiles, 8-bit level inputs (hi planes only) and arbitrary floats (hi + lo planes)."""
    from waternet_b200 import _lib
    sd = ofw.synthetic_state_dict(6, 3.0)
    m = _model(6, 3.0, precision)
    eng = m.engine()
    mode = m._mode()
    for n, h, w, exact in [(1, 16, 1, True), (1, 5, 2, False), (2, 23, 7, True), (1, 40, 61, False), (1, 64, 96, True),
                           (1, 130, 200, True)]:
        if exact:
            ins = _inputs_from_rgb([ofw.synthetic_image(700 + h + i, h, w, "noise") for i in range(n)])
        else:
            torch.manual_seed(h * w)
            ins = [torch.rand(n, 3, h, w) for _ in range(4)]
        cu = [t.cuda() for t in ins]
        res = {}
        with torch.no_grad():
            for flags in (0, 2048):
                eng.set_debug_flags(flags)
                try:
                    res[flags] = (eng.debug_layer(*cu, layer=0, mode=mode).cpu().numpy(),
                                  eng.debug_layer(*cu, layer=8, mode=mode).cpu().numpy(), m(*cu).cpu().numpy())
                finally:
                    eng.set_debug_flags(0)
        tol = 3e-4 if precision == "bf16_fp8" else 2e-5   # default mode: the hi + fp8 format is discontinuous (see the tail test)
        for got, want in zip(res[0], res[2048]):
            _assert_close(got, want, tol=tol)
        _assert_close(res[0][2], ofw.waternet_forward(sd, *ins, dtype=torch.float64).numpy())
    # the uint8 end-to-end path writes the K-packed planes from the preprocess kernel
    rgbs = np.stack([ofw.synthetic_image(800 + i, 37, 53, "smooth") for i in range(2)])
    dev = torch.from_numpy(rgbs).cuda()
    a = eng.enhance(dev, mode=mode).cpu().numpy()
    eng.set_debug_flags(2048)
    try:
        b = eng.enhance(dev, mode=mode).cpu().numpy()
    finally:
        eng.set_debug_flags(0)
    assert np.abs(a.astype(int) - b.astype(int)).max() <= 1 and (a != b).mean() < 0.02
