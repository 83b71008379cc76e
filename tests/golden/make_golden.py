"""Generate the fixtures under tests/golden/ from the UNMODIFIED reference.

Run once, with the path of a checkout of the reference::

    python tests/golden/make_golden.py REFERENCE_CHECKOUT

It imports the reference's ``waternet/{data,net}.py`` and ``hubconf.py`` by file
path (never copied), feeds them seeded synthetic inputs / weights
(``oracle.forward.synthetic_image`` / ``synthetic_state_dict``) and stores what
they return, so that the tests compare with the reference without needing it.
"""
import hashlib
import importlib.util
import json
import os
import sys
import types

import numpy as np
import torch

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle.forward import synthetic_image, synthetic_state_dict  # noqa: E402


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def load_reference(ref):
    pkg = types.ModuleType("waternet")
    pkg.__path__ = [os.path.join(ref, "waternet")]
    sys.modules["waternet"] = pkg
    data = _load("waternet.data", os.path.join(ref, "waternet", "data.py"))
    net = _load("waternet.net", os.path.join(ref, "waternet", "net.py"))
    hub = _load("ref_hubconf", os.path.join(ref, "hubconf.py"))
    return data, net, hub


def sha256(arr):
    return hashlib.sha256(np.ascontiguousarray(arr).tobytes()).hexdigest()


PRE_CASES = [
    ("noise_112x112", 0, 112, 112, "noise"),
    ("smooth_112x112", 1, 112, 112, "smooth"),
    ("noise_113x117", 2, 113, 117, "noise"),
    ("smooth_64x96", 3, 64, 96, "smooth"),
    ("noise_115x112", 4, 115, 112, "noise"),
    ("smooth_120x200", 5, 120, 200, "smooth"),
]

# (name, [(img seed, kind)], H, W, weight seed, gain)
FWD_CASES = [
    ("c1_1x112x112", [(10, "smooth")], 112, 112, 0, 1.0),
    ("n2_112x112", [(11, "noise"), (12, "smooth")], 112, 112, 0, 1.0),
    ("gain3_1x40x56", [(13, "noise")], 40, 56, 1, 3.0),
    # BASELINE.json configs[1]: batch 16, 112x112 (stress weights; mixed noise / smooth frames)
    ("c2_16x112x112", [(100 + i, "noise" if i % 4 == 0 else "smooth") for i in range(16)], 112, 112, 2, 3.0),
]

# test_oracle.py::test_preprocess_matches_live_reference: (H, W) x kind, SHA-256 of the reference's outputs
DIGEST_SHAPES = [(112, 112), (113, 117), (112, 117), (115, 112), (48, 200), (270, 480)]


def reference_digests(data):
    """SHA-256 digests of the reference's uint8 outputs: transform() on seeded colour frames, and the 2-D branch of
    white_balance_transform() on the inputs test_grayscale_white_balance_matches_live_reference draws."""
    pre = {}
    for i, (h, w) in enumerate(DIGEST_SHAPES):
        for j, kind in enumerate(("noise", "smooth")):
            seed = 300 + 2 * i + j
            wb, gc, he = data.transform(synthetic_image(seed, h, w, kind))
            pre[f"{h}x{w}_{kind}"] = {"seed": seed, "wb": sha256(wb), "gc": sha256(gc), "he": sha256(he)}
    gray = []
    rng = np.random.default_rng(0)
    for shape in [(40, 56), (7, 9), (33, 17), (112, 112)]:
        for k in range(2):
            g = rng.integers(0, 256, shape, dtype=np.uint8) if k == 0 else (rng.random(shape) * 90 + 40).astype(np.uint8)
            gray.append({"shape": list(shape), "kind": k, "sha256": sha256(data.white_balance_transform(g.copy()))})
    return {"preprocess": pre, "white_balance_gray": gray}


def reference_train_curve(data, net):
    """BASELINE configs[4] in miniature: the reference's train / eval loops (tests/ref_train_loop.py) driving the
    reference's WaterNet in fp32 on the host, per-item preprocess by the reference's transform.  Same synthetic pairs,
    initial weights, seeded VGG19, Adam 1e-3 and StepLR as test_training_loss_curve_matches_the_reference_loop."""
    sys.path.insert(0, os.path.dirname(HERE))
    import ref_train_loop
    from waternet_b200 import metrics
    from waternet_b200.training import PerceptualModel
    from waternet_b200.training_utils import SyntheticUIEB, arr2ten

    ds = SyntheticUIEB(length=80, im_height=64, im_width=64, seed=4)

    def batches(indices, size=16):  # DataLoader(Subset(ds, indices), batch_size=16) of the reference's items
        out = []
        for a in range(0, len(indices), size):
            items = []
            for i in indices[a:a + size]:
                raw, ref = ds.pair(i)
                wb, gc, he = data.transform(raw)
                items.append({"raw": arr2ten(raw), "wb": arr2ten(wb), "gc": arr2ten(gc), "he": arr2ten(he),
                              "ref": arr2ten(ref)})
            out.append(torch.utils.data.default_collate(items))
        return out

    train, val = batches(list(range(64))), batches(list(range(64, 80)))
    model = net.WaterNet()
    model.load_state_dict(synthetic_state_dict(11, 1.0), strict=True)
    model.train()
    vgg = PerceptualModel(pretrained=False).eval()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    sch = torch.optim.lr_scheduler.StepLR(opt, step_size=10000, gamma=0.1)
    curve = []
    for epoch in range(4):
        tr = ref_train_loop.train_one_epoch(model, train, opt, sch, vgg, "cpu", metrics)
        vr = ref_train_loop.eval_one_epoch(model, val, vgg, "cpu", metrics)
        curve.append({"train": tr, "val": vr})
        print("train curve epoch", epoch, round(tr["loss"], 3))
    return curve


def main():
    if len(sys.argv) != 2 or not os.path.isfile(os.path.join(sys.argv[1], "waternet", "net.py")):
        raise SystemExit("usage: python tests/golden/make_golden.py REFERENCE_CHECKOUT")
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    data, net, hub = load_reference(sys.argv[1])
    for name, seed, h, w, kind in PRE_CASES:
        rgb = synthetic_image(seed, h, w, kind)
        wb, gc, he = data.transform(rgb)
        np.savez_compressed(os.path.join(HERE, f"preprocess_{name}.npz"), rgb=rgb, wb=wb, gc=gc, he=he)
        print("preprocess", name, rgb.shape)

    preprocess, postprocess, model = hub.waternet(pretrained=False)
    model.eval()
    for name, imgs, h, w, wseed, gain in FWD_CASES:
        sd = synthetic_state_dict(wseed, gain)
        model.load_state_dict(sd, strict=True)
        rgbs = [synthetic_image(s, h, w, k) for s, k in imgs]
        parts = [preprocess(r) for r in rgbs]
        x, wb, he, gc = (torch.cat([p[i] for p in parts], dim=0) for i in range(4))
        with torch.no_grad():
            out = model(x, wb, he, gc)
        post = postprocess(out)
        np.savez_compressed(
            os.path.join(HERE, f"forward_{name}.npz"),
            rgb=np.stack(rgbs),
            out=out.numpy(),
            post=post,
            weight_seed=np.int64(wseed),
            gain=np.float64(gain),
            in_strides=np.array(parts[0][0].stride(), dtype=np.int64),
        )
        print("forward", name, tuple(out.shape), float(out.max()))

    for fname, content in (("reference_digests.json", reference_digests(data)),
                           ("reference_train_curve.json", reference_train_curve(data, net))):
        with open(os.path.join(HERE, fname), "w") as f:
            json.dump(content, f, indent=1)
            f.write("\n")
        print("wrote", fname)


if __name__ == "__main__":
    main()
