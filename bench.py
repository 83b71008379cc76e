#!/usr/bin/env python
"""Headline benchmark: images/sec of the WaterNet hot path at 1080p, batch 16 per GPU.

    python bench.py --gpus 1 --steps K --warmup W              # this repo's CUDA path
    python bench.py --impl reference --gpus 1 --steps K ...    # the UNMODIFIED reference on the host cores (baseline/_ref)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch: uint8 RGB images ->
WB/GC/HE preprocess -> gated-fusion forward -> uint8 enhanced images
(BASELINE.json configs[2]: batch 16, 1920x1080, preprocess+forward end to end).
`value` times that with the uint8 batch already resident in HBM; `e2e` times the
public host-buffer call (pinned host uint8 in, uint8 out) with both copies inside
the timed region (pipelined pass by pass on side streams).  At N>1 every rank
processes its own batch (weak scaling); the all-gather of the uint8 output (SURVEY.md 8e) is
fused into the launch that writes it -- NVLink stores into every rank's IPC-mapped buffer
(waternet_b200.dist.PeerGather; --gather peer / nccl: copy-engine pushes / NCCL per pass).
Before timing, image 0 of the batch is checked against the CPU reference (the line
carries `parity`; the run fails above the 1e-3 bar).  Rank 0 prints ONE JSON line.
`--dump-outputs DIR` writes the uint8 images of the last timed step as DIR/enhanced.npy (float32;
above 64 MB a fixed seeded sample of image rows), so that two builds can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "images/sec at 1080p batch16 (preprocess + gated-fusion forward, uint8 in -> uint8 out)"
UNIT = "images/s"


def workload_config(args, world):
    """`config` keys shared by both arms (same strings for the same command line)."""
    return {"workload": f"batch {args.batch} x {args.width}x{args.height} RGB uint8 per GPU: WB/GC/HE preprocess + "
                        "WaterNet forward + uint8 postprocess (BASELINE configs[2])",
            "global_batch": world * args.batch, "weights": "random init (torch.manual_seed(0))",
            "cache": "no L2 flush needed: each step streams GBs of inputs + intermediates (>> 126 MB L2)",
            "sampled_images_per_step": "product arm: every image of the batch; reference arm: 1 image per step "
                                       "(images are independent units, images/s does not depend on the batch)"}

# multiply-accumulates per pixel of every convolution, state-dict order (SURVEY.md 2.1)
CONV_MACS = [75264, 409600, 147456, 8192, 200704, 102400, 36864, 1728] + [9408, 25600, 864] * 3
CONV_NAMES = [f"cmg.conv{i}" for i in range(1, 9)] + [f"{r}.conv{i}" for r in ("wb_refiner", "ce_refiner", "gc_refiner")
                                                      for i in (1, 2, 3)]
TOTAL_MACS = sum(CONV_MACS)  # 1,089,824


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--mode", choices=["default", "fp32", "bf16x3", "bf16_fp8"], default="default")
    ap.add_argument("--batch", type=int, default=16, help="images per GPU per step")
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gather", choices=["fused", "peer", "nccl"], default="fused",
                    help="N > 1: how the uint8 output is all-gathered (fused = NVLink stores from the kernel that "
                         "writes the output; peer = copy-engine pushes per pass; nccl = NCCL all_gather per pass)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the uint8 images of the last timed step to DIR/enhanced.npy as float32 (all of them "
                         "up to 64 MB, else a fixed seeded sample of image rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computed (--impl ours)")
    return args


def synthetic_batch(n, h, w, seed):
    """Blue-green underwater-like frames: low-frequency structure + noise (deterministic)."""
    rng = np.random.default_rng(seed)
    coarse = rng.random((n, h // 40 + 2, w // 40 + 2, 3))
    up = np.repeat(np.repeat(coarse, 40, axis=1), 40, axis=2)[:, :h, :w]
    img = up * np.array([90.0, 200.0, 230.0]) + rng.integers(0, 24, (n, h, w, 3))
    return np.clip(img, 1, 255).astype(np.uint8)


DUMP_LIMIT_BYTES = 64 * 10**6


def dump_outputs(out_dir, images):
    """`images` (uint8 N x H x W x 3) -> out_dir/enhanced.npy in float32: the whole batch when it fits in
    DUMP_LIMIT_BYTES, else the rows of a fixed seeded sample of its N*H image rows, in order, shaped (rows, W, 3)."""
    n, h, w, c = images.shape
    rows = images.reshape(n * h, w * c)
    keep = min(n * h, DUMP_LIMIT_BYTES // (w * c * 4))
    idx = np.sort(np.random.default_rng(0).choice(n * h, keep, replace=False))
    sample = rows[torch.from_numpy(idx).to(rows.device)].float().cpu().numpy()
    sample = sample.reshape((n, h, w, c) if keep == n * h else (keep, w, c))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "enhanced.npy"), sample)
    return {"dir": out_dir, "enhanced": list(sample.shape),
            "sample": None if keep == n * h else f"{keep} of the {n * h} image rows "
                                                 f"(sorted numpy default_rng(0).choice({n * h}, {keep}, replace=False))"}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "tf_burst": p["bf16_tflops"], "tf_sustained": p["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [s for s, p in zip(sm, power) if p > 0.5 * max(power)] or sm
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power)}


# ------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the unmodified reference (baseline/_ref, copied from /root/reference by
# __graft_entry__.build()) on the host cores; the oracle port only when that copy or cv2 is missing
# ------------------------------------------------------------------------------------------
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def load_reference():
    """(transform, WaterNet class, arr2ten, ten2arr) of the unmodified reference, imported by file path under
    private module names (the repo's own `waternet` package keeps its name).  None when unavailable."""
    import importlib.util
    import types
    if not os.path.isfile(os.path.join(REF_DIR, "waternet", "net.py")):
        return None, "baseline/_ref is absent (run __graft_entry__.build() where /root/reference exists)"
    try:
        import cv2  # noqa: F401  (waternet/data.py needs it)
    except Exception as e:  # pragma: no cover
        return None, f"cv2 unavailable: {e}"

    def load(name, path):
        spec = importlib.util.spec_from_file_location(name, path)
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
        return mod

    sys.dont_write_bytecode = True
    pkg = types.ModuleType("_wn_reference")
    pkg.__path__ = [os.path.join(REF_DIR, "waternet")]
    sys.modules["_wn_reference"] = pkg
    data = load("_wn_reference.data", os.path.join(REF_DIR, "waternet", "data.py"))
    net = load("_wn_reference.net", os.path.join(REF_DIR, "waternet", "net.py"))
    hub = load("_wn_reference_hubconf", os.path.join(REF_DIR, "hubconf.py"))  # arr2ten / ten2arr helpers
    return (data.transform, net.WaterNet, hub.arr2ten_noeinops, hub.ten2arr_noeinops), None


class CpuReference:
    """One image through the reference on the CPU: transform -> arr2ten x4 -> WaterNet -> ten2arr."""

    def __init__(self, state_dict):
        ref, why = load_reference()
        self.kind = "reference" if ref else "port"
        self.note = why
        torch.set_num_threads(os.cpu_count() or 1)
        if ref:
            self.transform, net_cls, self.arr2ten, self.ten2arr = ref
            self.model = net_cls()
            self.model.load_state_dict(state_dict, strict=True)
            self.model.eval()
        else:
            self.sd = state_dict

    def step(self, rgb):
        """rgb uint8 HWC -> (fp32 output (1,3,H,W) ndarray, uint8 output HWC)."""
        if self.kind == "reference":
            wb, gc, he = self.transform(rgb)
            ins = [self.arr2ten(a) for a in (rgb, wb, he, gc)]
            with torch.no_grad():
                out = self.model(*ins)
            return out.numpy(), self.ten2arr(out)[0]
        from oracle import forward as ofw
        from oracle import preprocess as opre
        wb, gc, he = opre.transform(rgb)
        ins = [torch.from_numpy(opre.arr2ten(a).copy()) for a in (rgb, wb, he, gc)]
        out = ofw.waternet_forward(self.sd, *ins).numpy()
        return out, opre.ten2arr(out)[0]


def bench_state_dict():
    """The weights both arms use: WaterNet() default init under torch.manual_seed(0), as a CPU state dict."""
    from waternet_b200.net import WaterNet
    torch.manual_seed(0)
    return {k: v.detach().clone() for k, v in WaterNet().state_dict().items()}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    ref = CpuReference(bench_state_dict())
    frames = synthetic_batch(1, args.height, args.width, 0)
    for _ in range(args.warmup):
        ref.step(frames[0])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ref.step(frames[0])
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    value = 1.0 / dt
    sample = (f"1 image {args.width}x{args.height} per step (of the batch-{args.batch} workload; images are independent, "
              f"so images/s does not depend on the batch), "
              + ("unmodified reference: waternet.data.transform (numpy+cv2) + WaterNet.forward (torch CPU fp32)"
                 if ref.kind == "reference" else f"oracle port ({ref.note})"))
    # how the reference itself would run on this box (inference.py:85,185-191: preprocess on the host, model and
    # tensors on CUDA when available -- torch/cuDNN kernels, TF32 convolutions by default): reported beside the CPU
    # arm, not instead of it; nothing of this repository is on that path either
    on_gpu = None
    if ref.kind == "reference" and torch.cuda.is_available():
        try:
            dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
            model = ref.model.to(dev)
            pre_s = fwd_s = 0.0
            for i in range(3):  # first pass = warm-up (cuDNN algorithm selection)
                t0 = time.perf_counter()
                wb, gc, he = ref.transform(frames[0])
                ins = [ref.arr2ten(a).to(dev) for a in (frames[0], wb, he, gc)]
                torch.cuda.synchronize(dev)
                t1 = time.perf_counter()
                with torch.no_grad():
                    out = model(*ins)
                arr = ref.ten2arr(out)
                t2 = time.perf_counter()
                if i:
                    pre_s += (t1 - t0) / 2
                    fwd_s += (t2 - t1) / 2
            on_gpu = {"value": 1.0 / (pre_s + fwd_s), "unit": UNIT, "preprocess_ms_per_image": pre_s * 1e3,
                      "forward_and_postprocess_ms_per_image": fwd_s * 1e3,
                      "note": "unmodified reference, model.to(cuda) as inference.py does: transform on the host cores, "
                              "forward by torch/cuDNN on one GPU (allow_tf32 default), ten2arr on the host"}
            ref.model.to("cpu")
        except Exception as e:  # informational only
            on_gpu = {"unavailable": str(e)[:200]}
    config = workload_config(args, world)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": ref.kind,
                         "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "reference_with_cuda_forward": on_gpu,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); there is no CPU fallback for the product arm")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    import torch.distributed as dist
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=device)
    if args.gpus != world and rank == 0 and world > 1:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE {world}", file=sys.stderr)

    from waternet_b200 import _lib
    from waternet_b200.api import Enhancer
    from waternet_b200.dist import PassGather, PeerGather
    from waternet_b200.net import WaterNet

    sd = bench_state_dict()  # random init of the reference architecture, the same tensors the reference arm loads
    model = WaterNet(precision=args.mode)
    model.load_state_dict(sd, strict=True)
    model = model.to(device).eval()
    enh = Enhancer(model, device=device)
    eng = enh.engine
    mode = model._mode()

    B, H, W = args.batch, args.height, args.width
    host = synthetic_batch(B, H, W, seed=rank)
    dev_in = torch.from_numpy(host).to(device)
    dev_out = torch.empty_like(dev_in)
    nb = eng.chunk_images(B, H, W)
    gather = None
    if world > 1:  # peer memory over CUDA IPC (fused stores or copy-engine pushes); --gather nccl = all_gather per pass
        gather = (PassGather((B, H, W, 3), torch.uint8, device) if args.gather == "nccl"
                  else PeerGather.create((B, H, W, 3), torch.uint8, device))
    fused_gather = args.gather == "fused" and isinstance(gather, PeerGather)
    side = torch.cuda.Stream(device)

    push_done = {}

    def step_resident():
        """One step with the batch resident in HBM.  N > 1, fused: the last kernel of every pass stores its output
        into every rank's buffer; the completion signal follows the last pass on the compute stream, the wait for the
        peers' signals sits on a side stream.  peer / nccl: the exchange of a pass's output on the side stream, under
        the next pass's kernels.  The compute stream never waits for the exchange as such -- only, one step later, for
        the previous step's completion (fused) or for the push that still reads the slice of `dev_out` a pass is about
        to overwrite -- so the ranks are not lock-stepped."""
        cur = torch.cuda.current_stream(device)
        if fused_gather and "step" in push_done:
            cur.wait_event(push_done["step"])  # peers have signalled the step before the previous one
        for a in range(0, B, nb):
            b = min(B, a + nb)
            if fused_gather:
                eng.enhance(dev_in[a:b], mode=mode, out_u8=dev_out[a:b], peer_out=gather.addresses(a))
                continue
            if gather is not None and a in push_done:
                cur.wait_event(push_done[a])
            eng.enhance(dev_in[a:b], mode=mode, out_u8=dev_out[a:b])
            if gather is not None:
                ev = torch.cuda.Event()
                ev.record(cur)
                with torch.cuda.stream(side):
                    side.wait_event(ev)
                    gather.on_pass(dev_out[a:b], a, b)
                    done = torch.cuda.Event()
                    done.record(side)
                    push_done[a] = done
        if fused_gather:
            gather.signal()
            if "waited" in push_done:
                push_done["step"] = push_done["waited"]
            with torch.cuda.stream(side):
                gather.wait()
                done = torch.cuda.Event()
                done.record(side)
                push_done["waited"] = done
        elif gather is not None:
            with torch.cuda.stream(side):
                gather.finish()

    pins = [(torch.from_numpy(host).pin_memory(), torch.empty(host.shape, dtype=torch.uint8).pin_memory())
            for _ in range(2)]
    on_pass = gather.on_pass if gather is not None and not fused_gather else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(run, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(steps)
        e1.record()
        barrier()
        ms_local = e0.elapsed_time(e1)
        if world > 1:
            every = torch.zeros(world, device=device)
            every[rank] = ms_local
            dist.all_reduce(every, op=dist.ReduceOp.SUM)
            per_rank = [float(v) for v in every.tolist()]
        else:
            per_rank = [float(ms_local)]
        return max(per_rank), per_rank

    def run_resident(steps):
        for _ in range(steps):
            step_resident()

    def run_e2e(steps):
        """The public host-buffer call, as a video loop uses it: submit step i+1, then wait for step i.  Every
        step's input is copied H2D from pinned memory and its result D2H inside the timed region."""
        cur = torch.cuda.current_stream(device)
        prev = None
        for i in range(steps):
            ticket = enh.submit(*pins[i % 2], on_pass=on_pass, exchange=gather if fused_gather else None)
            if gather is not None and not fused_gather:
                with torch.cuda.stream(enh._s_out):
                    gather.finish()
            if prev is not None:
                enh.wait(prev)
            prev = ticket
        enh.wait(prev)
        cur.wait_stream(enh._s_out)

    # ---- parity before timing: image 0 of rank 0's batch against the CPU reference (both outputs) ----
    parity = None
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ref = CpuReference(sd)
        t0 = time.perf_counter()
        ref_f32, ref_u8 = ref.step(host[0])
        dt = time.perf_counter() - t0
        cpu_baseline = {"value": 1.0 / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": ref.kind,
                        "sample": f"1 image {W}x{H} of the batch ("
                                  + ("unmodified reference from baseline/_ref: numpy+cv2 preprocess, torch-CPU fp32 forward"
                                     if ref.kind == "reference" else f"oracle port: {ref.note}") + f"), {dt:.1f} s"}
        got_f32 = torch.empty((B, 3, H, W), dtype=torch.float32, device=device)
        for a in range(0, B, nb):  # the same pass structure as the timed step
            eng.enhance(dev_in[a:min(B, a + nb)], mode=mode, out_u8=dev_out[a:min(B, a + nb)], out_f32=got_f32[a:min(B, a + nb)])
        g32 = got_f32[0].cpu().numpy()
        g8 = dev_out[0].cpu().numpy()
        del got_f32
        scale = float(np.max(np.abs(ref_f32)))
        max_rel = float(np.max(np.abs(g32 - ref_f32[0])) / scale)
        d8 = np.abs(g8.astype(np.int16) - ref_u8.astype(np.int16))
        parity = {"against": cpu_baseline["kind"], "image": 0, "max_rel_err": max_rel, "tolerance": 1e-3,
                  "u8_mismatch_frac": float((d8 != 0).mean()), "u8_max_abs_diff": int(d8.max()),
                  "f8_overflowed": bool(eng.f8_overflowed())}
        if not (max_rel <= 1e-3 and d8.max() <= 1):
            print(json.dumps({"error": "parity check failed before timing", "parity": parity}), flush=True)
            raise SystemExit(2)

    for _ in range(max(args.warmup, 3) if args.warmup > 0 else 0):
        step_resident()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    eng.enable_timing(True)
    launches0 = eng.launch_count
    total_ms, per_rank_ms = timed(run_resident, args.steps)
    launches = eng.launch_count - launches0
    slot_ms, slot_cnt = eng.read_timings()
    eng.enable_timing(False)
    clocks = sampler.stop() if rank == 0 else None
    dumped = None
    if args.dump_outputs and rank == 0:  # timed() ended in a barrier: every rank's last step has landed
        dumped = dump_outputs(args.dump_outputs, gather.result() if gather is not None else dev_out)

    # the collective's own cost: the same step without it, same box, right after
    nogather_ms = None
    if world > 1:
        saved, gather, fused_gather = (gather, fused_gather), None, False
        nogather_ms, _ = timed(run_resident, args.steps)
        gather, fused_gather = saved

    run_e2e(2)
    e2e_ms, e2e_per_rank = timed(run_e2e, args.steps)
    if world > 1:  # what was gathered is what every rank computed: my own block bitwise, every rank's block by checksum
        last_out = enh._slots[(enh._next - 1) % len(enh._slots)].dev_out
        same = torch.equal(gather.gathered[rank], last_out)
        own = torch.zeros(world, dtype=torch.int64, device=device)
        own[rank] = last_out.view(-1).view(torch.int32).sum(dtype=torch.int64)
        dist.all_reduce(own)                                   # own[r] = checksum of what rank r computed
        got = torch.stack([gather.gathered[r].view(-1).view(torch.int32).sum(dtype=torch.int64) for r in range(world)])
        same = same and torch.equal(own, got)
        flag = torch.tensor([1 if same else 0], device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        gather_ok = bool(flag.item())
    else:
        gather_ok = None

    ms_per_step = total_ms / args.steps
    value = world * B * args.steps / (total_ms / 1e3)
    e2e_value = world * B * args.steps / (e2e_ms / 1e3)

    if rank == 0:
        peaks = load_peaks()
        conv_ms = slot_ms[:17]
        macs_by_slot = list(CONV_MACS)
        names_by_slot = list(CONV_NAMES)
        if mode != _lib.MODE_FP32_SIMT:
            # tensor-core path: ten launches.  slot 0 = cmg.conv1 + the three refiner conv1 (one 16->224 GEMM),
            # slot 9 = the three refiner conv2 (block-diagonal 96->96), slot 10 = the three conv3 + gated sum
            macs_by_slot = CONV_MACS[:8] + [0] * 9
            macs_by_slot[0] += 3 * 9408
            macs_by_slot[9] = 3 * 25600
            macs_by_slot[10] = 3 * 864
            names_by_slot[0] = "cmg.conv1+refiner.conv1x3"
            names_by_slot[9] = "refiner.conv2x3"
            names_by_slot[10] = "refiner.conv3x3+gate"
            flags = int(os.environ.get("WATERNET_B200_DEBUG_FLAGS", "0"), 0)
            if mode != _lib.MODE_BF16X3 and not flags & 256:   # conv4 runs as the tail GEMM of conv3's launch
                macs_by_slot[2] += macs_by_slot[3]
                macs_by_slot[3] = 0
                names_by_slot[2] = "cmg.conv3+conv4"
            if mode != _lib.MODE_BF16X3 and not flags & 1024:  # refiner conv3 tap-stacked behind conv2 + gather/gate kernel
                macs_by_slot[9] += macs_by_slot[10]
                macs_by_slot[10] = 0
                names_by_slot[9] = "refiner.conv2x3+conv3x3(taps)"
                names_by_slot[10] = "refiner.conv3.gather+gate"
            if mode != _lib.MODE_BF16X3 and not flags & 512:   # conv8 tap-stacked behind conv7 + a gather kernel
                macs_by_slot[6] += macs_by_slot[7]
                macs_by_slot[7] = 0
                names_by_slot[6] = "cmg.conv7+conv8(taps)"
                names_by_slot[7] = "cmg.conv8.gather+sigmoid"
        top = int(np.argmax(conv_ms))
        n_launch = max(slot_cnt[top], 1)
        avg_ms = conv_ms[top] / n_launch
        # how many images one bracketed launch group covers: steps*B images / count
        imgs_per_launch = args.steps * B / n_launch
        macs = macs_by_slot[top]
        fused = [names_by_slot[top]]
        traffic, traffic_total_per_image, traffic_src = None, None, None
        for cand in ("r2_traffic.json", "r1_traffic.json"):
            tpath = os.path.join(ROOT, "profiles", cand)
            if mode != _lib.MODE_FP32_SIMT and os.path.exists(tpath):
                with open(tpath) as f:
                    tj = json.load(f)
                ent = tj["kernels"].get(fused[0])
                if ent and (tj["height"], tj["width"]) == (H, W):  # measured per 1080p image; scales with images per launch
                    traffic = ent["dram_bytes_per_image"] * imgs_per_launch
                    traffic_total_per_image = sum(k["dram_bytes_per_image"] for k in tj["kernels"].values())
                    traffic_src = cand
                    break
        flops = 2.0 * macs * H * W * imgs_per_launch
        achieved = flops / (avg_ms * 1e-3) / 1e12
        peak = peaks["tf_sustained"]
        conv_total = sum(conv_ms)
        fwd_alg_bytes_per_image = 60.0 * H * W  # 4 fp32 inputs + 1 fp32 output (SURVEY 8d)
        roofline = {
            "bound": "tensor", "kernel": "+".join(fused), "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
            "frac": achieved / peak, "traffic": traffic,
            "traffic_note": f"DRAM bytes per launch from the committed ncu --set full capture (profiles/{traffic_src})",
            # FUSED definition (SURVEY 8d): the whole forward is one logical op of 60 B/px; a layer's share is
            # its share of the forward's FLOPs.  Everything above that is intermediate round trips through HBM.
            "algorithmic_bytes_per_launch": fwd_alg_bytes_per_image * imgs_per_launch * macs / TOTAL_MACS,
            "forward_dram_bytes_per_image": {"measured_ncu": traffic_total_per_image,
                                             "algorithmic_fused": fwd_alg_bytes_per_image,
                                             "ratio": (traffic_total_per_image / fwd_alg_bytes_per_image
                                                       if traffic_total_per_image else None)},
            "peak_source": peaks["source"] + ", bf16 dense sustained (kernel timed inside a long step)",
            "avg_launch_ms": avg_ms, "launches_timed": n_launch, "share_of_step": conv_ms[top] / (ms_per_step * args.steps),
            "forward_all_convs": {"achieved": 2.0 * TOTAL_MACS * H * W * B * args.steps / (conv_total * 1e-3) / 1e12,
                                  "unit": "TFLOP/s", "ms_per_step": conv_total / args.steps},
            # BASELINE.json's "fused-fwd HBM GB/s vs roofline": the forward's API-faithful bytes (4 fp32 inputs +
            # 1 fp32 output = 60 B/px, SURVEY 8d) over the time of all convolutions.  The forward is a dense
            # contraction (36 kFLOP/B), so this figure cannot come near the HBM roofline; reported for completeness.
            "forward_hbm_algorithmic": {
                "achieved": 60.0 * H * W * B * args.steps / (conv_total * 1e-3) / 1e9, "peak": peaks["hbm_gbs"],
                "unit": "GB/s", "frac": 60.0 * H * W * B * args.steps / (conv_total * 1e-3) / 1e9 / peaks["hbm_gbs"],
                "bytes_per_px": 60, "note": "tensor-bound, not HBM-bound: see bound/frac above"},
            "preprocess_apply_hbm": None,
        }
        if slot_cnt[21]:
            apply_ms = slot_ms[21] / slot_cnt[21]
            # folded path: 3 B/px read + 32 B/px of first-layer operand planes written (fp32 mode: 3 + 48)
            bpp = 51.0 if mode == _lib.MODE_FP32_SIMT else 35.0
            gbs = bpp * H * W * (args.steps * B / slot_cnt[21]) / (apply_ms * 1e-3) / 1e9
            roofline["preprocess_apply_hbm"] = {"achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                                "frac": gbs / peaks["hbm_gbs"], "bytes_per_px": bpp}
        config = workload_config(args, world)  # identical in both arms
        detail = {"mode": args.mode, "images_per_pass": nb,
                  "collective": ("none" if world == 1 else
                                 "all-gather of the uint8 output, pass by pass: " +
                                 ("NVLink stores into every rank's buffer (CUDA IPC) from the kernel that writes the output"
                                  if fused_gather else "copy-engine pushes into peer memory over NVLink (CUDA IPC)"
                                  if isinstance(gather, PeerGather) else "NCCL all_gather") +
                                 ("; per step one flag word pushed to every peer and a stream wait-value on theirs "
                                  "(no kernel)" if isinstance(gather, PeerGather) else ""))}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None,
            "dtype": {_lib.MODE_FP32_SIMT: "f32", _lib.MODE_BF16X3: "bf16x3 (3-term bf16 split operands, fp32 accumulate)"}.get(
                mode, "bf16 + fp8 corrections (v = hi + lo: hi x hi in bf16, both correction terms of the heavy "
                      "layers as one e4m3 MMA; fp32 accumulate; 3-term bf16 elsewhere)"),
            "data": "synthetic",
            "config": config,
            "detail": detail,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms / args.steps,
                    "h2d_bytes_per_step": int(pins[0][0].numel()), "d2h_bytes_per_step": int(pins[0][1].numel()),
                    "api": "Enhancer.submit/wait (pinned host uint8 in/out; H2D, kernels, D2H pipelined per pass on three streams)"},
            "gpu_launches": int(launches),
            "parity": parity,
            "roofline": roofline,
            "kernel_ms_per_step": {name: round(slot_ms[i] / args.steps, 4) for i, name in enumerate(
                names_by_slot + ["pack", "gate", "pre_stats", "pre_luts", "pre_apply", "post"]) if slot_cnt[i]},
            "kernel_tflops": {name: round(2.0 * macs_by_slot[i] * H * W * B * args.steps / (slot_ms[i] * 1e-3) / 1e12, 1)
                              for i, name in enumerate(names_by_slot) if slot_cnt[i] and slot_ms[i] > 0 and macs_by_slot[i]},
            "cpu_baseline": cpu_baseline,
        }
        if dumped is not None:
            line["dump_outputs"] = dumped
        if world > 1:
            line["multi_gpu"] = {
                "per_rank_ms_per_step": [round(v / args.steps, 3) for v in per_rank_ms],
                "per_rank_ms_per_step_e2e": [round(v / args.steps, 3) for v in e2e_per_rank],
                "ms_per_step_without_collective": nogather_ms / args.steps,
                "collective_cost_ms_per_step": ms_per_step - nogather_ms / args.steps,
                "gathered_equals_local": gather_ok,
                "gather_bytes_received_per_step": int((world - 1) * B * H * W * 3),
            }
        print(json.dumps(line), flush=True)
    if world > 1:
        if isinstance(gather, PeerGather):
            gather.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
