"""Times the encoder's 3x3 convolutions in training: forward, dgrad and wgrad of conv3x3 (libcdrhead, f16x2 tensor cores)
against cuDNN (F.conv2d + torch.autograd.grad, TF32 off and on), for every distinct 3x3 conv of ResNet-50 at 256 x 256
images and 64 images per call (forward_train runs the encoder once per view), and the whole CDRNet(trainable=True)
forward_train + backward step at torch's default TF32 flags with the encoder on libcdrhead (CDRNet(train_encoder_on_library=True):
ResNet.forward_train) and on torch (the default: cuDNN convs, torch BatchNorm), alternated in one run.  Then, in a separate profiled
step, the device time of the library encoder's step split into GEMMs, amax / fp16-plane encode passes, weight packs,
wgrad reductions and the rest.  CUDA events; the L2 is overwritten before every timed repetition of a single conv.
Prints one JSON line and writes it to --out.

    python devtools/conv3x3_train_bench.py [--reps 20] [--step-reps 5] [--out profiles/conv3x3_train_b200.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch                                   # noqa: E402
import torch.nn.functional as F                # noqa: E402

import fast_3d_human_pose_estimation_b200 as pkg          # noqa: E402
from fast_3d_human_pose_estimation_b200 import _lib, synth   # noqa: E402

# C, input H = W, stride: the distinct 3x3 convs of ResNet-50 at 256 x 256 images
LAYERS = {"layer1": (64, 64, 1), "layer2.0": (128, 64, 2), "layer2": (128, 32, 1), "layer3.0": (256, 32, 2),
          "layer3": (256, 16, 1), "layer4.0": (512, 16, 2), "layer4": (512, 8, 1)}


def timed(fn, reps, flush):
    """median ms of fn over reps, each preceded (outside the timed window) by an L2 overwrite"""
    fn()
    fn()                                        # first launches: module load, algorithm choice
    ts = []
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts)


def layer(name, n, reps, flush):
    c, h, s = LAYERS[name]
    ho = h // s
    flop = 2.0 * n * c * c * 9 * ho * ho
    x = torch.randn((n, c, h, h), device="cuda")
    w = torch.randn((c, c, 3, 3), device="cuda") * (9 * c) ** -0.5
    dy = torch.randn((n, c, ho, ho), device="cuda")
    L = _lib.lib()
    sb, wb = C.c_size_t(), C.c_size_t()
    _lib.check(L.cdr_conv3x3_train_workspace_bytes(n, c, c, h, h, s, C.byref(sb), C.byref(wb)))
    saved = torch.empty(sb.value, dtype=torch.uint8, device="cuda")
    ws = torch.empty(wb.value, dtype=torch.uint8, device="cuda")
    y = torch.empty((n, c, ho, ho), device="cuda")
    dx = torch.empty_like(x)
    dw = torch.empty_like(w)
    st = _lib.current_stream_ptr()
    P = _lib.ptr

    def fwd():
        _lib.check(L.cdr_conv3x3_train_forward(P(x), P(w), n, c, c, h, h, s, P(y), P(saved), sb.value, P(ws), wb.value,
                                               st))

    def bwd(gx, gw):
        return lambda: _lib.check(L.cdr_conv3x3_train_backward(P(saved), P(w), P(dy), n, c, c, h, h, s, P(gx), P(gw),
                                                               P(ws), wb.value, st))
    fwd()
    # forward times include the x encoding, dgrad / wgrad times the dy encoding (NCHW fp32 -> fp16 planes), paid once
    # per call
    ours = {"forward_ms": timed(fwd, reps, flush), "dgrad_ms": timed(bwd(dx, None), reps, flush),
            "wgrad_ms": timed(bwd(None, dw), reps, flush), "backward_all_ms": timed(bwd(dx, dw), reps, flush)}
    res = {"shape": {"n": n, "cin": c, "cout": c, "h": h, "w": h, "stride": s}, "flop_per_pass": flop,
           "libcdrhead_f16x2": ours}
    for tf32 in (False, True):
        torch.backends.cudnn.allow_tf32 = tf32
        xr, wg = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
        yd = F.conv2d(xr, w, stride=s, padding=1)        # graph for the data gradient only
        yw = F.conv2d(x, wg, stride=s, padding=1)        # graph for the weight gradient only
        ya = F.conv2d(xr, wg, stride=s, padding=1)
        r = {"forward_ms": timed(lambda: F.conv2d(x, w, stride=s, padding=1), reps, flush),
             "dgrad_ms": timed(lambda: torch.autograd.grad(yd, xr, dy, retain_graph=True), reps, flush),
             "wgrad_ms": timed(lambda: torch.autograd.grad(yw, wg, dy, retain_graph=True), reps, flush),
             "backward_all_ms": timed(lambda: torch.autograd.grad(ya, (xr, wg), dy, retain_graph=True), reps, flush)}
        res["cudnn_tf32_on" if tf32 else "cudnn_tf32_off"] = r
        del xr, wg, yd, yw, ya
    torch.backends.cudnn.allow_tf32 = True
    for k in ("libcdrhead_f16x2", "cudnn_tf32_off", "cudnn_tf32_on"):
        for p in ("forward", "dgrad", "wgrad"):
            res[k][p + "_tflops"] = round(flop / (res[k][p + "_ms"] * 1e-3) / 1e12, 2)
    # the timed outputs against cuDNN with TF32 off (the fp64 comparison is tests/test_gpu_conv3x3_train.py)
    torch.backends.cudnn.allow_tf32 = False
    fwd()
    bwd(dx, dw)()
    xr, wr = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
    yr = F.conv2d(xr, wr, stride=s, padding=1)
    gx, gw = torch.autograd.grad(yr, (xr, wr), dy)
    torch.backends.cudnn.allow_tf32 = True
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max())     # noqa: E731
    res["max_rel_diff_vs_cudnn_fp32"] = {"y": rel(y, yr.detach()), "dx": rel(dx, gx), "dw": rel(dw, gw)}
    return res


def _model_and_step(b):
    torch.manual_seed(0)
    m = pkg.CDRNet(synth.make_cfg(50, 19), trainable=True).cuda().train()
    imgs = [x.cuda() for x in synth.make_images(b, seed=1)]
    cams = synth.make_cameras(b, seed=2)
    Ps = [torch.from_numpy(cams["P_l"]).cuda(), torch.from_numpy(cams["P_r"]).cuda()]

    def step():
        m.zero_grad(set_to_none=True)
        kps, xyz = m(imgs, Ps)
        (kps[0].square().mean() + kps[1].square().mean() + xyz.abs().mean()).backward()
    return m, step


def _encoder_on_library(m, on):
    """the model's own switch: CDRNet(train_encoder_on_library=...)"""
    m.train_encoder_on_library = on


def train_step(b, reps):
    """forward_train + backward of CDRNet(trainable=True) at B pairs and torch's default TF32 flags, the encoder on torch
    ("before": cuDNN convs, torch BatchNorm) and on libcdrhead ("after"), alternated"""
    m, step = _model_and_step(b)
    times = {"before_torch_encoder": [], "after_libcdrhead_encoder": []}
    for rep in range(reps + 1):
        for key, lib in (("before_torch_encoder", False), ("after_libcdrhead_encoder", True)):
            _encoder_on_library(m, lib)
            torch.cuda.synchronize()
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step()
            e.record()
            e.synchronize()
            if rep:                                                    # rep 0 warms both up
                times[key].append(a.elapsed_time(e))
    _encoder_on_library(m, False)
    return {"batch_pairs": b, "cudnn_allow_tf32": torch.backends.cudnn.allow_tf32,
            "matmul_allow_tf32": torch.backends.cuda.matmul.allow_tf32,
            **{k: {"median_ms": statistics.median(v), "all_ms": [round(t, 2) for t in v]} for k, v in times.items()}}


def _category(name):
    if "tap_gemm_tc_kernel" in name:
        return "gemm"
    if "amax" in name or "rows_f16p" in name or "nchw_to_rows16" in name:
        return "amax_and_encode"
    if "pack_rows_f16" in name:
        return "weight_pack"
    if "wgrad_reduce" in name:
        return "wgrad_reduce"
    if "bn_train" in name or "batch_norm" in name.lower() or "bn_" in name:
        return "batchnorm"
    return "other"


def step_profile(b):
    """device time of one library-encoder step by kernel category (torch.profiler, a run of its own)"""
    from torch.profiler import ProfilerActivity, profile
    m, step = _model_and_step(b)
    _encoder_on_library(m, True)
    step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    cats = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t <= 0:
            continue
        k = _category(ev.key)
        cats[k] = cats.get(k, 0.0) + t / 1e3
    total = sum(cats.values())
    return {"batch_pairs": b, "device_ms_by_category": {k: round(v, 3) for k, v in sorted(cats.items())},
            "share": {k: round(v / total, 4) for k, v in sorted(cats.items())}, "device_ms_total": round(total, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=64, help="images per call (per view)")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--step-batch", type=int, default=64)
    ap.add_argument("--step-reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "conv3x3_train_b200.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("conv3x3_train_bench: needs a CUDA device")
    torch.cuda.set_device(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"nvidia-smi unavailable: {e}"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # 256 MB > the 126 MB L2
    out = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": q,
           "layers": {k: layer(k, a.n, a.reps, flush) for k in LAYERS}}
    del flush
    if a.step_reps > 0:
        out["train_step"] = train_step(a.step_batch, a.step_reps)
        out["train_step_profile_libcdrhead_encoder"] = step_profile(a.step_batch)
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
