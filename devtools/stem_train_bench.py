"""Times the encoder's stem in training: the 7x7 stride-2 conv's forward and weight gradient (stem_conv: libcdrhead,
fp16 hi/lo operands on mma.sync) and the 3x3 stride-2 max-pool's forward and backward (max_pool3x3) against torch
(cuDNN F.conv2d + torch.autograd.grad, TF32 off and on; F.max_pool2d), at N images of 256 x 256 per call (forward_train
runs the encoder once per view); then the whole CDRNet(trainable=True, train_encoder_on_library=True) forward_train +
backward step at torch's default TF32 flags with the stem on torch and on libcdrhead (train_stem_on_library), alternated
in one run; then, in a separate profiled step with the stem on libcdrhead, every device kernel whose name marks it as a
torch / cuDNN convolution or pooling kernel (there should be none).  CUDA events; the L2 is overwritten before every
timed repetition of a single op.  Prints one JSON line and writes it to --out.

    python devtools/stem_train_bench.py [--n 64] [--reps 20] [--step-reps 5] [--out profiles/stem_train_b200.json]
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


def stem(n, reps, flush):
    h = w = 256
    ho, wo = h // 2, w // 2
    pixels = n * ho * wo
    x = torch.randn((n, 3, h, w), device="cuda")
    wt = torch.randn((64, 3, 7, 7), device="cuda") / 147 ** 0.5
    dy = torch.randn((n, 64, ho, wo), device="cuda")
    L = _lib.lib()
    sb, wb = C.c_size_t(), C.c_size_t()
    _lib.check(L.cdr_stem_train_workspace_bytes(n, 3, 64, h, w, C.byref(sb), C.byref(wb)))
    saved = torch.empty(sb.value, dtype=torch.uint8, device="cuda")
    ws = torch.empty(wb.value, dtype=torch.uint8, device="cuda")
    y = torch.empty((n, 64, ho, wo), device="cuda")
    dw = torch.empty_like(wt)
    st = _lib.current_stream_ptr()
    P = _lib.ptr

    def fwd():
        _lib.check(L.cdr_stem_train_forward(P(x), P(wt), n, 3, 64, h, w, P(y), P(saved), sb.value, P(ws), wb.value, st))

    def wgrad():
        _lib.check(L.cdr_stem_train_backward(P(saved), P(wt), P(dy), n, 3, 64, h, w, None, P(dw), P(ws), wb.value, st))
    # the forward includes x's amax and fp16-plane encode and the weight pack; the weight gradient dy's amax pass
    conv = {"libcdrhead_f16x2": {"forward_ms": timed(fwd, reps, flush), "wgrad_ms": timed(wgrad, reps, flush)}}
    for tf32 in (False, True):
        torch.backends.cudnn.allow_tf32 = tf32
        wg = wt.clone().requires_grad_(True)
        yw = F.conv2d(x, wg, stride=2, padding=3)
        conv["cudnn_tf32_on" if tf32 else "cudnn_tf32_off"] = {
            "forward_ms": timed(lambda: F.conv2d(x, wt, stride=2, padding=3), reps, flush),
            "wgrad_ms": timed(lambda: torch.autograd.grad(yw, wg, dy, retain_graph=True), reps, flush)}
        del wg, yw
    torch.backends.cudnn.allow_tf32 = True
    flop = 2.0 * pixels * 64 * 147
    for r in conv.values():
        for p in ("forward", "wgrad"):
            r[p + "_tflops_fp32_equivalent"] = round(flop / (r[p + "_ms"] * 1e-3) / 1e12, 2)
    # the timed outputs against cuDNN with TF32 off (the fp64 comparison is tests/test_gpu_stem_train.py)
    torch.backends.cudnn.allow_tf32 = False
    fwd()
    wgrad()
    wr = wt.clone().requires_grad_(True)
    yr = F.conv2d(x, wr, stride=2, padding=3)
    (gw,) = torch.autograd.grad(yr, (wr,), dy)
    torch.backends.cudnn.allow_tf32 = True
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max())     # noqa: E731
    conv["max_rel_diff_vs_cudnn_fp32"] = {"y": rel(y, yr.detach()), "dw": rel(dw, gw)}
    conv["bytes_floor"] = {"forward": 4 * (x.numel() + y.numel()), "wgrad_dy_twice": 8 * dy.numel()}
    del x, dy, saved, ws, yr

    # max-pool on the stem conv's output shape, post-ReLU
    a = torch.randn((n, 64, ho, wo), device="cuda").clamp_min_(0)
    py = torch.randn((n, 64, (ho - 1) // 2 + 1, (wo - 1) // 2 + 1), device="cuda")
    ar, ao = a.clone().requires_grad_(True), a.clone().requires_grad_(True)
    yt, yo = F.max_pool2d(ar, 3, 2, 1), pkg.max_pool3x3(ao)
    pool = {
        "libcdrhead": {"forward_ms": timed(lambda: pkg.max_pool3x3(a), reps, flush),
                       "backward_ms": timed(lambda: torch.autograd.grad(yo, ao, py, retain_graph=True), reps, flush)},
        "torch": {"forward_ms": timed(lambda: F.max_pool2d(a, 3, 2, 1), reps, flush),
                  "backward_ms": timed(lambda: torch.autograd.grad(yt, ar, py, retain_graph=True), reps, flush)},
        "bytes": {"libcdrhead_forward": 4 * a.numel() + 5 * py.numel(), "libcdrhead_backward": 4 * a.numel() + 5 * py.numel(),
                  "torch_forward": 4 * a.numel() + 12 * py.numel(), "torch_backward": 4 * a.numel() + 12 * py.numel()},
        "bits_equal_torch": bool(torch.equal(yt.detach().view(torch.int32), yo.detach().view(torch.int32)) and torch.equal(
            torch.autograd.grad(yt, ar, py, retain_graph=True)[0].view(torch.int32),
            torch.autograd.grad(yo, ao, py, retain_graph=True)[0].view(torch.int32)))}
    return {"shape": {"n": n, "h": h, "w": w}, "conv": conv, "maxpool": pool}


def _model_and_step(b):
    torch.manual_seed(0)
    m = pkg.CDRNet(synth.make_cfg(50, 19), trainable=True, train_encoder_on_library=True).cuda().train()
    imgs = [x.cuda() for x in synth.make_images(b, seed=1)]
    cams = synth.make_cameras(b, seed=2)
    Ps = [torch.from_numpy(cams["P_l"]).cuda(), torch.from_numpy(cams["P_r"]).cuda()]

    def step():
        m.zero_grad(set_to_none=True)
        kps, xyz = m(imgs, Ps)
        (kps[0].square().mean() + kps[1].square().mean() + xyz.abs().mean()).backward()
    return m, step


def train_step(b, reps):
    """forward_train + backward of CDRNet(trainable=True, train_encoder_on_library=True) at B pairs and torch's default
    TF32 flags, the stem on torch ("before") and on libcdrhead ("after", the model's train_stem_on_library), alternated"""
    m, step = _model_and_step(b)
    times = {"before_torch_stem": [], "after_libcdrhead_stem": []}
    for rep in range(reps + 1):
        for key, lib in (("before_torch_stem", False), ("after_libcdrhead_stem", True)):
            m.train_stem_on_library = lib
            torch.cuda.synchronize()
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step()
            e.record()
            e.synchronize()
            if rep:                                                    # rep 0 warms both up
                times[key].append(a.elapsed_time(e))
    return {"batch_pairs": b, "cudnn_allow_tf32": torch.backends.cudnn.allow_tf32,
            "matmul_allow_tf32": torch.backends.cuda.matmul.allow_tf32,
            **{k: {"median_ms": statistics.median(v), "all_ms": [round(t, 2) for t in v]} for k, v in times.items()}}


def torch_conv_pool_kernels(b):
    """names of the device kernels of one step with the stem on libcdrhead that are torch / cuDNN convolution or pooling
    kernels (torch.profiler, a run of its own)"""
    from torch.profiler import ProfilerActivity, profile
    m, step = _model_and_step(b)
    m.train_stem_on_library = True
    step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    names = sorted({ev.key for ev in prof.key_averages()})
    ours = ("tap_gemm", "stem_", "maxpool3x3_train", "wgrad_reduce", "pack_")
    marks = ("conv", "cudnn", "pool", "wgrad", "dgrad", "sm90_", "sm100_", "implicit", "winograd")
    hits = [k for k in names if any(t in k.lower() for t in marks) and not any(o in k for o in ours)]
    return {"batch_pairs": b, "kernels": len(names), "torch_conv_or_pool_kernels": hits}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=64, help="images per call (per view)")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--step-batch", type=int, default=64)
    ap.add_argument("--step-reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "stem_train_b200.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("stem_train_bench: needs a CUDA device")
    torch.cuda.set_device(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"nvidia-smi unavailable: {e}"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # 256 MB > the 126 MB L2
    out = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": q,
           "stem": stem(a.n, a.reps, flush)}
    del flush
    if a.step_reps > 0:
        out["train_step"] = train_step(a.step_batch, a.step_reps)
        out["train_step_profile_libcdrhead_stem"] = torch_conv_pool_kernels(a.step_batch)
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
