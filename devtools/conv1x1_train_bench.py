"""Times the head's 1x1 convolutions in training: forward, dgrad and wgrad (+ bias gradient) of conv1x1 (libcdrhead, f16x2
tensor cores) against cuDNN (F.conv2d + torch.autograd.grad, TF32 off and on), per layer at the training shape (64
images per view: forward_train runs the fusion out_layer and the decoder once per view), and the whole
CDRNet(trainable=True) forward_train + backward step at torch's default TF32 flags with the 1x1 convs on cuDNN and on
libcdrhead, alternated in one run.  CUDA events; the L2 is overwritten before every timed repetition.  Prints one JSON
line and writes it to --out.

    python devtools/conv1x1_train_bench.py [--reps 20] [--step-reps 5] [--out profiles/conv1x1_train_b200.json]
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
from fast_3d_human_pose_estimation_b200 import autograd as AG   # noqa: E402

# Cin, Cout, H, W at the default fusion widths (fusion_hid_ch1 = 300, fusion_hid_ch2 = 400)
LAYERS = {"CF.conv_layer1": (2048, 300, 8, 8), "CF.conv_layer2.0": (800, 400, 8, 8),
          "CF.conv_layer2.3": (400, 400, 8, 8), "CF.out_layer": (300, 2048, 8, 8),
          "decoder.final_layer": (256, 19, 64, 64)}


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
    cin, cout, h, wd = LAYERS[name]
    flop = 2.0 * n * cin * cout * h * wd
    x = torch.randn((n, cin, h, wd), device="cuda")
    w = torch.randn((cout, cin, 1, 1), device="cuda") * cin ** -0.5
    bias = torch.randn((cout,), device="cuda") * 0.1
    dy = torch.randn((n, cout, h, wd), device="cuda")
    L = _lib.lib()
    sb, wb = C.c_size_t(), C.c_size_t()
    _lib.check(L.cdr_conv1x1_train_workspace_bytes(n, cin, cout, h, wd, C.byref(sb), C.byref(wb)))
    saved = torch.empty(sb.value, dtype=torch.uint8, device="cuda")
    ws = torch.empty(wb.value, dtype=torch.uint8, device="cuda")
    y = torch.empty((n, cout, h, wd), device="cuda")
    dx = torch.empty_like(x)
    dw = torch.empty_like(w)
    db = torch.empty_like(bias)
    st = _lib.current_stream_ptr()
    P = _lib.ptr

    def fwd():
        _lib.check(L.cdr_conv1x1_train_forward(P(x), P(w), P(bias), n, cin, cout, h, wd, P(y), P(saved), sb.value, P(ws),
                                               wb.value, st))

    def bwd(gx, gw, gb):
        return lambda: _lib.check(L.cdr_conv1x1_train_backward(P(saved), P(w), P(dy), n, cin, cout, h, wd, P(gx), P(gw),
                                                               P(gb), P(ws), wb.value, st))
    fwd()
    # dgrad / wgrad times include the dy encoding (NCHW fp32 -> fp16 planes), paid once per backward; wgrad includes
    # the bias gradient on both sides
    ours = {"forward_ms": timed(fwd, reps, flush), "dgrad_ms": timed(bwd(dx, None, None), reps, flush),
            "wgrad_ms": timed(bwd(None, dw, db), reps, flush), "backward_all_ms": timed(bwd(dx, dw, db), reps, flush)}
    res = {"shape": {"n": n, "cin": cin, "cout": cout, "h": h, "w": wd}, "flop_per_pass": flop, "libcdrhead_f16x2": ours}
    for tf32 in (False, True):
        torch.backends.cudnn.allow_tf32 = tf32
        xr, wg, bg = x.clone().requires_grad_(True), w.clone().requires_grad_(True), bias.clone().requires_grad_(True)
        yd = F.conv2d(xr, w, bias)                  # graph for the data gradient only
        yw = F.conv2d(x, wg, bg)                    # graph for the weight and bias gradients only
        ya = F.conv2d(xr, wg, bg)
        r = {"forward_ms": timed(lambda: F.conv2d(x, w, bias), reps, flush),
             "dgrad_ms": timed(lambda: torch.autograd.grad(yd, xr, dy, retain_graph=True), reps, flush),
             "wgrad_ms": timed(lambda: torch.autograd.grad(yw, (wg, bg), dy, retain_graph=True), reps, flush),
             "backward_all_ms": timed(lambda: torch.autograd.grad(ya, (xr, wg, bg), dy, retain_graph=True), reps, flush)}
        res["cudnn_tf32_on" if tf32 else "cudnn_tf32_off"] = r
        del xr, wg, bg, yd, yw, ya
    torch.backends.cudnn.allow_tf32 = True
    for k in ("libcdrhead_f16x2", "cudnn_tf32_off", "cudnn_tf32_on"):
        for p in ("forward", "dgrad", "wgrad"):
            res[k][p + "_tflops"] = round(flop / (res[k][p + "_ms"] * 1e-3) / 1e12, 2)
    # the timed outputs against cuDNN with TF32 off (the fp64 comparison is tests/test_gpu_conv1x1_train.py)
    torch.backends.cudnn.allow_tf32 = False
    fwd()
    bwd(dx, dw, db)()
    xr, wr, br = x.clone().requires_grad_(True), w.clone().requires_grad_(True), bias.clone().requires_grad_(True)
    yr = F.conv2d(xr, wr, br)
    gx, gw, gb = torch.autograd.grad(yr, (xr, wr, br), dy)
    torch.backends.cudnn.allow_tf32 = True
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max())     # noqa: E731
    res["max_rel_diff_vs_cudnn_fp32"] = {"y": rel(y, yr.detach()), "dx": rel(dx, gx), "dw": rel(dw, gw), "db": rel(db, gb)}
    return res


def train_step(b, reps):
    """forward_train + backward of CDRNet(trainable=True) at B pairs and torch's default TF32 flags, the head's 1x1
    convs on cuDNN ("before") and on libcdrhead ("after"), alternated"""
    torch.manual_seed(0)
    m = pkg.CDRNet(synth.make_cfg(50, 19), trainable=True).cuda().train()
    imgs = [x.cuda() for x in synth.make_images(b, seed=1)]
    cams = synth.make_cameras(b, seed=2)
    Ps = [torch.from_numpy(cams["P_l"]).cuda(), torch.from_numpy(cams["P_r"]).cuda()]
    ours = AG.conv1x1

    def cudnn(x, w, bias=None):
        return F.conv2d(x, w, bias)

    def step():
        m.zero_grad(set_to_none=True)
        kps, xyz = m(imgs, Ps)
        (kps[0].square().mean() + kps[1].square().mean() + xyz.abs().mean()).backward()

    times = {"before_cudnn": [], "after_libcdrhead": []}
    try:
        for rep in range(reps + 1):
            for key, op in (("before_cudnn", cudnn), ("after_libcdrhead", ours)):
                AG.conv1x1 = op
                torch.cuda.synchronize()
                a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                step()
                e.record()
                e.synchronize()
                if rep:                                                    # rep 0 warms both up
                    times[key].append(a.elapsed_time(e))
    finally:
        AG.conv1x1 = ours
    return {"batch_pairs": b, "cudnn_allow_tf32": torch.backends.cudnn.allow_tf32,
            "matmul_allow_tf32": torch.backends.cuda.matmul.allow_tf32,
            **{k: {"median_ms": statistics.median(v), "all_ms": [round(t, 2) for t in v]} for k, v in times.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=64, help="images per call (per view)")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--step-batch", type=int, default=64)
    ap.add_argument("--step-reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "conv1x1_train_b200.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("conv1x1_train_bench: needs a CUDA device")
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
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
