"""Times the decoder's transposed convolutions in training: forward, dgrad and wgrad of conv_transpose2d (libcdrhead,
f16x2 tensor cores) against cuDNN (F.conv_transpose2d + torch.autograd.grad, TF32 off and on), per layer at the training
shape (64 images per view: forward_train runs the decoder once per view), and the whole CDRNet(trainable=True)
forward_train + backward step with the decoder's convolutions on cuDNN and on libcdrhead, alternated in one run.
CUDA events; the L2 is overwritten before every timed repetition.  Prints one JSON line and writes it to --out.

    python devtools/deconv_train_bench.py [--reps 20] [--step-reps 5] [--out profiles/deconv_train_b200.json]
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

LAYERS = {"deconv1": (2048, 256, 8), "deconv2": (256, 256, 16), "deconv3": (256, 256, 32)}


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
    cin, cout, h = LAYERS[name]
    flop = 2.0 * n * cin * cout * 16 * h * h
    x = torch.randn((n, cin, h, h), device="cuda")
    w = torch.randn((cin, cout, 4, 4), device="cuda") * (cin * 4) ** -0.5
    dy = torch.randn((n, cout, 2 * h, 2 * h), device="cuda")
    L = _lib.lib()
    sb, wb = C.c_size_t(), C.c_size_t()
    _lib.check(L.cdr_deconv_train_workspace_bytes(n, cin, cout, h, h, C.byref(sb), C.byref(wb)))
    saved = torch.empty(sb.value, dtype=torch.uint8, device="cuda")
    ws = torch.empty(wb.value, dtype=torch.uint8, device="cuda")
    y = torch.empty((n, cout, 2 * h, 2 * h), device="cuda")
    dx = torch.empty_like(x)
    dw = torch.empty_like(w)
    st = _lib.current_stream_ptr()
    P = _lib.ptr

    def fwd():
        _lib.check(L.cdr_deconv_train_forward(P(x), P(w), n, cin, cout, h, h, P(y), P(saved), sb.value, P(ws), wb.value, st))

    def bwd(gx, gw):
        return lambda: _lib.check(L.cdr_deconv_train_backward(P(saved), P(w), P(dy), n, cin, cout, h, h, P(gx), P(gw),
                                                              P(ws), wb.value, st))
    fwd()
    ours = {"forward_ms": timed(fwd, reps, flush), "dgrad_ms": timed(bwd(dx, None), reps, flush),
            "wgrad_ms": timed(bwd(None, dw), reps, flush)}
    # dgrad / wgrad times include the shared dy encoding (NCHW fp32 -> fp16 planes), paid once per backward
    ours["backward_both_ms"] = timed(bwd(dx, dw), reps, flush)
    res = {"shape": {"n": n, "cin": cin, "cout": cout, "h": h, "w": h}, "flop_per_pass": flop, "libcdrhead_f16x2": ours}
    for tf32 in (False, True):
        torch.backends.cudnn.allow_tf32 = tf32
        xr, wg = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
        yd = F.conv_transpose2d(xr, w, stride=2, padding=1)          # graph for the data gradient only
        yw = F.conv_transpose2d(x, wg, stride=2, padding=1)          # graph for the weight gradient only
        r = {"forward_ms": timed(lambda: F.conv_transpose2d(x, w, stride=2, padding=1), reps, flush),
             "dgrad_ms": timed(lambda: torch.autograd.grad(yd, xr, dy, retain_graph=True), reps, flush),
             "wgrad_ms": timed(lambda: torch.autograd.grad(yw, wg, dy, retain_graph=True), reps, flush)}
        res["cudnn_tf32_on" if tf32 else "cudnn_tf32_off"] = r
        del xr, wg, yd, yw
    torch.backends.cudnn.allow_tf32 = True
    for k in ("libcdrhead_f16x2", "cudnn_tf32_off", "cudnn_tf32_on"):
        for p in ("forward", "dgrad", "wgrad"):
            res[k][p + "_tflops"] = round(flop / (res[k][p + "_ms"] * 1e-3) / 1e12, 1)
    # the timed outputs against cuDNN with TF32 off (the fp64 comparison is tests/test_gpu_deconv_train.py)
    torch.backends.cudnn.allow_tf32 = False
    fwd()
    bwd(dx, dw)()
    xr, wr = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
    yr = F.conv_transpose2d(xr, wr, stride=2, padding=1)
    gx, gw = torch.autograd.grad(yr, (xr, wr), dy)
    torch.backends.cudnn.allow_tf32 = True
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max())     # noqa: E731
    res["max_rel_diff_vs_cudnn_fp32"] = {"y": rel(y, yr.detach()), "dx": rel(dx, gx), "dw": rel(dw, gw)}
    return res


def train_step(b, reps):
    """forward_train + backward of CDRNet(trainable=True) at B pairs, decoder convs on cuDNN ("before") and on
    libcdrhead ("after"), alternated"""
    torch.manual_seed(0)
    m = pkg.CDRNet(synth.make_cfg(50, 19), trainable=True).cuda().train()
    imgs = [x.cuda() for x in synth.make_images(b, seed=1)]
    cams = synth.make_cameras(b, seed=2)
    Ps = [torch.from_numpy(cams["P_l"]).cuda(), torch.from_numpy(cams["P_r"]).cuda()]
    ours = AG.conv_transpose2d

    def cudnn(x, w):
        return F.conv_transpose2d(x, w, stride=2, padding=1)

    def step():
        m.zero_grad(set_to_none=True)
        kps, xyz = m(imgs, Ps)
        (kps[0].square().mean() + kps[1].square().mean() + xyz.abs().mean()).backward()

    times = {"before_cudnn": [], "after_libcdrhead": []}
    try:
        for rep in range(reps + 1):
            for key, op in (("before_cudnn", cudnn), ("after_libcdrhead", ours)):
                AG.conv_transpose2d = op
                torch.cuda.synchronize()
                a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                step()
                e.record()
                e.synchronize()
                if rep:                                                    # rep 0 warms both up
                    times[key].append(a.elapsed_time(e))
    finally:
        AG.conv_transpose2d = ours
    return {"batch_pairs": b, "cudnn_allow_tf32": torch.backends.cudnn.allow_tf32,
            "matmul_allow_tf32": torch.backends.cuda.matmul.allow_tf32,
            **{k: {"median_ms": statistics.median(v), "all_ms": [round(t, 2) for t in v]} for k, v in times.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=64, help="images per decoder call (per view)")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--step-batch", type=int, default=64)
    ap.add_argument("--step-reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "deconv_train_b200.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("deconv_train_bench: needs a CUDA device")
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
