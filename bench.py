#!/usr/bin/env python
"""bench.py — CDRNet post-backbone hot path on B200 (contract: see task statement / DESIGN.md).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--batch B] [--precision fp32|bf16]

One "step" = one pass of the head (canonical fusion -> decoder -> soft-argmax -> DLT -> MPJPE
partial sums [-> all-gather when N>1]) over one batch of B synthetic stereo pairs per GPU.
N=1 workload = BASELINE.json configs[1]: "CDRNet head fp32 batch 64 stereo pairs on 1xB200".
Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "cdrnet_head_stereo_pairs_per_sec"
UNIT = "stereo pairs/s"
JOINTS = 19
# algorithmic work per stereo pair (SURVEY.md §8d)
FLOP_PER_PAIR = {"deconv1": 2147.5e6, "deconv2": 1073.7e6, "deconv3": 4295.0e6, "final_1x1": 79.7e6,
                 "deconv3_tail": 4295.0e6 + 79.7e6,      # fused deconv3 + final 1x1 (+ soft-argmax partials)
                 "cf_conv1": 157.3e6, "cf_conv2": 61.5e6, "cf_out": 157.3e6}
HEAD_FLOP_PER_PAIR = 7972.5e6
SOFTARGMAX_DLT_BYTES_PER_POSE = 623220.0


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "tflops_burst": p["bf16_tflops"],
                "tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback"}


def ncu_traffic():
    """DRAM bytes per launch from the latest committed ncu capture (profiles/rNN_traffic.json)."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))
    return json.load(open(files[-1])) if files else {}


class ClockSampler:
    """SM clock / power / throttle reasons DURING the timed region (B200_PROFILING.md).  Sampled through NVML
    (nvidia-ml-py — the library nvidia-smi itself reads) from a thread every ~2 ms, because the timed region of a
    20-step run lasts ~30 ms and `nvidia-smi -lms` cannot loop faster than ~20 ms; falls back to the nvidia-smi
    loop when NVML cannot be loaded."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index, period_ms=2.0):
        self.index, self.rows, self.proc, self.period = index, [], None, period_ms / 1e3
        self.mode, self._stop, self._thread = None, threading.Event(), None

    @staticmethod
    def _nvml_index(local):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis and all(v.strip().isdigit() for v in vis.split(",")) and local < len(vis.split(",")):
            return int(vis.split(",")[local])
        return local

    def start(self):
        try:
            import pynvml as N
            N.nvmlInit()
            h = N.nvmlDeviceGetHandleByIndex(self._nvml_index(self.index))
            mx = float(N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM))
            bits = [(getattr(N, "nvmlClocksEventReasonHwSlowdown", 0x8), "hw_slowdown"),
                    (getattr(N, "nvmlClocksEventReasonHwThermalSlowdown", 0x40), "hw_thermal_slowdown"),
                    (getattr(N, "nvmlClocksEventReasonSwThermalSlowdown", 0x20), "sw_thermal_slowdown"),
                    (getattr(N, "nvmlClocksEventReasonSwPowerCap", 0x4), "sw_power_cap")]
            get_reasons = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
            N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM); get_reasons(h)         # fail here, not in the thread

            def loop():
                while not self._stop.is_set():
                    t = time.perf_counter()
                    try:
                        sm = float(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM))
                        r = int(get_reasons(h))
                        pw = N.nvmlDeviceGetPowerUsage(h) / 1e3
                        self.rows.append((t, sm, mx, pw, [n for b, n in bits if r & b]))
                    except Exception:
                        pass
                    rest = self.period - (time.perf_counter() - t)
                    if rest > 0:
                        time.sleep(rest)
            self._thread = threading.Thread(target=loop, daemon=True)
            self._thread.start()
            self.mode = "nvml"
            return
        except Exception:
            self.mode = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self._nvml_index(self.index))], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            self.mode, self.period = "nvidia-smi", 0.02
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            c = [x.strip() for x in line.split(",")]
            try:
                self.rows.append((time.perf_counter(), float(c[1]), float(c[2]), float(c[3]),
                                  [n for n, v in zip(self.NAMES, c[5:9]) if v.lower().startswith("active")]))
            except Exception:
                continue

    @property
    def running(self):
        return self.mode is not None

    def stop(self, t0=None, t1=None):
        """Summarise the samples taken inside the host-time window [t0, t1] (the timed region); the sampler is
        started before the warm-up so that it is already streaming when the region begins."""
        if self.mode is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML / nvidia-smi"], "samples": 0}
        time.sleep(2 * self.period)
        self._stop.set()
        if self.proc is not None:
            self.proc.terminate()
        rows = [r for r in self.rows if t0 is None or (t0 <= r[0] <= t1 + self.period)]
        window = "timed region"
        if not rows:                      # region shorter than one sampling period: nearest samples around it
            rows = [r for r in self.rows if t0 - 0.1 <= r[0] <= t1 + 0.1] or self.rows[-3:]
            window = "nearest samples (region shorter than the sampling period)"
        sm = [r[1] for r in rows]
        reasons = sorted({n for r in rows for n in r[4]})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(r[2] for r in rows) if rows else None,
                "reasons": reasons, "samples": len(sm), "power_w_max": max(r[3] for r in rows) if rows else None,
                "sm_mhz_min": min(sm) if sm else None, "window": window, "period_ms": 1e3 * self.period,
                "source": self.mode}


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


# ----------------------------------------------------------------------------------------------
def bench_config(batch, world):
    """The `config` object of the JSON line — ONE function for `--impl ours` and `--impl reference`, so the driver's
    same_config check compares like with like.  Run-specific facts (host binding, CPU model, the reference arm's
    bounded sample) live in other keys."""
    return {"workload": ("CDRNet head (post-encoder) fp32 batch 64 stereo pairs per GPU, BASELINE configs[1]"
                         if batch == 64 else f"CDRNet head (post-encoder) fp32 batch {batch} stereo pairs per GPU"),
            "pairs_per_gpu": batch, "global_pairs": batch * world, "joints": JOINTS, "views": 2,
            "weights": "seeded random init (final_layer x0.1)",
            "inputs": "seeded synthetic encoder latents (B,2048,8,8) x2 + per-sample 90-degree stereo rigs",
            "l2": "flushed between steps (256 MB write)",
            "collective": "1 all-gather of (B,19,3)+32 B per step" if world > 1 else "none",
            "parallelism": f"dp{world}"}


def oracle_head_runner(batch):
    """CPU arm, kind "port": the oracle port (oracle/cdr_oracle.py — the reference's own torch calls on a
    state_dict) of the same head on the same synthetic inputs, fp32, all host threads."""
    from oracle import cdr_oracle as O
    from fast_3d_human_pose_estimation_b200 import synth
    sd = synth.make_head_state_dict(seed=0, calibrated=True)
    feats = synth.make_features(batch, seed=1)
    cams = synth.make_cameras(batch, seed=2)
    gt = synth.make_gt(cams, seed=3)
    Ps = [torch.from_numpy(cams["P_l"]), torch.from_numpy(cams["P_r"])]

    def step():
        with torch.no_grad():
            p2, p3 = O.head_forward(sd, feats, Ps)
        return O.calc_mpjpe([x.numpy() for x in p2], p3.numpy(), gt["gt3d"], gt["gt2d_l"], gt["gt2d_r"], gt["vis"])
    return step


def reference_head_runner(batch):
    """CPU arm, kind "reference": the UNMODIFIED reference (oracle/refload.py: /root/reference, or its verbatim
    git-ignored copy baseline/_ref/ on the GPU box) through its own public API — ``CDRNet.forward`` (models/cdrnet.py:
    224-268) with the encoder replaced by a stub that returns the given latents, then ``calc_mpjpe``
    (models/metrics.py:65-97) — on the same weights and inputs as the GPU arm.  None when it is not present."""
    from oracle import refload
    if not refload.available():
        return None
    from fast_3d_human_pose_estimation_b200 import synth
    ref = refload.load()
    sd = synth.make_head_state_dict(seed=0, calibrated=True)
    feats = synth.make_features(batch, seed=1)
    cams = synth.make_cameras(batch, seed=2)
    gt = synth.make_gt(cams, seed=3)
    Ps = [torch.from_numpy(cams["P_l"]), torch.from_numpy(cams["P_r"])]
    m = ref.CDRNet(synth.make_cfg(18, JOINTS))
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.startswith("encoder.") for k in missing)
    m.encoder = refload.feature_stub(feats)
    m = m.eval()
    imgs = [torch.zeros(batch, 3, 256, 256) for _ in range(2)]        # only their size is read (img_size, :229)

    def step():
        with torch.no_grad():
            p2, p3 = m(imgs, Ps)
        return ref.calc_mpjpe([x.numpy() for x in p2], p3.numpy(), gt["gt3d"], gt["gt2d_l"], gt["gt2d_r"], gt["vis"])
    return step


def reference_head_on_gpu(batch, dev, reps=5):
    """Context number SURVEY §8d asks for: the UNMODIFIED reference head (CDRNet.forward with the encoder stubbed, then the
    .cpu() + calc_mpjpe of inference.py:62-66,98-101) as torch runs it on the SAME GPU — eager ATen / cuDNN / cuSOLVER
    kernels, 19 batched SVDs — with TF32 off (the parity configuration) and on.  Not the reference arm: that is the CPU."""
    from oracle import refload
    if not refload.available():
        return None
    from fast_3d_human_pose_estimation_b200 import synth
    ref = refload.load()
    sd = synth.make_head_state_dict(seed=0, calibrated=True)
    feats = [f.to(dev) for f in synth.make_features(batch, seed=1)]
    cams = synth.make_cameras(batch, seed=2)
    gt = synth.make_gt(cams, seed=3)
    Ps = [torch.from_numpy(cams["P_l"]).to(dev), torch.from_numpy(cams["P_r"]).to(dev)]
    m = ref.CDRNet(synth.make_cfg(18, JOINTS))
    m.load_state_dict(sd, strict=False)
    m.encoder = refload.feature_stub(feats)
    m = m.to(dev).eval()
    imgs = [torch.zeros(batch, 3, 256, 256, device=dev) for _ in range(2)]

    def step():
        with torch.no_grad():
            p2, p3 = m(imgs, Ps)
        return ref.calc_mpjpe([x.cpu().numpy() for x in p2], p3.cpu().numpy(), gt["gt3d"], gt["gt2d_l"], gt["gt2d_r"], gt["vis"])
    out = {}
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    try:
        for tag, flag in (("tf32_off", False), ("tf32_on", True)):
            torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = flag
            step(); step()
            torch.cuda.synchronize()
            ts = []
            for _ in range(reps):
                t0 = time.perf_counter(); step(); torch.cuda.synchronize(); ts.append(time.perf_counter() - t0)
            out[tag] = {"pairs_per_s": batch / float(np.median(ts)), "ms_per_step": 1e3 * float(np.median(ts))}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
    out["what"] = (f"unmodified reference CDRNet.forward (encoder stubbed) + .cpu() + calc_mpjpe, {batch} pairs per step, torch "
                   f"{torch.__version__} eager on this GPU, wall clock incl. the result read-back")
    return out


def cpu_head_runner(batch):
    """(step, kind): the reference itself when it is present, else the oracle port."""
    try:
        step = reference_head_runner(batch)
        if step is not None:
            return step, "reference"
    except Exception as e:                                             # never lose the arm over an import problem
        sys.stderr.write(f"bench: reference not usable ({e!r}); timing the oracle port instead\n")
    return oracle_head_runner(batch), "port"


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path, all host threads, on a bounded sample of the
    same workload (unmodified reference from baseline/_ref when present, else the oracle port)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    # bounded sample: size the per-step batch so warmup+steps stay within ~2 minutes
    probe, kind = cpu_head_runner(4)
    probe()
    t0 = time.perf_counter(); probe(); t_pair = (time.perf_counter() - t0) / 4
    budget = 120.0 / max(1, args.steps + args.warmup)
    b = int(max(1, min(args.batch, budget / max(t_pair, 1e-6))))
    step, kind = cpu_head_runner(b)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = b * args.steps / dt
    what = ("unmodified reference CDRNet.forward (encoder stubbed) + calc_mpjpe" if kind == "reference"
            else "oracle port of the reference head")
    sample = f"{b} of {args.batch} stereo pairs per step, head only, fp32, {what}, torch CPU {torch.__version__}"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32",
        "data": "synthetic", "gpu_launches": 0,
        "config": bench_config(args.batch, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
                         "pairs_per_step": b, "cpu": cpu_model()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ----------------------------------------------------------------------------------------------
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """One float32 / float64 DIR/<name>.npy per array (what a caller of the timed path receives), at most
    DUMP_LIMIT_BYTES in all."""
    arrays = {name: t.detach().cpu().numpy() for name, t in arrays.items()}
    arrays = {name: a if a.dtype in (np.float32, np.float64) else a.astype(np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure(args, precision, ctx, dump_dir=None):
    """Time the head at one precision.  Returns the per-precision part of the JSON line.  ``dump_dir``: write the
    outputs of the last timed step there (rank 0; with N > 1 the 2D joints are rank 0's shard)."""
    import torch.distributed as dist
    import fast_3d_human_pose_estimation_b200 as pkg
    from fast_3d_human_pose_estimation_b200 import synth, dist as cdist, _lib
    world, rank, dev, B, K, W = ctx["world"], ctx["rank"], ctx["dev"], args.batch, args.steps, ctx["W"]
    feats_h, P_h, feats, Ps = ctx["feats_h"], ctx["P_h"], ctx["feats"], ctx["Ps"]
    g3, g2l, g2r, vis, flush = ctx["g3"], ctx["g2l"], ctx["g2r"], ctx["vis"], ctx["flush"]
    n_total = B * world

    model = pkg.CDRNet(synth.make_cfg(18, JOINTS), precision=precision)   # encoder unused here
    model.load_state_dict(ctx["sd"], strict=False)
    model = model.to(dev).eval()

    # N > 1: the 3D joints and MPJPE sums land directly in this rank's slot of a pre-allocated gather buffer; the ONE
    # collective of the path is an in-place ncclAllGather of that buffer — no packing / unpacking kernels (dist.GatherBuffer)
    gb = cdist.GatherBuffer(n_total, JOINTS, dev) if world > 1 else None

    def step(f, p):
        if gb is None:
            (kl, kr), xyz = model.head(f, p)
            return kl, kr, xyz, pkg.mpjpe_sums([kl, kr], xyz, g3, g2l, g2r, vis)
        (kl, kr), xyz = model.head(f, p, out_xyz=gb.xyz_slot)
        pkg.mpjpe_sums([kl, kr], xyz, g3, g2l, g2r, vis, out=gb.sums_slot)
        gb.all_gather()
        return kl, kr, gb

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(ctx["local"])
    if rank == 0:
        sampler.start()                 # already streaming when the timed region begins
    for _ in range(W):
        flush.fill_(1)
        out = step(feats, Ps)
    barrier()

    if rank == 0 and sampler.running:               # the sampler needs a moment to produce its first sample
        t_wait = time.perf_counter()
        while not sampler.rows and time.perf_counter() - t_wait < 1.0:
            time.sleep(0.01)

    # ---- device-resident timing: K steps, L2 flushed between steps (outside the event pairs)
    L = _lib.lib()
    L.cdr_launch_count_reset()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    barrier()
    t_wall = t_region0 = time.perf_counter()
    for i in range(K):
        flush.fill_(i & 0xff)
        starts[i].record()
        out = step(feats, Ps)
        ends[i].record()
    barrier()
    t_wall = time.perf_counter() - t_wall
    launches = L.cdr_launch_count()
    dev_ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
    clocks = sampler.stop(t_region0, t_region0 + t_wall) if rank == 0 else None
    if gb is not None:                      # outside the timed region: one D2H of the gathered buffer, host-side unpack
        gb.to_host()
        torch.cuda.synchronize()
        xyz, sums = gb.unpack_host()
        xyz, sums = xyz.clone(), sums.clone()
        kl, kr = out[:2]
    else:
        kl, kr, xyz, sums = out
    if dump_dir is not None and rank == 0:
        dump_outputs(dump_dir, {"kp_l": kl, "kp_r": kr, "xyz": xyz, "mpjpe_sums": sums})
    e2d, e3d = cdist.mpjpe_from_sums(sums)

    # ---- N > 1, outside every timed region: the gathered result of the sharded run against an UNSHARDED recompute —
    # rank 0 regenerates every rank's seeded shard and runs all N*B pairs through the same model on its one GPU
    shard_check = None
    if world > 1 and rank == 0:
        xs, ss = [], torch.zeros(4, dtype=torch.float64, device=dev)
        for r in range(world):
            f_r = [f.to(dev) for f in synth.make_features(B, seed=1 + r)]
            cams_r = synth.make_cameras(B, seed=2 + r)
            gt_r = synth.make_gt(cams_r, seed=3 + r)
            P_r = [torch.from_numpy(cams_r["P_l"]).to(dev), torch.from_numpy(cams_r["P_r"]).to(dev)]
            (kl_r, kr_r), x_r = model.head(f_r, P_r)
            ss += pkg.mpjpe_sums([kl_r, kr_r], x_r, *[torch.from_numpy(gt_r[k]).to(dev) for k in ("gt3d", "gt2d_l", "gt2d_r", "vis")])
            xs.append(x_r)
        x_all = torch.cat(xs, 0).cpu()
        ss = ss.cpu()
        shard_check = {"sharded_equals_unsharded": bool(torch.equal(x_all, xyz) and torch.equal(ss, sums)),
                       "xyz_max_abs_diff_mm": float((x_all - xyz).abs().max()),
                       "mpjpe_sums_max_abs_diff": float((ss - sums).abs().max()), "pairs": int(x_all.shape[0]),
                       "how": "rank 0 recomputes all ranks' seeded shards unsharded on one GPU; bit-exact compare of the "
                              "all-gathered (N*B,19,3) joints and the rank-ordered fp64 MPJPE sums"}

    # ---- end to end through the public API with HOST buffers (H2D + D2H inside the timed region)
    h2d = sum(t.numel() * t.element_size() for t in feats_h + P_h)
    xyz_h = torch.empty((n_total, JOINTS, 3), dtype=torch.float32).pin_memory()
    sums_h = torch.empty(4, dtype=torch.float64).pin_memory()
    d2h = xyz_h.numel() * 4 + 32
    e_s, e_e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # public API for host buffers: pkg.HeadPipeline — per batch: H2D of the pinned latents / P on a copy
    # stream, one CUDA graph (head -> MPJPE sums -> D2H of 2D/3D joints + sums) on the compute stream;
    # batch i+1 crosses PCIe while batch i computes (depth 2).  Every step copies its inputs in and its
    # results out; a step's results are read on the host one submit later.
    pipe = pkg.HeadPipeline(model, B, gt={"gt3d": g3, "gt2d_l": g2l, "gt2d_r": g2r, "vis": vis},
                            gather_total=n_total if world > 1 else None)
    if world > 1:
        d2h = pipe.gather[0].host.numel()              # the gathered buffer: N slots of (B,19,3) fp32 + 32 B

    def first(res):                                    # the caller reads every step's result on the host
        return float(res.host[:4].view(torch.float32)[0]) if world > 1 else float(res[0, 0, 0])

    def e2e_run(k):
        checksum = 0.0
        pipe.submit(feats_h, P_h)
        for _ in range(k - 1):
            pipe.submit(feats_h, P_h)
            _, _, x_h, s_h = pipe.collect()
            checksum += first(x_h)
        _, _, x_h, s_h = pipe.collect()
        return checksum + first(x_h)
    e2e_run(3)
    barrier()
    e_s.record()
    e2e_run(K)
    e_e.record()
    barrier()
    e2e_ms = e_s.elapsed_time(e_e)
    # bf16 head: the same end-to-end step fed bf16 pixel-major latent rows from the host (what a bf16 producer holds; the
    # bf16 head rounds fp32 latents to bf16 anyway) — half the PCIe bytes of the reference-shaped fp32 tensors
    e2e_rows = None
    if precision == "bf16" and world == 1:
        rows_h = torch.cat([f.permute(0, 2, 3, 1).reshape(-1, 2048) for f in feats_h], 0).to(torch.bfloat16).contiguous().pin_memory()
        pipe_r = pkg.HeadPipeline(model, B, gt={"gt3d": g3, "gt2d_l": g2l, "gt2d_r": g2r, "vis": vis}, latents="rows_bf16")

        def rows_run(k):
            pipe_r.submit(rows_h, P_h)
            for _ in range(k - 1):
                pipe_r.submit(rows_h, P_h)
                x = pipe_r.collect()[2]
                float(x[0, 0, 0])
            return float(pipe_r.collect()[2][0, 0, 0])
        rows_run(3)
        torch.cuda.synchronize()
        r_s, r_e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r_s.record()
        rows_run(K)
        r_e.record()
        torch.cuda.synchronize()
        r_ms = r_s.elapsed_time(r_e) / K
        e2e_rows = {"value": B / (r_ms / 1e3), "unit": UNIT, "ms_per_step": r_ms,
                    "h2d_bytes_per_step": rows_h.numel() * 2 + sum(t.numel() * 4 for t in P_h),
                    "api": "HeadPipeline(latents='rows_bf16'): bf16 pixel-major latent rows (2B*64, 2048) from pinned host memory"}
        pipe_r.close()
        del pipe_r
    # latency form (no cross-step overlap): one CUDA graph of H2D -> head -> D2H, synchronised per step
    hg = pkg.HeadGraph(model, feats_h, P_h, gt={"gt3d": g3, "gt2d_l": g2l, "gt2d_r": g2r, "vis": vis})
    for _ in range(2):
        hg.replay(sync=True)
    l_s, l_e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l_s.record()
    for _ in range(K):
        hg.replay(sync=True)
    l_e.record()
    torch.cuda.synchronize()
    e2e_latency_ms = l_s.elapsed_time(l_e) / K
    d2h += 2 * B * JOINTS * 2 * 4                      # the graph also returns the two 2D joint sets

    # ---- per-kernel durations, live, with CUDA events on the launching stream
    stage_ms = {}
    reps = 5
    for _ in range(reps):
        flush.fill_(3)
        torch.cuda.synchronize()
        _lib.stage_timing_begin(dev)
        model.head(feats, Ps)
        for name, ms in _lib.stage_timing_end():
            stage_ms[name] = stage_ms.get(name, 0.0) + ms / reps

    # ---- sustained form (N=1): the same step back to back for ~2 s, no L2 flush, clocks / power sampled all along.
    # The K-step region above lasts tens of ms with flushes in between; under continuous load the B200 reaches its
    # power cap and lowers the SM clock (DESIGN.md §3), which this number shows and the headline cannot.
    sustained = None
    if world == 1 and not args.no_sustained:
        s2 = ClockSampler(ctx["local"])
        s2.start()
        tw = time.perf_counter()
        while s2.running and not s2.rows and time.perf_counter() - tw < 1.0:
            time.sleep(0.01)
        torch.cuda.synchronize()
        n_s, t_s0 = 0, time.perf_counter()
        a, bnd = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        while time.perf_counter() - t_s0 < 2.0:
            for _ in range(25):
                step(feats, Ps)
            n_s += 25
            torch.cuda.synchronize()
        bnd.record()
        torch.cuda.synchronize()
        t_s1 = time.perf_counter()
        ms_s = a.elapsed_time(bnd) / n_s
        sustained = {"value": B / (ms_s / 1e3), "unit": UNIT, "ms_per_step": ms_s, "steps": n_s,
                     "window_s": t_s1 - t_s0, "l2": "not flushed (weights and some activations stay in L2)",
                     "clocks": s2.stop(t_s0 + 0.5, t_s1)}

    t = torch.tensor([dev_ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = float(t[0]), float(t[1])
    if rank != 0:
        return None

    pk = peaks()
    value = n_total * K / (dev_ms / 1e3)
    top = max(stage_ms, key=stage_ms.get)
    share = stage_ms[top] / sum(stage_ms.values())
    if top in FLOP_PER_PAIR:
        ach = FLOP_PER_PAIR[top] * B / (stage_ms[top] / 1e3) / 1e12
        roof = {"kernel": top, "bound": "tensor", "achieved": ach, "peak": pk["tflops_sustained"],
                "unit": "TFLOP/s", "frac": ach / pk["tflops_sustained"],
                "traffic": ncu_traffic().get(precision, {}).get(top) if B == 64 else None,
                "traffic_source": ncu_traffic().get("source"),
                "peak_source": pk["source"] + " bf16 sustained (cuBLAS)", "launch_ms": stage_ms[top],
                "share_of_step": share,
                "fused": "deconv3 + final 1x1 + soft-argmax partial sums in one kernel" if top == "deconv3_tail" else None,
                "note": {"bf16": "tcgen05 kind::f16, bf16 operands",
                         "fp32": "tcgen05 kind::f16 on fp16 two-term operands, 3 MMAs per product at the full 16-bit "
                                 "rate: at most 1/3 of the bf16 peak in algorithmic FLOPs",
                         "tf32x3": "tcgen05 kind::tf32, 3 MMAs per product (3xTF32 split) at half the bf16 rate: "
                                   "at most 1/6 of the bf16 peak in algorithmic FLOPs",
                         "fp32_ffma": "fp32 FFMA kernel on CUDA cores; fp32 FFMA peak is 74.4 TFLOP/s"}[precision]}
    else:
        ach = SOFTARGMAX_DLT_BYTES_PER_POSE * B / (stage_ms[top] / 1e3) / 1e9
        roof = {"kernel": top, "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": ach / pk["hbm_gbs"], "traffic": None, "peak_source": pk["source"],
                "launch_ms": stage_ms[top], "share_of_step": share}
    sa = stage_ms.get("softargmax_dlt")          # absent when the decoder tail is fused (deconv3_tail + merge_dlt)
    hbm = None
    if sa:
        a = SOFTARGMAX_DLT_BYTES_PER_POSE * B / (sa / 1e3) / 1e9
        hbm = {"kernel": "softargmax_dlt", "bound": "hbm", "achieved": a, "peak": pk["hbm_gbs"],
               "unit": "GB/s", "frac": a / pk["hbm_gbs"], "launch_ms": sa,
               "note": "latency-bound launch at this batch (64 CTAs on 148 SMs, 40 MB of logits still in L2); the "
                       "kernel's HBM roofline is roofline_hbm_stream / config4_softargmax_dlt_1m_poses"}
    dec_ms = sum(stage_ms.get(k, 0.0) for k in ("deconv1", "deconv2", "deconv3", "final_1x1", "deconv3_tail"))
    dec_tf = 7595.9e6 * B / (dec_ms / 1e3) / 1e12 if dec_ms else None
    return {
        "value": value, "ms_per_step": dev_ms / K, "dtype": precision,
        "e2e": {"value": n_total * K / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / K,
                "api": "HeadPipeline (depth-2: H2D of batch i+1 overlaps compute of batch i)"
                       + ("; in-place all-gather %s" % ("captured in the step's CUDA graph" if pipe.gather_in_graph
                                                        else "issued after the graph replay") if world > 1 else ""),
                "unpipelined_ms_per_step": e2e_latency_ms},
        "gpu_launches": int(launches), "launches_per_step": launches / K,
        "roofline": roof, "roofline_hbm": hbm, "stages_ms": stage_ms,
        "decoder_tflops": dec_tf, "decoder_frac_of_peak": dec_tf / pk["tflops_sustained"] if dec_tf else None,
        "head_tflops": HEAD_FLOP_PER_PAIR * value / 1e12,
        "clocks": clocks, "wall_s_timed_region": t_wall, "sustained": sustained,
        "mpjpe": {"error_2d_px": e2d, "error_3d_mm": e3d},
        "sharded_check": shard_check, "e2e_bf16_rows": e2e_rows,
    }


def stream_microbench(dev, poses=8192, reps=5):
    """BASELINE configs[3] in miniature: the fused soft-argmax + DLT kernel streaming `poses` stereo
    poses x 19 joints x 2 views x 64x64 fp32 logits (>> L2) — its HBM roofline at scale (the B=64
    head launch is latency-bound: 64 CTAs, 40 MB)."""
    from fast_3d_human_pose_estimation_b200 import synth, _lib
    L = _lib.lib()
    cams = synth.make_cameras(64, seed=4)
    P_l = torch.from_numpy(cams["P_l"]).to(dev).repeat(poses // 64, 1, 1).contiguous()
    P_r = torch.from_numpy(cams["P_r"]).to(dev).repeat(poses // 64, 1, 1).contiguous()
    g = torch.Generator(device=dev).manual_seed(0)
    heat = torch.empty((2, poses, JOINTS, 64, 64), dtype=torch.float32, device=dev)
    for v in range(2):
        for lo in range(0, poses, 1024):
            heat[v, lo:lo + 1024].normal_(0.0, 3.0, generator=g)
    kl = torch.empty((poses, JOINTS, 2), device=dev)
    kr = torch.empty_like(kl)
    xyz = torch.empty((poses, JOINTS, 3), device=dev)
    st = _lib.current_stream_ptr(dev)

    def run():
        _lib.check(L.cdr_softargmax_dlt(_lib.ptr(heat[0]), _lib.ptr(heat[1]), 0, _lib.ptr(P_l), _lib.ptr(P_r), poses,
                                        JOINTS, 64, 64, 4.0, _lib.ptr(kl), _lib.ptr(kr), _lib.ptr(xyz), None, None,
                                        None, None, None, st))
    for _ in range(2):
        run()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); run(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ms = float(np.median(ts))
    pk = peaks()
    gbs = SOFTARGMAX_DLT_BYTES_PER_POSE * poses / (ms / 1e3) / 1e9
    del heat
    return {"kernel": "softargmax_dlt (streaming microbench)", "bound": "hbm", "poses": poses,
            "bytes_per_pose": SOFTARGMAX_DLT_BYTES_PER_POSE, "launch_ms": ms, "poses_per_s": poses / (ms / 1e3),
            "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"],
            "peak_source": pk["source"], "input": "resident in HBM (5.1 GB, >> L2), fp32 logits N(0,3)",
            "algorithmic_bytes": SOFTARGMAX_DLT_BYTES_PER_POSE * poses,
            "traffic": ncu_traffic().get("softargmax_dlt_stream") if poses == 8192 else None}


def config4_1m_poses(dev, chunk=8192, total=1 << 20):
    """BASELINE configs[3]: soft-argmax + DLT over 2^20 stereo poses x 19 joints x 2 views x 64x64 fp32 logits
    (653 GB of heat-maps: does not fit HBM).  SURVEY §8d recipe: `total/chunk` launches of `chunk` poses each
    over two alternating device buffers (2 x 5.1 GB, each >> L2), kernels only, one CUDA-event pair around
    all of them.  Heat-maps = Gaussian blobs (sigma 3 px, amplitude 10) on the projections of a synthetic
    3D ground truth + N(0,0.1) noise, so the triangulation has a truth to land on (reported, not gated)."""
    from fast_3d_human_pose_estimation_b200 import synth, _lib
    L = _lib.lib()
    cams = synth.make_cameras(chunk, seed=4)
    gt = synth.make_gt(cams, seed=5)
    P_l = torch.from_numpy(cams["P_l"]).to(dev)
    P_r = torch.from_numpy(cams["P_r"]).to(dev)
    bufs = []
    for b in range(2):
        heat = torch.empty((2, chunk, JOINTS, 64, 64), dtype=torch.float32, device=dev)
        for v, key in enumerate(("gt2d_l", "gt2d_r")):
            c = torch.from_numpy(gt[key] / 4.0).float().to(dev)
            for lo in range(0, chunk, 512):
                heat[v, lo:lo + 512] = synth.blob_heatmaps(c[lo:lo + 512], seed=100 * b + 10 * v + lo)
        bufs.append(heat)
    kl = torch.empty((chunk, JOINTS, 2), device=dev)
    kr = torch.empty_like(kl)
    xyz = torch.empty((chunk, JOINTS, 3), device=dev)
    st = _lib.current_stream_ptr(dev)
    n_launch = total // chunk

    def run(k):
        for i in range(k):
            h = bufs[i & 1]
            _lib.check(L.cdr_softargmax_dlt(_lib.ptr(h[0]), _lib.ptr(h[1]), 0, _lib.ptr(P_l), _lib.ptr(P_r), chunk,
                                            JOINTS, 64, 64, 4.0, _lib.ptr(kl), _lib.ptr(kr), _lib.ptr(xyz), None, None,
                                            None, None, None, st))
    run(4)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); run(n_launch); b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b)
    err = (xyz.double().cpu().numpy() - gt["gt3d"])
    err3 = float(np.sqrt((err ** 2).sum(-1)).mean())
    err2 = float(np.abs(kl.double().cpu().numpy() - gt["gt2d_l"]).mean())
    pk = peaks()
    gbs = SOFTARGMAX_DLT_BYTES_PER_POSE * total / (ms / 1e3) / 1e9
    del bufs
    torch.cuda.empty_cache()
    return {"workload": "BASELINE configs[3]: soft-argmax + DLT, 2^20 poses x 19 joints x 2 views x 64x64 fp32",
            "poses": total, "launches": n_launch, "poses_per_launch": chunk, "ms_total": ms,
            "poses_per_s": total / (ms / 1e3), "bytes_per_pose": SOFTARGMAX_DLT_BYTES_PER_POSE,
            "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"], "bound": "hbm",
            "input": "two alternating 5.1 GB device buffers of Gaussian-blob logits (each >> 126 MB L2)",
            "mean_3d_err_vs_truth_mm": err3, "mean_2d_err_vs_truth_px": err2}


def ftl_stream(dev, n=4096, reps=5):
    """CanonicalFusion.ftl (models/cdrnet.py:45-56) at a size that leaves L2: n samples x 64 pixels, fp32
    rows, through the C ABI `cdr_ftl`.  Algorithmic bytes per sample and direction = (300 + 400) channels x
    64 pixels x 4 B = 179 200 (SURVEY §8d: 76 800 + 102 400).  The B=64 head launches are latency-bound."""
    from fast_3d_human_pose_estimation_b200 import _lib
    L = _lib.lib()
    st = _lib.current_stream_ptr(dev)
    g = torch.Generator(device=dev).manual_seed(0)
    x3 = torch.zeros((n * 64, 304), device=dev)
    x3[:, :300].normal_(generator=g)
    x4 = torch.empty((n * 64, 400), device=dev)
    m43 = torch.randn((n, 4, 3), device=dev, generator=g)
    m34 = torch.randn((n, 3, 4), device=dev, generator=g)
    out = {}
    pk = peaks()
    for name, (src, sp, mats, r, c, dst, dp, fill) in {"inverse_4x3": (x3, 304, m43, 4, 3, x4, 400, 400),
                                                       "forward_3x4": (x4, 400, m34, 3, 4, x3, 304, 304)}.items():
        def run():
            _lib.check(L.cdr_ftl(_lib.ptr(src), sp, _lib.ptr(mats), r, c, 100, n, 64, _lib.ptr(dst), dp, fill, st))
        run(); run()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); run(); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ms = float(np.median(ts))
        gbs = 179200.0 * n / (ms / 1e3) / 1e9
        out[name] = {"launch_ms": ms, "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"]}
    # spot check against the definition: out[row, r*100+c] = sum_k m[r,k] * in[row, k*100+c]   (last launch: forward)
    rows = torch.arange(0, n * 64, max(1, n * 64 // 257), device=dev)
    want = torch.einsum("nrk,nkc->nrc", m34[rows // 64].double(), x4[rows].double().reshape(-1, 4, 100)).reshape(-1, 300)
    out["max_abs_err_vs_fp64"] = float((x3[rows, :300].double() - want).abs().max())
    out.update({"kernel": "ftl_vec_kernel<float> via cdr_ftl", "bound": "hbm", "samples": n, "bytes_per_sample": 179200,
                "input": f"{n} samples x 64 px fp32 rows ({x3.numel() * 4 / 1e6:.0f} + {x4.numel() * 4 / 1e6:.0f} MB, >> L2)"})
    return out


def backward_stream(dev, poses=4096, reps=5):
    """SURVEY §8f rank 3 (first slice): backward of soft-argmax (HBM-bound: 16 KB of logits in, 16 KB of gradient out
    per map) and of the DLT, at a size that leaves L2.  Algorithmic bytes per pose = 2 * 19 * (2 * 16384 + 8)."""
    from fast_3d_human_pose_estimation_b200 import synth, _lib
    L = _lib.lib()
    st = _lib.current_stream_ptr(dev)
    n_maps = 2 * poses * JOINTS
    g = torch.Generator(device=dev).manual_seed(0)
    heat = torch.empty((n_maps, 64, 64), dtype=torch.float32, device=dev)
    for lo in range(0, n_maps, 16384):
        heat[lo:lo + 16384].normal_(0.0, 3.0, generator=g)
    gk = torch.randn((n_maps, 2), device=dev, generator=g)
    gh = torch.empty_like(heat)
    cams = synth.make_cameras(64, seed=4)
    P_l = torch.from_numpy(cams["P_l"]).to(dev).repeat(poses // 64, 1, 1).contiguous()
    P_r = torch.from_numpy(cams["P_r"]).to(dev).repeat(poses // 64, 1, 1).contiguous()
    kl = torch.rand((poses, JOINTS, 2), device=dev, generator=g) * 256
    kr = torch.rand((poses, JOINTS, 2), device=dev, generator=g) * 256
    gx = torch.randn((poses, JOINTS, 3), device=dev, generator=g)
    gl, gr = torch.empty_like(kl), torch.empty_like(kr)

    def timed(fn):
        fn(); fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts))
    ms_sa = timed(lambda: _lib.check(L.cdr_softargmax_backward(_lib.ptr(heat), _lib.ptr(gk), n_maps, 64, 64, 4.0,
                                                               _lib.ptr(gh), st)))
    ms_dlt = timed(lambda: _lib.check(L.cdr_dlt_backward(_lib.ptr(P_l), _lib.ptr(P_r), _lib.ptr(kl), _lib.ptr(kr),
                                                         _lib.ptr(gx), poses, JOINTS, _lib.ptr(gl), _lib.ptr(gr), st)))
    pk = peaks()
    bytes_sa = n_maps * (2 * 16384 + 8)
    gbs = bytes_sa / (ms_sa / 1e3) / 1e9
    # train-mode BatchNorm2d + ReLU (second slice) on deconv3's activation at B = 64: (128, 256, 64, 64) fp32 = 537 MB.
    # forward: x read twice (statistics, normalise) + y written = 3 passes; backward: x and dy read twice + dx written = 5
    del heat, gh
    torch.cuda.empty_cache()
    n, c, hw = 128, 256, 4096
    xb = torch.randn((n, c, 64, 64), device=dev, generator=g)
    yb, dyb, dxb = torch.empty_like(xb), torch.randn((n, c, 64, 64), device=dev, generator=g), torch.empty_like(xb)
    gam, bet = torch.ones(c, device=dev), torch.zeros(c, device=dev)
    rm, rv = torch.zeros(c, device=dev), torch.ones(c, device=dev)
    sm, si = torch.empty(c, device=dev), torch.empty(c, device=dev)
    dg, db = torch.empty(c, device=dev), torch.empty(c, device=dev)
    ms_bf = timed(lambda: _lib.check(L.cdr_bn_train_forward(_lib.ptr(xb), n, c, hw, _lib.ptr(gam), _lib.ptr(bet), 1e-5, 0.1,
                                                            _lib.ptr(rm), _lib.ptr(rv), 1, _lib.ptr(yb), _lib.ptr(sm),
                                                            _lib.ptr(si), st)))
    ms_bb = timed(lambda: _lib.check(L.cdr_bn_train_backward(_lib.ptr(xb), _lib.ptr(dyb), n, c, hw, _lib.ptr(gam),
                                                             _lib.ptr(bet), _lib.ptr(sm), _lib.ptr(si), 1, _lib.ptr(dxb),
                                                             _lib.ptr(dg), _lib.ptr(db), st)))
    tb = xb.numel() * 4
    bn = {"tensor": "(128, 256, 64, 64) fp32 (deconv3's activation at B = 64)",
          "forward": {"launch_ms": ms_bf, "algorithmic_bytes": 3 * tb, "achieved": 3 * tb / (ms_bf / 1e3) / 1e9,
                      "frac": 3 * tb / (ms_bf / 1e3) / 1e9 / pk["hbm_gbs"]},
          "backward": {"launch_ms": ms_bb, "algorithmic_bytes": 5 * tb, "achieved": 5 * tb / (ms_bb / 1e3) / 1e9,
                       "frac": 5 * tb / (ms_bb / 1e3) / 1e9 / pk["hbm_gbs"]},
          "peak": pk["hbm_gbs"], "unit": "GB/s", "bound": "hbm"}
    return {"bn_train_relu": bn, "softargmax_backward": {"launch_ms": ms_sa, "maps": n_maps, "algorithmic_bytes": bytes_sa, "achieved": gbs,
                                    "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"], "bound": "hbm"},
            "dlt_backward": {"launch_ms": ms_dlt, "joints_per_s": poses * JOINTS / (ms_dlt / 1e3), "bound": "latency / fp64"},
            "input": f"{poses} poses x 19 joints x 2 views of 64x64 fp32 logits ({n_maps * 16384 / 1e9:.1f} GB in, the same out)"}


def config5(args, ctx, precision, total=1024, encoder_precision="bf16"):
    """BASELINE configs[4]: the full pipeline (uint8 stereo frames in pinned HOST memory -> ResNet-101 encoder
    + head on this repo's kernels -> 3D joints + MPJPE sums on the host) over a batch of `total` stereo pairs
    sharded across the ranks (strong scaling: total/N pairs per GPU), processed in chunks of --batch pairs
    through FramePipeline, ONE final all-gather of every rank's (total/N,19,3) joints + MPJPE sums."""
    import torch.distributed as dist
    import fast_3d_human_pose_estimation_b200 as pkg
    from fast_3d_human_pose_estimation_b200 import synth, dist as cdist
    dev, B, world, rank = ctx["dev"], args.batch, ctx["world"], ctx["rank"]
    per = total // world
    n_chunks = max(1, per // B)
    per = n_chunks * B
    pipe, err = None, None
    try:
        torch.manual_seed(0)
        m = pkg.CDRNet(synth.make_cfg(101, JOINTS), precision=precision, encoder_precision=encoder_precision)
        m.load_state_dict(ctx["sd"], strict=False)
        m = m.to(dev).eval()
        gen = torch.Generator().manual_seed(7 + rank)
        frames_h = [torch.randint(0, 256, (2, B, 256, 256, 3), dtype=torch.uint8, generator=gen).pin_memory()
                    for _ in range(n_chunks)]
        pipe = pkg.FramePipeline(m, B, gt={"gt3d": ctx["g3"], "gt2d_l": ctx["g2l"], "gt2d_r": ctx["g2r"], "vis": ctx["vis"]})
    except Exception as e:
        err = repr(e)[:200]
    if world > 1:
        ok = torch.tensor([0.0 if pipe is None else 1.0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)        # enter the collective section only if every rank is ready
        if float(ok[0]) < 1.0:
            return {"error": err or "another rank failed to build the pipeline"}
    elif pipe is None:
        return {"error": err}
    xyz_all = torch.zeros((per, JOINTS, 3), dtype=torch.float32, device=dev)
    sums_all = torch.zeros(4, dtype=torch.float64, device=dev)
    xyz_h = torch.empty((per * world, JOINTS, 3), dtype=torch.float32).pin_memory()
    sums_h = torch.empty(4, dtype=torch.float64).pin_memory()
    state = {"i": 0}

    def post(slot):                       # on the compute stream, after the chunk's graph
        i = state["i"]
        xyz_all[i * B:(i + 1) * B].copy_(pipe.xyz_dev[slot])
        sums_all.add_(pipe.sums_dev[slot])
        state["i"] = i + 1

    def run():
        state["i"] = 0
        sums_all.zero_()
        pipe.submit(frames_h[0], ctx["P_h"], post)
        for c in range(1, n_chunks):
            pipe.submit(frames_h[c], ctx["P_h"], post)
            pipe.collect()
        pipe.collect()
        with torch.cuda.stream(pipe.compute_stream):
            x, s = cdist.gather_results(xyz_all, sums_all, per * world)
            xyz_h.copy_(x, non_blocking=True)
            sums_h.copy_(s, non_blocking=True)
        pipe.compute_stream.synchronize()
        return float(sums_h[3])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    run()
    barrier()
    reps, ms = 3, []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        with torch.cuda.stream(pipe.compute_stream):
            a.record()
        count = run()
        with torch.cuda.stream(pipe.compute_stream):
            b.record()
        barrier()
        t = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms.append(float(t[0]))
    best = float(np.median(ms))
    # N > 1, outside the timed region: the gathered result of the sharded run against an UNSHARDED recompute — rank 0
    # regenerates every rank's seeded frames / cameras / ground truth and pushes all the pairs through its own pipeline
    shard_check = None
    if world > 1 and rank == 0:
        xs, total = [], None
        for r in range(world):
            gen_r = torch.Generator().manual_seed(7 + r)
            fr = [torch.randint(0, 256, (2, B, 256, 256, 3), dtype=torch.uint8, generator=gen_r).pin_memory()
                  for _ in range(n_chunks)]
            cams_r = synth.make_cameras(B, seed=2 + r)
            gt_r = synth.make_gt(cams_r, seed=3 + r)
            P_r = [torch.from_numpy(cams_r["P_l"]).pin_memory(), torch.from_numpy(cams_r["P_r"]).pin_memory()]
            g_r = [torch.from_numpy(gt_r[k]).to(dev) for k in ("gt3d", "gt2d_l", "gt2d_r", "vis")]
            s_r = torch.zeros(4, dtype=torch.float64, device=dev)
            for c in range(n_chunks):
                pipe.submit(fr[c], P_r)
                _, kp_h, x_h, _ = pipe.collect()
                xs.append(x_h.clone())
                s_r += pkg.mpjpe_sums([kp_h[0].to(dev), kp_h[1].to(dev)], x_h.to(dev), *g_r)
            total = s_r.clone() if total is None else total + s_r
        x_all = torch.cat(xs, 0)
        torch.cuda.synchronize()
        shard_check = {"sharded_equals_unsharded": bool(torch.equal(x_all, xyz_h) and torch.equal(total.cpu(), sums_h)),
                       "xyz_max_abs_diff_mm": float((x_all - xyz_h).abs().max()),
                       "mpjpe_sums_max_abs_diff": float((total.cpu() - sums_h).abs().max()), "pairs": int(x_all.shape[0])}
    if world > 1:
        dist.barrier()
    return {"sharded_check": shard_check,
            "workload": "BASELINE configs[4]: full pipeline, %d stereo pairs sharded over %d GPU(s)" % (per * world, world),
            "pairs_per_s": per * world / (best / 1e3), "ms_total": best, "n_gpus": world, "pairs_per_gpu": per,
            "chunk_pairs": B, "chunks_per_gpu": n_chunks, "scaling": "strong", "head_precision": precision,
            "encoder_precision": {"bf16": "bf16 (tcgen05, below the reference's fp32)",
                                  "fp32": "f16x2 (tcgen05, fp32-accurate: the reference's precision)"}[encoder_precision],
            "mpjpe_count": count, "h2d_bytes_per_gpu": n_chunks * (frames_h[0].numel() + 2 * B * 48),
            "collective": "1 all-gather of (%d,19,3) fp32 + 32 B per rank at the end" % per,
            "api": "FramePipeline per rank (uint8 frames in pinned host memory; ResNet-101 encoder + head on this repo's kernels)"}


def full_pipeline(args, ctx, precision):
    """SURVEY §8d: pairs/s of the whole CDRNet.forward — ResNet-101 encoder on torch/cuDNN (not
    ours, by decree) + our head — on device-resident (B,3,256,256) image pairs.  Two encoder
    settings: torch default fp32 (cuDNN may use TF32) and bf16 autocast + channels_last."""
    import fast_3d_human_pose_estimation_b200 as pkg
    from fast_3d_human_pose_estimation_b200 import synth, _lib
    dev, B = ctx["dev"], args.batch
    torch.manual_seed(0)
    model = pkg.CDRNet(synth.make_cfg(101, JOINTS), precision=precision)
    model.load_state_dict(ctx["sd"], strict=False)
    model = model.to(dev).eval()
    g = torch.Generator(device=dev).manual_seed(1)
    xs = [torch.randn((B, 3, 256, 256), generator=g, device=dev) for _ in range(2)]
    out = {}

    def timed(fn, reps=5):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    ms = timed(lambda: model(xs, ctx["Ps"]))
    enc_ms = timed(lambda: [model.encoder(x) for x in xs])
    out["encoder_fp32_cudnn"] = {"pairs_per_s": B / (ms / 1e3), "ms_per_step": ms, "encoder_ms": enc_ms,
                                 "head_share": max(0.0, 1.0 - enc_ms / ms)}
    enc = model.encoder.to(memory_format=torch.channels_last)
    xcl = [x.contiguous(memory_format=torch.channels_last) for x in xs]

    def bf16_step():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            zs = [enc(x) for x in xcl]
        return model.head([z.float() for z in zs], ctx["Ps"])

    def bf16_enc():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            return [enc(x) for x in xcl]
    ms = timed(bf16_step)
    enc_ms = timed(bf16_enc)
    out["encoder_bf16_autocast_channels_last"] = {"pairs_per_s": B / (ms / 1e3), "ms_per_step": ms,
                                                  "encoder_ms": enc_ms, "head_share": max(0.0, 1.0 - enc_ms / ms)}
    # SURVEY §8f rank 1: the whole encoder on this repo's kernels (stem: warp-MMA, layer1-4: tcgen05 tap-GEMM),
    # with the fp32-accurate head and with the bf16 head (the natural partner of a bf16 encoder)
    del enc, xcl
    x2 = torch.cat(xs, 0)
    gt = {"gt3d": ctx["g3"], "gt2d_l": ctx["g2l"], "gt2d_r": ctx["g2r"], "vis": ctx["vis"]}
    # (encoder precision, head precision): the bf16 encoder with this run's head and with the bf16 head; and — the
    # pipeline at the REFERENCE's precision end to end — the f16x2 encoder feeding the fp32 head fp16 planes
    combos = [("bf16", hp) for hp in dict.fromkeys([precision, "bf16"])]
    if precision in ("fp32", "f16x2"):
        combos.append(("fp32", precision))
    for enc_prec, head_prec in combos:
        torch.manual_seed(0)
        m2 = pkg.CDRNet(synth.make_cfg(101, JOINTS), precision=head_prec, encoder_precision=enc_prec)
        m2.load_state_dict(ctx["sd"], strict=False)
        m2 = m2.to(dev).eval()
        ms = timed(lambda: m2(xs, ctx["Ps"]))
        enc_ms = timed(lambda: m2._tc_encoder.rows(x2))
        _lib.stage_timing_begin(dev)
        m2._tc_encoder.rows(x2)
        blocks = {}
        for name, t in _lib.stage_timing_end():
            blocks[name] = blocks.get(name, 0.0) + t
        rec = {"pairs_per_s": B / (ms / 1e3), "ms_per_step": ms, "encoder_ms": enc_ms,
               "stem_ms": blocks.get("enc_stem", 0.0), "head_share": max(0.0, 1.0 - enc_ms / ms),
               "encoder_tflops": 40747.7e6 * B / (enc_ms / 1e3) / 1e12,
               "layer_ms": {f"layer{i + 1}": sum(v for k, v in blocks.items()
                                                 if k.startswith("enc_block") and lo <= int(k[9:].split(".")[0]) < hi)
                            for i, (lo, hi) in enumerate(((0, 3), (3, 7), (7, 30), (30, 33)))}}
        # production-shaped end to end: raw uint8 stereo frames in pinned HOST memory -> 3D joints on the host
        for bb in (B, 2 * B):
            try:
                gen = torch.Generator().manual_seed(7)
                frames_h = torch.randint(0, 256, (2, bb, 256, 256, 3), dtype=torch.uint8, generator=gen).pin_memory()
                P_h = [p.repeat(bb // B, 1, 1).pin_memory() for p in ctx["P_h"]]
                pipe = pkg.FramePipeline(m2, bb, gt={k: v.repeat(bb // B, *([1] * (v.dim() - 1))) for k, v in gt.items()})

                def run(k):
                    pipe.submit(frames_h, P_h)
                    for _ in range(k - 1):
                        pipe.submit(frames_h, P_h)
                        pipe.collect()
                    return pipe.collect()
                run(3)
                torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                kk = 10
                a.record()
                run(kk)
                b.record()
                torch.cuda.synchronize()
                e_ms = a.elapsed_time(b) / kk
                rec["e2e_uint8_frames_host" + ("" if bb == B else f"_batch{bb}")] = {
                    "pairs_per_s": bb / (e_ms / 1e3), "ms_per_step": e_ms, "pairs_per_step": bb,
                    "h2d_bytes_per_step": frames_h.numel() + 2 * bb * 48,
                    "d2h_bytes_per_step": bb * JOINTS * (3 + 2 + 2) * 4 + 32,
                    "api": "FramePipeline: H2D of uint8 frames (copy stream) overlapped with one CUDA graph of "
                           "normalise+stem+layer1-4+head+MPJPE+D2H (depth 2)"}
                del pipe, frames_h
            except Exception as e:
                rec["e2e_uint8_frames_host" + ("" if bb == B else f"_batch{bb}")] = {"error": repr(e)[:200]}
        if enc_prec == "fp32":
            rec["precision"] = ("encoder: scaled fp16 hi/lo planes, 3 kind::f16 MMAs per product, three-term fp16 mma.sync stem (latents "
                                "1.5e-6 of max vs fp64 on ResNet-50); head: fp32 mode")
            rec["encoder_tflops_issued_mma"] = 3 * rec["encoder_tflops"]
            out["encoder_f16x2_tcgen05"] = rec
        else:
            out["encoder_bf16_tcgen05" + ("" if head_prec == precision else "_head_bf16")] = rec
        del m2
        torch.cuda.empty_cache()
    del x2
    # BASELINE configs[2]: baseline.py — PoseResNet-101 2D heat-maps on both views, arg-max x4 -> uint8, DLT
    # triangulation; 256 images (128 pairs), bf16, all on this library (frames as uint8 in HBM)
    try:
        torch.manual_seed(0)
        pr = pkg.PoseResNet(synth.make_cfg(101, JOINTS), precision="bf16", encoder_precision="bf16").to(dev).eval()
        nb = 128
        frames = torch.randint(0, 256, (2 * nb, 256, 256, 3), dtype=torch.uint8, device=dev)
        cams = synth.make_cameras(nb, seed=5)
        row4 = np.tile([[[0, 0, 0, 1.0]]], (nb, 1, 1))
        P1 = torch.from_numpy(np.concatenate([cams["P_l"], row4], 1).astype(np.float64)).to(dev)
        P2 = torch.from_numpy(np.concatenate([cams["P_r"], row4], 1).astype(np.float64)).to(dev)

        def baseline_step():
            pts = pkg.baseline_keypoints(pr(frames))
            return pkg.triangulation(P1, P2, pts[:nb], pts[nb:])
        ms = timed(baseline_step)
        out["baseline_poseresnet101_bf16_batch256"] = {"pairs_per_s": nb / (ms / 1e3), "images_per_s": 2 * nb / (ms / 1e3),
                                                       "ms_per_step": ms, "images_per_step": 2 * nb}
        del pr, frames
        torch.cuda.empty_cache()
    except Exception as e:
        out["baseline_poseresnet101_bf16_batch256"] = {"error": repr(e)[:200]}
    out["note"] = ("ResNet-101 encoder = 40.7 GF/pair on torch/cuDNN (out of scope, SURVEY §8f rank 1); head = "
                   f"{precision} kernels of this repo; images resident in HBM")
    del model, xs
    torch.cuda.empty_cache()
    return out


def full_pipeline_sharded(args, ctx, precision, encoder_precision="bf16"):
    """BASELINE configs[4] shape at N GPUs: every rank runs the whole pipeline (uint8 frames in pinned host
    memory -> FramePipeline -> 3D joints) on its shard, one all-gather of the 3D joints + MPJPE sums per
    step; aggregate pairs/s = all ranks' pairs / max-over-ranks device time."""
    import torch.distributed as dist
    import fast_3d_human_pose_estimation_b200 as pkg
    from fast_3d_human_pose_estimation_b200 import synth, dist as cdist
    dev, B, world, rank = ctx["dev"], args.batch, ctx["world"], ctx["rank"]
    pipe, err = None, None
    try:
        torch.manual_seed(0)
        m = pkg.CDRNet(synth.make_cfg(101, JOINTS), precision=precision, encoder_precision=encoder_precision)
        m.load_state_dict(ctx["sd"], strict=False)
        m = m.to(dev).eval()
        gen = torch.Generator().manual_seed(7 + rank)
        frames_h = torch.randint(0, 256, (2, B, 256, 256, 3), dtype=torch.uint8, generator=gen).pin_memory()
        pipe = pkg.FramePipeline(m, B, gt={"gt3d": ctx["g3"], "gt2d_l": ctx["g2l"], "gt2d_r": ctx["g2r"], "vis": ctx["vis"]})
    except Exception as e:
        err = repr(e)[:200]
    ok = torch.tensor([0.0 if pipe is None else 1.0], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)            # enter the collective section only if every rank is ready
    if float(ok[0]) < 1.0:
        return {"error": err or "another rank failed to build the pipeline"}
    n_total = B * world
    xyz_h = torch.empty((n_total, JOINTS, 3), dtype=torch.float32).pin_memory()
    sums_h = torch.empty(4, dtype=torch.float64).pin_memory()

    def post(slot):
        x, s = cdist.gather_results(pipe.xyz_dev[slot], pipe.sums_dev[slot], n_total)
        xyz_h.copy_(x, non_blocking=True)
        sums_h.copy_(s, non_blocking=True)

    def run(k):
        pipe.submit(frames_h, ctx["P_h"], post)
        for _ in range(k - 1):
            pipe.submit(frames_h, ctx["P_h"], post)
            pipe.collect()
        pipe.collect()
    run(3)
    dist.barrier(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kk = 10
    a.record()
    run(kk)
    b.record()
    dist.barrier(); torch.cuda.synchronize()
    t = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0]) / kk
    return {"e2e_uint8_frames_host": {"pairs_per_s": n_total / (ms / 1e3), "ms_per_step": ms, "n_gpus": world,
                                      "encoder_precision": encoder_precision,
                                      "pairs_per_gpu": B, "h2d_bytes_per_step_per_gpu": frames_h.numel() + 2 * B * 48,
                                      "collective": "1 all-gather of (B,19,3)+32 B per step",
                                      "api": "FramePipeline per rank (ResNet-101 encoder + head on this repo's kernels)"}}


def run_ours(args):
    import torch.distributed as dist
    from fast_3d_human_pose_estimation_b200 import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from fast_3d_human_pose_estimation_b200 import dist as cdist
    orig_affinity = os.sched_getaffinity(0)
    numa_cpus = cdist.bind_to_gpu_numa(local)      # before any pinned allocation (first touch)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, K, W = args.batch, args.steps, max(3, args.warmup)

    ctx = {"world": world, "rank": rank, "local": local, "dev": dev, "W": W,
           "sd": synth.make_head_state_dict(seed=0, calibrated=True)}
    ctx["feats_h"] = [f.pin_memory() for f in synth.make_features(B, seed=1 + rank)]
    cams = synth.make_cameras(B, seed=2 + rank)
    gt = synth.make_gt(cams, seed=3 + rank)
    ctx["P_h"] = [torch.from_numpy(cams["P_l"]).pin_memory(), torch.from_numpy(cams["P_r"]).pin_memory()]
    ctx["feats"] = [f.to(dev) for f in ctx["feats_h"]]
    ctx["Ps"] = [p.to(dev) for p in ctx["P_h"]]
    ctx["g3"] = torch.from_numpy(gt["gt3d"]).to(dev)
    ctx["g2l"] = torch.from_numpy(gt["gt2d_l"]).to(dev)
    ctx["g2r"] = torch.from_numpy(gt["gt2d_r"]).to(dev)
    ctx["vis"] = torch.from_numpy(gt["vis"]).to(dev)
    ctx["flush"] = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    ctx["numa_cpus"] = numa_cpus
    main_res = measure(args, args.precision, ctx, dump_dir=args.dump_outputs)
    other = None
    if args.precision != "bf16" and not args.single_precision:
        other = measure(args, "bf16", ctx)      # the tensor-core configuration, reported alongside

    fp_multi = None
    if world > 1 and not args.no_full_pipeline:
        # every rank takes part (collectives).  fp32 head: the reference-precision pipeline (f16x2 encoder) and, beside
        # it, the bf16 encoder
        if args.precision in ("fp32", "f16x2"):
            fp_multi = full_pipeline_sharded(args, ctx, args.precision, "fp32")
            extra = full_pipeline_sharded(args, ctx, args.precision, "bf16")
            fp_multi["e2e_uint8_frames_host_encoder_bf16"] = extra.get("e2e_uint8_frames_host", extra)
        else:
            fp_multi = full_pipeline_sharded(args, ctx, args.precision)
    c5, c5_bf16 = None, None
    if not args.no_full_pipeline and not args.no_config5:
        # at the reference's precision end to end (f16x2 encoder + fp32 head) when this run's head is the fp32 one; the
        # bf16 encoder (faster, below the reference's precision) is reported next to it
        ref_prec = args.precision in ("fp32", "f16x2")
        try:
            c5 = config5(args, ctx, args.precision, encoder_precision="fp32" if ref_prec else "bf16")   # every rank takes part
            if ref_prec:
                c5_bf16 = config5(args, ctx, args.precision, encoder_precision="bf16")
        except Exception as e:
            if world > 1:
                raise
            c5 = {"error": repr(e)[:200]}
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            # CPU baseline on a bounded sample of the same workload (rank 0, N=1 only)
            os.sched_setaffinity(0, orig_affinity)      # the CPU arm uses every host core again
            cores = os.cpu_count() or 1
            torch.set_num_threads(cores)
            cb = min(B, 32)
            cstep, ckind = cpu_head_runner(cb)
            cstep()
            ts = []
            for _ in range(3):
                t0 = time.perf_counter(); cstep(); ts.append(time.perf_counter() - t0)
            cpu = {"value": cb / float(np.median(ts)), "unit": UNIT, "cores": cores, "kind": ckind,
                   "sample": f"{cb} of {B} stereo pairs, head only, fp32, "
                             + ("unmodified reference CDRNet.forward (encoder stubbed) + calc_mpjpe"
                                if ckind == "reference" else "oracle port") + " on torch CPU, median of 3",
                   "cpu": cpu_model()}
        ref_gpu = None
        if world == 1 and not args.no_cpu_baseline:
            try:
                ref_gpu = reference_head_on_gpu(B, dev)
            except Exception as e:
                ref_gpu = {"error": repr(e)[:200]}
        line = {
            "metric": METRIC, "value": main_res["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": main_res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "config": bench_config(B, world),
            "host_binding": (f"rank 0 bound to {len(numa_cpus)} CPUs local to its GPU (NVML affinity)"
                             if numa_cpus else "none"),
        }
        for k in ("e2e", "gpu_launches", "launches_per_step", "roofline", "roofline_hbm", "stages_ms",
                  "decoder_tflops", "decoder_frac_of_peak", "head_tflops", "clocks", "wall_s_timed_region", "sustained",
                  "mpjpe", "sharded_check"):
            line[k] = main_res[k]
        line["cpu_baseline"] = cpu
        if world == 1 and not args.no_stream_microbench:
            line["roofline_hbm_stream"] = stream_microbench(dev)
            for key, fn in (("config4_softargmax_dlt_1m_poses", config4_1m_poses), ("roofline_hbm_ftl", ftl_stream),
                            ("backward_ops", backward_stream)):
                try:
                    line[key] = fn(dev)
                except Exception as e:                  # secondary numbers: never lose the main line
                    line[key] = {"error": repr(e)[:200]}
        if other is not None:
            line["bf16"] = other
        if world == 1 and not args.no_full_pipeline:
            try:
                line["full_pipeline"] = full_pipeline(args, ctx, args.precision)
            except Exception as e:                      # secondary number: never lose the main line
                line["full_pipeline"] = {"error": repr(e)[:200]}
        if fp_multi is not None:
            line["full_pipeline"] = fp_multi
        if c5 is not None:
            line["config5_full_pipeline_1024_pairs"] = c5
            if c5_bf16 is not None:
                line["config5_full_pipeline_1024_pairs_encoder_bf16"] = c5_bf16
        if ref_gpu is not None:
            line["reference_head_same_gpu"] = ref_gpu
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    # stdout carries the one JSON line; NCCL's own log (version banner, "comm ... nranks N" lines when the caller
    # sets NCCL_DEBUG=INFO) stays enabled but goes to stderr unless the caller chose a file
    if "CDR_NCCL_DEBUG" in os.environ:
        os.environ["NCCL_DEBUG"] = os.environ["CDR_NCCL_DEBUG"]
    if os.environ.get("NCCL_DEBUG"):
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="stereo pairs per GPU per step")
    ap.add_argument("--precision", default="fp32", choices=["fp32", "tf32x3", "fp32_ffma", "bf16"],
                    help="fp32 = fp32 results on tcgen05: decoder on scaled fp16 two-term operands, fusion block 3xTF32 "
                         "(default); tf32x3 = 3xTF32 everywhere; fp32_ffma = CUDA cores; bf16 = tcgen05 bf16")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stream-microbench", action="store_true")
    ap.add_argument("--no-full-pipeline", action="store_true")
    ap.add_argument("--no-sustained", action="store_true", help="skip the 2 s back-to-back (power-capped) measurement")
    ap.add_argument("--no-config5", action="store_true", help="skip the 1024-pair sharded full-pipeline run")
    ap.add_argument("--single-precision", action="store_true",
                    help="fp32 run only: skip the bf16 tensor-core measurement reported alongside")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs (2D joints per view, 3D joints, MPJPE sums) as DIR/<name>.npy; "
                         "the inputs are seeded, so runs with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs dumps the timed GPU path: it needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
