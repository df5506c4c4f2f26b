"""Host-side pieces of bench.py that must not break the one JSON line (CPU), and what --dump-outputs writes (GPU)."""
import importlib.util
import json
import os
import subprocess
import sys
import time

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


class _FakeProc:
    def terminate(self):
        pass


def test_clock_sampler_window_and_reasons():
    b = _bench()
    s = b.ClockSampler(0)
    s.mode, s.proc = "nvidia-smi", _FakeProc()
    t0 = time.perf_counter()
    row = lambda t, sm, pw, cap: (t, float(sm), 1965.0, pw, ["sw_power_cap"] if cap else [])
    s.rows = [row(t0 - 1.0, 1965, 250.0, False),                    # before the window: ignored
              row(t0 + 0.01, 1700, 990.0, True), row(t0 + 0.03, 1680, 1001.5, True),
              row(t0 + 5.0, 1965, 200.0, False)]                    # after: ignored
    c = s.stop(t0, t0 + 0.04)
    assert c["samples"] == 2 and c["sm_mhz"] == 1690.0 and c["sm_max_mhz"] == 1965.0 and c["sm_mhz_min"] == 1680.0
    assert c["reasons"] == ["sw_power_cap"] and c["power_w_max"] == 1001.5 and c["window"] == "timed region"
    # a region shorter than the sampling period falls back to the nearest samples and says so
    s2 = b.ClockSampler(0)
    s2.mode, s2.proc = "nvidia-smi", _FakeProc()
    s2.rows = [row(t0 - 0.05, 1965, 300.0, False)]
    c2 = s2.stop(t0, t0 + 0.001)
    assert c2["samples"] == 1 and c2["window"].startswith("nearest")
    # the nvidia-smi fallback parses its csv rows into the same tuples
    s4 = b.ClockSampler(0)

    class _P:
        stdout = ["0, 1700, 1965, 990.0, 0x4, Not Active, Not Active, Not Active, Active\n", "garbage\n"]
    s4.proc = _P()
    s4._read()
    assert len(s4.rows) == 1 and s4.rows[0][1:] == (1700.0, 1965.0, 990.0, ["sw_power_cap"])
    # no NVML / nvidia-smi at all
    s3 = b.ClockSampler(0)
    assert s3.stop(t0, t0 + 1)["sm_mhz"] is None


def test_both_arms_share_one_config():
    """The driver compares the `config` of `--impl ours` and `--impl reference` (same_config): one function."""
    b = _bench()
    c = b.bench_config(64, 1)
    assert c == b.bench_config(64, 1) and c["workload"].startswith("CDRNet head") and "BASELINE configs[1]" in c["workload"]
    assert b.bench_config(64, 8)["parallelism"] == "dp8" and json.dumps(c)


def test_dump_outputs_writes_float_npy(tmp_path):
    """--dump-outputs: one DIR/<name>.npy per output, float32 / float64 kept, anything else widened to float64."""
    import numpy as np
    import torch
    b = _bench()
    xyz = torch.arange(12, dtype=torch.float32).reshape(1, 4, 3)
    b.dump_outputs(str(tmp_path / "d"), {"xyz": xyz, "sums": torch.ones(4, dtype=torch.float64),
                                         "u8": torch.full((2, 2), 7, dtype=torch.uint8)})
    assert sorted(os.listdir(tmp_path / "d")) == ["sums.npy", "u8.npy", "xyz.npy"]
    a = np.load(tmp_path / "d" / "xyz.npy")
    assert a.dtype == np.float32 and np.array_equal(a, xyz.numpy())
    assert np.load(tmp_path / "d" / "sums.npy").dtype == np.float64
    u8 = np.load(tmp_path / "d" / "u8.npy")
    assert u8.dtype == np.float64 and (u8 == 7).all()
    # more than the limit in all: refused before anything is written
    big = torch.zeros(b.DUMP_LIMIT_BYTES // 8 + 1, dtype=torch.float64)
    with pytest.raises(ValueError, match="limit"):
        b.dump_outputs(str(tmp_path / "big"), {"big": big})
    assert not (tmp_path / "big").exists()
    # only the GPU arm is timed with outputs to dump
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs",
                        str(tmp_path / "r")], capture_output=True, text=True)
    assert r.returncode != 0 and "--impl ours" in r.stderr and not (tmp_path / "r").exists()


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(cuda_pkg, tmp_path):
    """bench.py --steps 1 --dump-outputs: the dumped arrays are what CDRNet.head + mpjpe_sums return on the bench's
    seeded inputs (the same model, weights and batch rebuilt here), bit for bit."""
    import numpy as np
    import torch
    from fast_3d_human_pose_estimation_b200 import synth
    d = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1",
                        "--dump-outputs", str(d), "--single-precision", "--no-cpu-baseline", "--no-stream-microbench",
                        "--no-full-pipeline", "--no-sustained", "--no-config5"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 1
    b = 64
    m = cuda_pkg.CDRNet(synth.make_cfg(18, 19), precision="fp32")
    m.load_state_dict(synth.make_head_state_dict(seed=0, calibrated=True), strict=False)
    m = m.cuda().eval()
    feats = [f.cuda() for f in synth.make_features(b, seed=1)]
    cams = synth.make_cameras(b, seed=2)
    gt = synth.make_gt(cams, seed=3)
    Ps = [torch.from_numpy(cams["P_l"]).cuda(), torch.from_numpy(cams["P_r"]).cuda()]
    (kl, kr), xyz = m.head(feats, Ps)
    g = [torch.from_numpy(gt[k]).cuda() for k in ("gt3d", "gt2d_l", "gt2d_r", "vis")]
    sums = cuda_pkg.mpjpe_sums([kl, kr], xyz, *g)
    got = {n: np.load(d / (n + ".npy")) for n in ("kp_l", "kp_r", "xyz", "mpjpe_sums")}
    assert got["xyz"].dtype == np.float32 and got["mpjpe_sums"].dtype == np.float64
    for n, want in (("kp_l", kl), ("kp_r", kr), ("xyz", xyz), ("mpjpe_sums", sums)):
        assert np.array_equal(got[n], want.cpu().numpy()), n


def test_peaks_and_constants():
    b = _bench()
    p = b.peaks()
    assert p["hbm_gbs"] > 1000 and p["tflops_sustained"] <= p["tflops_burst"]
    # algorithmic work per stereo pair (SURVEY §8d): decoder 7595.9 MF, fused soft-argmax + DLT 623 220 B
    dec = sum(b.FLOP_PER_PAIR[k] for k in ("deconv1", "deconv2", "deconv3", "final_1x1"))
    assert b.FLOP_PER_PAIR["deconv3_tail"] == b.FLOP_PER_PAIR["deconv3"] + b.FLOP_PER_PAIR["final_1x1"]
    assert abs(dec - 7595.9e6) < 1e5 and b.SOFTARGMAX_DLT_BYTES_PER_POSE == 2 * 19 * 4096 * 4 + 96 + 304 + 228
    t = b.ncu_traffic()
    top = t["fp32"].get("deconv3_tail", t["fp32"].get("deconv3"))          # r02: fused tail; r01: deconv3
    assert "fp32" in t and top > 1e8 and json.dumps(t)
