"""SURVEY §8f rank 4: the extracted-MADS frame reader and the inference.py evaluation loop on this library
(fast_3d_human_pose_estimation_b200/mads.py) against the reference's own LoadMADSData (tools/load.py:15-102) and its
own per-frame loop (inference.py:70-101,130-152) on a small synthetic dataset written in extract_data.py's layout."""
import json
import os

import numpy as np
import pytest
import torch

import refdrivers as RD
from fast_3d_human_pose_estimation_b200 import mads, synth
from oracle import refload


def _write_dataset(root, n_frames=5, hw=(300, 420), seed=3):
    import cv2
    rng = np.random.default_rng(seed)
    cams = synth.make_cameras(1, seed=seed + 1)
    K = np.array([[900.0, 0, hw[1] / 2], [0, 900.0, hw[0] / 2], [0, 0, 1]])      # intrinsics of the UNcropped frame
    base = os.path.join(root, "valid", "HipHop", "seq_01")
    for sub in ("left", "right", "pose"):
        os.makedirs(os.path.join(base, sub), exist_ok=True)
    calibs = {f"cam_{v}": {"intrinsics": K.tolist(), "rotation": cams[f"R_{v[0]}"][0].tolist(),
                           "translation": cams[f"T_{v[0]}"][0].tolist(), "distortion_coeffs": [0.0] * 5}
              for v in ("left", "right")}
    for i in range(n_frames):
        for sub in ("left", "right"):
            img = cv2.GaussianBlur(rng.integers(0, 256, (*hw, 3), dtype=np.uint8), (9, 9), 3)
            cv2.imwrite(os.path.join(base, sub, f"{sub}_{i:04d}.jpg"), img)
        pose = rng.uniform([-500, -800, -300], [500, 800, 300], size=(19, 3))
        if i == 1:
            pose[7] = np.nan
        with open(os.path.join(base, "pose", f"gt_pose_{i:04d}.json"), "w") as f:
            json.dump({"calibs_info": calibs, "pose_3d": pose.tolist()}, f, indent=4, sort_keys=True)
    return os.path.join(root, "valid")


def test_mads_frames_match_reference_loader(tmp_path):
    data = _write_dataset(str(tmp_path))
    ours = mads.MADSFrames(data, [256, 256], "HipHop")
    assert len(ours) == 5
    items = list(ours)
    l, r, meta = items[0]
    assert l.shape == (256, 256, 3) and l.dtype == np.uint8 and meta["cam_left"]["intrinsics"].shape == (3, 3)
    # the crop keeps the principal point at the centre of the 256-px frame and scales the focal length by 256 / 300
    np.testing.assert_allclose(meta["cam_left"]["intrinsics"], [[768.0, 0, 128], [0, 768.0, 128], [0, 0, 1]], atol=1e-3)
    with pytest.raises(AssertionError):
        os.remove(ours.pose[0])
        mads.MADSFrames(data, [256, 256], "HipHop")
    if not refload.available():
        pytest.skip("reference sources not present: structural checks only")
    data = _write_dataset(str(tmp_path / "again"))
    ours = list(mads.MADSFrames(data, [256, 256], "HipHop"))
    load_mod = refload._import(["tools.load"])[0]
    ref = list(load_mod.LoadMADSData(data, [256, 256], "HipHop"))
    assert len(ref) == len(ours)
    for (l, r, m), (rl, rr, rm) in zip(ours, ref):
        assert np.array_equal(l, rl) and np.array_equal(r, rr)
        for cam in ("cam_left", "cam_right"):
            assert np.array_equal(m[cam]["intrinsics"], rm[cam]["intrinsics"])
            assert m[cam]["rotation"] == rm[cam]["rotation"] and m[cam]["translation"] == rm[cam]["translation"]
        assert np.array_equal(np.array(m["pose_3d"]), np.array(rm["pose_3d"]), equal_nan=True)


@pytest.mark.gpu
def test_evaluate_sequence_matches_reference_loop(cuda_pkg, tmp_path):
    """The loop of inference.py:130-152 (CDRNetInferencer.estimate per frame, errors averaged over frames) run by the
    UNMODIFIED reference on this GPU, against evaluate_sequence (batched, device-side P construction and MPJPE sums).
    Where the reference's sources are absent: against that loop's recorded result (tests/golden/reference_recorded.json)."""
    data = _write_dataset(str(tmp_path / "d"), n_frames=4)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    if RD.available():
        inference_mod, _ = refload.load_drivers()
        cfg = refload.load_config("mads_3d.yaml")
        sd = RD.seeded_state_dict(cuda_pkg.CDRNet, cfg)
        RD._blank_plot(inference_mod)
        with RD.workdir_with_checkpoint(tmp_path, cfg, sd, "best.pth"):
            inf = inference_mod.CDRNetInferencer(cfg)
            errs = []
            with torch.no_grad():
                for l, r, meta in mads.MADSFrames(data, cfg.MODEL.IMAGE_SIZE, "HipHop"):
                    errs.append(inf.estimate(l, r, meta)[1])
        want = np.mean(np.array(errs, dtype=np.float64), axis=0)
    else:
        cfg = synth.make_cfg(101, 19)                      # the two values of configs/mads_3d.yaml the models read
        cfg.MODEL.IMAGE_SIZE = [256, 256]
        sd = RD.seeded_state_dict(cuda_pkg.CDRNet, cfg)
        rec = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_recorded.json")))["mads_sequence"]
        want = np.array([rec["mpjpe_2d"], rec["mpjpe_3d"]])
    m = cuda_pkg.CDRNet(cfg)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    got = mads.evaluate_sequence(m, mads.MADSFrames(data, cfg.MODEL.IMAGE_SIZE, "HipHop"), batch=3)
    print(f"\nMADS loop: ours MPJPE2D {got['mpjpe_2d']:.6f} MPJPE3D {got['mpjpe_3d']:.6f} | reference loop {want[0]:.6f} {want[1]:.6f}")
    assert got["frames"] == 4 and got["pred_3d"].shape == (4, 19, 3) and got["pred_2d"].shape == (2, 4, 19, 2)
    assert abs(got["mpjpe_2d"] - want[0]) <= 1e-3
    assert abs(got["mpjpe_3d"] - want[1]) <= max(1e-2, 1e-4 * want[1])
    # the same loop with the ENCODER on this library too, at the reference's precision (raw uint8 frames -> fused
    # normalisation -> f16x2 ResNet -> fp32 head): the whole of inference.py's arithmetic without torch kernels
    m2 = cuda_pkg.CDRNet(cfg, encoder_precision="fp32")
    m2.load_state_dict(sd)
    m2 = m2.cuda().eval()
    got2 = mads.evaluate_sequence(m2, mads.MADSFrames(data, cfg.MODEL.IMAGE_SIZE, "HipHop"), batch=3)
    print(f"MADS loop, f16x2 encoder: MPJPE2D {got2['mpjpe_2d']:.6f} MPJPE3D {got2['mpjpe_3d']:.6f}")
    assert abs(got2["mpjpe_2d"] - want[0]) <= 1e-3
    assert abs(got2["mpjpe_3d"] - want[1]) <= max(1e-2, 1e-4 * want[1])
