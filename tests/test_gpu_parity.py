"""GPU parity: the CUDA path (through the C ABI / the reference-shaped shim) against the oracle
on the same seeded inputs, against the reference's golden vectors, and through size-independent
properties at BASELINE.json's sizes.  Tolerances are the north-star's: 2D <= 1e-3 px,
3D <= 1e-2 mm, MPJPE <= 1e-3 mm for the fp32 path against the fp64 oracle on the calibrated
90-degree rig (SURVEY.md §8d); integer/index work is bit-exact."""
import ctypes as C

import numpy as np
import pytest
import torch

from fast_3d_human_pose_estimation_b200 import synth
from oracle import cdr_oracle as O

pytestmark = pytest.mark.gpu

TOL_2D_PX, TOL_3D_MM, TOL_MPJPE_MM = 1e-3, 1e-2, 1e-3


def _model(pkg, sd, joints=19, precision="fp32"):
    m = pkg.CDRNet(synth.make_cfg(18, joints), nj=joints, precision=precision)
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected
    return m.cuda().eval()


def _oracle64(sd, feats, cams, taps=None):
    sd64 = O.cast_state_dict(sd, torch.float64)
    Ps = [torch.from_numpy(cams["P_l"]).double(), torch.from_numpy(cams["P_r"]).double()]
    with torch.no_grad():
        p2, p3 = O.head_forward(sd64, [f.double() for f in feats], Ps, taps=taps)
    return [x.numpy() for x in p2], p3.numpy()


def _run_head(m, feats, cams, taps=False):
    Ps = [torch.from_numpy(cams["P_l"]).cuda(), torch.from_numpy(cams["P_r"]).cuda()]
    out = m.head([f.cuda() for f in feats], Ps, taps=taps)
    torch.cuda.synchronize()
    return out


def _dlt64(cams, kp_l, kp_r):
    """fp64 oracle DLT (models/cdrnet.py:151-179 looped over joints) on given 2D joints."""
    projs = torch.stack([torch.from_numpy(cams["P_l"]).double(), torch.from_numpy(cams["P_r"]).double()], 1)
    kl, kr = torch.as_tensor(kp_l).double(), torch.as_tensor(kp_r).double()
    return np.stack([O.dlt(projs, torch.stack([kl[:, k], kr[:, k]], 1)).numpy() for k in range(kl.shape[1])], 1)


def _dlt_sensitivity(cams, kp_l, kp_r, delta=1e-3):
    """mm of 3D motion per px of 2D motion, per joint (finite differences through the oracle).
    Random-init heads predict 2D joints that violate the epipolar constraint, which makes the
    un-normalised DLT of the reference badly conditioned for some joints (thousands of mm/px);
    the 3D gate has to be read against this."""
    base = _dlt64(cams, kp_l, kp_r)
    k = np.zeros(base.shape[:2])
    for view in range(2):
        for c in range(2):
            pl, pr = np.array(kp_l, dtype=np.float64), np.array(kp_r, dtype=np.float64)
            (pl if view == 0 else pr)[..., c] += delta
            k = np.maximum(k, np.abs(_dlt64(cams, pl, pr) - base).max(-1) / delta)
    return k


def check_3d(cams, kl, kr, xyz, o2, o3, label="", flat=True):
    """The 3D gates: (1) our DLT against the fp64 oracle DLT on OUR 2D joints: <= 1e-2 mm
    (isolates the kernel); (2) end to end against the fp64 oracle: <= 1e-2 mm plus what the
    2D difference explains through the oracle's own sensitivity."""
    kl, kr, xyz = kl.cpu().numpy(), kr.cpu().numpy(), xyz.cpu().numpy()
    same2d = np.abs(xyz - _dlt64(cams, kl, kr)).max(-1)
    kappa = _dlt_sensitivity(cams, o2[0], o2[1])
    d2 = np.maximum(np.abs(kl - o2[0]).max(-1), np.abs(kr - o2[1]).max(-1))
    d3 = np.abs(xyz - o3).max(-1)
    ulp3 = np.abs(o3).max(-1) * 2.0 ** -23          # fp32 output rounding of the coordinates
    print(f"\n{label} DLT on identical 2D: max {same2d.max():.2e} mm | end-to-end d3D max {d3.max():.2e} mm, "
          f"d2D max {d2.max():.2e} px, kappa median {np.median(kappa):.1f} max {kappa.max():.1f} mm/px; "
          f"well-conditioned joints (kappa<=25): {int((kappa <= 25).sum())}/{kappa.size}, "
          f"their d3D max {d3[kappa <= 25].max() if (kappa <= 25).any() else float('nan'):.2e} mm")
    assert np.all(same2d <= TOL_3D_MM + ulp3 + 4 * kappa * 2.0 ** -24 * 256)   # 2D inputs are fp32
    assert np.all(d3 <= TOL_3D_MM + ulp3 + 4 * kappa * d2)
    good = kappa <= 25
    if flat and good.any():
        # the flat north-star tolerance, end to end, wherever the reference's own DLT is well conditioned
        assert d3[good].max() <= TOL_3D_MM, f"{label} well-conditioned joints: {d3[good].max():.2e} mm > {TOL_3D_MM}"
        assert d2[good].max() <= TOL_2D_PX
    return d2.max(), d3.max()


def _nhwc_to_nchw(t, c):  # (..., 64, C) -> (..., C, 8, 8)
    return t.reshape(*t.shape[:-2], 8, 8, c).permute(*range(t.dim() - 2), -1, -3, -2)


@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "fp32_ffma"])
def test_head_fp32_vs_fp64_oracle_stagewise(cuda_pkg, precision):
    """fp32 results: 'fp32' = tcgen05 with the fusion block and the decoder on scaled fp16 two-term operands (f16x2,
    default); 'tf32x3' = 3xTF32 everywhere; 'fp32_ffma' = CUDA cores."""
    b = 4
    sd = synth.make_head_state_dict(seed=0, calibrated=True, randomize_bn=True)
    feats, cams = synth.make_features(b, seed=1), synth.make_cameras(b, seed=2)
    gt = synth.make_gt(cams, seed=3)
    otaps = {}
    o2, o3 = _oracle64(sd, feats, cams, otaps)
    m = _model(cuda_pkg, sd, precision=precision)
    (kl, kr), xyz, taps = _run_head(m, feats, cams, taps=True)

    def rel(got, want):
        return float(np.abs(got - want).max() / np.abs(want).max())

    pinv = torch.stack(otaps["pinv"]).numpy()
    cat = _nhwc_to_nchw(taps["cf_cat"].cpu(), 800).numpy()
    f = _nhwc_to_nchw(taps["cf_f"].cpu(), 400).numpy()
    fo = _nhwc_to_nchw(taps["f_out"].cpu(), 2048).numpy()
    hm = taps["heatmaps"].cpu().numpy()
    r = {"pinv": rel(taps["pinv"].cpu().numpy(), pinv), "cf_cat": rel(cat, otaps["cf_cat"].numpy()),
         "cf_f": rel(f, otaps["cf_f"].numpy()), "f_out": rel(fo, torch.stack(otaps["f_out"]).numpy()),
         "heat": rel(hm, torch.stack(otaps["heatmaps"]).numpy())}
    print(f"\nstage taps [{precision}] max|err|/max|ref|: " + " ".join(f"{k}={v:.2e}" for k, v in r.items()))
    assert r["pinv"] < 1e-6
    assert r["cf_cat"] < 2e-5 and r["cf_f"] < 2e-5 and r["f_out"] < 2e-5 and r["heat"] < 2e-5

    d2, d3 = check_3d(cams, kl, kr, xyz, o2, o3, f"head B=4 [{precision}]:")
    # the reference's own fp32 rounding, for context (printed with -s)
    with torch.no_grad():
        r2, r3 = O.head_forward(sd, feats, [torch.from_numpy(cams["P_l"]), torch.from_numpy(cams["P_r"])])
    ref_d2 = max(np.abs(r2[0].numpy() - o2[0]).max(), np.abs(r2[1].numpy() - o2[1]).max())
    ref_d3 = np.abs(r3.numpy() - o3).max()
    print(f"\nCUDA {precision} vs fp64 oracle: d2D={d2:.2e}px d3D={d3:.2e}mm | reference fp32 vs fp64: "
          f"d2D={ref_d2:.2e}px d3D={ref_d3:.2e}mm")
    assert d2 <= TOL_2D_PX
    assert d3 <= max(TOL_3D_MM, 3 * ref_d3), "worse than 3x the reference's own fp32 rounding"
    e_gpu = cuda_pkg.calc_mpjpe([kl, kr], xyz, gt["gt3d"], gt["gt2d_l"], gt["gt2d_r"], gt["vis"])
    e_ora = O.calc_mpjpe(o2, o3, gt["gt3d"], gt["gt2d_l"], gt["gt2d_r"], gt["vis"])
    assert abs(e_gpu[0] - e_ora[0]) <= TOL_2D_PX
    # MPJPE on OUR outputs: device kernel vs the oracle's numpy formula, the stated 1e-3 mm
    e_same = O.calc_mpjpe([kl.cpu().numpy(), kr.cpu().numpy()], xyz.cpu().numpy(), gt["gt3d"], gt["gt2d_l"],
                          gt["gt2d_r"], gt["vis"])
    assert abs(e_gpu[1] - e_same[1]) <= 1e-9 and abs(e_gpu[0] - e_same[0]) <= 1e-9
    assert abs(e_gpu[1] - e_ora[1]) <= max(TOL_MPJPE_MM, d3)


@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "fp32_ffma", "bf16"])
@pytest.mark.parametrize("hid", [(96, 128), (192, 256), (444, 592)])
def test_head_other_fusion_widths(cuda_pkg, precision, hid):
    """CDRNet(cfg, fusion_hid_ch1=h1, fusion_hid_ch2=h2) (models/cdrnet.py:89-101) for widths other than the default
    300 / 400, every precision, stage taps and joints against the fp64 oracle (the oracle is shape-generic)."""
    b = 3
    sd = synth.make_head_state_dict(seed=4, calibrated=True, randomize_bn=True, hid=hid)
    feats, cams = synth.make_features(b, seed=1), synth.make_cameras(b, seed=2)
    otaps = {}
    o2, o3 = _oracle64(sd, feats, cams, otaps)
    m = cuda_pkg.CDRNet(synth.make_cfg(18, 19), precision=precision, fusion_hid_ch1=hid[0], fusion_hid_ch2=hid[1])
    assert not m.load_state_dict(sd, strict=False).unexpected_keys
    m = m.cuda().eval()
    (kl, kr), xyz, taps = _run_head(m, feats, cams, taps=True)

    def rel(got, want):
        return float(np.abs(got - want).max() / np.abs(want).max())
    cat = _nhwc_to_nchw(taps["cf_cat"].cpu(), 2 * hid[1]).numpy()
    f = _nhwc_to_nchw(taps["cf_f"].cpu(), hid[1]).numpy()
    fo = _nhwc_to_nchw(taps["f_out"].cpu(), 2048).numpy()
    r = {"cf_cat": rel(cat, otaps["cf_cat"].numpy()), "cf_f": rel(f, otaps["cf_f"].numpy()),
         "f_out": rel(fo, torch.stack(otaps["f_out"]).numpy()),
         "heat": rel(taps["heatmaps"].cpu().numpy(), torch.stack(otaps["heatmaps"]).numpy())}
    d2 = max(np.abs(kl.cpu().numpy() - o2[0]).max(), np.abs(kr.cpu().numpy() - o2[1]).max())
    print(f"\nfusion widths {hid} [{precision}]: " + " ".join(f"{k}={v:.2e}" for k, v in r.items()) + f" d2D={d2:.2e} px")
    if precision == "bf16":
        assert max(r.values()) < 3e-2 and d2 <= 2.0      # bf16 noise of a random-init head (flat heat-maps); taps are the gate
    else:
        assert max(r.values()) < 2e-5 and d2 <= TOL_2D_PX
        check_3d(cams, kl, kr, xyz, o2, o3, f"widths {hid} [{precision}]:", flat=False)
    with pytest.raises(ValueError):
        cuda_pkg.CDRNet(synth.make_cfg(18, 19), fusion_hid_ch1=300, fusion_hid_ch2=300)    # the reference's ftl cannot reshape
    with pytest.raises(NotImplementedError):
        cuda_pkg.CDRNet(synth.make_cfg(18, 19), n_views=3)


@pytest.mark.parametrize("name,b,joints,calib,rbn,rig,t2,t3", [
    ("head_b2", 2, 19, True, True, "wide", TOL_2D_PX, TOL_3D_MM),
    ("head_b3_default_init", 3, 19, False, False, "wide", 5e-2, None),   # stress: logit std ~34
    ("head_b1_j16_narrow", 1, 16, True, True, "narrow", TOL_2D_PX, None),  # ill-conditioned rig
])
def test_head_vs_reference_golden(cuda_pkg, golden, name, b, joints, calib, rbn, rig, t2, t3):
    sd = synth.make_head_state_dict(seed=0, joints=joints, calibrated=calib, randomize_bn=rbn)
    feats, cams = synth.make_features(b, seed=1), synth.make_cameras(b, seed=2, rig=rig)
    m = _model(cuda_pkg, sd, joints)
    (kl, kr), xyz = _run_head(m, feats, cams)
    d2 = max(np.abs(kl.cpu().numpy() - golden[f"{name}.f64.kp_l"]).max(),
             np.abs(kr.cpu().numpy() - golden[f"{name}.f64.kp_r"]).max())
    ref = golden[f"{name}.f64.xyz"]
    d3 = np.abs(xyz.cpu().numpy() - ref).max()
    ref32 = np.abs(golden[f"{name}.f32.xyz"] - ref).max()
    print(f"\n{name}: d2D={d2:.2e}px d3D={d3:.2e}mm (reference fp32 vs fp64 d3D={ref32:.2e}mm)")
    assert d2 <= t2
    o2 = [golden[f"{name}.f64.kp_l"], golden[f"{name}.f64.kp_r"]]
    if t3 is not None:
        check_3d(cams, kl, kr, xyz, o2, ref, name)
        assert d3 <= max(t3, 3 * ref32)
    else:  # un-gated conditioning cases: we must not be worse than the reference's own fp32
        assert d3 <= max(10 * ref32, 1.0)


@pytest.mark.parametrize("kind", ["randn3", "randn30", "blob", "flat", "onehot"])
def test_softargmax_kernel(cuda_pkg, kind):
    n = 37
    g = torch.Generator().manual_seed(5)
    if kind == "randn3":
        h = 3 * torch.randn(n, 64, 64, generator=g)
    elif kind == "randn30":
        h = 30 * torch.randn(n, 64, 64, generator=g)
    elif kind == "blob":
        h = synth.blob_heatmaps(torch.rand(n, 2, generator=g) * 63, seed=1)
    elif kind == "flat":
        h = torch.full((n, 64, 64), -2.5)
    else:
        h = torch.full((n, 64, 64), -1e4)
        h[torch.arange(n), torch.arange(n) % 64, (torch.arange(n) * 7) % 64] = 50.0
    want = (O.process_heatmap(h.double().unsqueeze(0))[0] * 4.0).numpy()
    hd = h.cuda().contiguous()
    kp = torch.empty(n, 2, device="cuda")
    L = cuda_pkg._lib
    L.check(L.lib().cdr_softargmax(L.ptr(hd), n, 64, 64, 4.0, L.ptr(kp), L.current_stream_ptr()))
    torch.cuda.synchronize()
    np.testing.assert_allclose(kp.cpu().numpy(), want, rtol=0, atol=1e-4)   # px


def test_softargmax_edge_sizes(cuda_pkg):
    L = cuda_pkg._lib
    kp = torch.zeros(1, 2, device="cuda")
    h = torch.zeros(1, 64, 64, device="cuda")
    L.check(L.lib().cdr_softargmax(L.ptr(h), 0, 64, 64, 4.0, L.ptr(kp), L.current_stream_ptr()))  # empty
    # non-square / smaller maps (ragged relative to the 16 KB tile)
    g = torch.Generator().manual_seed(6)
    h = torch.randn(5, 32, 48, generator=g) * 4
    b, j, hh, ww = 1, 5, 32, 48
    hm = torch.softmax(h.double().reshape(5, -1), 1).reshape(5, hh, ww)
    cx = (hm.sum(1) * torch.arange(ww)).sum(1)
    cy = (hm.sum(2) * torch.arange(hh)).sum(1)
    kp = torch.empty(5, 2, device="cuda")
    hd = h.cuda()
    L.check(L.lib().cdr_softargmax(L.ptr(hd), 5, hh, ww, 1.0, L.ptr(kp), L.current_stream_ptr()))
    torch.cuda.synchronize()
    np.testing.assert_allclose(kp.cpu().numpy(), torch.stack([cx, cy], 1).numpy(), atol=1e-4)
    with pytest.raises(cuda_pkg.CdrError):     # larger than a tile
        L.check(L.lib().cdr_softargmax(L.ptr(hd), 1, 128, 128, 1.0, L.ptr(kp), L.current_stream_ptr()))


def _dlt_oracle(cams, kp_l, kp_r):
    projs = torch.stack([torch.from_numpy(cams["P_l"]).double(), torch.from_numpy(cams["P_r"]).double()], 1)
    j = kp_l.shape[1]
    return np.stack([O.dlt(projs, torch.stack([torch.from_numpy(kp_l[:, k]).double(),
                                               torch.from_numpy(kp_r[:, k]).double()], 1)).numpy()
                     for k in range(j)], 1)


def test_dlt_kernel(cuda_pkg):
    b, j = 33, 19
    cams = synth.make_cameras(b, seed=7)
    gt = synth.make_gt(cams, seed=8)
    rng = np.random.default_rng(9)
    kp_l = (gt["gt2d_l"] + rng.normal(scale=1.5, size=(b, j, 2))).astype(np.float32)
    kp_r = (gt["gt2d_r"] + rng.normal(scale=1.5, size=(b, j, 2))).astype(np.float32)
    want = _dlt_oracle(cams, kp_l, kp_r)
    L = cuda_pkg._lib
    d = [torch.from_numpy(x).cuda() for x in (cams["P_l"], cams["P_r"], kp_l, kp_r)]
    xyz = torch.empty(b, j, 3, device="cuda")
    L.check(L.lib().cdr_dlt(*[L.ptr(t) for t in d], b, j, L.ptr(xyz), L.current_stream_ptr()))
    torch.cuda.synchronize()
    np.testing.assert_allclose(xyz.cpu().numpy(), want, rtol=0, atol=1e-3)   # mm (fp32 output ulp)
    # exact projections recover the ground truth (KAT T2) to fp32 input rounding
    d[2] = torch.from_numpy(gt["gt2d_l"].astype(np.float32)).cuda().contiguous()
    d[3] = torch.from_numpy(gt["gt2d_r"].astype(np.float32)).cuda().contiguous()
    L.check(L.lib().cdr_dlt(*[L.ptr(t) for t in d], b, j, L.ptr(xyz), L.current_stream_ptr()))
    torch.cuda.synchronize()
    assert np.abs(xyz.cpu().numpy() - gt["gt3d"]).max() < 5.0     # P and 2D were rounded to fp32


@pytest.mark.parametrize("bf16,b", [(False, 21), (True, 21), (False, 64)])
def test_fused_softargmax_dlt_mpjpe(cuda_pkg, bf16, b):
    """Blob heat-maps centred on consistent projections (a well-conditioned DLT) through the whole fused
    soft-argmax + DLT + MPJPE kernel, at B = 64 too: the flat tolerances end to end against the oracle chain
    process_heatmap -> dlt -> calc_mpjpe."""
    j = 19
    cams = synth.make_cameras(b, seed=10)
    gt = synth.make_gt(cams, seed=11)
    cl = torch.from_numpy(gt["gt2d_l"] / 4.0).float()
    cr = torch.from_numpy(gt["gt2d_r"] / 4.0).float()
    hl, hr = synth.blob_heatmaps(cl, seed=1), synth.blob_heatmaps(cr, seed=2)
    if bf16:
        hl, hr = hl.bfloat16(), hr.bfloat16()
    o_l = (O.process_heatmap(hl.double()) * 4.0)
    o_r = (O.process_heatmap(hr.double()) * 4.0)
    want3 = _dlt_oracle(cams, o_l.numpy(), o_r.numpy())
    L = cuda_pkg._lib
    dev = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to("cuda", dt)
    Pl, Pr = dev(cams["P_l"], torch.float32), dev(cams["P_r"], torch.float32)
    g3, g2l, g2r = dev(gt["gt3d"], torch.float64), dev(gt["gt2d_l"], torch.float64), dev(gt["gt2d_r"], torch.float64)
    vis = dev(gt["vis"][..., 0], torch.float64)
    hld, hrd = hl.cuda().contiguous(), hr.cuda().contiguous()
    kl, kr = torch.empty(b, j, 2, device="cuda"), torch.empty(b, j, 2, device="cuda")
    xyz = torch.empty(b, j, 3, device="cuda")
    perr = torch.empty(b, 3, dtype=torch.float64, device="cuda")
    st = L.current_stream_ptr()
    L.check(L.lib().cdr_softargmax_dlt(L.ptr(hld), L.ptr(hrd), int(bf16), L.ptr(Pl), L.ptr(Pr), b, j, 64, 64, 4.0,
                                       L.ptr(kl), L.ptr(kr), L.ptr(xyz), L.ptr(g3), L.ptr(g2l), L.ptr(g2r),
                                       L.ptr(vis), L.ptr(perr), st))
    sums = torch.empty(4, dtype=torch.float64, device="cuda")
    scratch = torch.empty(L.lib().cdr_mpjpe_scratch_bytes(b), dtype=torch.uint8, device="cuda")
    L.check(L.lib().cdr_mpjpe_reduce(L.ptr(perr), b, j, L.ptr(sums), L.ptr(scratch), st))
    torch.cuda.synchronize()
    np.testing.assert_allclose(kl.cpu().numpy(), o_l.numpy(), atol=1e-4)
    np.testing.assert_allclose(kr.cpu().numpy(), o_r.numpy(), atol=1e-4)
    e2, e3 = O.calc_mpjpe([kl.cpu().numpy(), kr.cpu().numpy()], xyz.cpu().numpy(), gt["gt3d"], gt["gt2d_l"],
                          gt["gt2d_r"], gt["vis"])
    s = sums.cpu().numpy()
    assert s[3] == b * j
    np.testing.assert_allclose([(s[0] + s[1]) / (2 * s[3]), s[2] / s[3]], [e2, e3], rtol=1e-10)
    o2e, o3e = O.calc_mpjpe([o_l.numpy(), o_r.numpy()], want3, gt["gt3d"], gt["gt2d_l"], gt["gt2d_r"], gt["vis"])
    d3 = np.abs(xyz.cpu().numpy() - want3).max()
    print(f"\nfused kernel B={b} bf16={bf16}: d3D {d3:.2e} mm, MPJPE kernel ({(s[0] + s[1]) / (2 * s[3]):.6f}, {s[2] / s[3]:.6f}) "
          f"oracle chain ({o2e:.6f}, {o3e:.6f})")
    assert d3 <= TOL_3D_MM
    assert abs(s[2] / s[3] - o3e) <= TOL_MPJPE_MM and abs((s[0] + s[1]) / (2 * s[3]) - o2e) <= TOL_2D_PX
    # blobs sit on the projections of the ground truth -> triangulation lands near it
    if not bf16:
        assert np.abs(xyz.cpu().numpy() - gt["gt3d"]).mean() < 25.0   # blob truncation at the borders biases a few mm


def test_argmax_and_triangulation_bit_exact(cuda_pkg, golden):
    from test_oracle_golden import baseline_inputs
    heat, heat_r, cams = baseline_inputs()
    preds, maxv = cuda_pkg.get_max_preds(heat)
    assert preds.dtype == np.float32
    assert np.array_equal(preds, golden["base.preds"]) and np.array_equal(maxv, golden["base.maxvals"])
    u8_l, u8_r = cuda_pkg.baseline_keypoints(heat), cuda_pkg.baseline_keypoints(heat_r)
    assert u8_l.dtype == np.uint8
    assert np.array_equal(u8_l, golden["base.u8_l"]) and np.array_equal(u8_r, golden["base.u8_r"])
    PL = np.stack([O.get_projection_matrix(cams["K"], cams["R_l"][i], cams["T_l"][i]) for i in range(3)])
    PR = np.stack([O.get_projection_matrix(cams["K"], cams["R_r"][i], cams["T_r"][i]) for i in range(3)])
    one = cuda_pkg.triangulation(PL[0], PR[0], u8_l[0], u8_r[0])          # the reference's per-frame call
    assert one.shape == (19, 3) and one.dtype == np.float64
    np.testing.assert_allclose(one, golden["base.xyz"][0], rtol=0, atol=1e-2)
    allb = cuda_pkg.triangulation(PL, PR, u8_l, u8_r)                     # batched extension
    np.testing.assert_allclose(allb, golden["base.xyz"], rtol=1e-6, atol=1e-2)
    gt = synth.make_gt(cams, seed=6)
    e = cuda_pkg.calc_mpjpe([u8_l[0], u8_r[0]], one, gt["gt3d"][0], gt["gt2d_l"][0], gt["gt2d_r"][0],
                            gt["vis"][0].astype(bool))
    np.testing.assert_allclose(np.array(e), golden["base.mpjpe0"], rtol=1e-9)
    # random maps with planted ties: identical to numpy's first-index rule
    rng = np.random.default_rng(3)
    h = rng.integers(-3, 4, size=(7, 19, 64, 64)).astype(np.float32)     # many exact ties
    p, mv = cuda_pkg.get_max_preds(h)
    op, omv = O.get_max_preds(h)
    assert np.array_equal(p, op) and np.array_equal(mv, omv)


def test_mpjpe_call_styles(cuda_pkg, golden):
    for name, b, joints, rig in [("head_b2", 2, 19, "wide"), ("head_b1_j16_narrow", 1, 16, "narrow")]:
        cams = synth.make_cameras(b, seed=2, rig=rig)
        gt = synth.make_gt(cams, joints=joints, seed=3)
        p2 = [golden[f"{name}.f32.kp_l"], golden[f"{name}.f32.kp_r"]]
        e = cuda_pkg.calc_mpjpe(p2, golden[f"{name}.f32.xyz"], gt["gt3d"], gt["gt2d_l"], gt["gt2d_r"],
                                gt["vis"].astype(np.float32))
        np.testing.assert_allclose(np.array(e), golden[f"{name}.mpjpe"], rtol=1e-12)
        e = cuda_pkg.calc_mpjpe([p2[0][0], p2[1][0]], golden[f"{name}.f32.xyz"][0], gt["gt3d"][0],
                                gt["gt2d_l"][0], gt["gt2d_r"][0], gt["vis"][0].astype(bool))
        np.testing.assert_allclose(np.array(e), golden[f"{name}.mpjpe_frame0"], rtol=1e-12)
    np.testing.assert_allclose(golden["kat.t3"], [(18 / 19 * np.sqrt(2)) / 2, 5 * 18 / 19])
    p3 = np.zeros((19, 3)); g3 = np.zeros((19, 3)); g3[:, 0] = 3; g3[:, 1] = 4
    p2l = np.ones((19, 2)); g2 = np.zeros((19, 2)); vis = np.ones((19, 1), bool); vis[4] = False
    np.testing.assert_allclose(np.array(cuda_pkg.calc_mpjpe([p2l, g2.copy()], p3, g3, g2, g2, vis)), golden["kat.t3"], rtol=1e-14)
    np.testing.assert_allclose(np.array(cuda_pkg.calc_mpjpe([p2l, g2.copy()], p3, g3, g2, g2)),
                               [np.sqrt(2) / 2, 5.0], rtol=1e-14)            # no weights


def test_ftl_identity_and_oracle(cuda_pkg):
    """KAT T6 on the device + FTL against the oracle's reshape/bmm (channel-block layout)."""
    b = 3
    cams = synth.make_cameras(b, seed=12)
    P = torch.from_numpy(cams["P_l"])
    Pinv = torch.linalg.pinv(P.double()).float()
    x = torch.randn(b, 300, 8, 8, generator=torch.Generator().manual_seed(1))
    want = O.ftl(x.double(), Pinv.double())                                # (b,400,8,8)
    L = cuda_pkg._lib
    rows = torch.zeros(b, 64, 304)
    rows[:, :, :300] = x.permute(0, 2, 3, 1).reshape(b, 64, 300)
    xin, out = rows.cuda(), torch.full((b, 64, 400), float("nan"), device="cuda")
    st = L.current_stream_ptr()
    Pinv_d, P_d = Pinv.cuda().contiguous(), P.cuda().contiguous()
    L.check(L.lib().cdr_ftl(L.ptr(xin), 304, L.ptr(Pinv_d), 4, 3, 100, b, 64, L.ptr(out), 400, 400, st))
    back = torch.full((b, 64, 304), float("nan"), device="cuda")
    L.check(L.lib().cdr_ftl(L.ptr(out), 400, L.ptr(P_d), 3, 4, 100, b, 64, L.ptr(back), 304, 304, st))
    torch.cuda.synchronize()
    got = out.cpu().reshape(b, 8, 8, 400).permute(0, 3, 1, 2)
    assert float((got - want).abs().max() / want.abs().max()) < 1e-5
    assert torch.all(back[:, :, 300:] == 0)
    assert float((back.cpu()[:, :, :300] - rows[:, :, :300]).abs().max()) < 5e-3 * float(x.abs().max())
    with pytest.raises(cuda_pkg.CdrError):
        L.check(L.lib().cdr_ftl(L.ptr(xin), 304, L.ptr(P_d), 2, 2, 100, b, 64, L.ptr(out), 400, 400, st))


def test_ftl_scalar_and_vector_paths(cuda_pkg):
    """The 128-bit FTL kernel (blk, pitches, pad multiples of 4 channels) and the scalar kernel
    (anything else: blk = 25 here, and a mis-aligned plane) against the definition
    out[row, r*blk + c] = sum_k m[r,k] * in[row, k*blk + c]  (models/cdrnet.py:45-56)."""
    L = cuda_pkg._lib
    st = L.current_stream_ptr()
    g = torch.Generator().manual_seed(9)
    n, hw = 5, 64
    for blk, in_pitch, out_pitch, out_fill, off in [(100, 304, 400, 400, 0), (100, 304, 800, 400, 400),
                                                    (25, 80, 101, 101, 0), (100, 304, 401, 400, 1)]:
        x = torch.randn(n * hw, in_pitch, generator=g)
        m = torch.randn(n, 4, 3, generator=g)
        xd, md = x.cuda(), m.cuda()
        out = torch.full((n * hw, out_pitch), float("nan"), device="cuda")
        L.check(L.lib().cdr_ftl(L.ptr(xd), in_pitch, L.ptr(md), 4, 3, blk, n, hw, out.data_ptr() + 4 * off, out_pitch,
                                out_fill, st))
        torch.cuda.synchronize()
        want = torch.einsum("nrk,npkc->nprc", m.double(), x[:, :3 * blk].double().reshape(n, hw, 3, blk)).reshape(n * hw, 4 * blk)
        got = out.cpu()
        got = got[:, off:off + out_fill]
        assert float((got[:, :4 * blk].double() - want).abs().max()) < 1e-5 * float(want.abs().max()), (blk, in_pitch)
        assert torch.all(got[:, 4 * blk:] == 0)
        if off == 0 and out_fill < out_pitch:
            assert torch.isnan(out.cpu()[:, out_fill:]).all()       # never writes past out_fill


def test_softargmax_nonfinite_logits_propagate(cuda_pkg):
    """torch.softmax gives NaN for a map that holds NaN or +Inf (models/cdrnet.py:131-133); the 64x64 fast
    path widens its partial sums on the integer pipe, which alone would lose them."""
    L = cuda_pkg._lib
    h = torch.randn(6, 64, 64, generator=torch.Generator().manual_seed(2))
    h[1, 3, 5] = float("nan")
    h[2, 60, 1] = float("inf")
    h[4, 0, 0] = float("-inf")                      # -Inf is an ordinary zero-weight pixel
    want = (O.process_heatmap(h.double().unsqueeze(0))[0] * 4.0).numpy()
    assert np.isnan(want[1]).all() and np.isnan(want[2]).all() and np.isfinite(want[[0, 3, 4, 5]]).all()
    hd, kp = h.cuda(), torch.empty(6, 2, device="cuda")
    L.check(L.lib().cdr_softargmax(L.ptr(hd), 6, 64, 64, 4.0, L.ptr(kp), L.current_stream_ptr()))
    torch.cuda.synchronize()
    got = kp.cpu().numpy()
    assert np.isnan(got[1]).all() and np.isnan(got[2]).all()
    np.testing.assert_allclose(got[[0, 3, 4, 5]], want[[0, 3, 4, 5]], rtol=0, atol=1e-4)


@pytest.mark.parametrize("gain", [1.0, 3.0e4, 1.0e-5])
def test_decoder_f16x2_dynamic_range(cuda_pkg, gain):
    """The f16x2 decoder scales every tensor by a data-dependent power of two: the relative error of
    the heat-maps must not depend on the magnitude of the latents (fp16 alone would overflow at
    gain 3e4 and flush to zero at 1e-5).  BN is the identity here so the network stays positively
    homogeneous up to the final bias."""
    n, joints = 2, 19
    sd = synth.make_head_state_dict(seed=5, joints=joints, calibrated=True, randomize_bn=False, decoder_only=True)
    feats = synth.make_features(n, seed=6)[0] * gain
    want = O.decoder(O.cast_state_dict(sd, torch.float64), feats.double()).numpy()
    dec = cuda_pkg.PoseDecoder(synth.make_cfg(18, joints), precision="f16x2")
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items()})
    dec = dec.cuda().eval()
    got = dec(feats.cuda()).cpu().numpy()
    rel = np.abs(got - want).max() / np.abs(want).max()
    print(f"\ndecoder [f16x2] latents x{gain:g}: rel err {rel:.2e}, max |heat| {np.abs(want).max():.3e}")
    assert np.isfinite(got).all()
    assert rel < 2e-5


@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "fp32_ffma"])
def test_decoder_forward_vs_oracle(cuda_pkg, precision):
    """PoseResNet's decoder half (models/poseresnet.py:17-21) incl. an odd image count."""
    n, joints = 3, 16
    sd = synth.make_head_state_dict(seed=3, joints=joints, calibrated=True, randomize_bn=True, decoder_only=True)
    feats = synth.make_features(n, seed=4)[0]
    want = O.decoder(O.cast_state_dict(sd, torch.float64), feats.double()).numpy()
    dec = cuda_pkg.PoseDecoder(synth.make_cfg(18, joints), precision=precision)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items()})
    dec = dec.cuda().eval()
    got = dec(feats.cuda()).cpu().numpy()
    print(f"\ndecoder [{precision}] rel err {np.abs(got - want).max() / np.abs(want).max():.2e}")
    assert got.shape == (n, joints, 64, 64)
    assert np.abs(got - want).max() / np.abs(want).max() < 2e-5


def test_repack_on_parameter_change(cuda_pkg):
    sd = synth.make_head_state_dict(seed=0)
    feats, cams = synth.make_features(1, seed=1), synth.make_cameras(1, seed=2)
    m = _model(cuda_pkg, sd)
    (a, _), _ = _run_head(m, feats, cams)
    with torch.no_grad():
        m.decoder.final_layer.weight.mul_(2.0)
    (b2, _), _ = _run_head(m, feats, cams)
    assert not torch.equal(a, b2)
    sd2 = dict(sd)
    m.load_state_dict(sd2, strict=False)
    (c, _), _ = _run_head(m, feats, cams)
    assert torch.equal(a, c)


def test_full_size_properties(cuda_pkg):
    """BASELINE config 2 size (B=64): determinism and per-sample independence (batch
    permutation equivariance, shard == slice of the full batch) — size-independent properties
    that hold only if every kernel indexes the batch correctly."""
    b = 64
    sd = synth.make_head_state_dict(seed=0, calibrated=True)
    feats, cams = synth.make_features(b, seed=1), synth.make_cameras(b, seed=2)
    m = _model(cuda_pkg, sd)
    (kl, kr), xyz = _run_head(m, feats, cams)
    (kl2, kr2), xyz2 = _run_head(m, feats, cams)
    assert torch.equal(kl, kl2) and torch.equal(kr, kr2) and torch.equal(xyz, xyz2)
    assert torch.isfinite(xyz).all()
    perm = torch.randperm(b, generator=torch.Generator().manual_seed(0))
    cams_p = {k: (v[perm.numpy()] if isinstance(v, np.ndarray) and v.shape[:1] == (b,) else v) for k, v in cams.items()}
    (klp, krp), xyzp = _run_head(m, [f[perm] for f in feats], cams_p)
    assert torch.equal(klp, kl[perm.cuda()]) and torch.equal(xyzp, xyz[perm.cuda()])
    lo, hi = 40, 53
    cams_s = {k: (v[lo:hi] if isinstance(v, np.ndarray) and v.shape[:1] == (b,) else v) for k, v in cams.items()}
    (kls, _), xyzs = _run_head(m, [f[lo:hi] for f in feats], cams_s)
    assert torch.equal(kls, kl[lo:hi]) and torch.equal(xyzs, xyz[lo:hi])
    # 8 of the 64 pairs, spread over the batch (every 128-row tile of the fusion block holds one), against the fp64 oracle
    idx = np.arange(3, b, 8)
    sub = lambda v: ([v[i] for i in idx] if isinstance(v, list) and len(v) == b else
                     v[idx] if isinstance(v, np.ndarray) and v.shape[:1] == (b,) else v)
    cams8 = {k: sub(v) for k, v in cams.items()}
    o2, o3 = _oracle64(sd, [f[idx] for f in feats], cams8)
    ti = torch.from_numpy(idx).cuda()
    assert np.abs(kl[ti].cpu().numpy() - o2[0]).max() <= TOL_2D_PX and np.abs(kr[ti].cpu().numpy() - o2[1]).max() <= TOL_2D_PX
    check_3d(cams8, kl[ti], kr[ti], xyz[ti], o2, o3, "B=64, 8 pairs spread over the batch:")


def test_full_pipeline_vs_reference_golden(cuda_pkg, golden):
    """BASELINE config 1 shape: ResNet-101 encoder on torch/cuDNN + the CUDA head, against the
    reference's fp64 forward.  The encoder runs in fp32 on the GPU (TF32 off), so the gate is
    the reference's own fp32-vs-fp64 distance with headroom, not the head-only tolerance."""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    cfg = synth.make_cfg(101, 19)
    torch.manual_seed(0)
    m = cuda_pkg.CDRNet(cfg)
    with torch.no_grad():
        m.decoder.final_layer.weight.mul_(0.1)
    m = m.cuda().eval()
    imgs = [i.cuda() for i in synth.make_images(1, seed=1)]
    cams = synth.make_cameras(1, seed=2)
    (kl, kr), xyz = m(imgs, [torch.from_numpy(cams["P_l"]).cuda(), torch.from_numpy(cams["P_r"]).cuda()])
    d2 = max(np.abs(kl.cpu().numpy() - golden["full_b1.f64.kp_l"]).max(), np.abs(kr.cpu().numpy() - golden["full_b1.f64.kp_r"]).max())
    d3 = np.abs(xyz.cpu().numpy() - golden["full_b1.f64.xyz"]).max()
    r2 = max(np.abs(golden["full_b1.f32.kp_l"] - golden["full_b1.f64.kp_l"]).max(), np.abs(golden["full_b1.f32.kp_r"] - golden["full_b1.f64.kp_r"]).max())
    r3 = np.abs(golden["full_b1.f32.xyz"] - golden["full_b1.f64.xyz"]).max()
    print(f"\nfull pipeline: d2D={d2:.2e}px d3D={d3:.2e}mm | reference fp32 vs fp64: {r2:.2e}px {r3:.2e}mm")
    assert kl.shape == (1, 19, 2) and xyz.shape == (1, 19, 3) and kl.is_cuda
    # flat north-star tolerances against the reference's fp64 forward (the reference's own fp32 sits at r2 / r3)
    assert d2 <= TOL_2D_PX and d3 <= TOL_3D_MM


# ------------------------------------------------------------------------------------------
# bf16 tensor-core path (tcgen05 / TMEM / TMA)
def test_bf16_decoder_vs_emulated_oracle(cuda_pkg):
    """The tcgen05 implicit-GEMM decoder against the oracle with bf16 rounding at the same points."""
    from bf16_emulation import decoder_bf16
    n, joints = 3, 19
    sd = synth.make_head_state_dict(seed=3, joints=joints, calibrated=True, randomize_bn=True, decoder_only=True)
    feats = synth.make_features(n, seed=4)[0]
    with torch.no_grad():
        want = decoder_bf16(sd, feats.bfloat16().double()).numpy()
    dec = cuda_pkg.PoseDecoder(synth.make_cfg(18, joints), precision="bf16")
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items()})
    dec = dec.cuda().eval()
    got = dec(feats.cuda()).cpu().numpy()
    err = np.abs(got - want)
    print(f"\nbf16 decoder vs emulated oracle: max {err.max():.3e} mean {err.mean():.3e} (|h| max {np.abs(want).max():.2f})")
    assert err.max() / np.abs(want).max() < 1e-2 and err.mean() / np.abs(want).std() < 1e-3


def test_bf16_head_vs_emulated_and_fp64_oracle(cuda_pkg):
    from bf16_emulation import head_bf16
    b = 5     # odd: M = 320 / 640 rows exercise the partial last 128-row tile
    sd = synth.make_head_state_dict(seed=0, calibrated=True, randomize_bn=True)
    feats, cams = synth.make_features(b, seed=1), synth.make_cameras(b, seed=2)
    m = _model(cuda_pkg, sd, precision="bf16")
    (kl, kr), xyz, taps = _run_head(m, feats, cams, taps=True)
    Ps = [torch.from_numpy(cams["P_l"]), torch.from_numpy(cams["P_r"])]
    pinvs = [taps["pinv"][0].cpu(), taps["pinv"][1].cpu()]
    et = {}
    with torch.no_grad():
        ek, exyz = head_bf16(sd, feats, Ps, pinvs, et)

    def rel(got, want):
        return float(np.abs(got - want).max() / np.abs(want).max())

    r_cat = rel(_nhwc_to_nchw(taps["cf_cat"].cpu(), 800).numpy(), et["cf_cat"].numpy())
    r_f = rel(_nhwc_to_nchw(taps["cf_f"].cpu(), 400).numpy(), et["cf_f"].numpy())
    r_fo = rel(_nhwc_to_nchw(taps["f_out"].cpu(), 2048).numpy(), torch.stack(et["f_out"]).numpy())
    r_hm = rel(taps["heatmaps"].cpu().numpy(), torch.stack(et["heatmaps"]).numpy())
    d2e = max(np.abs(kl.cpu().numpy() - ek[0].numpy()).max(), np.abs(kr.cpu().numpy() - ek[1].numpy()).max())
    o2, o3 = _oracle64(sd, feats, cams)
    d2 = np.concatenate([np.abs(kl.cpu().numpy() - o2[0]).ravel(), np.abs(kr.cpu().numpy() - o2[1]).ravel()])
    print(f"\nbf16 head vs emulated oracle: cat {r_cat:.2e} f {r_f:.2e} f_out {r_fo:.2e} heat {r_hm:.2e} "
          f"2D {d2e:.3e}px | vs fp64 oracle: 2D max {d2.max():.3f} mean {d2.mean():.3f} px")
    assert r_cat < 1e-2 and r_f < 1e-2 and r_fo < 1e-2 and r_hm < 1e-2
    assert d2e < 0.5        # bf16 ties flip a few activations in the fusion block (f_out 3e-3)
    # stated looser bf16 bounds against the fp64 reference (SURVEY.md §8d)
    assert d2.max() <= 1.0 and d2.mean() <= 0.15
    kappa = _dlt_sensitivity(cams, o2[0], o2[1])
    good = kappa <= 25
    d3 = np.abs(xyz.cpu().numpy() - o3).max(-1)
    print(f"bf16 3D on well-conditioned joints: max {d3[good].max():.2f} mean {d3[good].mean():.2f} mm")
    assert d3[good].max() <= 10.0 and d3[good].mean() <= 3.0


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_decoder_many_joints(cuda_pkg, precision):
    """A joint count other than MADS's 19 (24: final layer padded to 32 columns)."""
    n, joints = 2, 24
    sd = synth.make_head_state_dict(seed=7, joints=joints, calibrated=True, randomize_bn=True, decoder_only=True)
    feats = synth.make_features(n, seed=8)[0]
    want = O.decoder(O.cast_state_dict(sd, torch.float64), feats.double()).numpy()
    dec = cuda_pkg.PoseDecoder(synth.make_cfg(18, joints), precision=precision)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items()})
    got = dec.cuda().eval()(feats.cuda()).cpu().numpy()
    rel = np.abs(got - want).max() / np.abs(want).max()
    print(f"\ndecoder [{precision}] 24 joints: rel err {rel:.2e}")
    assert rel < (2e-5 if precision == "fp32" else 2e-2)


def test_head_pipeline_matches_eager(cuda_pkg):
    """HeadPipeline (bench.py's e2e path): depth-2 submit/collect over changing batches returns, per
    batch, exactly what the eager call returns."""
    b = 3
    sd = synth.make_head_state_dict(seed=0, calibrated=True)
    m = _model(cuda_pkg, sd, precision="fp32")
    batches = []
    for i in range(4):
        feats = [f.pin_memory() for f in synth.make_features(b, seed=10 + i)]
        cams = synth.make_cameras(b, seed=20 + i)
        Ps = [torch.from_numpy(cams["P_l"]).pin_memory(), torch.from_numpy(cams["P_r"]).pin_memory()]
        batches.append((feats, Ps))
    gt = synth.make_gt(synth.make_cameras(b, seed=2), seed=3)
    gtd = {k: torch.from_numpy(gt[k]).cuda() for k in ("gt3d", "gt2d_l", "gt2d_r", "vis")}
    pipe = cuda_pkg.HeadPipeline(m, b, gt=gtd)
    got = []
    pipe.submit(*batches[0])
    for i in range(1, 4):
        pipe.submit(*batches[i])
        _, kp, xyz, sums = pipe.collect()
        got.append((kp[0].clone(), kp[1].clone(), xyz.clone(), sums.clone()))
    with pytest.raises(RuntimeError):
        pipe.submit(*batches[0]); pipe.submit(*batches[0])
    while pipe.n_collected < pipe.n_submitted:
        _, kp, xyz, sums = pipe.collect()
        if len(got) < 4:
            got.append((kp[0].clone(), kp[1].clone(), xyz.clone(), sums.clone()))
    for (feats, Ps), (kl_h, kr_h, xyz_h, sums_h) in zip(batches, got):
        (kl, kr), xyz = m.head([f.cuda() for f in feats], [p.cuda() for p in Ps])
        sums = cuda_pkg.mpjpe_sums([kl, kr], xyz, gtd["gt3d"], gtd["gt2d_l"], gtd["gt2d_r"], gtd["vis"])
        torch.cuda.synchronize()
        assert torch.equal(kl.cpu(), kl_h) and torch.equal(kr.cpu(), kr_h) and torch.equal(xyz.cpu(), xyz_h)
        assert torch.equal(sums.cpu(), sums_h)


def test_head_graph_replay_matches_eager(cuda_pkg):
    """CUDA-graph capture of H2D -> head -> MPJPE -> D2H (the e2e path of bench.py): bit-identical to
    the eager call, and re-playable after the pinned inputs are refilled."""
    b = 3
    sd = synth.make_head_state_dict(seed=0, calibrated=True)
    m = _model(cuda_pkg, sd, precision="bf16")
    feats = [f.pin_memory() for f in synth.make_features(b, seed=1)]
    cams = synth.make_cameras(b, seed=2)
    gt = synth.make_gt(cams, seed=3)
    Ps = [torch.from_numpy(cams["P_l"]).pin_memory(), torch.from_numpy(cams["P_r"]).pin_memory()]
    gtd = {k: torch.from_numpy(gt[k]).cuda() for k in ("gt3d", "gt2d_l", "gt2d_r", "vis")}
    hg = cuda_pkg.HeadGraph(m, feats, Ps, gt=gtd)
    (kl, kr), xyz = m.head([f.cuda() for f in feats], [p.cuda() for p in Ps])
    sums = cuda_pkg.mpjpe_sums([kl, kr], xyz, gtd["gt3d"], gtd["gt2d_l"], gtd["gt2d_r"], gtd["vis"])
    kp_h, xyz_h, sums_h = hg.replay()
    assert torch.equal(kp_h[0], kl.cpu()) and torch.equal(kp_h[1], kr.cpu()) and torch.equal(xyz_h, xyz.cpu())
    assert torch.equal(sums_h, sums.cpu())
    new = synth.make_features(b, seed=7)                 # refill the same pinned tensors
    feats[0].copy_(new[0]); feats[1].copy_(new[1])
    (kl2, _), xyz2 = m.head([f.cuda() for f in feats], [p.cuda() for p in Ps])
    kp_h, xyz_h, _ = hg.replay()
    assert torch.equal(kp_h[0], kl2.cpu()) and torch.equal(xyz_h, xyz2.cpu()) and not torch.equal(xyz2, xyz)


def _seeded_resnet(layers, seed=0, randomize_bn=True):
    from fast_3d_human_pose_estimation_b200.encoder import ResNet
    torch.manual_seed(seed)
    r = ResNet(synth.make_cfg(layers, 19))
    if randomize_bn:
        g = torch.Generator().manual_seed(seed + 77)
        for m in r.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                n = m.num_features
                m.weight.data = 1.0 + 0.2 * (torch.rand(n, generator=g) - 0.5)
                m.bias.data = 0.05 * (torch.rand(n, generator=g) - 0.5)
                m.running_mean.data = 0.05 * (torch.rand(n, generator=g) - 0.5)
                m.running_var.data = 1.0 + 0.4 * (torch.rand(n, generator=g) - 0.5)
    return r.eval()


def test_tc_encoder_resnet50_vs_emulated_and_fp32(cuda_pkg):
    """SURVEY §8f rank 1: layer1..layer4 of the encoder on the tcgen05 tap-GEMM kernel (3x3 = 9 shifted
    TMA taps, stride 2 through element-strided tensor maps, residual add in the epilogue) against
    (i) the fp64 evaluation with bf16 rounding at the same points, (ii) the fp32 torch module."""
    from bf16_emulation import encoder_bf16
    from fast_3d_human_pose_estimation_b200.encoder import TcEncoder
    r = _seeded_resnet(50)
    x = torch.randn(3, 3, 256, 256, generator=torch.Generator().manual_seed(5))      # odd image count
    with torch.no_grad():
        want_e = encoder_bf16(r, x.double()).numpy()
        want_32 = r(x).numpy()
    enc = TcEncoder(r.cuda())
    got = enc(x.cuda()).cpu().numpy()
    assert got.shape == (3, 2048, 8, 8)
    enc.torch_stem = True                       # the cuDNN-stem fallback feeds the same kernels
    got_t = enc(x.cuda()).cpu().numpy()
    assert np.abs(got_t - got).max() / np.abs(got).max() < 2e-2
    e_e = np.abs(got - want_e).max() / np.abs(want_e).max()
    e_32 = np.abs(got - want_32).max() / np.abs(want_32).max()
    m_32 = np.abs(got - want_32).mean() / np.abs(want_32).mean()
    print(f"\ntcgen05 ResNet-50 encoder: vs bf16-emulated fp64 {e_e:.2e} | vs fp32 torch max {e_32:.2e} mean {m_32:.2e}")
    assert e_e < 2e-2
    assert e_32 < 6e-2 and m_32 < 2e-2          # stated bf16 bounds for ~50 layers of bf16 activations


def test_tc_encoder_fp32_resnet50_vs_fp64(cuda_pkg):
    """SURVEY §8f rank 1 at the reference's precision: the f16x2 tcgen05 encoder (scaled fp16 hi/lo planes, 3 MMAs
    per product, residual add on planes in the epilogue, three-term fp16 tensor-core stem) against the fp64 evaluation of the same
    network, beside the reference's own fp32 module (torch, TF32 off) against that fp64."""
    from fast_3d_human_pose_estimation_b200.encoder import TcEncoder
    r = _seeded_resnet(50)
    x = torch.randn(3, 3, 256, 256, generator=torch.Generator().manual_seed(5))      # odd image count
    with torch.no_grad():
        import copy
        want = copy.deepcopy(r).double()(x.double()).numpy()
        ref32 = r(x).numpy()
    enc = TcEncoder(r.cuda(), precision="fp32")
    got = enc(x.cuda()).cpu().numpy()
    assert got.shape == (3, 2048, 8, 8)
    e = np.abs(got - want).max() / np.abs(want).max()
    e_ref = np.abs(ref32 - want).max() / np.abs(want).max()
    print(f"\ntcgen05 f16x2 ResNet-50 encoder vs fp64: {e:.2e} of max (reference's own fp32 on CPU: {e_ref:.2e})")
    assert e <= 2e-5
    # uint8 frames: the fused ToTensor + Normalize stem gives the latents of the preprocessed fp32 tensor bit for bit
    from fast_3d_human_pose_estimation_b200.encoder import IMAGENET_MEAN, IMAGENET_STD
    fr = torch.randint(0, 256, (2, 256, 256, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(3))
    mean = torch.tensor(IMAGENET_MEAN).reshape(1, 3, 1, 1)
    std = torch.tensor(IMAGENET_STD).reshape(1, 3, 1, 1)
    pre = fr.permute(0, 3, 1, 2).float().div(255).sub_(mean).div_(std)
    b_u8, _ = enc.rows(fr.cuda())
    b_f32, _ = enc.rows(pre.cuda())
    torch.cuda.synchronize()
    used = 2 * (2 * 64 * 2048 * 2) + 8                # two planes + {amax, scale}; the rest of the buffer is padding
    assert torch.equal(b_u8[:used], b_f32[:used])


def test_full_pipeline_fp32_tc_encoder(cuda_pkg):
    """CDRNet.forward entirely on this library at the reference's precision (encoder_precision='fp32': the encoder's
    fp16 planes feed conv_layer1 without a conversion pass) against the fp64 oracle pipeline; flat north-star
    tolerance on the 2D joints, 3D through the sensitivity-aware gate of check_3d."""
    b = 2
    torch.manual_seed(0)
    m = cuda_pkg.CDRNet(synth.make_cfg(50, 19), precision="fp32", encoder_precision="fp32")
    m.load_state_dict(synth.make_head_state_dict(seed=0, calibrated=True), strict=False)
    cams = synth.make_cameras(b, seed=2)
    P_cpu = [torch.from_numpy(cams["P_l"]), torch.from_numpy(cams["P_r"])]
    g = torch.Generator().manual_seed(1)
    xs_cpu = [torch.randn(b, 3, 256, 256, generator=g) for _ in range(2)]
    sd = _head_sd_of(m)
    with torch.no_grad():
        import copy
        e64 = copy.deepcopy(m.encoder).double().eval()
        lat = [e64(x.double()) for x in xs_cpu]
        o2, o3 = O.head_forward(O.cast_state_dict(sd, torch.float64), lat, [p.double() for p in P_cpu])
    m = m.cuda().eval()
    (kl, kr), xyz = m([x.cuda() for x in xs_cpu], [p.cuda() for p in P_cpu])
    torch.cuda.synchronize()
    d2 = max(float((kl.cpu().double() - o2[0]).abs().max()), float((kr.cpu().double() - o2[1]).abs().max()))
    print(f"\nfull pipeline, f16x2 encoder + fp32 head vs the fp64 oracle pipeline: d2D max {d2:.2e} px")
    assert d2 <= 1e-3
    check_3d(cams, kl, kr, xyz, [o.numpy() for o in o2], o3.numpy(), label="full pipeline f16x2 encoder", flat=False)
    # PoseResNet on the same encoder: heat-maps vs the fp64 oracle decoder
    pr = cuda_pkg.PoseResNet(synth.make_cfg(50, 19), precision="fp32", encoder_precision="fp32")
    pr.encoder.load_state_dict(m.encoder.state_dict())
    pr.decoder.load_state_dict(m.decoder.state_dict())
    pr = pr.cuda().eval()
    hm = pr(xs_cpu[0].cuda()).cpu().double()
    with torch.no_grad():
        want = O.decoder(O.cast_state_dict(sd, torch.float64), lat[0])
    e = float((hm - want).abs().max() / want.abs().max())
    print(f"PoseResNet f16x2 encoder + decoder heat-maps vs fp64: {e:.2e} of max")
    assert e <= 2e-5


def _head_sd_of(m):
    return {k: v.detach().cpu() for k, v in m.state_dict().items() if k.startswith(("CF.", "decoder."))}


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_full_pipeline_tc_encoder(cuda_pkg, precision):
    """CDRNet.forward with encoder_precision='bf16' (encoder rows feed cdr_head_forward_rows directly) against
    the ORACLE of the same pipeline: the reference network evaluated in fp64 with bf16 rounding where the
    tcgen05 encoder rounds (tests/bf16_emulation.py: encoder_bf16), followed by the fp64 oracle head (fp32
    head) or the bf16-emulated oracle head (bf16 head).  Gate: the stated bf16 bound, 2D <= 1 px."""
    from bf16_emulation import encoder_bf16, head_bf16
    b = 2
    torch.manual_seed(0)
    m = cuda_pkg.CDRNet(synth.make_cfg(50, 19), precision=precision, encoder_precision="bf16")
    m.load_state_dict(synth.make_head_state_dict(seed=0, calibrated=True), strict=False)
    cams = synth.make_cameras(b, seed=2)
    P_cpu = [torch.from_numpy(cams["P_l"]), torch.from_numpy(cams["P_r"])]
    g = torch.Generator().manual_seed(1)
    xs_cpu = [torch.randn(b, 3, 256, 256, generator=g) for _ in range(2)]
    sd = _head_sd_of(m)
    with torch.no_grad():
        lat = [encoder_bf16(m.encoder.eval(), x.double()) for x in xs_cpu]          # fp64 values on the bf16 grid
        if precision == "fp32":
            o2, _ = O.head_forward(O.cast_state_dict(sd, torch.float64), lat, [p.double() for p in P_cpu])
        else:
            pinvs = [torch.linalg.pinv(p.double()).float() for p in P_cpu]
            o2, _ = head_bf16(sd, [x.float() for x in lat], P_cpu, pinvs)
    m = m.cuda().eval()
    Ps = [p.cuda() for p in P_cpu]
    xs = [x.cuda() for x in xs_cpu]
    (kl, kr), xyz = m(xs, Ps)
    with torch.no_grad():
        zs = [m.encoder(x) for x in xs]
    (rl, rr), rxyz = m.head(zs, Ps)
    torch.cuda.synchronize()
    d2o = max(float((kl.cpu().double() - o2[0]).abs().max()), float((kr.cpu().double() - o2[1]).abs().max()))
    d2 = max(float((kl - rl).abs().max()), float((kr - rr).abs().max()))
    print(f"\nfull pipeline [{precision}] tcgen05 bf16 encoder: vs bf16-emulated oracle pipeline d2D max {d2o:.3f} px | "
          f"vs the same head on the torch fp32 encoder {d2:.3f} px")
    assert torch.isfinite(xyz).all() and kl.shape == (b, 19, 2) and xyz.shape == (b, 19, 3)
    assert d2o <= 1.0
    assert d2 <= 1.0


def test_frames_u8_match_reference_preprocessing(cuda_pkg):
    """SURVEY §8f rank 2: uint8 HWC frames through the fused ToTensor + Normalize stem give exactly
    the latents of the reference's host-side preprocessing (inference.py:40-44) fed as fp32 tensors,
    and FramePipeline (graph replay, H2D/compute overlap) returns the eager forward_frames result."""
    from fast_3d_human_pose_estimation_b200.encoder import TcEncoder, IMAGENET_MEAN, IMAGENET_STD
    b = 2
    torch.manual_seed(0)
    m = cuda_pkg.CDRNet(synth.make_cfg(50, 19), precision="fp32", encoder_precision="bf16")
    m.load_state_dict(synth.make_head_state_dict(seed=0, calibrated=True), strict=False)
    m = m.cuda().eval()
    g = torch.Generator().manual_seed(3)
    frames = [torch.randint(0, 256, (b, 256, 256, 3), dtype=torch.uint8, generator=g) for _ in range(2)]
    mean = torch.tensor(IMAGENET_MEAN).reshape(1, 3, 1, 1)
    std = torch.tensor(IMAGENET_STD).reshape(1, 3, 1, 1)
    pre = [(f.permute(0, 3, 1, 2).float().div(255).sub_(mean).div_(std)) for f in frames]   # ToTensor + Normalize
    rows_u8, _ = m._tc_encoder.rows(torch.cat(frames, 0).cuda())
    rows_f32, _ = m._tc_encoder.rows(torch.cat(pre, 0).cuda())
    torch.cuda.synchronize()
    assert torch.equal(rows_u8, rows_f32), "fused normalisation must be bit-identical to the reference's preprocessing"
    cams = synth.make_cameras(b, seed=2)
    Ps = [torch.from_numpy(cams["P_l"]), torch.from_numpy(cams["P_r"])]
    (kl, kr), xyz = m.forward_frames([f.cuda() for f in frames], [p.cuda() for p in Ps])
    pipe = cuda_pkg.FramePipeline(m, b)
    fh = torch.stack(frames, 0).pin_memory()
    pipe.submit(fh, [p.pin_memory() for p in Ps])
    pipe.submit([f.pin_memory() for f in frames], [p.pin_memory() for p in Ps])
    for _ in range(2):
        _, kp_h, xyz_h, _ = pipe.collect()
        assert torch.equal(kp_h[0], kl.cpu()) and torch.equal(kp_h[1], kr.cpu()) and torch.equal(xyz_h, xyz.cpu())


def test_frame_pipeline_reference_precision(cuda_pkg):
    """The reference-precision pipeline as a service: uint8 frames in pinned host memory -> FramePipeline on the f16x2
    encoder + fp32 head (one CUDA graph per slot: fused normalisation, three-term stem, planes through layer1-4 into
    conv_layer1, MPJPE sums) gives the eager forward_frames result bit for bit, replay after replay; PoseResNet on raw
    frames equals PoseResNet on the preprocessed tensor."""
    from fast_3d_human_pose_estimation_b200.encoder import IMAGENET_MEAN, IMAGENET_STD
    b = 3
    torch.manual_seed(0)
    m = cuda_pkg.CDRNet(synth.make_cfg(50, 19), precision="fp32", encoder_precision="fp32")
    m.load_state_dict(synth.make_head_state_dict(seed=0, calibrated=True), strict=False)
    m = m.cuda().eval()
    g = torch.Generator().manual_seed(3)
    frames = [torch.randint(0, 256, (b, 256, 256, 3), dtype=torch.uint8, generator=g) for _ in range(2)]
    cams = synth.make_cameras(b, seed=2)
    gt = synth.make_gt(cams, seed=3)
    Ps = [torch.from_numpy(cams["P_l"]), torch.from_numpy(cams["P_r"])]
    gtd = {k: torch.from_numpy(gt[k]).cuda() for k in ("gt3d", "gt2d_l", "gt2d_r", "vis")}
    (kl, kr), xyz = m.forward_frames([f.cuda() for f in frames], [p.cuda() for p in Ps])
    sums = cuda_pkg.mpjpe_sums([kl, kr], xyz, gtd["gt3d"], gtd["gt2d_l"], gtd["gt2d_r"], gtd["vis"])
    pipe = cuda_pkg.FramePipeline(m, b, gt=gtd)
    fh = torch.stack(frames, 0).pin_memory()
    for _ in range(2):
        pipe.submit(fh, [p.pin_memory() for p in Ps])
        pipe.submit([f.pin_memory() for f in frames], [p.pin_memory() for p in Ps])
        for _ in range(2):
            _, kp_h, xyz_h, sums_h = pipe.collect()
            assert torch.equal(kp_h[0], kl.cpu()) and torch.equal(kp_h[1], kr.cpu()) and torch.equal(xyz_h, xyz.cpu())
            assert torch.equal(sums_h, sums.cpu())
    # the same images as floats through CDRNet.forward (host-side ToTensor + Normalize, inference.py:40-44)
    mean = torch.tensor(IMAGENET_MEAN).reshape(1, 3, 1, 1)
    std = torch.tensor(IMAGENET_STD).reshape(1, 3, 1, 1)
    pre = [(f.permute(0, 3, 1, 2).float().div(255).sub_(mean).div_(std)).cuda() for f in frames]
    (kl2, kr2), xyz2 = m(pre, [p.cuda() for p in Ps])
    assert torch.equal(kl2, kl) and torch.equal(kr2, kr) and torch.equal(xyz2, xyz)


def test_tc_encoder_shapes_and_errors(cuda_pkg):
    """Other image sizes / batch 1 through the tcgen05 encoder; unsupported geometry fails loudly."""
    from fast_3d_human_pose_estimation_b200.encoder import TcEncoder
    r = _seeded_resnet(50, seed=3).cuda()
    enc = TcEncoder(r)
    for n, hw in ((1, (256, 256)), (2, (128, 256)), (1, (512, 512))):
        x = torch.randn(n, 3, *hw, generator=torch.Generator().manual_seed(n)).cuda()
        with torch.no_grad():
            want = r(x)
        got = enc(x)
        assert got.shape == want.shape == (n, 2048, hw[0] // 32, hw[1] // 32)
        rel = float((got - want).abs().max() / want.abs().max())
        print(f"\ntcgen05 encoder {n}x{hw}: rel err vs fp32 torch {rel:.2e}")
        assert rel < 6e-2
    with pytest.raises(cuda_pkg.CdrError):
        enc(torch.randn(1, 3, 192, 192).cuda())        # 48-wide feature maps do not tile into 128-pixel boxes
    with pytest.raises(RuntimeError):
        enc(torch.randn(1, 3, 256, 256))               # no CPU path
    with pytest.raises(NotImplementedError):
        TcEncoder(_seeded_resnet(18))                  # BasicBlock ResNets stay on torch


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_poseresnet_tc_encoder_baseline_path(cuda_pkg, precision):
    """baseline.py's path (BASELINE configs[2]) on this library end to end: PoseResNet with the tcgen05
    encoder feeding cdr_decoder_forward_rows, then get_max_preds x4 -> uint8 -> triangulation, against the
    ORACLE of the same pipeline (fp64 evaluation with bf16 rounding where the kernels round).  Heat-maps stay
    within the stated bf16 bound and the uint8 key points are identical wherever the oracle's top-2 logit gap
    exceeds the heat-map error."""
    n, joints = 4, 19
    torch.manual_seed(0)
    m = cuda_pkg.PoseResNet(synth.make_cfg(50, joints), precision=precision, encoder_precision="bf16")
    sd = synth.make_head_state_dict(seed=3, joints=joints, calibrated=True, decoder_only=True)
    m.decoder.load_state_dict({k[len("decoder."):]: v for k, v in sd.items()})
    from bf16_emulation import encoder_bf16, decoder_bf16
    x_cpu = torch.randn(n, 3, 256, 256, generator=torch.Generator().manual_seed(2))
    with torch.no_grad():                                   # the ORACLE of this pipeline (CPU, fp64, bf16 grid)
        lat = encoder_bf16(m.encoder.cpu().eval(), x_cpu.double())
        if precision == "bf16":
            want = decoder_bf16(sd, lat)
        else:
            want = O.decoder(O.cast_state_dict(sd, torch.float64), lat)
    m = m.cuda().eval()
    x = x_cpu.cuda()
    got = m(x)
    torch.cuda.synchronize()
    ref = want.float().cuda()
    rel = float((got - ref).abs().max() / ref.abs().max())
    pts = cuda_pkg.baseline_keypoints(got)
    pts_ref = torch.from_numpy((O.get_max_preds(want.float().numpy())[0] * 4.0).astype(np.uint8)).cuda()   # baseline.py:51-53
    top2 = torch.topk(ref.reshape(n, joints, -1), 2, dim=-1).values
    decisive = (top2[..., 0] - top2[..., 1]) > 4 * float((got - ref).abs().max())
    agree = (pts == pts_ref).all(-1)
    print(f"\nPoseResNet-50 [{precision}] tcgen05 encoder + decoder vs the bf16-emulated oracle pipeline: heat rel {rel:.2e}, "
          f"arg-max agree {int(agree.sum())}/{agree.numel()} (decisive {int(decisive.sum())})")
    assert got.shape == (n, joints, 64, 64) and rel < 6e-2
    assert bool(agree[decisive].all())
    P = synth.make_cameras(n // 2, seed=2)
    P1 = np.concatenate([P["P_l"], np.tile([[[0, 0, 0, 1.0]]], (n // 2, 1, 1))], 1).astype(np.float64)
    P2 = np.concatenate([P["P_r"], np.tile([[[0, 0, 0, 1.0]]], (n // 2, 1, 1))], 1).astype(np.float64)
    xyz = cuda_pkg.triangulation(torch.from_numpy(P1), torch.from_numpy(P2), pts[: n // 2], pts[n // 2:])
    assert tuple(xyz.shape) == (n // 2, joints, 3) and bool(torch.isfinite(xyz).all())


def test_baseline_config3_full_size(cuda_pkg):
    """BASELINE configs[2] at its full size — PoseResNet-101, 256 uint8 frames (128 stereo pairs), bf16 — through
    size-independent properties: determinism, per-image independence (a 16-image slice run alone gives the same bits),
    and for ALL 128 pairs the arg-max x4 -> uint8 -> triangulation chain against the reference's functions
    (tools/utils.py:30-58, baseline.py:51-53, tools/common.py:51-71): key points bit-exact on the SAME heat-maps, 3D
    <= 1e-2 mm on view-consistent uint8 points."""
    n, joints = 256, 19
    torch.manual_seed(0)
    m = cuda_pkg.PoseResNet(synth.make_cfg(101, joints), precision="bf16", encoder_precision="bf16")
    sd = synth.make_head_state_dict(seed=3, joints=joints, calibrated=True, decoder_only=True)
    m.decoder.load_state_dict({k[len("decoder."):]: v for k, v in sd.items()})
    m = m.cuda().eval()
    frames = torch.randint(0, 256, (n, 256, 256, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(9)).cuda()
    hm = m(frames)
    hm2 = m(frames)
    assert hm.shape == (n, joints, 64, 64) and torch.equal(hm, hm2) and bool(torch.isfinite(hm).all())
    part = m(frames[96:112].contiguous())
    assert torch.equal(part, hm[96:112])
    pts = cuda_pkg.baseline_keypoints(hm)
    h_np = hm.cpu().numpy()
    want_pts = (O.get_max_preds(h_np)[0] * 4.0).astype(np.uint8)
    assert np.array_equal(pts.cpu().numpy(), want_pts)
    nb = n // 2
    cams = synth.make_cameras(nb, seed=5)
    row4 = np.tile([[[0, 0, 0, 1.0]]], (nb, 1, 1))
    P1 = np.concatenate([cams["P_l"], row4], 1).astype(np.float64)
    P2 = np.concatenate([cams["P_r"], row4], 1).astype(np.float64)
    xyz = cuda_pkg.triangulation(torch.from_numpy(P1).cuda(), torch.from_numpy(P2).cuda(), pts[:nb], pts[nb:])
    assert tuple(xyz.shape) == (nb, joints, 3)
    # triangulation at this size against the reference's function: on view-consistent uint8 points (the key points of
    # a random-init network point at rays that barely intersect: both answers are then noise of eig / SVD)
    gt = synth.make_gt(cams, seed=6)
    u_l = np.clip(np.rint(gt["gt2d_l"]), 0, 255).astype(np.uint8)
    u_r = np.clip(np.rint(gt["gt2d_r"]), 0, 255).astype(np.uint8)
    got = cuda_pkg.triangulation(torch.from_numpy(P1).cuda(), torch.from_numpy(P2).cuda(), torch.from_numpy(u_l).cuda(),
                                 torch.from_numpy(u_r).cuda()).cpu().numpy()
    want = np.stack([O.triangulation(P1[i], P2[i], u_l[i], u_r[i]) for i in range(nb)])
    err = np.abs(got - want).max()
    print(f"\nconfigs[2] full size: {pts.numel() // 2} key points bit-exact; triangulation of {nb} pairs vs the reference's "
          f"eig form: max {err:.2e} mm")
    assert err <= TOL_3D_MM


@pytest.mark.parametrize("precision,b", [("bf16", 3), ("fp32", 3), ("fp32", 64), ("bf16", 64)])
def test_fused_decoder_tail_matches_unfused_and_oracle(cuda_pkg, precision, b, monkeypatch):
    """deconv3 -> ReLU -> final 1x1 -> soft-argmax partials as ONE kernel (bf16: tail_tc.cuh; fp32: the cta_group::2 pair
    kernel of tail_pair_tc.cuh; a second tcgen05.mma on the ReLU'd tile, per-row online-softmax partials merged in fp64)
    against the three-launch path of the same library (CDR_FUSED_TAIL=0) — heat-maps to accumulation-order rounding, 2D
    joints <= 1e-4 px — and, at B = 3, against the fp64 oracle with the flat tolerance."""
    sd = synth.make_head_state_dict(seed=0, calibrated=True, randomize_bn=True)
    feats, cams = synth.make_features(b, seed=1), synth.make_cameras(b, seed=2)
    m = _model(cuda_pkg, sd, precision=precision)
    L = cuda_pkg._lib.lib()
    monkeypatch.setenv("CDR_FUSED_TAIL", "1")
    (kl, kr), xyz, taps = _run_head(m, feats, cams, taps=True)      # (the first call also packs the weights)
    L.cdr_launch_count_reset()
    (kl_nt, kr_nt), xyz_nt = _run_head(m, feats, cams)              # without taps: heat-maps never written
    n_fused = L.cdr_launch_count()
    monkeypatch.setenv("CDR_FUSED_TAIL", "0")
    (ul, ur), uxyz, utaps = _run_head(m, feats, cams, taps=True)
    L.cdr_launch_count_reset()
    _run_head(m, feats, cams)
    n_unfused = L.cdr_launch_count()
    monkeypatch.setenv("CDR_FUSED_TAIL", "1")
    assert torch.equal(kl, kl_nt) and torch.equal(kr, kr_nt) and torch.equal(xyz, xyz_nt)
    hm, uhm = taps["heatmaps"], utaps["heatmaps"]
    rel = float((hm - uhm).abs().max() / uhm.abs().max())
    d2 = max(float((kl - ul).abs().max()), float((kr - ur).abs().max()))
    print(f"\nfused tail [{precision}, B={b}]: heat-maps vs unfused rel {rel:.2e}, 2D {d2:.2e} px; launches {n_fused} vs {n_unfused}")
    assert rel <= (1e-6 if precision == "fp32" else 1e-5)
    assert d2 <= 1e-4
    assert n_fused < n_unfused
    if b <= 4:
        o2, o3 = _oracle64(sd, feats, cams)
        d2o = max(np.abs(kl.cpu().numpy() - o2[0]).max(), np.abs(kr.cpu().numpy() - o2[1]).max())
        print(f"fused tail [{precision}] vs fp64 oracle: d2D {d2o:.2e} px")
        if precision == "fp32":
            assert d2o <= TOL_2D_PX
            check_3d(cams, kl, kr, xyz, o2, o3, f"fused tail B={b}:")
        else:
            assert d2o <= 1.0


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_fused_tail_decoder_only_heatmaps(cuda_pkg, precision, monkeypatch):
    """PoseDecoder.forward (PoseResNet's decoder half) through the fused tail: same heat-maps as the unfused path."""
    n, joints = 3, 19
    sd = synth.make_head_state_dict(seed=3, joints=joints, calibrated=True, randomize_bn=True, decoder_only=True)
    feats = synth.make_features(n, seed=4)[0].cuda()
    dec = cuda_pkg.PoseDecoder(synth.make_cfg(18, joints), precision=precision)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items()})
    dec = dec.cuda().eval()
    monkeypatch.setenv("CDR_FUSED_TAIL", "1")
    a = dec(feats)
    monkeypatch.setenv("CDR_FUSED_TAIL", "0")
    bb = dec(feats)
    monkeypatch.setenv("CDR_FUSED_TAIL", "1")
    torch.cuda.synchronize()
    rel = float((a - bb).abs().max() / bb.abs().max())
    print(f"\nfused tail decoder-only [{precision}]: heat-maps vs unfused rel {rel:.2e}")
    assert rel <= (1e-6 if precision == "fp32" else 1e-5)


def test_projection_matrices_on_device(cuda_pkg):
    """SURVEY §8f rank 2 remainder: P = T @ K @ [R | t] built on the device against the reference's host construction
    (tools/common.py:28-32 get_projection_matrix, dataset/mads_3d.py:223-226 `T @ P`, inference.py:53-56 `[:3]` float32)."""
    n = 37
    cams = synth.make_cameras(n, seed=31)
    rng = np.random.default_rng(32)
    trans = np.stack([np.array([[s * np.cos(a), -s * np.sin(a), tx], [s * np.sin(a), s * np.cos(a), ty]])
                      for s, a, tx, ty in zip(rng.uniform(0.3, 1.2, n), rng.uniform(-0.5, 0.5, n),
                                              rng.uniform(-40, 40, n), rng.uniform(-40, 40, n))])
    for view in ("l", "r"):
        R, T = np.stack(cams[f"R_{view}"]), np.stack(cams[f"T_{view}"])
        want_plain = np.stack([O.get_projection_matrix(cams["K"], R[i], T[i])[:3] for i in range(n)])
        got = cuda_pkg.projection_matrices(cams["K"], R, T).cpu().numpy()
        assert got.dtype == np.float32 and got.shape == (n, 3, 4)
        assert np.array_equal(got, want_plain.astype(np.float32))
        assert np.array_equal(got, cams[f"P_{view}"])                 # what every other test feeds the head
        want_t = []
        for i in range(n):
            Tm = np.eye(4)
            Tm[:2, :3] = trans[i]
            want_t.append((Tm @ O.get_projection_matrix(cams["K"], R[i], T[i]))[:3])
        got_t = cuda_pkg.projection_matrices(np.stack([cams["K"]] * n), torch.from_numpy(R), T, trans=trans).cpu().numpy()
        want32 = np.stack(want_t).astype(np.float32)
        ulp = np.abs(got_t.view(np.int32) - want32.view(np.int32)).max()
        assert ulp <= 1, f"{ulp} ulp"                                  # BLAS may contract / reorder a sum; never more than 1 fp32 ulp
