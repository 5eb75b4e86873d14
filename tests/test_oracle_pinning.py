"""Pin the oracle: against the reference's own code (FPS .cpp and the vendored-Ceres uncertainty PnP compiled into
oracle/_ref, Python head/PnP/pose classes imported with stubbed third-party deps; their outputs stored under
tests/golden/), and against independent formulations elsewhere."""
import ctypes
import math
import os
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import gdrn_model_oracle as O
from oracle import ops_oracle as OO

GOLD = os.path.join(ROOT, "tests", "golden")
GOLD_CPU = os.path.join(GOLD, "ref_cpu_ops.npz")   # tools/make_golden_ref_ops.py cpu


def test_fps_oracle_matches_survey_vector():
    # SURVEY.md §8c: reference build, RandomState(0).rand(5000,3) f32, init_center, 8 samples
    pts = np.random.RandomState(0).rand(5000, 3).astype(np.float32)
    assert OO.fps(pts, 8).tolist() == [2895, 884, 2241, 4602, 3356, 3779, 3096, 4550]


def test_fps_oracle_matches_golden_fixture():
    g = np.load(os.path.join(GOLD, "fps_golden.npz"))
    for i in range(int(g["n_cases"])):
        pts, idx = g[f"pts_{i}"], g[f"idx_{i}"]
        assert (OO.fps(pts, len(idx)) == idx).all(), i


def fps_ref_cases():
    rs = np.random.RandomState(5)
    for pn, sn in ((1, 1), (7, 7), (100, 16), (3000, 64), (20000, 128)):
        pts = (rs.rand(pn, 3).astype(np.float32) - 0.5) * 0.3
        if pn == 100:
            pts[10:20] = pts[0]  # duplicates -> zero distances / ties
        yield pn, sn, pts


def test_fps_oracle_matches_reference_build_when_present():
    """Against the REFERENCE's own FPS (core/csrc/fps/src/farthest_point_sampling.cpp built into oracle/_ref), whose
    indices on these clouds are stored in tests/golden/ref_cpu_ops.npz."""
    g = np.load(GOLD_CPU)
    for pn, sn, pts in fps_ref_cases():
        assert (OO.fps(pts, sn) == g["fps/%d_%d" % (pn, sn)]).all(), (pn, sn)


def test_head_pnp_pose_oracle_matches_reference_classes():
    """tests/golden/ref_heads.npz was produced by tools/make_golden_ref_heads.py, which imports the reference's
    own TopDownDoubleMaskXyzRegionHead / ConvPnPNet / rot6d / pose_from_predictions_test / allo->ego code."""
    path = os.path.join(GOLD, "ref_heads.npz")
    g = np.load(path)
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd/")}
    feat = torch.from_numpy(g["in/feat"])
    with torch.no_grad():
        outs = O.geo_head(sd, feat, num_classes=int(g["num_classes"]))
    for name, o in zip(("vis", "full", "cx", "cy", "cz", "region"), outs):
        assert torch.allclose(o, torch.from_numpy(g["out/" + name]), atol=2e-5, rtol=1e-4), name
    with torch.no_grad():
        rot, t = O.conv_pnp_net(sd, torch.from_numpy(g["in/coor_feat"]), torch.from_numpy(g["in/region"]),
                                torch.from_numpy(g["in/extents"]))
    assert torch.allclose(rot, torch.from_numpy(g["out/pnp_rot"]), atol=1e-5, rtol=1e-4)
    assert torch.allclose(t, torch.from_numpy(g["out/pnp_t_raw"]), atol=1e-5, rtol=1e-4)
    Rm = O.rot6d_to_mat_batch(torch.from_numpy(g["out/pnp_rot"]))
    assert torch.allclose(Rm, torch.from_numpy(g["out/rot_m"]), atol=1e-6)
    ego, trans = O.pose_from_predictions_test(
        torch.from_numpy(g["out/rot_m"]), torch.from_numpy(g["out/pnp_t"])[:, :2], torch.from_numpy(g["out/pnp_t"])[:, 2:3],
        torch.from_numpy(g["in/cams"]), torch.from_numpy(g["in/centers"]), torch.from_numpy(g["in/ratios"]),
        torch.from_numpy(g["in/whs"]))
    assert np.allclose(ego.numpy(), g["out/ego_rot"], atol=1e-6)
    assert np.allclose(trans.numpy(), g["out/trans"], atol=1e-7)


def test_backbone_oracle_param_count_and_fp64_agreement():
    from gdrnpp_bop2022_b200.synthetic import make_batch, make_state_dict

    sd = make_state_dict("convnext_tiny")
    batch = make_batch(B=1, seed=2)
    with torch.no_grad():
        f32 = O.convnext_features(sd, batch["roi_img"], "convnext_tiny")
        f64 = O.convnext_features(O.cast_state_dict(sd, torch.float64), batch["roi_img"].double(), "convnext_tiny")
    assert f32.shape == (1, 768, 8, 8)
    assert (f32.double() - f64).abs().max() / f64.abs().max() < 1e-4
    sdb = make_state_dict("convnext_base")
    assert sum(v.numel() for k, v in sdb.items() if k.startswith("backbone.")) == 87564416  # SURVEY.md Appendix A


@pytest.mark.parametrize("arch,res", [("convnext_tiny", 96), ("convnext_base", 64)])
def test_backbone_oracle_pinned_to_torchvision(arch, res):
    """Pins the ConvNeXt restatement: timm 0.6.7 (the reference's un-vendored dependency, core/utils/timm_utils.py:9-35)
    cannot be installed here, but torchvision ships an independent implementation of the same published network.
    With the timm-named weights remapped (oracle.torchvision_convnext) the two must agree BIT FOR BIT on the stage-3
    feature map (features_only, out_indices=(3,): no final norm), and convnext_base must have timm's 87,564,416
    backbone parameters (SURVEY.md Appendix A)."""
    pytest.importorskip("torchvision")
    from gdrnpp_bop2022_b200.synthetic import make_state_dict

    sd = make_state_dict(arch)
    net = O.torchvision_convnext(sd, arch)
    x = torch.rand(2, 3, res, res, generator=torch.Generator().manual_seed(res))
    with torch.no_grad():
        tv = net(x)
        mine = O.convnext_features(sd, x, arch)
    assert tv.shape == mine.shape == (2, O.CONVNEXT_ARCH[arch][1][3], res // 32, res // 32)
    assert torch.equal(tv, mine), float((tv - mine).abs().max())
    n_params = sum(p.numel() for p in net.parameters())
    n_sd = sum(v.numel() for k, v in sd.items() if k.startswith("backbone."))
    assert n_params == n_sd
    if arch == "convnext_base":
        assert n_params == 87_564_416


def test_gelu_epilogue_fit_accuracy():
    hdr = open(os.path.join(ROOT, "gdrnpp_bop2022_b200", "csrc", "gelu_coeffs.h")).read()
    c = [float(l.split()[2].rstrip("f")) for l in hdr.splitlines() if l.startswith("#define GELU_C") and "CLAMP" not in l]
    clamp = float([l for l in hdr.splitlines() if "GELU_CLAMP" in l][0].split()[2].rstrip("f"))
    x = np.linspace(-8, 8, 40001)
    xc = np.clip(x, -clamp, clamp)
    p = ((c[3] * xc**2 + c[2]) * xc**2 + c[1]) * xc**2 + c[0]
    g = x / (1 + np.exp2(xc * p))
    ref = torch.nn.functional.gelu(torch.from_numpy(x)).numpy()
    assert np.abs(g - ref).max() < 3e-5


def test_gelu_erf_epilogue_forms_accuracy():
    """The parity-mode (split-bf16) epilogue GELU: both evaluation orders of the A&S 7.1.26 erfc form (scalar gelu_erf and the
    packed gelu_erf2 the fc1 epilogue runs), emulated in float32, stay within 6e-7 of the float64 erf GELU."""
    pytest.importorskip("scipy")
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import check_erf as CE
    from scipy.special import erf as erf64
    x = np.linspace(-12, 12, 400001).astype(np.float32)
    ref = 0.5 * x.astype(np.float64) * (1 + erf64(x.astype(np.float64) / np.sqrt(2)))
    assert np.abs(CE.gelu_as(x) - ref).max() < 6e-7
    assert np.abs(CE.gelu_as_packed(x) - ref).max() < 6e-7


def test_nnd_oracle_vs_cdist():
    rs = np.random.RandomState(1)
    a, b = rs.rand(2, 200, 3).astype(np.float32), rs.rand(2, 300, 3).astype(np.float32)
    d1, d2, i1, i2 = OO.nnd_forward(a, b)
    cd = torch.cdist(torch.from_numpy(a).double(), torch.from_numpy(b).double()) ** 2
    assert np.abs(d1 - cd.min(2)[0].numpy()).max() < 1e-6
    assert (i1 == cd.argmin(2).numpy()).mean() > 0.999


def test_voting_oracle_geometry():
    # all pixels point exactly at a known keypoint -> every valid hypothesis is that keypoint and all vote for it
    rs = np.random.RandomState(2)
    tn, vn, hn = 500, 3, 32
    coords = rs.rand(tn, 2).astype(np.float32) * 100
    kp = np.array([[50.3, 40.2], [10.0, 90.0], [70.5, 20.25]], np.float32)
    d = kp[None] - coords[:, None]
    direct = (d / np.linalg.norm(d, axis=2, keepdims=True)).astype(np.float32)
    idxs = rs.randint(0, tn, (hn, vn, 2)).astype(np.int32)
    hyp = OO.generate_hypothesis(direct, coords, idxs)
    ok = np.abs(hyp).sum(2) > 0
    assert ok.mean() > 0.9
    assert np.abs(hyp[ok] - np.broadcast_to(kp[None], hyp.shape)[ok]).max() < 0.05
    inl, cnt = OO.voting(direct, coords, hyp, 0.999)
    assert (cnt[ok] > 0.95 * tn).all()
    assert (inl.sum(2) == cnt).all()


def test_raster_oracle_sphere_depth():
    from gdrnpp_bop2022_b200.synthetic import make_icosphere_mesh

    v, f = make_icosphere_mesh(3, (0.1, 0.1, 0.1))
    pose = np.hstack([np.eye(3), [[0.0], [0.0], [0.5]]]).astype(np.float32)
    K = np.array([[100, 0, 32], [0, 100, 32], [0, 0, 1]], np.float32)
    d = OO.render_depth(v, f, pose, K, 64, 64)
    assert abs(d[32, 32] - 0.45) < 2e-3 and d[0, 0] == 0
    # silhouette radius: r/z*f = 0.05/sqrt(0.5^2-0.05^2)*100 ~ 10.05 px -> area ~ 317 px
    assert abs((d > 0).sum() - 317) < 20


def test_upnp_oracle_known_answer():
    # recipe of the reference's own main() (uncertainty_pnp.cpp:98-156)
    rs = np.random.RandomState(3)
    rt = rs.rand(6)
    p3 = rs.rand(8, 3)
    K = np.array([[400.0, 0, 128], [0, 400, 128], [0, 0, 1]])
    p2 = np.zeros((8, 2))
    for i in range(8):
        q = OO._rodrigues_point(rt[:3], p3[i]) + rt[3:]
        p2[i] = [K[0, 0] * q[0] / q[2] + K[0, 2], K[1, 1] * q[1] / q[2] + K[1, 2]]
    w = np.tile(np.array([[1.0, 0.0, 1.0]]), (8, 1))
    init = rt + rs.rand(6) * 0.1
    sol = OO.uncertainty_pnp(p2, p3, w, K, init)
    assert np.abs(sol - rt).max() < 1e-5


# ---------------------------------------------------------------------------------------------------------------
# ROI crop + resize: the arithmetic lives in OpenCV (un-vendored dependency of the reference).  opencv-python is in
# this image, so the oracle is pinned against cv2.warpAffine itself, exactly as crop_resize_by_warp_affine calls it
# (core/utils/data_utils.py:115-133), and against a committed golden crop for boxes without cv2.
# ---------------------------------------------------------------------------------------------------------------
def _crop_cases(rng, n, W=640, H=480):
    for i in range(n):
        cx, cy = rng.uniform(-40, W + 40), rng.uniform(-40, H + 40)
        scale = float(rng.uniform(24, 720))
        out = 256 if i % 2 == 0 else 64
        s = out / scale
        M = np.array([[s, 0, out * 0.5 - cx * s], [0, s, out * 0.5 - cy * s]], np.float64)
        if i % 5 == 0:   # a rotated crop (the data loader's augmentation path uses rot != 0)
            a = rng.uniform(-0.6, 0.6)
            M[:, :2] = np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]) * s
        yield M, out


def test_warp_affine_oracle_bit_exact_vs_cv2():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.RandomState(0)
    img = rng.randint(0, 256, (480, 640, 3)).astype(np.uint8)
    coord = rng.rand(480, 640, 2).astype(np.float32)
    depth = (rng.rand(480, 640) * 2).astype(np.float32)
    for M, out in _crop_cases(rng, 24):
        ref = cv2.warpAffine(img, M, (out, out), flags=cv2.INTER_LINEAR)
        assert np.array_equal(ref, OO.warp_affine_u8(img, M, (out, out)))
        ref = cv2.warpAffine(coord, M, (out, out), flags=cv2.INTER_LINEAR)
        got = OO.warp_affine_f32(coord, M, (out, out))
        assert np.abs(ref - got).max() <= 1e-6            # measured 0 with the scalar float path of cv2 4.13
        ref = cv2.warpAffine(depth, M, (out, out), flags=cv2.INTER_NEAREST)
        assert np.array_equal(ref, OO.warp_affine_f32(depth, M, (out, out), nearest=True)[:, :, 0])


def test_warp_affine_oracle_matches_golden_fixture():
    """tests/golden/crop_golden.npz was written by tools/make_golden_crop.py from cv2.warpAffine outputs."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "crop_golden.npz"))
    for i in range(g["M"].shape[0]):
        out = int(g["out"][i])
        assert np.array_equal(OO.warp_affine_u8(g["img"], g["M"][i], (out, out)), g["crop_%d" % i])


def test_get_affine_transform_matches_reference_formula():
    """Host mirror of get_affine_transform (data_utils.py:136-189) vs the cv2.getAffineTransform-based original."""
    cv2 = pytest.importorskip("cv2")
    from gdrnpp_bop2022_b200.native_ops import get_affine_transform

    def ref(center, scale, rot, out):
        if isinstance(center, (tuple, list)):   # the reference converts sequences only; arrays keep their dtype (float64 bbox
            center = np.array(center, np.float32)   # arithmetic is rounded ONCE, into the float32 point array)
        scale = np.array([scale, scale], np.float32)
        rot_rad = np.pi * rot / 180
        sn, cs = np.sin(rot_rad), np.cos(rot_rad)
        sp = [0, scale[0] * -0.5]
        src_dir = [sp[0] * cs - sp[1] * sn, sp[0] * sn + sp[1] * cs]
        dst_dir = np.array([0, out * -0.5], np.float32)
        src, dst = np.zeros((3, 2), np.float32), np.zeros((3, 2), np.float32)
        src[0, :], src[1, :] = center, center + src_dir
        dst[0, :] = [out * 0.5, out * 0.5]
        dst[1, :] = np.array([out * 0.5, out * 0.5], np.float32) + dst_dir
        t3 = lambda a, b: b + np.array([-(a - b)[1], (a - b)[0]], np.float32)
        src[2, :], dst[2, :] = t3(src[0], src[1]), t3(dst[0], dst[1])
        return cv2.getAffineTransform(np.float32(src), np.float32(dst))

    rng = np.random.RandomState(3)
    for _ in range(100):
        c, s = rng.uniform(0, 640, 2), float(rng.uniform(20, 700))
        rot, out = float(rng.choice([0, 0, 15, -30])), int(rng.choice([64, 256]))
        for cc in (c, c.astype(np.float32), tuple(c.tolist())):   # float64 array, float32 array, python sequence
            assert np.abs(get_affine_transform(cc, s, rot, out) - ref(cc, s, rot, out)).max() < 1e-9


def test_baseline_config0_cpu_plumbing():
    """BASELINE.json configs[0] / SURVEY.md 8d config 1: one 256x256 synthetic ROI through a random-init ConvNeXt-tiny
    model, one FPS (pn = 8192 in U[-0.1, 0.1]^3, sn = 64, init_center), one RANSAC voting round (tn = 2048, vn = 9,
    hn = 128, unit-norm directions, threshold 0.999) and the Patch-PnP forward, CPU only.  Pass = runs, finite,
    self-consistent (rotation orthonormal, FPS indices distinct and equal to the reference build when present,
    vote counts bounded by tn)."""
    from gdrnpp_bop2022_b200.synthetic import make_batch, make_state_dict

    sd = make_state_dict("convnext_tiny", seed=0)
    batch = make_batch(B=1, seed=0)
    with torch.no_grad():
        out = O.gdrn_forward(sd, batch, arch="convnext_tiny", return_maps=True)
    R = out["rot"][0].double()
    assert torch.isfinite(out["trans"]).all() and (R @ R.T - torch.eye(3, dtype=torch.float64)).abs().max() < 1e-5
    assert abs(float(torch.det(R)) - 1.0) < 1e-5 and out["region"].shape == (1, 65, 64, 64)

    rng = np.random.RandomState(0)
    pts = rng.uniform(-0.1, 0.1, (8192, 3)).astype(np.float32)
    idx = OO.fps(pts, 64)
    assert len(set(idx.tolist())) == 64 and idx.min() >= 0 and idx.max() < 8192
    assert np.array_equal(np.load(GOLD_CPU)["fps/config0"], idx)   # the reference build's indices

    tn, vn, hn = 2048, 9, 128
    coords = rng.uniform(0, 64, (tn, 2)).astype(np.float32)
    direct = rng.normal(size=(tn, vn, 2)).astype(np.float32)
    direct /= np.linalg.norm(direct, axis=2, keepdims=True)
    idxs = rng.randint(0, tn, (hn, vn, 2)).astype(np.int32)
    hypo = OO.generate_hypothesis(direct, coords, idxs)
    inl, cnt = OO.voting(direct, coords, hypo, 0.999)
    assert hypo.shape == (hn, vn, 2) and cnt.shape == (hn, vn) and cnt.min() >= 0 and cnt.max() <= tn
    assert np.array_equal(inl.sum(axis=2).astype(np.int64), cnt.astype(np.int64))


def _gl_window_coords(K, X, W, H, nc, fc):
    """The reference's GL pipeline restated in numpy: lib/render_vispy/renderer.py:461-476 (projective_matrix; its
    transpose is uploaded, so clip = proj @ view_point), camera-space OpenCV point -> GL view by the y/z flip the
    renderer applies (:67-69, 377), perspective divide, viewport transform (0, 0, W, H), window depth in [0, 1]."""
    q = -(fc + nc) / float(fc - nc)
    qn = -2 * (fc * nc) / float(fc - nc)
    proj = np.array([[2 * K[0, 0] / W, -2 * K[0, 1] / W, (-2 * K[0, 2] + W) / W, 0],
                     [0, 2 * K[1, 1] / H, (2 * K[1, 2] - H) / H, 0],
                     [0, 0, q, qn],
                     [0, 0, -1, 0]], np.float64)
    view = np.array([X[0], -X[1], -X[2], 1.0])          # OpenCV (x right, y down, z forward) -> GL (y up, z backward)
    clip = proj @ view
    ndc = clip[:3] / clip[3]
    xw, yw = (ndc[0] + 1) * W / 2, (ndc[1] + 1) * H / 2  # glViewport(0, 0, W, H); window origin = lower left
    return xw, yw, (ndc[2] + 1) / 2


def test_raster_conventions_pinned_to_the_gl_pipeline():
    """Pins the rasteriser's conventions (SURVEY.md Appendix B) against the reference's own matrices rather than against
    our reading of them: for random cameras and points, the GL pipeline of lib/render_vispy/renderer.py (projective_matrix
    :461-476, glReadPixels + [::-1] row flip :155-174, depth decode mult / (d + addi) :176-182) puts a camera-space point
    in the image row / column where u = fx X/Z + s Y/Z + cx, v = fy Y/Z + cy says, samples pixels at their centres
    (c + 0.5, r + 0.5), and decodes exactly its camera-space Z."""
    rs = np.random.RandomState(0)
    W, H, nc, fc = 64, 48, 0.1, 100.0
    for _ in range(200):
        K = np.array([[rs.uniform(80, 140), rs.uniform(-2, 2), rs.uniform(20, 44)], [0, rs.uniform(80, 140), rs.uniform(14, 34)], [0, 0, 1]])
        X = np.array([rs.uniform(-0.3, 0.3), rs.uniform(-0.2, 0.2), rs.uniform(0.3, 3.0)])
        xw, yw, d = _gl_window_coords(K, X, W, H, nc, fc)
        # our convention
        u = (K[0, 0] * X[0] + K[0, 1] * X[1]) / X[2] + K[0, 2]
        v = K[1, 1] * X[1] / X[2] + K[1, 2]
        # NOTE the reference negates the skew term (-2*cam[0,1]/w with y already flipped): same sign as ours
        assert abs(xw - u) < 1e-9
        # glReadPixels row 0 = bottom window row; rgb/dep are flipped with [::-1]: image row r covers window y in
        # [H - 1 - r, H - r), i.e. image v = H - yw, pixel centres at r + 0.5
        assert abs((H - yw) - v) < 1e-9
        mult, addi = (nc * fc) / (nc - fc), fc / (nc - fc)
        assert abs(mult / (d + addi) - X[2]) < 1e-9 * max(1.0, X[2]) * 100
    # the oracle rasteriser on an analytic case: a tilted plane quad -> depth = ray / plane intersection at pixel centres
    K = np.array([[110.0, 0, 31.5], [0, 112.0, 30.25], [0, 0, 1]])
    n_pl, d_pl = np.array([0.2, -0.1, 1.0]), 0.8           # plane n.X = d
    corners = []
    for sx, sy in ((-1, -1), (1, -1), (1, 1), (-1, 1)):
        ray = np.array([sx * 0.5, sy * 0.5, 1.0])
        corners.append(ray * (d_pl / (n_pl @ ray)))
    verts = np.array(corners, np.float32)
    faces = np.array([[0, 1, 2], [0, 2, 3]], np.int32)
    pose = np.hstack([np.eye(3), np.zeros((3, 1))]).astype(np.float32)
    dep = OO.render_depth(verts, faces, pose, K.astype(np.float32), 64, 64)
    cc, rr = np.meshgrid(np.arange(64) + 0.5, np.arange(64) + 0.5)
    rays = np.stack([(cc - K[0, 2]) / K[0, 0], (rr - K[1, 2]) / K[1, 1], np.ones_like(cc)], -1)
    z_true = d_pl / (rays @ n_pl)
    assert (dep > 0).all()                                  # the quad covers the whole 64 x 64 window
    assert np.abs(dep - z_true).max() < 2e-6


def _upnp_problem(rs, pn, noise):
    K = np.array([[400.0, 0, 128], [0, 400, 128], [0, 0, 1]])
    while True:   # the reference recipe (rt ~ U(0,1)^6, points ~ U(0,1)^3) with the points safely in front of the camera
        rt = rs.rand(6)
        p3 = rs.rand(pn, 3)
        q = np.stack([OO._rodrigues_point(rt[:3], p3[i]) + rt[3:] for i in range(pn)])
        if q[:, 2].min() > 0.4:
            break
    p2 = np.stack([K[0, 0] * q[:, 0] / q[:, 2] + K[0, 2], K[1, 1] * q[:, 1] / q[:, 2] + K[1, 2]], 1)
    p2 += rs.randn(pn, 2) * noise
    w = np.stack([1 + rs.rand(pn), 0.1 * rs.randn(pn), 1 + rs.rand(pn)], 1)
    return K, rt, p2, p3, w, rt + rs.rand(6) * 0.05


def upnp_ceres_ref(p2, p3, w, K, init):
    """oracle/_ref/libupnp_ceres_ref.so: the reference's vendored Ceres (Jet autodiff + TinySolver LM); None if not built."""
    so = os.path.join(ROOT, "oracle", "_ref", "libupnp_ceres_ref.so")
    if not os.path.exists(so):
        return None
    L = ctypes.CDLL(so)
    L.upnp_ceres_ref.restype = ctypes.c_int
    c = lambda a: np.ascontiguousarray(a, np.float64).ctypes.data_as(ctypes.c_void_p)
    res = np.zeros(6)
    a2, a3, aw, aK, ai = (np.ascontiguousarray(x, np.float64) for x in (p2, p3, w, K, init))
    L.upnp_ceres_ref(a2.ctypes.data_as(ctypes.c_void_p), a3.ctypes.data_as(ctypes.c_void_p), aw.ctypes.data_as(ctypes.c_void_p),
                     aK.ctypes.data_as(ctypes.c_void_p), ai.ctypes.data_as(ctypes.c_void_p), res.ctypes.data_as(ctypes.c_void_p),
                     int(p2.shape[0]), None)
    return res


UPNP_REF_FIELDS = ("K", "rt", "p2", "p3", "w", "init", "ref")


def upnp_ref_problems(prefix):
    """The stored problems {K, rt, p2, p3, w, init} and the reference's solution ``ref`` of each (ref_cpu_ops.npz)."""
    g = np.load(GOLD_CPU)
    return [{f: g["%s/%d/%s" % (prefix, i, f)] for f in UPNP_REF_FIELDS} for i in range(int(g[prefix + "/n"]))]


def test_upnp_oracle_pinned_to_vendored_ceres():
    """Pins the uncertainty-PnP oracle (numpy LM) against the REFERENCE's own vendored Ceres 2.0: ceres::Jet autodiff of
    the residual of uncertainty_pnp.cpp:16-34 + ceres::AngleAxisRotatePoint + ceres::TinySolver, built from the headers
    under the reference's core/csrc/uncertainty_pnp/include (oracle/build_ref.py); its solutions are stored in
    tests/golden/ref_cpu_ops.npz.  Noise-free (the reference main() recipe, :98-156) and noisy problems: same minimiser
    to 1e-7."""
    for trial, p in enumerate(upnp_ref_problems("upnp_cpu")):
        K, rt, p2, p3, w, init, ref = (p[f] for f in UPNP_REF_FIELDS)
        mine = OO.uncertainty_pnp(p2, p3, w, K, init)
        assert np.abs(ref - mine).max() < 1e-7, (trial, ref, mine)
        if trial % 2 == 0:
            assert np.abs(ref - rt).max() < 1e-9
