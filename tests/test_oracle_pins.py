"""Pin the oracle against the reference's own known-answer tests (SURVEY.md section 8(c)).

Each test cites the reference test it replays (paths relative to a Kimera-VIO checkout).  They read
the reference's fixtures stored under tests/golden/reference (PNG images as lossless WebP); the
committed golden vectors in tests/golden/ are produced by the oracle pinned here.
"""
import os

import cv2
import numpy as np
import pytest

from conftest import REF_DATA
from kimera_vio_b200.params import CameraParams, FrontendParams
from oracle import frontend as ofe
from oracle.rig import StereoRig


def _frame(img_rel):
    img = cv2.imread(os.path.join(REF_DATA, img_rel), cv2.IMREAD_GRAYSCALE)
    cam = CameraParams.from_yaml(os.path.join(REF_DATA, "sensor.yaml"))
    return ofe.Frame(0, 123, img, cam)


def _bins(fr, p):
    brs = np.float32(fr.img.shape[0]) / np.float32(p.nr_vertical_bins)
    bcs = np.float32(fr.img.shape[1]) / np.float32(p.nr_horizontal_bins)
    cnt = np.zeros((p.nr_vertical_bins, p.nr_horizontal_bins), int)
    for x, y in fr.keypoints:
        cnt[int(np.float32(y) / brs), int(np.float32(x) / bcs)] += 1
    return cnt


# tests/testFeatureDetector.cpp:26-52
def test_detector_no_nms_393():
    p = FrontendParams.from_yaml(os.path.join(REF_DATA, "ForFeatureDetector/frontendParams-noNMS.yaml"))
    f = _frame("ForStereoFrame/left_fisheye_img_0.webp")
    ofe.FeatureDetector(p).feature_detection(f, None)
    assert len(f.keypoints) == 393


# tests/testFeatureDetector.cpp:55-80
def test_detector_no_nms_400():
    p = FrontendParams.from_yaml(os.path.join(REF_DATA, "ForFeatureDetector/frontendParams-noNMS.yaml"))
    p.quality_level = 1e-10
    f = _frame("ForStereoFrame/left_fisheye_img_0.webp")
    ofe.FeatureDetector(p).feature_detection(f, None)
    assert len(f.keypoints) == 400


# tests/testFeatureDetector.cpp:83-106
def test_detector_topn_300():
    p = FrontendParams.from_yaml(os.path.join(REF_DATA, "ForFeatureDetector/frontendParams-NMS-TopN.yaml"))
    f = _frame("ForStereoFrame/left_fisheye_img_0.webp")
    ofe.FeatureDetector(p).feature_detection(f, None)
    assert len(f.keypoints) == 300


# tests/testFeatureDetector.cpp:109-150
def test_detector_binning_20():
    p = FrontendParams.from_yaml(os.path.join(REF_DATA, "ForFeatureDetector/frontendParams-NMS-Binning.yaml"))
    f = _frame("ForStereoFrame/left_fisheye_img_0.webp")
    ofe.FeatureDetector(p).feature_detection(f, None)
    assert len(f.keypoints) == 20
    assert np.all(_bins(f, p) == 1)


# tests/testFeatureDetector.cpp:153-200
def test_detector_binning_200():
    p = FrontendParams.from_yaml(os.path.join(REF_DATA, "ForFeatureDetector/frontendParams-NMS-Binning.yaml"))
    p.max_features_per_frame = 200
    p.quality_level = 1e-10
    p.enable_subpixel_corner_refinement = False
    f = _frame("ForStereoFrame/left_fisheye_img_0.webp")
    ofe.FeatureDetector(p).feature_detection(f, None)
    assert len(f.keypoints) == 200
    assert np.all(_bins(f, p) == 10)


# tests/testFeatureDetector.cpp:203-258
def test_detector_binning_mask_140():
    p = FrontendParams.from_yaml(os.path.join(REF_DATA, "ForFeatureDetector/frontendParams-NMS-Binning2.yaml"))
    p.quality_level = 1e-10
    p.enable_subpixel_corner_refinement = False
    f = _frame("ForStereoFrame/left_fisheye_img_0.webp")
    ofe.FeatureDetector(p).feature_detection(f, None)
    assert len(f.keypoints) == 140
    cnt = _bins(f, p)
    assert np.all(cnt[p.binning_mask == 1] == 10) and np.all(cnt[p.binning_mask == 0] == 0)


# tests/testStereoMatcher.cpp:148 (baseline) -- Euroc rig
def test_rig_baseline_euroc():
    rig = StereoRig(CameraParams.euroc_left(), CameraParams.euroc_right())
    assert abs(rig.baseline - 0.110078) < 1e-4
    # tests/testStereoCamera.cpp:374-440: P2[0,3] = -fx * b
    assert abs(rig.P2[0, 3] + rig.fx * rig.baseline) < 1e-9


# tests/testStereoMatcher.cpp:272-388 -- getRightKeypointsRectified on a synthetically shifted image
def test_stereo_matcher_shifted_849_of_900():
    d = os.path.join(REF_DATA, "ForStereoFrame")
    left = CameraParams.from_yaml(os.path.join(d, "sensorLeft.yaml"))
    right = CameraParams.from_yaml(os.path.join(d, "sensorRight.yaml"))
    rig = StereoRig(left, right)
    assert abs(rig.baseline - 0.110078) < 1e-4            # tests/testStereoMatcher.cpp:148
    p = FrontendParams()                                  # struct defaults, as in the fixture
    m = ofe.StereoMatcher(p, rig)
    img = cv2.imread(os.path.join(d, "left_img_0.webp"), cv2.IMREAD_GRAYSCALE)
    corners = cv2.goodFeaturesToTrack(img, 100, 0.01, 10, blockSize=3, useHarrisDetector=False, k=0.04)
    corners = corners.reshape(-1, 2)
    count_valid = total = 0
    for offset in (-20, -10, -5):
        M = np.eye(3)
        M[0, 2] = offset
        right_img = cv2.warpPerspective(img, M, (img.shape[1], img.shape[0]), flags=cv2.INTER_NEAREST)
        lk = []
        for t in range(2):
            if t == 1:
                lk += [(ofe.KP_VALID, (np.float32(ofe.c_round(x)), np.float32(ofe.c_round(y)))) for x, y in corners]
            else:
                lk += [(ofe.KP_VALID, (np.float32(x), np.float32(y))) for x, y in corners]
            rk = m.get_right_keypoints_rectified(img, right_img, lk, 458.654, rig.baseline)
            for (ls, lp), (rs_, rp) in zip(lk, rk):
                total += 1
                y_left, x_exp, x_act = float(lp[1]), float(lp[0]) + offset, float(rp[0])
                stripe_rows = 11 + 4
                if y_left <= (stripe_rows - 1) // 2 or y_left + (stripe_rows - 1) // 2 >= img.shape[0]:
                    assert rs_ == ofe.KP_NO_RIGHT_RECT
                elif x_exp >= 50 and x_exp + 50 < img.shape[1]:
                    assert rs_ == ofe.KP_VALID
                    assert abs(x_exp - x_act) <= 0.5
                    assert abs(float(lp[1]) - float(rp[1])) <= 0.5
                    count_valid += 1
    assert count_valid == 849
    assert total == 900


# tests/testStereoVisionImuFrontend.cpp:455-661 -- processFirstFrame on the 35-corner synthetic pair
def test_process_first_frame_35_corners():
    d = os.path.join(REF_DATA, "ForStereoTracker")
    left = CameraParams.from_yaml(os.path.join(d, "camLeft.yaml"))
    right = CameraParams.from_yaml(os.path.join(d, "camRight.yaml"))
    rig = StereoRig(left, right)
    p = FrontendParams()                       # struct defaults
    p.min_distance = int(0.05)                 # the test assigns 0.05 to an int member
    p.quality_level = 0.1
    p.max_point_dist = 500
    p.templ_cols = 9
    p.subpixel_refinement_stereo = True
    imgl = cv2.imread(os.path.join(d, "img_distort_left.webp"), cv2.IMREAD_GRAYSCALE)
    imgr = cv2.imread(os.path.join(d, "img_distort_right.webp"), cv2.IMREAD_GRAYSCALE)

    def load(path):
        vals = open(path).read().split()
        n = int(vals[0])
        return np.array([float(v) for v in vals[1:]]).reshape(n, -1)

    gl, gr = load(os.path.join(d, "corners_normal_left.txt")), load(os.path.join(d, "corners_normal_right.txt"))
    depth = load(os.path.join(d, "depth_left.txt")).reshape(-1)
    fe = ofe.StereoFrontend(p, rig)
    out = fe.spin(ofe.StereoFrame.make(0, 0, imgl, imgr, rig), np.eye(3))
    sf = out.frame
    n = len(sf.left_frame.keypoints)
    assert n == len(sf.left_frame.landmarks) == len(sf.left_frame.versors) > 0
    assert all(a == 1 for a in sf.left_frame.landmarks_age)
    assert sf.is_keyframe and sf.is_rectified
    for i in range(n):
        kp = np.array(sf.left_frame.keypoints[i], float)
        dist = np.abs(gl - kp).max(axis=1)
        j = int(np.argmin(dist))
        assert dist[j] < 3                      # findPointInVector tolerance
        assert np.all(np.abs(gl[j] - kp) <= 2)
        assert np.all(np.abs(gr[j] - np.array(sf.right_frame.keypoints[i], float)) <= 2)
        assert sf.left_keypoints_rectified[i][0] == ofe.KP_VALID
        assert sf.right_keypoints_rectified[i][0] == ofe.KP_VALID
        assert abs(depth[j] - sf.keypoints_3d[i][2]) <= 4


def test_getrectsubpix_border_model_matches_cv2():
    """The arithmetic subpix.cuh implements for cv::getRectSubPix (u8 -> f32) windows that leave the
    image, restated in numpy and pinned against cv2 on random border / corner centres: pair-wise 4-tap
    blend inside, 2-tap vertical blend in columns outside (rows above the image take column W-2 on
    the right), fma(P01, a, P00*(1-a)) in rows outside."""
    import cv2
    f32 = np.float32
    rng = np.random.default_rng(11)
    Hh, Ww = 96, 128
    img = cv2.GaussianBlur((rng.random((Hh, Ww)) * 255).astype(np.uint8), (0, 0), 1.5)
    I = img.astype(f32)

    def model(cxf, cyf, pw=23, ph=23):
        cx = f32(f32(cxf) - f32((pw - 1) * 0.5)); cy = f32(f32(cyf) - f32((ph - 1) * 0.5))
        ipx = int(np.floor(cx)); ipy = int(np.floor(cy))
        a = f32(cx - f32(ipx)); b = f32(cy - f32(ipy))
        a11 = f32((f32(1) - a) * (f32(1) - b)); a12 = f32(a * (f32(1) - b)); a21 = f32((f32(1) - a) * b); a22 = f32(a * b)
        a1 = f32(f32(1) - a); b1 = f32(f32(1) - b)
        rx = min(max(-ipx, 0), pw); rw = pw if ipx + pw < Ww else max(Ww - ipx - 1, 0)
        ry = max(-ipy, 0); rh = ph if ipy + ph < Hh else max(Hh - ipy - 1, 0)
        out = np.zeros((ph, pw), f32)
        for i in range(ph):
            outside = i < ry or i >= rh
            y0 = 0 if i < ry else (Hh - 1 if i >= rh else ipy + i)
            y1 = y0 if outside else y0 + 1
            for j in range(pw):
                if j < rx or j >= rw:
                    xc = 0 if j < rx else Ww - 1
                    if i < ry and j >= rw:
                        xc = Ww - 2
                    out[i, j] = f32(f32(I[y0, xc] * b1) + f32(I[y1, xc] * b))
                else:
                    x = ipx + j
                    if outside:
                        out[i, j] = f32(np.float64(I[y0, x + 1]) * np.float64(a) + np.float64(f32(I[y0, x] * a1)))
                    else:
                        out[i, j] = f32(f32(I[y0, x] * a11) + f32(I[y0, x + 1] * a12)) + f32(f32(I[y1, x] * a21) + f32(I[y1, x + 1] * a22))
        return out

    bad = 0
    for k in range(48):
        side = k % 8
        cx = rng.uniform(0, 12) if side in (0, 4, 5) else (rng.uniform(Ww - 12, Ww - 1) if side in (1, 6, 7) else rng.uniform(20, Ww - 20))
        cy = rng.uniform(0, 12) if side in (2, 4, 6) else (rng.uniform(Hh - 12, Hh - 1) if side in (3, 5, 7) else rng.uniform(20, Hh - 20))
        cx, cy = float(f32(cx)), float(f32(cy))
        ref = cv2.getRectSubPix(img, (23, 23), (cx, cy), patchType=cv2.CV_32F)
        bad += int((model(cx, cy) != ref).sum())
    assert bad == 0


def test_rotational_flow_predictor_reference_numbers():
    """RotationalOpticalFlowPredictor::predictSparseFlow on the cube scene of
    tests/testOpticalFlowPredictor.cpp:40-76,566-612 (cam 1 at z = -4 looking at a unit cube, cam 2
    rotated by the quaternion (0.985, 0, 0, 0.174) about z): the sixteen coordinates the reference
    test lists, tolerance 1e-1 px as there."""
    from oracle import frontend as ofe
    fx, W, H = 458.654, 752, 480
    K = np.array([[fx, 0, W // 2], [0, fx, H // 2], [0, 0, 1.0]])
    lmks = [(0, 0, 0), (0, 1, 0), (1, 0, 0), (1, 1, 0), (0, 0, 1), (0, 1, 1), (1, 0, 1), (1, 1, 1)]
    kps = []
    for X, Y, Z in lmks:                       # cam 1: identity rotation, position (0, 0, -4)
        zc = Z + 4.0
        kps.append((fx * X / zc + W // 2, fx * Y / zc + H // 2))
    qw, qx, qy, qz = 0.985, 0.0, 0.0, 0.174    # gtsam::Rot3(w, x, y, z) normalises the quaternion
    n = np.sqrt(qw * qw + qx * qx + qy * qy + qz * qz)
    qw, qx, qy, qz = qw / n, qx / n, qy / n, qz / n
    R = np.array([[1 - 2 * (qy * qy + qz * qz), 2 * (qx * qy - qz * qw), 2 * (qx * qz + qy * qw)],
                  [2 * (qx * qy + qz * qw), 1 - 2 * (qx * qx + qz * qz), 2 * (qy * qz - qx * qw)],
                  [2 * (qx * qz - qy * qw), 2 * (qy * qz + qx * qw), 1 - 2 * (qx * qx + qy * qy)]])
    out = ofe.predict_sparse_flow(kps, R, K, W, H, 1)
    expected = [(376.00003051757812, 239.99998474121094), (415.302001953125, 347.7138671875),
                (483.71389770507812, 200.69801330566406), (523.015869140625, 308.41189575195312),
                (376.00003051757812, 239.99998474121094), (407.44161987304688, 326.17108154296875),
                (462.17111206054688, 208.55841064453125), (493.61270141601562, 294.7294921875)]
    assert len(out) == 8
    for (x, y), (ex, ey) in zip(out, expected):
        assert abs(float(x) - ex) <= 1e-1 and abs(float(y) - ey) <= 1e-1, ((x, y), (ex, ey))


def test_mesher_create_mesh_2d_reference_fixture():
    """tests/testMesher.cpp:147-197: the four corners of chessboard_small.png (UtilsOpenCV::ExtractCorners =
    goodFeaturesToTrack(100, 0.01, 10, blockSize 3)) give two triangles, vertices in the order
    (kp2, kp1, kp3) and (kp1, kp2, kp0); no keypoints -> no triangle."""
    import cv2
    from oracle import mesher
    img = cv2.imread(os.path.join(REF_DATA, "chessboard_small.webp"), cv2.IMREAD_GRAYSCALE)
    kps = cv2.goodFeaturesToTrack(img, 100, 0.01, 10, None, None, 3, False, 0.04).reshape(-1, 2)
    assert len(kps) == 4
    size = (img.shape[1], img.shape[0])
    tri = mesher.create_mesh_2d(size, [tuple(k) for k in kps], list(range(len(kps))), list(range(len(kps))))
    assert tri.shape == (2, 6)
    assert np.array_equal(tri[0], np.concatenate([kps[2], kps[1], kps[3]]))
    assert np.array_equal(tri[1], np.concatenate([kps[1], kps[2], kps[0]]))
    assert mesher.create_mesh_2d(size, [tuple(k) for k in kps], list(range(4)), []).shape == (0, 6)


def test_mesher_stereo_filters_invalid_keypoints():
    from oracle import mesher
    rng = np.random.default_rng(4)
    kps = [(float(x), float(y)) for x, y in rng.uniform(5, 95, (30, 2)).astype(np.float32)]
    lmk = list(range(30))
    status = [0] * 30
    lmk[3] = -1
    status[7] = 2
    tri, l3d = mesher.create_mesh_2d_stereo((100, 100), lmk, status, kps, rng.normal(size=(30, 3)))
    verts = {(float(t[2 * j]), float(t[2 * j + 1])) for t in tri for j in range(3)}
    assert kps[3] not in verts and kps[7] not in verts and len(verts) == 28 and len(l3d) == 28
    # Delaunay: no input point strictly inside any triangle's circumcircle
    P = np.array([k for i, k in enumerate(kps) if i not in (3, 7)], np.float64)
    for t in tri.astype(np.float64):
        (ax, ay), (bx, by), (cx, cy) = t[0:2], t[2:4], t[4:6]
        d = 2 * (ax * (by - cy) + bx * (cy - ay) + cx * (ay - by))
        ux = ((ax * ax + ay * ay) * (by - cy) + (bx * bx + by * by) * (cy - ay) + (cx * cx + cy * cy) * (ay - by)) / d
        uy = ((ax * ax + ay * ay) * (cx - bx) + (bx * bx + by * by) * (ax - cx) + (cx * cx + cy * cy) * (bx - ax)) / d
        r2 = (ax - ux) ** 2 + (ay - uy) ** 2
        assert ((P[:, 0] - ux) ** 2 + (P[:, 1] - uy) ** 2 >= r2 * (1 - 1e-6)).all()
