"""Stores under tests/golden/reference/ the Kimera-VIO data fixtures that the known-answer tests
(tests/test_oracle_pins.py, tests/test_host_logic.py) and the Euroc pipeline parity test
(tests/test_gpu_long.py) read, so that the suite needs nothing outside the repository:

  params/<rig>/{FrontendParams,LeftCameraParams}.yaml   the shipped rig files, verbatim
  data/...                                              YAML / text fixtures of Kimera-VIO's tests/data, verbatim;
                                                        its PNG images re-encoded as lossless WebP (pixels identical)
  euroc_micro_rel_R.npy                                 frame-to-frame rotations camLrectKm1_R_camLrectK of the Euroc
                                                        pairs stored in euroc_micro.npz, integrated from the dataset's
                                                        gyroscope samples (imu0/data.csv, no bias correction)

The image data are Euroc V1_01_easy ((c) ASL/ETHZ) and Kimera-VIO's test images (BSD-2-Clause).

Run from the repository root:  python tests/golden/make_reference_fixtures.py <Kimera-VIO checkout>
"""
import glob
import os
import shutil
import sys

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from kimera_vio_b200.params import CameraParams  # noqa: E402
from kimera_vio_b200.rig import StereoRigSetup  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference")
PARAM_FILES = ["FrontendParams.yaml", "LeftCameraParams.yaml"]
DATA_FILES = ["sensor.yaml",
              "ForFeatureDetector/frontendParams-noNMS.yaml", "ForFeatureDetector/frontendParams-NMS-TopN.yaml",
              "ForFeatureDetector/frontendParams-NMS-Binning.yaml", "ForFeatureDetector/frontendParams-NMS-Binning2.yaml",
              "ForStereoFrame/sensorLeft.yaml", "ForStereoFrame/sensorRight.yaml",
              "ForStereoTracker/camLeft.yaml", "ForStereoTracker/camRight.yaml",
              "ForStereoTracker/corners_normal_left.txt", "ForStereoTracker/corners_normal_right.txt",
              "ForStereoTracker/depth_left.txt"]
DATA_IMAGES = ["chessboard_small.png", "ForStereoFrame/left_fisheye_img_0.png", "ForStereoFrame/left_img_0.png",
               "ForStereoTracker/img_distort_left.png", "ForStereoTracker/img_distort_right.png"]


def so3_exp(w):
    th = float(np.linalg.norm(w))
    if th < 1e-12:
        return np.eye(3)
    k = w / th
    K = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * (K @ K)


def euroc_rel_R(mav0, ts):
    """Rotation of the rectified left camera between consecutive timestamps (identity first)."""
    imu = np.loadtxt(os.path.join(mav0, "imu0/data.csv"), delimiter=",", skiprows=1)
    it, gyro = imu[:, 0].astype(np.int64), imu[:, 1:4]
    left = CameraParams.euroc_left()
    rig = StereoRigSetup(left, CameraParams.euroc_right())
    body_R_cam = left.T_BS[:3, :3]
    rel = [np.eye(3)]
    for k in range(1, len(ts)):
        sel = np.nonzero((it >= ts[k - 1]) & (it < ts[k]))[0]
        dR = np.eye(3)
        for i in sel:                          # forward integration of the raw gyro samples
            dt = (min(it[i + 1], ts[k]) - it[i]) * 1e-9
            dR = dR @ so3_exp(gyro[i] * dt)
        rel.append(rig.R1 @ (body_R_cam.T @ dR @ body_R_cam) @ rig.R1.T)
    return np.stack(rel)


def main(ref):
    for rig in sorted(os.listdir(os.path.join(ref, "params"))):
        for f in PARAM_FILES:
            src = os.path.join(ref, "params", rig, f)
            if os.path.exists(src):
                os.makedirs(os.path.join(OUT, "params", rig), exist_ok=True)
                shutil.copyfile(src, os.path.join(OUT, "params", rig, f))
    data = os.path.join(ref, "tests", "data")
    for f in DATA_FILES:
        os.makedirs(os.path.dirname(os.path.join(OUT, "data", f)), exist_ok=True)
        shutil.copyfile(os.path.join(data, f), os.path.join(OUT, "data", f))
    for f in DATA_IMAGES:
        img = cv2.imread(os.path.join(data, f), cv2.IMREAD_GRAYSCALE)
        ok, buf = cv2.imencode(".webp", img, [cv2.IMWRITE_WEBP_QUALITY, 101])      # quality > 100: lossless
        assert ok and np.array_equal(cv2.imdecode(buf, cv2.IMREAD_GRAYSCALE), img), f
        out = os.path.join(OUT, "data", f[:-4] + ".webp")
        os.makedirs(os.path.dirname(out), exist_ok=True)
        with open(out, "wb") as fh:
            fh.write(buf.tobytes())
    ts = np.load(os.path.join(ROOT, "tests", "golden", "euroc_micro.npz"))["timestamps"]
    np.save(os.path.join(OUT, "euroc_micro_rel_R.npy"), euroc_rel_R(os.path.join(data, "MicroEurocDataset", "mav0"), ts))
    print("wrote", OUT)


if __name__ == "__main__":
    main(sys.argv[1])
