"""Generates tests/golden/rgbd_frame1.npz from the reference's RGB-D test data: the second frame of tests/data/ForRgbd
(depth_img_1.tiff, CV_32FC1 720x480, and left_img_1.png), the frame that follows rgbd_pair.npz.  Frames 0 -> 1 drive the
frame-level RGB-D step in tests/test_gpu_rgbd_frontend.py.  The depth image is stored losslessly (float32).

Run from the repo root:  python tests/golden/make_rgbd_frame1.py <Kimera-VIO checkout>
"""
import os
import sys

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main(ref_root):
    src = os.path.join(ref_root, "tests", "data", "ForRgbd")
    depth = cv2.imread(os.path.join(src, "depth_img_1.tiff"), cv2.IMREAD_UNCHANGED)
    assert depth is not None and depth.dtype == np.float32 and depth.shape == (480, 720)
    # UtilsOpenCV::ReadAndConvertToGrayScale (UtilsOpenCV.cpp:390-403): imread, cvtColor BGR2GRAY for 3 channels
    img = cv2.imread(os.path.join(src, "left_img_1.png"), cv2.IMREAD_ANYCOLOR)
    if img.ndim == 3:
        img = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)
    out = os.path.join(ROOT, "tests", "golden", "rgbd_frame1.npz")
    np.savez_compressed(out, depth=depth, left=img)
    print("wrote", out, depth.shape, img.shape, os.path.getsize(out))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
