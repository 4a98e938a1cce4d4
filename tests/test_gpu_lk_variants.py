"""kvfe_track and kvfe_pyramid against cv2.calcOpticalFlowPyrLK / cv2.buildOpticalFlowPyramid away from the
Euroc default (752x480, window 24, 5 levels, lk_kernel_tma<24>):
  * 640x400, window 24      the coarsest level is 40x25, narrower than the TMA kernel's 28-px reflection limit:
                            lk_kernel_col<24>
  * 752x480, window 21/31/32  the generic lk_kernel; 31 and 32 also stop the pyramid after 4 levels, and 32 is
                            its largest shared-memory configuration
  * 640x360, window 24      the TMA kernel on a pyramid cv stops after 4 levels
  * 752x480, window 24, klt_max_level 0, and window 5
Statuses exact, positions within 1e-3 px, pyramids bit-exact with as many levels as cv2 returns."""
import dataclasses

import cv2
import numpy as np
import pytest

import helpers as H
import scenes
from kimera_vio_b200 import lib as kl
from kimera_vio_b200.params import CameraParams, FrontendParams
from kimera_vio_b200.rig import StereoRigSetup
from kimera_vio_b200.synth import SynthStream
from oracle import frontend as ofe
from oracle.rig import StereoRig

TOL_PX = 1e-3
KVFE_MAX_LEVELS = 8          # kvfe_internal.h
TMA_MIN_TOP = 28             # lk.cu launch_lk: the TMA kernel needs a coarsest level of at least 28 x 28

# (id, width, height, klt_win_size, klt_max_level, kernel launch_lk must pick, levels cv2 returns)
CASES = [
    ("640x400_win24", 640, 400, 24, 4, "col24", 4),
    ("752x480_win21", 752, 480, 21, 4, "generic", 4),
    ("752x480_win31", 752, 480, 31, 4, "generic", 3),
    ("752x480_win32", 752, 480, 32, 4, "generic", 3),
    ("640x360_win24", 640, 360, 24, 4, "tma24", 3),
    ("752x480_win24_level0", 752, 480, 24, 0, "tma24", 0),
    ("752x480_win5", 752, 480, 5, 4, "generic", 4),
]
IDS = [c[0] for c in CASES]


def pyramid_sizes(w, h, win, max_level):
    """Level sizes of kvfe_create's pyramid (cv::buildOpticalFlowPyramid's stopping rule, restated in api.cu)."""
    sizes = []
    for level in range(min(max_level, KVFE_MAX_LEVELS - 1) + 1):
        sizes.append((w, h))
        w, h = (w + 1) // 2, (h + 1) // 2
        if w <= win or h <= win:
            break
    return sizes


def lk_kernel_for(w, h, win, max_level):
    """launch_lk's choice for this geometry."""
    tw, th = pyramid_sizes(w, h, win, max_level)[-1]
    if win == 24:
        return "tma24" if tw >= TMA_MIN_TOP and th >= TMA_MIN_TOP else "col24"
    return "generic"


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_scene_kernel_and_levels(case):
    _, w, h, win, ml, kernel, levels = case
    assert lk_kernel_for(w, h, win, ml) == kernel
    assert len(pyramid_sizes(w, h, win, ml)) - 1 == levels
    n, pyr = cv2.buildOpticalFlowPyramid(np.zeros((h, w), np.uint8), (win, win), ml, withDerivatives=False)
    assert n == levels
    assert [p.shape[::-1] for p in pyr] == pyramid_sizes(w, h, win, ml)


def test_scene_level_rule_agrees_with_cv2():
    """The restated stopping rule gives cv2's level count across sensor sizes and windows."""
    for w, h in ((640, 400), (640, 360), (640, 480), (752, 480), (720, 480), (1280, 720), (320, 240), (100, 60)):
        for win in (3, 5, 13, 21, 24, 25, 31, 32):
            for ml in (0, 1, 3, 4, 7):
                n, _ = cv2.buildOpticalFlowPyramid(np.zeros((h, w), np.uint8), (win, win), ml, withDerivatives=False)
                assert n == len(pyramid_sizes(w, h, win, ml)) - 1, (w, h, win, ml)


def cameras(w, h):
    left, right = CameraParams.euroc_left(), CameraParams.euroc_right()
    if (w, h) != (left.width, left.height):
        left, right = left.scaled(w, h), right.scaled(w, h)
    return left, right


def image_pairs(w, h):
    """Euroc golden pairs (one and four frames apart) and a synthetic pair, resized with INTER_AREA when the
    case's sensor is smaller than 752x480."""
    _, lefts, _ = H.golden()
    _, frames = H.synth_frames(2)
    pairs = [("euroc", lefts[0], lefts[1]), ("euroc_gap", lefts[0], lefts[4]), ("synth", frames[0].left, frames[1].left)]
    if (w, h) == (752, 480):
        return pairs
    return [(n, cv2.resize(a, (w, h), interpolation=cv2.INTER_AREA), cv2.resize(b, (w, h), interpolation=cv2.INTER_AREA))
            for n, a, b in pairs]


def track_points(img, w, h, rng):
    c = cv2.goodFeaturesToTrack(img, 300, 0.001, 20).reshape(-1, 2)
    # border / textureless / off-grid points
    extra = np.array([[2.5, 3.5], [w - 2.8, h - 2.9], [w / 2 - 0.7, 1.2], [1.1, h / 2 + 0.9], [w - 51.3, 10.2]], np.float32)
    return np.concatenate([c, extra, c[:40] + rng.uniform(-0.5, 0.5, (40, 2)).astype(np.float32)]).astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_lk_variant_matches_cv2(case):
    name, w, h, win, ml, kernel, levels = case
    p = dataclasses.replace(FrontendParams.euroc(), klt_win_size=win, klt_max_level=ml)
    left, right = cameras(w, h)
    rig = StereoRigSetup(left, right)
    K = StereoRig(left, right).left.K
    cfg = kl.make_config(p, w, h, batch=1, sobel_cpu_tail_start=H.sobel_cpu_tail_start(w))
    ctx = kl.Context(cfg, rig.to_c())
    rng = np.random.default_rng(3)
    crit = (cv2.TERM_CRITERIA_COUNT + cv2.TERM_CRITERIA_EPS, p.klt_max_iter, p.klt_eps)
    try:
        for pair, A, B in image_pairs(w, h):
            lv = ctx.pyramid(A)
            n_ref, ref = cv2.buildOpticalFlowPyramid(A, (win, win), ml, withDerivatives=False)
            bad_lv = [i + 1 for i, g in enumerate(lv) if i + 1 >= len(ref) or g.shape != ref[i + 1].shape
                      or not np.array_equal(g, ref[i + 1])]
            H.diag("lk_variant_pyramid", case=name, pair=pair, n_gpu=len(lv), n_ref=int(n_ref), bad_levels=bad_lv)
            assert len(lv) == n_ref == levels
            assert not bad_lv
            pts = track_points(A, w, h, rng)
            for rot in (np.eye(3), scenes.expmap([0.004, -0.003, 0.002])):
                pred = ofe.predict_sparse_flow([tuple(q) for q in pts], rot, K, w, h, p.optical_flow_predictor_type)
                a = pts.reshape(-1, 1, 2)
                b = np.array(pred, np.float32).reshape(-1, 1, 2)
                nxt, st, _ = cv2.calcOpticalFlowPyrLK(A, B, a, b.copy(), winSize=(win, win), maxLevel=ml,
                                                      criteria=crit, flags=cv2.OPTFLOW_USE_INITIAL_FLOW)
                gp, gn, gs = ctx.track(A, B, rot, pts)
                pred_bad = int((gp != np.array(pred, np.float32)).sum())
                st_bad = int((gs != st.reshape(-1)).sum())
                ok = (st.reshape(-1) == 1) & (gs == 1)
                d = np.abs(gn - nxt.reshape(-1, 2))[ok]
                H.diag("lk_variant", case=name, kernel=kernel, pair=pair, rot=not np.allclose(rot, np.eye(3)),
                       n=len(pts), pred_mismatch=pred_bad, status_mismatch=st_bad,
                       n_fail_ref=int((st.reshape(-1) != 1).sum()), max_err=float(d.max()) if len(d) else 0.0,
                       n_over_tol=int((d.max(axis=1) > TOL_PX).sum()) if len(d) else 0,
                       n_exact=int((d.max(axis=1) == 0).sum()) if len(d) else 0)
                assert pred_bad == 0
                assert st_bad == 0
                assert len(d) == 0 or d.max() <= TOL_PX
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("rig_case", ["640x400_win24", "752x480_win21"])
def test_lk_variant_sequence(rig_case):
    """A short synthetic sequence through the whole front-end step with the fallback LK kernels, against the
    oracle's StereoFrontend: lk_kernel_col<24> on a 640x400 rig, the generic lk_kernel at window 21."""
    from test_gpu_sequence import run_sequence
    w, h, win = (640, 400, 24) if rig_case == "640x400_win24" else (752, 480, 21)
    p = dataclasses.replace(FrontendParams.euroc(), klt_win_size=win)
    left, right = cameras(w, h)
    rig = StereoRigSetup(left, right)
    cfg = kl.make_config(p, w, h, batch=1, sobel_cpu_tail_start=H.sobel_cpu_tail_start(w))
    ctx = kl.Context(cfg, rig.to_c())
    s = SynthStream(left, right, rig.R1, seed=515)
    fr = [s.frame(k) for k in range(8)]
    fe = ofe.StereoFrontend(p, StereoRig(left, right))
    try:
        ok = run_sequence(ctx, [fe], [[(f.left, f.right, f.timestamp) for f in fr]],
                          lambda b, k, l: s.kf_rotation(l, k), "lk_" + rig_case)
    finally:
        ctx.close()
    assert ok
