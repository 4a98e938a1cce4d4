"""Corner selection (cand_kernel, the top-K prefilter and sort_greedy_kernel in gftt.cu) against
cv2.goodFeaturesToTrack through the oracle's FeatureDetector, bit-exact: corner list and order.

The scenes are built to reach the selection branches that ordinary frames never take:
  * prefix redo       the best GREEDY_TOPK candidates yield fewer than maxCorners acceptances, so the selection
                      is repeated over the full list (pass 1); with a smaller min_distance more than
                      GREEDY_ACC_MAX corners are accepted and the accepted keys go to global memory
  * plateaus          a 2-px checkerboard: nearly every interior pixel is a candidate, in five distinct values,
                      so equal responses are ordered by address, the candidate list is far longer than one
                      entry per eight pixels, the threshold bin of the prefilter overflows GREEDY_SEL_CAP (the
                      prefix is abandoned) and the bookkeeping lives in global memory; min_distance 0 takes the
                      full bitonic sort
  * quality edge      quality levels whose threshold maxVal * qualityLevel, formed in double and rounded to
                      float once (cv::GFTTDetector keeps qualityLevel a double), differs from the one formed
                      from a float-rounded quality, on a local maximum of the response
Every scene has a CPU check (cv2 and numpy only) that proves it still reaches its branch, so the GPU test
cannot quietly stop covering it."""
import dataclasses
import functools

import cv2
import numpy as np
import pytest

import helpers as H
from kimera_vio_b200 import lib as kl
from kimera_vio_b200.params import CameraParams, FrontendParams
from kimera_vio_b200.rig import StereoRigSetup
from oracle import frontend as ofe

# gftt.cu
GREEDY_TOPK = 12288
GREEDY_SEL_CAP = 16384
GREEDY_ACC_MAX = 2048
SMEM_KEYS = 16384
CAND_HIST_BINS = 2048

SIZES = [(752, 480), (1280, 720)]


# ---------------------------------------------------------------------------------------------------------------
# plain restatement of cv::goodFeaturesToTrack (minEigenVal, blockSize 3)
# ---------------------------------------------------------------------------------------------------------------
def candidates(img, quality, mask=None):
    """(values, ys, xs, maxv) of the candidates -- interior local maxima (3x3, ties pass) above the threshold --
    in cv2's processing order: value descending, ties by address descending."""
    e = cv2.cornerMinEigenVal(img, 3, ksize=3)
    m = np.ones(img.shape, bool) if mask is None else mask > 0
    maxv = np.float32(e[m].max()) if m.any() else np.float32(0)
    thr = np.float32(np.float64(maxv) * np.float64(quality))
    h, w = e.shape
    pad = np.pad(e, 1, constant_values=-np.inf)
    nb = np.max(np.stack([pad[dy:dy + h, dx:dx + w] for dy in range(3) for dx in range(3) if (dy, dx) != (1, 1)]), 0)
    ok = (e > thr) & (e >= nb) & m
    ok[0, :] = ok[-1, :] = ok[:, 0] = ok[:, -1] = False
    ys, xs = np.nonzero(ok)
    v = e[ys, xs]
    order = np.lexsort((-(ys.astype(np.int64) * w + xs), -v))
    return v[order], ys[order], xs[order], maxv


def greedy(ys, xs, md, limit=None):
    """Indices (into the ordered candidate list) that the min-distance rule accepts, in acceptance order."""
    acc, grid = [], {}
    for i, (y, x) in enumerate(zip(ys.tolist(), xs.tolist())):
        gx, gy = x // md, y // md
        if any((px - x) ** 2 + (py - y) ** 2 < md * md
               for a in (-1, 0, 1) for b in (-1, 0, 1) for px, py in grid.get((gx + a, gy + b), ())):
            continue
        acc.append(i)
        grid.setdefault((gx, gy), []).append((x, y))
        if limit is not None and len(acc) >= limit:
            break
    return acc


def prefilter(v, maxv):
    """cand_hist_kernel / cand_compact_kernel: (number of candidates in bins <= the threshold bin, usable)."""
    if len(v) <= GREEDY_TOPK:
        return len(v), False
    bits = v.view(np.uint32) >> 16
    d = np.clip(int(np.float32(maxv).view(np.uint32) >> 16) - bits.astype(np.int64), 0, CAND_HIST_BINS - 1)
    cum = np.cumsum(np.bincount(d, minlength=CAND_HIST_BINS))
    t = int(np.argmax(cum >= GREEDY_TOPK))
    n_sel = int(cum[t])
    return n_sel, n_sel <= GREEDY_SEL_CAP


def list_cap_one_in_eight(w, h):
    """A candidate list sized for one entry in eight pixels (power of two, at least 8192)."""
    p = 8192
    while p < w * h // 8:
        p <<= 1
    return p


# ---------------------------------------------------------------------------------------------------------------
# scenes
# ---------------------------------------------------------------------------------------------------------------
def scene_prefix_redo(w, h):
    """Strong texture (sigma 60) in the left 400 columns, weak texture (sigma 6) elsewhere: the best candidates
    crowd into the left part, where min_distance rejects most of them."""
    rng = np.random.default_rng(5)
    img = np.full((h, w), 128, np.float32)
    img[:, :400] += rng.normal(0, 60, (h, 400))
    img[:, 400:] += rng.normal(0, 6, (h, w - 400))
    return np.clip(img, 0, 255).astype(np.uint8)


def checker(w, h):
    yy, xx = np.mgrid[0:h, 0:w]
    return ((((xx >> 1) + (yy >> 1)) & 1) * 200 + 20).astype(np.uint8)


def euroc_frame(w, h):
    _, lefts, _ = H.golden()
    img = lefts[0]
    return img if img.shape == (h, w) else cv2.resize(img, (w, h), interpolation=cv2.INTER_LINEAR)


def scene_checker_in_euroc(w, h):
    """A real frame with a checkerboard patch over its central quarter."""
    img = euroc_frame(w, h).copy()
    x0, y0, pw, ph = w // 4, h // 4, w // 2, h // 2
    img[y0:y0 + ph, x0:x0 + pw] = checker(pw, ph)
    return img


SCENES = {"prefix_redo": scene_prefix_redo, "checker": checker, "checker_in_euroc": scene_checker_in_euroc}

# (scene, maxCorners, min_distance): every case runs at quality_level 0.001
CASES = [("prefix_redo", 800, 20), ("prefix_redo", 3000, 10)] + \
        [(s, 2000, md) for s in ("checker", "checker_in_euroc") for md in (20, 8, 0)]


@functools.lru_cache(maxsize=None)
def scene(name, w, h):
    return SCENES[name](w, h)


def params(max_corners, min_distance, quality=0.001):
    return dataclasses.replace(FrontendParams.euroc(), max_nr_keypoints_before_anms=max_corners,
                               min_distance=min_distance, quality_level=quality)


def make_ctx(p, w, h):
    left, right = CameraParams.euroc_left(), CameraParams.euroc_right()
    if (w, h) != (left.width, left.height):
        left, right = left.scaled(w, h), right.scaled(w, h)
    rig = StereoRigSetup(left, right)
    cfg = kl.make_config(p, w, h, batch=1, sobel_cpu_tail_start=H.sobel_cpu_tail_start(w))
    return kl.Context(cfg, rig.to_c()), left


def oracle_raw(p, img, cam, kps=(), lmks=()):
    det = ofe.FeatureDetector(p)
    fr = ofe.Frame(0, 0, img, cam, keypoints=list(kps), landmarks=list(lmks))
    raw = det.raw_feature_detection(img, det.build_mask(fr))
    return np.array([k.pt for k in raw], np.float32).reshape(-1, 2)


# ---------------------------------------------------------------------------------------------------------------
# CPU scene checks
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,h", SIZES)
def test_scene_prefix_redo_reaches_pass1_and_global_accepts(w, h):
    img = scene("prefix_redo", w, h)
    v, ys, xs, maxv = candidates(img, 0.001)
    n_sel, usable = prefilter(v, maxv)
    assert usable, "the prefilter must produce a prefix for pass 0 to use it"
    for maxc, md in ((800, 20), (3000, 10)):
        pre = greedy(ys[:n_sel], xs[:n_sel], md)
        full = greedy(ys, xs, md)
        ref = cv2.goodFeaturesToTrack(img, maxc, 0.001, md, blockSize=3).reshape(-1, 2)
        assert len(pre) < maxc, "the prefix must fall short of maxCorners (pass 1 redo)"
        assert len(ref) == min(len(full), maxc)
        assert np.array_equal(ref, np.stack([xs, ys], 1)[full[:maxc]].astype(np.float32))
        if md == 20:
            assert len(ref) > len(pre), "the full list must accept more corners than the prefix"
        else:
            assert len(full) > GREEDY_ACC_MAX, "the accepted keys must overflow the shared-memory list"


@pytest.mark.parametrize("w,h", SIZES)
@pytest.mark.parametrize("name", ["checker", "checker_in_euroc"])
def test_scene_plateaus_overflow_list_and_prefilter(name, w, h):
    img = scene(name, w, h)
    v, ys, xs, maxv = candidates(img, 0.001)
    assert len(v) > list_cap_one_in_eight(w, h), "more candidates than one in eight pixels"
    assert len(v) > SMEM_KEYS, "the candidate keys must not fit in shared memory"
    n_sel, usable = prefilter(v, maxv)
    assert n_sel > GREEDY_SEL_CAP and not usable, "the threshold bin must overflow the prefix buffer"
    # equal responses: the order among them is decided by address alone
    top = v[:2000]
    assert len(np.unique(top)) < len(top) // 10
    # the restated rule is cv2's, including the tie order
    for md in (20, 8, 0):
        ref = cv2.goodFeaturesToTrack(img, 2000, 0.001, md, blockSize=3).reshape(-1, 2)
        sel = greedy(ys, xs, md, limit=2000) if md >= 1 else list(range(min(2000, len(v))))
        assert np.array_equal(ref, np.stack([xs, ys], 1)[sel].astype(np.float32)), md
        if md == 8:
            assert len(greedy(ys, xs, md)) > GREEDY_ACC_MAX


# ---------------------------------------------------------------------------------------------------------------
# quality threshold edge
# ---------------------------------------------------------------------------------------------------------------
def _gftt(img, maxc, q, md, mask):
    c = cv2.goodFeaturesToTrack(img, maxc, q, md, mask=mask, blockSize=3)
    return np.zeros((0, 2), np.float32) if c is None else c.reshape(-1, 2)


def search_quality_edges(img, maxc, md, mask=None, target=None, want=3, budget=20000):
    """Quality levels q at which a local maximum r lies between f32(maxv * q) and f32(maxv * f64(f32(q))), and
    cv2's corner list at q differs from its list at the float-rounded quality."""
    e = cv2.cornerMinEigenVal(img, 3, ksize=3)
    m = np.full(img.shape, 255, np.uint8) if mask is None else mask
    maxv = float(e[m > 0].max())
    h, w = e.shape
    pad = np.pad(e, 1, constant_values=-np.inf)
    nb = np.max(np.stack([pad[dy:dy + h, dx:dx + w] for dy in range(3) for dx in range(3) if (dy, dx) != (1, 1)]), 0)
    lm = (e >= nb) & (m > 0)
    lm[0, :] = lm[-1, :] = lm[:, 0] = lm[:, -1] = False
    vals = np.unique(e[lm])
    vals = vals[vals > 0]
    order = vals[::-1] if target is None else vals[np.argsort(np.abs(np.log(vals / maxv) - np.log(target)), kind="stable")]
    hits = []
    for r in order[:budget]:
        r = np.float32(r)
        q0 = float(r) / maxv
        for k in range(-40, 41):
            q = q0 * (1 + k * 1e-9)
            if (r > np.float32(maxv * q)) != (r > np.float32(maxv * float(np.float32(q)))):
                a = _gftt(img, maxc, q, md, mask)
                b = _gftt(img, maxc, float(np.float32(q)), md, mask)
                if a.shape != b.shape or not np.array_equal(a, b):
                    hits.append(q)
                break
        if len(hits) >= want:
            break
    return hits


def masked_keypoints(w, h):
    rng = np.random.default_rng(11)
    kps = [(np.float32(x), np.float32(y)) for x, y in zip(rng.uniform(0, w, 120), rng.uniform(0, h, 120))]
    lmks = [i if i % 5 else -1 for i in range(len(kps))]
    return kps, lmks


def quality_image(name):
    if name == "euroc":
        return euroc_frame(752, 480)
    _, frames = H.synth_frames(1)
    return frames[0].left


# (image, maxCorners, min_distance, masked, target quality): min_distance 1 with few corners near q ~ 1, and the
# shipped detector settings (min_distance 20, 2000 corners) near the shipped quality 1e-3
QUALITY_CASES = [("euroc", 4096, 1, False, None), ("synth", 4096, 1, False, None),
                 ("euroc", 2000, 20, False, 1e-3), ("euroc", 2000, 20, True, 1e-3)]


@functools.lru_cache(maxsize=None)
def quality_edges(name, maxc, md, masked, target):
    img = quality_image(name)
    kps, lmks = masked_keypoints(752, 480) if masked else ((), ())
    mask = None
    if masked:
        det = ofe.FeatureDetector(params(maxc, md))
        mask = det.build_mask(ofe.Frame(0, 0, img, CameraParams.euroc_left(), keypoints=list(kps), landmarks=list(lmks)))
    return img, kps, lmks, mask, tuple(search_quality_edges(img, maxc, md, mask, target))


@pytest.mark.parametrize("case", QUALITY_CASES, ids=lambda c: "%s_md%d%s" % (c[0], c[2], "_masked" if c[3] else ""))
def test_scene_quality_edges_found(case):
    img, kps, lmks, mask, qs = quality_edges(*case)
    assert len(qs) >= 3
    for q in qs:
        a, b = _gftt(img, case[1], q, case[2], mask), _gftt(img, case[1], float(np.float32(q)), case[2], mask)
        assert a.shape != b.shape or not np.array_equal(a, b)
        if case[4] is not None:
            assert 0.5 * case[4] < q < 2 * case[4]


def test_quality_edge_known_values():
    """Three quality levels on the Euroc golden frame 0 (min_distance 1, 4096 corners) whose corner counts
    differ between the double and the float-rounded threshold."""
    img = euroc_frame(752, 480)
    for q, n_double, n_float in ((0.9649973733580902, 2, 3), (0.9233312913650042, 6, 5), (0.8638855021376395, 11, 10)):
        assert len(_gftt(img, 4096, q, 1, None)) == n_double
        assert len(_gftt(img, 4096, float(np.float32(q)), 1, None)) == n_float


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("w,h", SIZES)
@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s_%d_md%d" % c)
def test_select_matches_cv2(case, w, h):
    name, maxc, md = case
    img = scene(name, w, h)
    p = params(maxc, md)
    ctx, cam = make_ctx(p, w, h)
    try:
        e = oracle_raw(p, img, cam)
        g, _ = ctx.detect_raw(img)
        g2, _ = ctx.detect_raw(img)
        same = g.shape == e.shape and bool(np.array_equal(g, e))
        first = -1
        if not same and len(g) and len(e):
            k = min(len(g), len(e))
            d = np.nonzero(np.any(g[:k] != e[:k], axis=1))[0]
            first = int(d[0]) if len(d) else k
        H.diag("gftt_select", scene=name, w=w, h=h, max_corners=maxc, min_distance=md, n_gpu=len(g), n_ref=len(e),
               same=same, first_diff=first, repeat_same=bool(np.array_equal(g, g2)))
        assert g.shape == e.shape
        assert np.array_equal(g, e)
        assert np.array_equal(g, g2), "two runs on the same input must select the same corners"
        if name == "prefix_redo" and md == 20:
            # the whole detector (ANMS binning + sub-pixel refinement) on top of the redone selection
            det = ofe.FeatureDetector(p)
            need = p.max_features_per_frame
            ed = det.detect_corners(ofe.Frame(0, 0, img, cam), need)
            gd = ctx.detect(img, [], [], need)
            assert len(gd) == len(ed)
            assert len(ed) == 0 or np.abs(gd - ed).max() <= 1e-3
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", QUALITY_CASES, ids=lambda c: "%s_md%d%s" % (c[0], c[2], "_masked" if c[3] else ""))
def test_quality_edge_matches_cv2(case):
    img, kps, lmks, mask, qs = quality_edges(*case)
    assert len(qs) >= 3
    _, maxc, md, _, _ = case
    cam = CameraParams.euroc_left()
    bad = []
    for q in qs:
        p = params(maxc, md, q)
        ctx, _ = make_ctx(p, 752, 480)
        try:
            e = oracle_raw(p, img, cam, kps, lmks)
            g, _ = ctx.detect_raw(img, kps, lmks)
        finally:
            ctx.close()
        same = g.shape == e.shape and bool(np.array_equal(g, e))
        H.diag("gftt_quality_edge", image=case[0], min_distance=md, masked=case[3], quality=q, n_gpu=len(g),
               n_ref=len(e), same=same)
        if not same:
            bad.append((q, len(g), len(e)))
    assert not bad, "corner lists differ from cv2 at quality (q, n_gpu, n_ref): %r" % bad
