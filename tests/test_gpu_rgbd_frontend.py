"""Row f2: the frame-level RGB-D front-end (frontend_type 2, kvfe_frontend_step_rgbd / kvfe_pipeline_push_rgbd) against
oracle/rgbd.py: RgbdFrontend, the line-by-line restatement of RgbdVisionImuFrontend.cpp:183-395, fed the same frames.

Every packet must equal the oracle's frame: keypoints (<= 1e-3 px), landmark ids, ages, versors (< 1e-5), the keyframe
decision and both tracking statuses; on keyframes also left_keypoints_rectified_ (Camera::undistortKeypoints), the
hallucinated right keypoints and their statuses, keypoints_depth_, keypoints_3d_, the distorted right keypoints, the
checkStatusRightKeypoints counters and the smart stereo measurements (uR present whenever the right keypoint is VALID).
Undistorted / right coordinates use the 2e-3 px bound test_gpu_mono.py uses for keypoints_undistorted_.

Scenes: a synthetic Euroc-left RGB-D stream (IMU rotation, identity rotation, uint16 millimetres, depth holes, a
textureless frame, use_stereo_tracking 0, use_ransac 0); the shipped KinectAzure rig with equalizeImage; the reference's
real RGB-D frames 0 -> 1 with a forced keyframe; a batch of three streams; the pipeline with depth in pageable, pinned and
device memory.  The CPU checks at the bottom make sure each oracle run still reaches the branch its scene is meant to cover.
"""
import dataclasses
import json
import math
import os

import cv2
import numpy as np
import pytest

import helpers as H
from kimera_vio_b200 import lib as kl
from kimera_vio_b200.params import CameraParams, FrontendParams
from kimera_vio_b200.rig import RgbdRigSetup
from kimera_vio_b200.synth import SynthStream
from oracle import frontend as ofe
from oracle import rgbd as org

f32 = np.float32
REF_PARAMS = os.path.join(H.ROOT, "tests", "golden", "reference", "params")
N_FRAMES = 16
TEXTURELESS_FRAME = 8            # flat image: the NEXT frame loses every track (LK needs the gradient of the previous frame)


# ---------------------------------------------------------------------------------------------------------------------
# scenes
# ---------------------------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class Scene:
    p: FrontendParams
    cam: CameraParams
    frames: list                  # (timestamp, intensity image, depth image)
    rotations: str                # "imu" or "identity"
    stream: SynthStream = None
    force: tuple = ()             # frames forced to be keyframes (Frame::isKeyframe_)
    equalize: bool = False        # the oracle sees cv2.equalizeHist of the image (the data provider's job)


def _patches(depth, k, dtype):
    """Depth holes: NaN, +inf and 0 squares (0 only for uint16) at places that change every frame, so that tracked keypoints
    fall into them (NO_DEPTH from a hole / below min_depth)."""
    rng = np.random.default_rng(1000 + k)
    H_, W_ = depth.shape
    vals = [0] if dtype == np.uint16 else [np.nan, np.inf, 0.0]
    for i in range(9):
        y, x = int(rng.integers(0, H_ - 48)), int(rng.integers(0, W_ - 48))
        depth[y:y + 48, x:x + 48] = vals[i % len(vals)]
    return depth


_scene_cache = {}


def synth_scene(variant: str) -> Scene:
    if variant in _scene_cache:
        return _scene_cache[variant]
    p = FrontendParams.euroc()
    left, right = CameraParams.euroc_left(), CameraParams.euroc_right()
    u16 = variant == "u16_mm"
    cam = dataclasses.replace(left, depth={"virtual_baseline": float(f32(0.2)), "depth_to_meters": 0.001 if u16 else 1.0,
                                           "min_depth": 0.3, "max_depth": 4.0, "is_registered": True})
    if variant == "no_stereo_tracking":
        p = dataclasses.replace(p, use_stereo_tracking=False)
    if variant == "no_ransac":
        p = dataclasses.replace(p, use_ransac=False)
    s = SynthStream(left, right, np.eye(3), seed=4242)
    frames = []
    for k in range(N_FRAMES):
        f, depth = s.frame_with_depth(k)
        img = f.left
        if variant == "textureless" and k == TEXTURELESS_FRAME:
            img = np.full_like(img, 128)
        if u16:
            depth = np.clip(np.rint(depth * 1000.0), 0, 65535).astype(np.uint16)
        if variant in ("holes", "u16_mm"):
            depth = _patches(depth, k, depth.dtype.type)
        frames.append((f.timestamp, img, np.ascontiguousarray(depth)))
    sc = Scene(p, cam, frames, "identity" if variant == "identity" else "imu", stream=s)
    _scene_cache[variant] = sc
    return sc


def kinect_scene() -> Scene:
    if "kinect" in _scene_cache:
        return _scene_cache["kinect"]
    p = FrontendParams.from_yaml(os.path.join(REF_PARAMS, "KinectAzure", "FrontendParams.yaml"))
    assert p.use_pnp_tracking and p.equalize_image
    p = dataclasses.replace(p, use_pnp_tracking=False)        # PnP is not built (out of the packet)
    cam = CameraParams.from_yaml(os.path.join(REF_PARAMS, "KinectAzure", "LeftCameraParams.yaml"))
    s = SynthStream(cam, cam, np.eye(3), seed=777)
    frames = []
    for k in range(N_FRAMES):
        f, depth = s.frame_with_depth(k)
        frames.append((f.timestamp, f.left, depth))
    sc = Scene(p, cam, frames, "imu", stream=s, equalize=True)
    _scene_cache["kinect"] = sc
    return sc


def real_scene(u16: bool) -> Scene:
    key = ("real", u16)
    if key in _scene_cache:
        return _scene_cache[key]
    g0 = np.load(os.path.join(H.ROOT, "tests", "golden", "rgbd_pair.npz"))
    g1 = np.load(os.path.join(H.ROOT, "tests", "golden", "rgbd_frame1.npz"))
    c = json.loads(str(g0["camera"]))
    c["T_BS"] = np.asarray(c["T_BS"], np.float64)
    cam = CameraParams(**c)
    depths = [g0["depth"], g1["depth"]]
    if u16:
        depths = [np.clip(np.rint(np.nan_to_num(d, nan=0.0, posinf=0.0) * 1000.0), 0, 65535).astype(np.uint16) for d in depths]
        cam = dataclasses.replace(cam, depth=dict(cam.depth, depth_to_meters=float(f32(0.001))))
    t0 = 1_000_000_000
    frames = [(t0, g0["left"], depths[0]), (t0 + 50_000_000, g1["left"], depths[1])]
    sc = Scene(FrontendParams.euroc(), cam, frames, "identity", force=(1,))
    _scene_cache[key] = sc
    return sc


def rotation(sc: Scene, lkf: int, k: int) -> np.ndarray:
    return np.eye(3) if sc.rotations == "identity" else sc.stream.kf_rotation(lkf, k)


# ---------------------------------------------------------------------------------------------------------------------
# the oracle run, recorded frame by frame (the lkf's right statuses change later: snapshot right after each spin)
# ---------------------------------------------------------------------------------------------------------------------
class _Forced(org.RgbdFrontend):
    force = ()

    def _stereo_frame(self, k, ts, img):
        sf = super()._stereo_frame(k, ts, img)
        sf.left_frame.is_keyframe = k in self.force
        return sf


def _snapshot(sf, is_kf, smart, fe):
    lf = sf.left_frame
    rec = dict(n=len(lf.keypoints), is_kf=bool(is_kf), mono=int(fe.mono_status), stereo=int(fe.stereo_status),
               kp=np.array(lf.keypoints, np.float32).reshape(-1, 2), lmk=np.array(lf.landmarks, np.int64),
               age=np.array(lf.landmarks_age, np.int64), versor=np.array(lf.versors, np.float64).reshape(-1, 3))
    if is_kf:
        rec["ls"] = np.array([st for st, _ in sf.left_keypoints_rectified], np.int32)
        rec["lxy"] = np.array([q for _, q in sf.left_keypoints_rectified], np.float32).reshape(-1, 2)
        rec["rs"] = np.array([st for st, _ in sf.right_keypoints_rectified], np.int32)
        rec["rxy"] = np.array([q for _, q in sf.right_keypoints_rectified], np.float32).reshape(-1, 2)
        rec["depth"] = np.array(sf.keypoints_depth, np.float64)
        rec["p3d"] = np.array(sf.keypoints_3d, np.float64).reshape(-1, 3)
        rec["rkp"] = np.array(sf.right_frame.keypoints, np.float32).reshape(-1, 2)
        rec["smart"] = list(smart)
    return rec


_oracle_cache = {}


def oracle_run(name: str, sc: Scene):
    if name in _oracle_cache:
        return _oracle_cache[name]
    fe = _Forced(sc.p, sc.cam)
    fe.force = sc.force
    out, lkf = [], 0
    for k, (ts, img, depth) in enumerate(sc.frames):
        R = rotation(sc, lkf, k)
        im = cv2.equalizeHist(img) if sc.equalize else img
        sf, is_kf, smart = fe.spin(k, ts, im, depth, R)
        rec = _snapshot(sf, is_kf, smart, fe)
        rec["R"] = R
        out.append(rec)
        if is_kf:
            lkf = k
    _oracle_cache[name] = out
    return out


def make_ctx(sc: Scene, batch: int = 1):
    rig = RgbdRigSetup(sc.cam)
    dtype = sc.frames[0][2].dtype
    dp = kl.make_depth_params(dtype, **{k: v for k, v in sc.cam.depth.items() if k != "is_registered"})
    cfg = kl.make_config(sc.p, rig.W, rig.H, batch=batch, sobel_cpu_tail_start=H.sobel_cpu_tail_start(rig.W), depth=dp)
    return cfg, rig


def compare(pk, o):
    """Returns the list of fields that differ between a packet and an oracle snapshot."""
    bad = []
    if pk["n"] != o["n"]:
        return ["n %d != %d" % (pk["n"], o["n"])]
    if bool(pk["is_keyframe"]) != o["is_kf"]:
        return ["is_keyframe"]
    n = o["n"]
    if n:
        if np.abs(np.stack([pk["kp_x"], pk["kp_y"]], 1) - o["kp"]).max() > 1e-3:
            bad.append("keypoints")
        if not np.array_equal(pk["landmark"], o["lmk"]):
            bad.append("landmark")
        if not np.array_equal(pk["age"].astype(np.int64), o["age"]):
            bad.append("age")
        if np.abs(pk["versor"] - o["versor"]).max() >= 1e-5:
            bad.append("versor")
    if pk["mono_status"] != o["mono"] or pk["stereo_status"] != o["stereo"]:
        bad.append("status (%d, %d) != (%d, %d)" % (pk["mono_status"], pk["stereo_status"], o["mono"], o["stereo"]))
    if not o["is_kf"]:
        if n and not ((pk["left_status"] == -1).all() and (pk["right_status"] == -1).all() and (pk["depth"] == 0).all()):
            bad.append("non-keyframe stereo fields")
        if pk["n_smart"] != 0:
            bad.append("non-keyframe smart measurements")
        return bad
    if n:
        if not np.array_equal(pk["left_status"], o["ls"]):
            bad.append("left_status")
        if np.abs(np.stack([pk["left_rect_x"], pk["left_rect_y"]], 1) - o["lxy"]).max() > 2e-3:
            bad.append("left_rect")
        if not np.array_equal(pk["right_status"], o["rs"]):
            bad.append("right_status")
        if np.abs(np.stack([pk["right_rect_x"], pk["right_rect_y"]], 1) - o["rxy"]).max() > 2e-3:
            bad.append("right_rect")
        if not np.array_equal(pk["depth"], o["depth"]):
            bad.append("depth")
        if np.abs(pk["point3d"] - o["p3d"]).max() > 1e-4 * (1.0 + np.abs(o["depth"]).max()):
            bad.append("point3d")
        if np.abs(np.stack([pk["right_x"], pk["right_y"]], 1) - o["rkp"]).max() > 2e-3:
            bad.append("right keypoints")
    cnt = [int((o["rs"] == s).sum()) for s in range(5)] if n else [0] * 5
    got = [pk["nr_valid_rkp"], pk["nr_no_left_rect_rkp"], pk["nr_no_right_rect_rkp"], pk["nr_no_depth_rkp"], pk["nr_failed_arun_rkp"]]
    if got != cnt:
        bad.append("nr_*_rkp %s != %s" % (got, cnt))
    sm = o["smart"]
    if pk["n_smart"] != len(sm):
        bad.append("n_smart %d != %d" % (pk["n_smart"], len(sm)))
    elif sm:
        if not np.array_equal(pk["smart_lmk"], np.array([m[0] for m in sm], np.int64)):
            bad.append("smart_lmk")
        uR = np.array([m[2] for m in sm])
        if not np.array_equal(np.isnan(pk["smart_uR"]), np.isnan(uR)):
            bad.append("smart_uR NaN pattern")
        else:
            v = ~np.isnan(uR)
            if v.any() and np.abs(pk["smart_uR"][v] - uR[v]).max() > 2e-3:
                bad.append("smart_uR")
        if np.abs(pk["smart_uL"] - np.array([m[1] for m in sm])).max() > 2e-3 or \
                np.abs(pk["smart_v"] - np.array([m[3] for m in sm])).max() > 2e-3:
            bad.append("smart_uL / v")
    return bad


def gpu_run(sc: Scene, orc):
    """Steps one context through the scene with the oracle's rotations and forced keyframes; returns the packets."""
    cfg, rig = make_ctx(sc)
    ctx = kl.Context(cfg, rig.to_c())
    pks = []
    for k, (ts, img, depth) in enumerate(sc.frames):
        if k in sc.force:
            ctx.force_keyframe([1])
        pks.append(ctx.step_rgbd([img], [depth], [ts], np.array([orc[k]["R"]]))[0])
    ctx.close()
    return pks


def check_scene(name, sc, min_kf=3):
    orc = oracle_run(name, sc)
    pks = gpu_run(sc, orc)
    bad = []
    for k, (pk, o) in enumerate(zip(pks, orc)):
        why = compare(pk, o)
        H.diag("rgbd_frontend", scene=name, k=k, n=int(pk["n"]), kf=int(pk["is_keyframe"]), why=why)
        if why:
            bad.append((k, why))
    assert not bad, (name, bad[:4])
    assert sum(o["is_kf"] for o in orc) >= min_kf


SYNTH_VARIANTS = ["imu", "identity", "u16_mm", "holes", "textureless", "no_stereo_tracking", "no_ransac"]


@pytest.mark.gpu
@pytest.mark.parametrize("variant", SYNTH_VARIANTS)
def test_rgbd_frontend_synthetic_euroc(variant):
    check_scene(variant, synth_scene(variant))


@pytest.mark.gpu
def test_rgbd_frontend_kinect_azure_rig():
    check_scene("kinect", kinect_scene())


@pytest.mark.gpu
@pytest.mark.parametrize("u16", [False, True])
def test_rgbd_frontend_real_frames(u16):
    check_scene("real_u16" if u16 else "real_f32", real_scene(u16), min_kf=2)


@pytest.mark.gpu
def test_rgbd_frontend_batch_equals_single_streams():
    """Three streams with different seeds in one context: each stream's packets equal its own single-stream run."""
    N, seeds = 10, (11, 22, 33)
    left, right = CameraParams.euroc_left(), CameraParams.euroc_right()
    cam = dataclasses.replace(left, depth={"virtual_baseline": float(f32(0.2)), "depth_to_meters": 1.0, "min_depth": 0.3,
                                           "max_depth": 4.0, "is_registered": True})
    streams = [SynthStream(left, right, np.eye(3), seed=s) for s in seeds]
    seqs = [[s.frame_with_depth(k) for k in range(N)] for s in streams]
    sc = Scene(FrontendParams.euroc(), cam, [], "imu")
    singles = []
    for b, (st, seq) in enumerate(zip(streams, seqs)):
        cfg, rig = make_ctx(dataclasses.replace(sc, frames=[(f.timestamp, f.left, d) for f, d in seq]))
        ctx = kl.Context(cfg, rig.to_c())
        out, lkf = [], 0
        for k, (f, d) in enumerate(seq):
            pk = ctx.step_rgbd([f.left], [d], [f.timestamp], np.array([st.kf_rotation(lkf, k)]))[0]
            lkf = k if pk["is_keyframe"] else lkf
            out.append(pk)
        ctx.close()
        singles.append(out)
    cfg, rig = make_ctx(dataclasses.replace(sc, frames=[(0, seqs[0][0][0].left, seqs[0][0][1])]), batch=3)
    ctx = kl.Context(cfg, rig.to_c())
    lkf, bad = [0, 0, 0], []
    for k in range(N):
        Rs = np.array([streams[b].kf_rotation(lkf[b], k) for b in range(3)])
        pks = ctx.step_rgbd([seqs[b][k][0].left for b in range(3)], [seqs[b][k][1] for b in range(3)],
                            [seqs[b][k][0].timestamp for b in range(3)], Rs)
        for b in range(3):
            ok, why = same_packet(pks[b], singles[b][k])
            if not ok:
                bad.append((b, k, why))
            if pks[b]["is_keyframe"]:
                lkf[b] = k
    ctx.close()
    assert not bad, bad[:5]
    assert sum(p["is_keyframe"] for p in singles[0]) >= 3


# ---------------------------------------------------------------------------------------------------------------------
# pipeline: byte-identical packets to the blocking step
# ---------------------------------------------------------------------------------------------------------------------
def mat3(a, b):
    """3x3 product in the device's operation order (common.cuh matmul3: a0*b0 + (a1*b1 + a2*b2))."""
    a, b = np.asarray(a, np.float64).reshape(3, 3), np.asarray(b, np.float64).reshape(3, 3)
    c = np.zeros((3, 3))
    for i in range(3):
        for j in range(3):
            c[i, j] = float(a[i, 0]) * float(b[0, j]) + (float(a[i, 1]) * float(b[1, j]) + float(a[i, 2]) * float(b[2, j]))
    return c


def same_packet(a, b):
    for name, _, _ in kl.PACKET_FIELDS:
        if a[name].shape != b[name].shape or not np.array_equal(a[name], b[name], equal_nan=True):
            return False, name
    for k, _ in kl.PacketHeader._fields_:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        if not np.array_equal(x, y):
            return False, k
    return True, ""


@pytest.mark.gpu
@pytest.mark.parametrize("memory", ["pageable", "pinned", "device"])
@pytest.mark.parametrize("split", [0, -1])
@pytest.mark.parametrize("rotation_mode", [0, 1])
def test_rgbd_pipeline_matches_blocking_step(memory, split, rotation_mode):
    import torch
    sc = synth_scene("holes")
    N = len(sc.frames)
    rel = [np.eye(3)] + [sc.stream.kf_rotation(k - 1, k) for k in range(1, N)]
    # blocking reference with the rotations the device forms: mode 0 lkf_R_k as given, mode 1 the accumulated product
    cfg, rig = make_ctx(sc)
    ctx = kl.Context(cfg, rig.to_c())
    refs, lkf, acc = [], 0, np.eye(3)
    for k, (ts, img, depth) in enumerate(sc.frames):
        if rotation_mode == 0:
            R = sc.stream.kf_rotation(lkf, k)
        else:
            R = mat3(np.eye(3) if (k == 0 or lkf == k - 1) else acc, rel[k])
            acc = R
        pk = ctx.step_rgbd([img], [depth], [ts], np.array([R]))[0]
        refs.append(pk)
        lkf = k if pk["is_keyframe"] else lkf
    ctx.close()
    pipe = kl.Pipeline(cfg, rig.to_c(), n_streams=2, n_workers=1, queue_depth=N, output_slots=4, want_rectified=True,
                       rotation_mode=rotation_mode, checksum_outputs=True, split_graphs=split)
    keep = []

    def buf(a):
        a = np.ascontiguousarray(a)
        if memory == "pageable":
            keep.append(a)
            return a.ctypes.data
        t = torch.from_numpy(a)
        t = t.pin_memory() if memory == "pinned" else t.cuda()
        keep.append(t)
        return t.data_ptr()

    def push(s, k, R):
        ts, img, depth = sc.frames[k]
        assert pipe.push_rgbd(s, buf(img), img.shape[1], buf(depth), depth.strides[0], ts, R, tag=k)

    lkf = [0, 0]
    if rotation_mode == 1:            # queue every frame up front
        for k in range(N):
            for s in range(2):
                push(s, k, rel[k])
    else:
        for s in range(2):
            push(s, 0, np.eye(3))
    done, bad = 0, []
    while done < 2 * N:
        outs = pipe.pop(timeout_ms=20000)
        assert outs, "pipeline stalled"
        for o in outs:
            s, k = o.stream, int(o.tag)
            d = pipe.parse(o)
            ok, why = same_packet(d, refs[k])
            if not ok:
                bad.append((s, k, why))
            if o.rect_left or o.rect_right:
                bad.append((s, k, "rectified images delivered"))
            lkf[s] = k if d["is_keyframe"] else lkf[s]
            done += 1
            if rotation_mode == 0 and k + 1 < N:
                push(s, k + 1, sc.stream.kf_rotation(lkf[s], k + 1))
        pipe.release(outs)
    st = pipe.stats()
    pipe.close()
    H.diag("rgbd_pipeline", memory=memory, split=split, rotation_mode=rotation_mode, bad=bad, **st)
    assert not bad, bad[:5]
    assert (st["staged_copies"] > 0) == (memory == "pageable")


# ---------------------------------------------------------------------------------------------------------------------
# rejections
# ---------------------------------------------------------------------------------------------------------------------
def _ok_rgbd_cfg():
    sc = synth_scene("imu")
    cfg, rig = make_ctx(sc)
    return sc, cfg, rig.to_c()


@pytest.mark.gpu
def test_rgbd_create_time_rejections():
    sc, cfg, rig = _ok_rgbd_cfg()
    kl.Context(cfg, rig).close()
    cases = []
    c = kl.Config.from_buffer_copy(cfg); c.depth.depth_type = 7; cases.append(("depth_type", c, rig))
    r = kl.Rig.from_buffer_copy(rig); r.baseline = 0.2; cases.append(("baseline", cfg, r))     # != (double)f32(0.2)
    c = kl.Config.from_buffer_copy(cfg); c.mesh_2d = 1; cases.append(("mesh_2d", c, rig))
    r = kl.Rig.from_buffer_copy(rig); r.distortion_model = 1; cases.append(("equidistant", cfg, r))
    for what, c, r in cases:
        with pytest.raises(kl.KvfeError) as e:
            kl.Context(c, r)
        assert "(-1)" in str(e.value), (what, str(e.value))


@pytest.mark.gpu
def test_rgbd_wrong_entry_points():
    import ctypes as C
    sc, cfg, rig = _ok_rgbd_cfg()
    ts, img, depth = sc.frames[0]
    lib = kl.load()
    R = np.eye(3).reshape(1, 9).copy()
    tsa = np.array([ts], np.int64)
    ctx = kl.Context(cfg, rig)
    buf = np.zeros(ctx.packet_bytes, np.uint8)
    ip = (C.c_void_p * 1)(img.ctypes.data)
    assert lib.kvfe_frontend_step(ctx.h, ip, ip, C.c_size_t(img.shape[1]), kl._p(tsa), kl._p(R), kl._p(buf), None, None, C.c_size_t(0)) == -1
    assert lib.kvfe_frontend_submit(ctx.h, ip, ip, C.c_size_t(img.shape[1]), kl._p(tsa), kl._p(R), kl._p(buf)) == -1
    assert lib.kvfe_frontend_step_dev(ctx.h, C.c_void_p(img.ctypes.data), C.c_void_p(img.ctypes.data), C.c_size_t(img.shape[1]),
                                      kl._p(tsa), kl._p(R)) == -1
    assert "RGB-D" in lib.kvfe_last_error(ctx.h).decode()
    up = C.c_void_p()
    arr = (C.c_void_p * 1)(ctx.h)
    assert lib.kvfe_upload_create(arr, 1, C.byref(up)) == -1
    ctx.step_rgbd([img], [depth], [ts], R)                   # the context is still usable
    ctx.close()
    # the RGB-D entry points on a stereo context
    p, srig, sctx = H.euroc_setup(batch=1)
    dp_ = (C.c_void_p * 1)(depth.ctypes.data)
    assert lib.kvfe_frontend_step_rgbd(sctx.h, ip, C.c_size_t(img.shape[1]), dp_, C.c_size_t(depth.strides[0]), kl._p(tsa), kl._p(R),
                                       kl._p(np.zeros(sctx.packet_bytes, np.uint8))) == -1
    sctx.close()
    # pipelines: push on an RGB-D pipeline, push_rgbd on a stereo one
    pipe = kl.Pipeline(cfg, rig, n_streams=1)
    with pytest.raises(kl.KvfeError):
        pipe.push(0, img.ctypes.data, img.ctypes.data, img.shape[1], ts, np.eye(3))
    assert pipe.push_rgbd(0, img.ctypes.data, img.shape[1], depth.ctypes.data, depth.strides[0], ts, np.eye(3))
    assert pipe.pop(timeout_ms=20000)
    pipe.close()
    spipe = kl.Pipeline(kl.make_config(p, srig.W, srig.H, sobel_cpu_tail_start=H.sobel_cpu_tail_start(srig.W)), srig.to_c(), n_streams=1)
    with pytest.raises(kl.KvfeError):
        spipe.push_rgbd(0, img.ctypes.data, img.shape[1], depth.ctypes.data, depth.strides[0], ts, np.eye(3))
    spipe.close()


# ---------------------------------------------------------------------------------------------------------------------
# CPU checks: marshalling, and the branches each scene's oracle run must reach
# ---------------------------------------------------------------------------------------------------------------------
def _lib_built():
    if not os.path.exists(kl.LIB_PATH):
        from kimera_vio_b200 import build
        build.build()


def test_make_config_rgbd_marshalling():
    _lib_built()
    p = FrontendParams.euroc()
    dp = kl.make_depth_params(np.uint16, virtual_baseline=0.3, depth_to_meters=0.001, min_depth=0.2, max_depth=5.0)
    c = kl.make_config(p, 640, 360, depth=dp)
    assert c.frontend_type == 2 and c.depth.depth_type == 0 and c.depth.virtual_baseline == f32(0.3)
    assert c.depth.depth_to_meters == f32(0.001) and c.depth.min_depth == f32(0.2) and c.depth.max_depth == f32(5.0)
    assert kl.make_config(p, 640, 360).frontend_type == 0 and kl.make_config(p, 640, 360, mono=True).frontend_type == 1
    d = kl.make_config(p, 640, 360).depth                  # kvfe_config_default: CameraParams::DepthParams defaults
    assert (d.depth_type, d.virtual_baseline, d.depth_to_meters, d.min_depth, d.max_depth) == (1, f32(1e-2), 1.0, 0.0, 10.0)
    with pytest.raises(ValueError):
        kl.make_config(dataclasses.replace(p, use_pnp_tracking=True), 640, 360, depth=dp)
    with pytest.raises(ValueError):
        kl.make_config(p, 640, 360, mono=True, depth=dp)


def _statuses(orc, key):
    return np.concatenate([o[key] for o in orc if o["is_kf"] and o["n"]])


def _uR_negative(sc, orc):
    """Keyframe keypoints with a finite depth whose virtual right keypoint falls left of the image (uR < 0)."""
    n, fx_b = 0, sc.cam.intrinsics[0] * float(f32(sc.cam.depth["virtual_baseline"]))
    for (ts, img, depth), o in zip(sc.frames, orc):
        if not o["is_kf"]:
            continue
        for i in np.flatnonzero((o["rs"] == ofe.KP_NO_DEPTH) & (o["ls"] == ofe.KP_VALID)):
            x, y = int(o["kp"][i, 0]), int(o["kp"][i, 1])
            d = float(depth[y, x]) * sc.cam.depth["depth_to_meters"]
            if math.isfinite(d) and d >= sc.cam.depth["min_depth"] and o["lxy"][i, 0] - f32(fx_b / d) < 0:
                n += 1
    return n


def _no_depth_from(sc, orc, pred):
    n = 0
    for (ts, img, depth), o in zip(sc.frames, orc):
        if o["is_kf"]:
            for i in np.flatnonzero(o["rs"] == ofe.KP_NO_DEPTH):
                n += pred(depth[int(o["kp"][i, 1]), int(o["kp"][i, 0])])
    return n


def test_rgbd_scenes_reach_their_branches():
    """The oracle runs the GPU tests compare against still cover: NO_DEPTH from a hole (NaN / +inf), from a depth below
    min_depth and from uR < 0; a NO_LEFT_RECT keypoint passed through to the right status; 1-point and 3-point stereo
    RANSAC keyframes; the frame after the textureless one, whose pyramid has no gradient, loses every track (no mode-3
    shortcut: it is an ordinary keyframe whose keypoints are all new detections); uR in the smart measurements without use_stereo_tracking; DISABLED statuses without RANSAC."""
    holes = synth_scene("holes")
    oh = oracle_run("holes", holes)
    assert _no_depth_from(holes, oh, lambda v: not math.isfinite(float(v))) > 0
    assert _no_depth_from(holes, oh, lambda v: math.isfinite(float(v)) and float(v) < holes.cam.depth["min_depth"]) > 0
    assert _uR_negative(holes, oh) > 0
    u16 = synth_scene("u16_mm")
    assert _no_depth_from(u16, oracle_run("u16_mm", u16), lambda v: int(v) == 0) > 0
    ls, rs = _statuses(oh, "ls"), _statuses(oh, "rs")
    assert ((ls == ofe.KP_NO_LEFT_RECT) & (rs == ofe.KP_NO_LEFT_RECT)).any()
    # 1-point (IMU rotation given) and 3-point (identity) keyframes with a computed stereo status
    imu, ident = oracle_run("imu", synth_scene("imu")), oracle_run("identity", synth_scene("identity"))
    assert any(o["is_kf"] and k > 0 and not ofe.rot_equals_identity(o["R"]) and o["stereo"] != ofe.INVALID for k, o in enumerate(imu))
    assert any(o["is_kf"] and k > 0 and o["stereo"] != ofe.INVALID for k, o in enumerate(ident))
    assert all(ofe.rot_equals_identity(o["R"]) for o in ident)
    tl = oracle_run("textureless", synth_scene("textureless"))
    lost = tl[TEXTURELESS_FRAME + 1]
    assert lost["is_kf"] and lost["n"] > 0 and (lost["age"] == 1).all() and (tl[TEXTURELESS_FRAME]["age"] > 1).any()
    nst = oracle_run("no_stereo_tracking", synth_scene("no_stereo_tracking"))
    kfs = [o for k, o in enumerate(nst) if o["is_kf"] and k > 0]
    assert kfs and all(o["stereo"] == ofe.INVALID for o in kfs)
    assert any(not math.isnan(m[2]) for o in kfs for m in o["smart"])
    nr = oracle_run("no_ransac", synth_scene("no_ransac"))
    assert all(o["mono"] == ofe.DISABLED and o["stereo"] == ofe.DISABLED for k, o in enumerate(nr) if o["is_kf"] and k > 0)


def test_rgbd_real_and_kinect_scenes_reach_their_branches():
    """The real frames: frame 1 is a keyframe only because it is forced; the KinectAzure scene runs with equalizeImage and
    the rig's 640x360 geometry and has keyframes with VALID right keypoints."""
    for u16 in (False, True):
        orc = oracle_run("real_u16" if u16 else "real_f32", real_scene(u16))
        assert orc[1]["is_kf"] and orc[1]["n"] > 0 and (orc[1]["rs"] == ofe.KP_VALID).any()
        sc = real_scene(u16)
        fe = org.RgbdFrontend(sc.p, sc.cam)                   # unforced: frame 1 (50 ms later) is no keyframe
        fe.spin(0, *sc.frames[0], np.eye(3))
        assert not fe.spin(1, *sc.frames[1], np.eye(3))[1]
    kin = kinect_scene()
    assert kin.p.equalize_image and (kin.cam.width, kin.cam.height) == (640, 360)
    orc = oracle_run("kinect", kin)
    assert sum(o["is_kf"] for o in orc) >= 3 and all((o["rs"] == ofe.KP_VALID).any() for o in orc if o["is_kf"])
