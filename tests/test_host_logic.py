"""CPU tests of the host-side pieces: parameter parsing (reference YAMLs), config marshalling,
the synthetic generator, stream sharding and the 2-rank gloo packet gather."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import REF, ROOT
from kimera_vio_b200 import dist as kd
from kimera_vio_b200.params import CameraParams, FrontendParams
from kimera_vio_b200.rig import StereoRigSetup
from kimera_vio_b200.synth import SynthStream


def test_euroc_yaml_equals_inlined_defaults():
    p = FrontendParams.from_yaml(os.path.join(REF, "params/Euroc/FrontendParams.yaml"))
    q = FrontendParams.euroc()
    for k, v in vars(q).items():
        w = getattr(p, k)
        if isinstance(v, np.ndarray):
            assert np.array_equal(v, w), k
        else:
            assert v == w, (k, v, w)
    l = CameraParams.from_yaml(os.path.join(REF, "params/Euroc/LeftCameraParams.yaml"))
    assert l.intrinsics == CameraParams.euroc_left().intrinsics
    assert np.allclose(l.T_BS, CameraParams.euroc_left().T_BS)
    assert l.distortion == CameraParams.euroc_left().distortion


@pytest.mark.parametrize("rig", ["Euroc", "uHumans2", "D455", "KinectAzure", "EurocMono", "RealSenseIR", "Kitti"])
def test_all_shipped_rigs_parse(rig):
    path = os.path.join(REF, "params", rig, "FrontendParams.yaml")
    if not os.path.exists(path):
        pytest.skip("rig not shipped")
    p = FrontendParams.from_yaml(path)
    assert p.feature_detector_type == 3 and p.non_max_suppression_type == 6   # SURVEY section 0


def test_config_marshalling_roundtrip():
    from kimera_vio_b200 import lib as kl
    if not os.path.exists(kl.LIB_PATH):
        from kimera_vio_b200 import build
        build.build()
    p = FrontendParams.euroc()
    c = kl.make_config(p, 752, 480, batch=32, sobel_cpu_tail_start=736)
    assert (c.width, c.height, c.batch) == (752, 480, 32)
    assert c.klt_win_size == 24 and c.klt_max_level == 4 and abs(c.klt_eps - 0.1) < 1e-15
    assert c.nr_horizontal_bins == 7 and c.nr_vertical_bins == 5 and sum(c.binning_mask[:35]) == 35
    assert c.min_intra_keyframe_time_ns == 200_000_000 and c.ransac_randomize == 0
    assert c.sobel_cpu_tail_start == 736


def test_synth_stream_deterministic_and_textured():
    rig = StereoRigSetup(CameraParams.euroc_left(), CameraParams.euroc_right())
    assert abs(rig.baseline - 0.110078) < 1e-4
    a = SynthStream(CameraParams.euroc_left(), CameraParams.euroc_right(), rig.R1, seed=7)
    b = SynthStream(CameraParams.euroc_left(), CameraParams.euroc_right(), rig.R1, seed=7)
    fa, fb = a.frame(3), b.frame(3)
    assert np.array_equal(fa.left, fb.left) and np.array_equal(fa.right, fb.right)
    assert fa.left.shape == (480, 752) and fa.left.std() > 10
    R = a.kf_rotation(0, 3)
    assert np.allclose(R @ R.T, np.eye(3), atol=1e-12)
    assert np.allclose(a.kf_rotation(2, 2), np.eye(3))


def test_stream_shard_partitions():
    for n, w in ((32, 1), (32, 2), (32, 8), (33, 8), (5, 8)):
        seen = []
        for r in range(w):
            b, e = kd.stream_shard(n, w, r)
            seen += list(range(b, e))
        assert seen == list(range(n))


def _gloo_worker(rank, world, port, q):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    b, e = kd.stream_shard(6, world, rank)
    local = torch.full((3, 16), rank + 1, dtype=torch.uint8)      # 3 streams x 16-byte "packets"
    local[:, 0] = torch.arange(b, e, dtype=torch.uint8)
    out = kd.gather_packets(local, dst=0)
    ms = kd.max_over_ranks(10.0 + rank)
    if rank == 0:
        q.put((torch.cat(out)[:, 0].tolist(), [int(t[0, 1]) for t in out], ms))
    dist.destroy_process_group()


def test_gloo_world2_gather_packets():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    ids, tags, ms = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert ids == [0, 1, 2, 3, 4, 5]          # stream-major order: rank 0's block, then rank 1's
    assert tags == [1, 2]
    assert ms == 11.0                          # max over ranks


def _dt_host_lib():
    """Builds tests/native/dt_host.cpp (the mesh kernel's quad-edge code, delaunay.cuh, compiled for the host)."""
    import ctypes as C
    import shutil
    import subprocess
    if not shutil.which("g++"):
        pytest.skip("g++ not available")
    out = os.path.join(ROOT, "tests", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libdt_host.so")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-o", so, os.path.join(ROOT, "tests", "native", "dt_host.cpp")])
    return C.CDLL(so)


def test_delaunay_restatement_matches_subdiv2d():
    """delaunay.cuh (what mesh_kernel executes) against cv2.Subdiv2D through oracle/mesher.py: identical triangle
    LISTS -- order and first vertex included -- on random sub-pixel points, integer corners (collinear and
    cocircular sets), a coarse grid with duplicates, and points partly outside the image."""
    import ctypes as C
    from oracle.mesher import create_mesh_2d_impl
    lib = _dt_host_lib()
    rng = np.random.default_rng(1)
    for trial in range(120):
        w, h = (752, 480) if trial % 2 else (1280, 720)
        n = int(rng.integers(1, 600))
        kind = trial % 4
        if kind == 0:
            pts = rng.uniform(0, [w, h], (n, 2))
        elif kind == 1:
            pts = np.floor(rng.uniform(0, [w, h], (n, 2)))
        elif kind == 2:
            pts = np.floor(rng.uniform(0, [w / 20, h / 20], (n, 2))) * 20
        else:
            pts = rng.uniform(-5, [w + 5, h + 5], (n, 2))
        pts = np.ascontiguousarray(pts, np.float32)
        tri = np.zeros((4 * n + 16, 6), np.float32)
        nq = C.c_int()
        m = lib.dt_host_mesh(w, h, pts.ctypes.data_as(C.c_void_p), n, tri.ctypes.data_as(C.c_void_p), len(tri), C.byref(nq))
        assert m >= 0
        ref = create_mesh_2d_impl((w, h), [tuple(p) for p in pts])
        assert tri[:m].shape == ref.shape and np.array_equal(tri[:m], ref), (trial, kind, n)
        assert nq.value <= 3 * n + 16


def test_find_and_remove_outliers_host_logic():
    """kvfe_find_outliers / kvfe_remove_outliers_{mono,stereo} (Tracker.cpp:836-917): pure host bookkeeping, no GPU."""
    import ctypes as C
    from kimera_vio_b200 import build as kb
    from oracle import ransac as ors
    lib = C.CDLL(kb.build())
    rng = np.random.default_rng(2)
    for n_matches, n_inl in ((40, 25), (7, 0), (5, 5), (0, 0)):
        inl = rng.permutation(n_matches)[:n_inl].astype(np.int32)          # unsorted on purpose
        out = np.zeros(max(n_matches, 1), np.int32)
        no = C.c_int()
        assert lib.kvfe_find_outliers(n_matches, inl.ctypes.data_as(C.c_void_p), n_inl, out.ctypes.data_as(C.c_void_p), C.byref(no)) == 0
        assert list(out[:no.value]) == ors.find_outliers(n_matches, sorted(int(v) for v in inl))
        # mono
        n_ref, n_cur = n_matches + 5, n_matches + 3
        mr = rng.permutation(n_ref)[:n_matches].astype(np.int32)
        mc = rng.permutation(n_cur)[:n_matches].astype(np.int32)
        lr = np.arange(100, 100 + n_ref, dtype=np.int64)
        lc = np.arange(500, 500 + n_cur, dtype=np.int64)
        elr, elc = lr.copy(), lc.copy()
        for o in ors.find_outliers(n_matches, sorted(int(v) for v in inl)):
            elr[mr[o]] = -1
            elc[mc[o]] = -1
        emr, emc = mr[inl].copy(), mc[inl].copy()
        mr2, mc2 = mr.copy(), mc.copy()
        nm = C.c_int(n_matches)
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        assert lib.kvfe_remove_outliers_mono(vp(inl), n_inl, vp(lr), n_ref, vp(lc), n_cur, vp(mr2), vp(mc2), C.byref(nm)) == 0
        assert nm.value == n_inl and np.array_equal(lr, elr) and np.array_equal(lc, elc)
        assert np.array_equal(mr2[:n_inl], emr) and np.array_equal(mc2[:n_inl], emc)
        # stereo
        rs, cs = np.zeros(n_ref, np.int32), np.zeros(n_cur, np.int32)
        rd, cd = np.ones(n_ref), np.ones(n_cur)
        rp, cp = np.ones((n_ref, 3)), np.ones((n_cur, 3))
        mr3, mc3 = mr.copy(), mc.copy()
        nm = C.c_int(n_matches)
        assert lib.kvfe_remove_outliers_stereo(vp(inl), n_inl, vp(rs), vp(rd), vp(rp), n_ref, vp(cs), vp(cd), vp(cp), n_cur,
                                               vp(mr3), vp(mc3), C.byref(nm)) == 0
        outl = ors.find_outliers(n_matches, sorted(int(v) for v in inl))
        assert sorted(np.nonzero(rs == 4)[0]) == sorted(int(mr[o]) for o in outl)
        assert sorted(np.nonzero(cd == 0)[0]) == sorted(int(mc[o]) for o in outl)
        assert all((rp[mr[o]] == 0).all() and (cp[mc[o]] == 0).all() for o in outl)
        assert nm.value == n_inl and np.array_equal(mr3[:n_inl], emr)


def test_find_matching_and_smart_measurements_host_logic():
    """kvfe_find_matching_keypoints / _stereo_keypoints (Tracker.cpp:919-989) and kvfe_smart_stereo_measurements
    (StereoVisionImuFrontend.cpp:485-531, RgbdVisionImuFrontend.cpp:368-395): host bookkeeping, no GPU; against the oracle,
    incl. the reference's own fillSmartStereoMeasurements scenario (tests/testRgbdVisionImuFrontend.cpp:140-230: 12 valid,
    12 without a right keypoint, 12 without a landmark -> 24 measurements, uR NaN where the right keypoint is missing)."""
    import ctypes as C
    from types import SimpleNamespace as NS
    from kimera_vio_b200 import lib as kl
    from oracle import frontend as ofe
    lib = kl.load()
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    rng = np.random.default_rng(3)
    for trial in range(20):
        n_ref, n_cur = int(rng.integers(0, 60)), int(rng.integers(0, 60))
        ids = rng.permutation(100)
        lr = np.where(rng.random(n_ref) < 0.2, -1, ids[:n_ref]).astype(np.int64)
        lc = np.where(rng.random(n_cur) < 0.2, -1, rng.permutation(ids)[:n_cur]).astype(np.int64)
        if n_ref > 3 and trial % 3 == 0:
            lr[1] = lr[0]                                   # a duplicated id: the later position wins (std::map assignment)
        exp = ofe.find_matching_keypoints(NS(landmarks=list(lr)), NS(landmarks=list(lc)))
        mr, mc, nm = np.zeros(max(n_cur, 1), np.int32), np.zeros(max(n_cur, 1), np.int32), C.c_int()
        assert lib.kvfe_find_matching_keypoints(vp(lr), n_ref, vp(lc), n_cur, vp(mr), vp(mc), C.byref(nm)) == 0
        assert list(zip(mr[:nm.value], mc[:nm.value])) == exp
        rs = rng.integers(0, 5, max(n_ref, 1)).astype(np.int32)
        cs = rng.integers(0, 3, max(n_cur, 1)).astype(np.int32)
        ref = NS(left_frame=NS(landmarks=list(lr)), right_keypoints_rectified=[(int(s), (0.0, 0.0)) for s in rs])
        cur = NS(left_frame=NS(landmarks=list(lc)), right_keypoints_rectified=[(int(s), (0.0, 0.0)) for s in cs])
        exps = ofe.find_matching_stereo_keypoints(ref, cur)
        sr, sc, ns = np.zeros(max(nm.value, 1), np.int32), np.zeros(max(nm.value, 1), np.int32), C.c_int()
        assert lib.kvfe_find_matching_stereo_keypoints(vp(rs), n_ref, vp(cs), n_cur, vp(mr), vp(mc), nm.value, vp(sr), vp(sc), C.byref(ns)) == 0
        assert list(zip(sr[:ns.value], sc[:ns.value])) == exps
    # the reference's fillSmartStereoMeasurements scenario
    n = 36
    lm = np.concatenate([np.arange(24), np.full(12, -1)]).astype(np.int64)
    lx, ly = rng.integers(0, 800, n).astype(np.float32), rng.integers(0, 600, n).astype(np.float32)
    rstat = np.concatenate([np.zeros(12), np.full(12, 2), np.zeros(12)]).astype(np.int32)      # VALID / NO_RIGHT_RECT / VALID
    rx = (lx - 7.25).astype(np.float32)
    for use_right in (1, 0):
        ol, ouL, ouR, ov, no = np.zeros(n, np.int64), np.zeros(n), np.zeros(n), np.zeros(n), C.c_int()
        assert lib.kvfe_smart_stereo_measurements(vp(lm), vp(lx), vp(ly), vp(rstat), vp(rx), n, use_right, vp(ol), vp(ouL), vp(ouR), vp(ov), C.byref(no)) == 0
        assert no.value == 24 and list(ol[:24]) == list(range(24))
        assert np.array_equal(ouL[:24], lx[:24].astype(np.float64)) and np.array_equal(ov[:24], ly[:24].astype(np.float64))
        if use_right:
            assert np.array_equal(ouR[:12], rx[:12].astype(np.float64)) and np.isnan(ouR[12:24]).all()
        else:
            assert np.isnan(ouR[:24]).all()
    # and against the oracle's getSmartStereoMeasurements
    fe = NS(p=NS(use_stereo_tracking=True))
    sf = NS(left_frame=NS(landmarks=list(lm)), left_keypoints_rectified=[(0, (x, y)) for x, y in zip(lx, ly)],
            right_keypoints_rectified=[(int(s), (x, 0.0)) for s, x in zip(rstat, rx)])
    exp = ofe.StereoFrontend.get_smart_stereo_measurements(fe, sf)
    ol, ouL, ouR, ov, no = np.zeros(n, np.int64), np.zeros(n), np.zeros(n), np.zeros(n), C.c_int()
    lib.kvfe_smart_stereo_measurements(vp(lm), vp(lx), vp(ly), vp(rstat), vp(rx), n, 1, vp(ol), vp(ouL), vp(ouR), vp(ov), C.byref(no))
    got = list(zip(ol[:no.value], ouL[:no.value], ouR[:no.value], ov[:no.value]))
    assert len(got) == len(exp) and all(a[0] == b[0] and a[1] == b[1] and a[3] == b[3] and (a[2] == b[2] or (np.isnan(a[2]) and np.isnan(b[2]))) for a, b in zip(got, exp))


def test_should_be_keyframe_host_logic():
    """kvfe_should_be_keyframe == VisionImuFrontend::shouldBeKeyframe (VisionImuFrontend.cpp:175-232), against the oracle's
    method over the whole truth table of its conditions."""
    import ctypes as C
    import itertools
    from types import SimpleNamespace as NS
    from kimera_vio_b200 import lib as kl
    from oracle import frontend as ofe
    lib = kl.load()
    lib.kvfe_should_be_keyframe.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_double, C.c_int, C.c_int, C.c_void_p]
    p = FrontendParams.euroc()
    cfg = kl.make_config(p, 752, 480, batch=1)
    t0 = 1403715273262142976
    n_true = 0
    for dt, nvalid, disp, status, user in itertools.product(
            (0, p.min_intra_keyframe_time_ns - 1, p.min_intra_keyframe_time_ns, p.max_intra_keyframe_time_ns - 1, p.max_intra_keyframe_time_ns),
            (0, p.min_number_features, p.min_number_features + 1, 200),
            (0.0, p.disparity_threshold - 1e-9, p.disparity_threshold, 50.0, p.max_disparity_since_lkf, p.max_disparity_since_lkf + 1e-6),
            (ofe.VALID, ofe.LOW_DISPARITY, ofe.INVALID), (0, 1)):
        # the oracle method reads disparity through its helpers: feed it one match with the wanted displacement
        lkf = ofe.Frame(0, t0, None, None, False, [(np.float32(10.0), np.float32(10.0))], [7], [1], [0.0], [np.zeros(3)])
        cur = ofe.Frame(1, t0 + dt, None, None, bool(user), [(np.float32(10.0 + disp), np.float32(10.0))], [7] + [], [1], [0.0], [np.zeros(3)])
        cur.landmarks = [7] + list(range(100, 100 + max(nvalid - 1, 0)))
        cur.keypoints = cur.keypoints + [(np.float32(0), np.float32(0))] * max(nvalid - 1, 0)
        if nvalid == 0:
            cur.landmarks, cur.keypoints = [-1], [(np.float32(0), np.float32(0))]
        fe = NS(p=p, mono_status=status, _last_disparity=0.0)
        want = ofe.StereoFrontend.should_be_keyframe(fe, cur, lkf)
        d_eff = float(fe._last_disparity)                    # what computeMedianDisparity returned (float32 pixel arithmetic)
        got = C.c_int(-1)
        assert lib.kvfe_should_be_keyframe(C.byref(cfg), t0 + dt, t0, sum(1 for l in cur.landmarks if l != -1), d_eff, status, user, C.byref(got)) == 0
        assert bool(got.value) == bool(want), (dt, nvalid, disp, status, user)
        n_true += bool(want)
    assert 50 < n_true < 700


def test_camera_yaml_distortion_models_and_depth_blocks():
    """CameraParams.from_yaml on the shipped camera files: distortion model names (CameraParams.cpp:114-140) and the RGB-D
    block (CameraParams.cpp:342-349)."""
    seen = {}
    for rig in ("Euroc", "uHumans2", "D455", "RealSenseIR", "KinectAzure", "EurocMono"):
        path = os.path.join(REF, "params", rig, "LeftCameraParams.yaml")
        if not os.path.exists(path):
            continue
        c = CameraParams.from_yaml(path)
        seen[rig] = (c.distortion_model, c.depth)
        assert c.distortion_model in ("radtan", "equidistant") and len(c.distortion) >= 4
    assert seen["RealSenseIR"][0] == "equidistant" and seen["Euroc"][0] == "radtan" and seen["Euroc"][1] is None
    d = seen["KinectAzure"][1]
    assert d and d["is_registered"] and abs(d["virtual_baseline"] - 0.3) < 1e-6 and d["max_depth"] == 10.0
