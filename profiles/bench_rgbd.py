"""RGB-D pipeline throughput (kvfe_pipeline_push_rgbd, frontend_type 2): N streams of synthetic RGB-D frames
(SynthStream.frame_with_depth, float32 metres) through one pipeline, for
  * the shipped KinectAzure rig (640x360, its FrontendParams with use_pnp_tracking off, equalizeImage on);
  * the Euroc left camera at 752x480 (Euroc FrontendParams, virtual baseline 0.1 m);
each with the frames (intensity and depth) in device memory and in pinned host memory, plus the stereo pipeline at
752x480 from pinned memory through the same harness as the yardstick.  Rotation mode 1 (frame-to-frame rotations, frames
queued ahead).  Per case: warm-up, then a timed region of at least --seconds; frames/s, keyframe share, depth bytes that
crossed into the step per frame (bootstrap + keyframes only) and the launch statistics.  Before timing, the first packets of
one stream are checked against oracle/rgbd.py.  Prints one JSON line (GPU name and power limit read in the same run).

    python profiles/bench_rgbd.py [--streams 32] [--seconds 2] [--out profiles/rgbd_bench.json]
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kimera_vio_b200 import build  # noqa: E402
from kimera_vio_b200 import lib as kl  # noqa: E402
from kimera_vio_b200.hostprobe import sobel_cpu_tail_start  # noqa: E402
from kimera_vio_b200.params import CameraParams, FrontendParams  # noqa: E402
from kimera_vio_b200.rig import RgbdRigSetup, StereoRigSetup  # noqa: E402
from kimera_vio_b200.synth import SynthStream  # noqa: E402

POOL = 24                       # rendered frames per sequence, replayed forth and back (continuous motion)


def mat3(a, b):
    """3x3 product in the device's operation order (common.cuh matmul3: a0*b0 + (a1*b1 + a2*b2))."""
    a, b = np.asarray(a, np.float64).reshape(3, 3), np.asarray(b, np.float64).reshape(3, 3)
    c = np.zeros((3, 3))
    for i in range(3):
        for j in range(3):
            c[i, j] = float(a[i, 0]) * float(b[0, j]) + (float(a[i, 1]) * float(b[1, j]) + float(a[i, 2]) * float(b[2, j]))
    return c


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        o = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,power.max_limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=10).stdout.strip()
        lim, mx = (float(v) for v in o.split(","))
    except Exception:
        lim = mx = None
    return {"gpu": name, "power_limit_w": lim, "power_max_limit_w": mx}


def case_setup(name):
    if name == "kinect":
        ref = os.path.join(ROOT, "tests", "golden", "reference", "params", "KinectAzure")
        p = dataclasses.replace(FrontendParams.from_yaml(os.path.join(ref, "FrontendParams.yaml")), use_pnp_tracking=False)
        cam = CameraParams.from_yaml(os.path.join(ref, "LeftCameraParams.yaml"))
        return p, cam, SynthStream(cam, cam, np.eye(3), seed=777)
    p = FrontendParams.euroc()
    left, right = CameraParams.euroc_left(), CameraParams.euroc_right()
    cam = dataclasses.replace(left, depth={"virtual_baseline": float(np.float32(0.1)), "depth_to_meters": 1.0, "min_depth": 0.3,
                                           "max_depth": 10.0, "is_registered": True})
    return p, cam, SynthStream(left, right, np.eye(3), seed=20240)


def pool_frames(stream, stereo=False):
    """POOL frames + their frame-to-frame rotations in the order 0..POOL-1, POOL-2..1 (a closed loop)."""
    fr = []
    for k in range(POOL):
        if stereo:
            f = stream.frame(k)
            fr.append((f.left, f.right))
        else:
            f, d = stream.frame_with_depth(k)
            fr.append((f.left, d))
    order = list(range(POOL)) + list(range(POOL - 2, 0, -1))
    rel = [stream.kf_rotation(order[i - 1], order[i]) for i in range(len(order))]
    return fr, order, rel


def oracle_check(p, cam, frames, order, rel, n_check=6):
    """First packets of one stream (one-stream pipeline) against oracle/rgbd.py fed the rotations the device accumulates."""
    from oracle import rgbd as org
    rig = RgbdRigSetup(cam)
    dp = kl.make_depth_params(np.float32, **{k: v for k, v in cam.depth.items() if k != "is_registered"})
    cfg = kl.make_config(p, rig.W, rig.H, sobel_cpu_tail_start=sobel_cpu_tail_start(rig.W), depth=dp)
    pipe = kl.Pipeline(cfg, rig.to_c(), n_streams=1, queue_depth=n_check, output_slots=n_check, want_rectified=False, rotation_mode=1)
    t0, dt = 1_000_000_000, 50_000_000
    for i in range(n_check):
        img, d = frames[order[i]]
        assert pipe.push_rgbd(0, img.ctypes.data, img.shape[1], d.ctypes.data, d.strides[0], t0 + i * dt, rel[i], tag=i)
    got = {}
    while len(got) < n_check:
        outs = pipe.pop(timeout_ms=20000)
        assert outs, "pipeline stalled"
        for o in outs:
            got[int(o.tag)] = pipe.parse(o)
        pipe.release(outs)
    pipe.close()
    import cv2
    fe = org.RgbdFrontend(p, cam)
    acc, lkf, bad = np.eye(3), 0, []
    for i in range(n_check):
        R = mat3(np.eye(3) if (i == 0 or lkf == i - 1) else acc, rel[i])
        acc = R
        img, d = frames[order[i]]
        sf, is_kf, smart = fe.spin(i, t0 + i * dt, cv2.equalizeHist(img) if p.equalize_image else img, d, R)
        pk = got[i]
        kp = np.array(sf.left_frame.keypoints, np.float32).reshape(-1, 2)
        ok = pk["n"] == len(kp) and bool(pk["is_keyframe"]) == bool(is_kf)
        ok = ok and (len(kp) == 0 or np.abs(np.stack([pk["kp_x"], pk["kp_y"]], 1) - kp).max() <= 1e-3)
        ok = ok and np.array_equal(pk["landmark"], np.array(sf.left_frame.landmarks, np.int64))
        ok = ok and pk["mono_status"] == fe.mono_status and pk["stereo_status"] == fe.stereo_status
        if ok and is_kf:
            ok = np.array_equal(pk["right_status"], np.array([s for s, _ in sf.right_keypoints_rectified], np.int32))
            ok = ok and pk["n_smart"] == len(smart)
        if is_kf:
            lkf = i
        if not ok:
            bad.append(i)
    return {"frames_checked": n_check, "mismatching_frames": bad}


def run_case(name, memory, n_streams, seconds, stereo=False):
    import torch
    p, cam, stream = case_setup(name)
    if stereo:
        rig = StereoRigSetup(CameraParams.euroc_left(), CameraParams.euroc_right())
        stream = SynthStream(rig.left, rig.right, rig.R1, seed=20240)      # rotations in the rectified frame
    frames, order, rel = pool_frames(stream, stereo)
    if stereo:
        cfg = kl.make_config(p, rig.W, rig.H, sobel_cpu_tail_start=sobel_cpu_tail_start(rig.W))
    else:
        rig = RgbdRigSetup(cam)
        dp = kl.make_depth_params(np.float32, **{k: v for k, v in cam.depth.items() if k != "is_registered"})
        cfg = kl.make_config(p, rig.W, rig.H, sobel_cpu_tail_start=sobel_cpu_tail_start(rig.W), depth=dp)
    W, Hh = rig.W, rig.H

    def put(a):
        t = torch.from_numpy(np.ascontiguousarray(a))
        return t.pin_memory() if memory == "pinned" else t.cuda()
    bufs = [(put(a), put(b)) for a, b in frames]
    ptrs = [(a.data_ptr(), b.data_ptr()) for a, b in bufs]
    dpitch = W * 4
    qd = 4
    pipe = kl.Pipeline(cfg, rig.to_c(), n_streams=n_streams, queue_depth=qd, output_slots=qd + 2, want_rectified=False,
                       rotation_mode=1)
    L = len(order)
    pos = [(7 * s) % L for s in range(n_streams)]        # streams start at different places of the loop
    nxt = [0] * n_streams
    t0, dt = 1_000_000_000, 50_000_000

    def push_all():
        for s in range(n_streams):
            while True:
                i = pos[s]
                j = order[i % L]
                # a stream's first frame is its bootstrap: its rotation is ignored
                R = rel[i % L] if nxt[s] else np.eye(3)
                if stereo:
                    ok = pipe.push(s, ptrs[j][0], ptrs[j][1], W, t0 + nxt[s] * dt, R, tag=nxt[s])
                else:
                    ok = pipe.push_rgbd(s, ptrs[j][0], W, ptrs[j][1], dpitch, t0 + nxt[s] * dt, R, tag=nxt[s])
                if not ok:
                    break
                pos[s] += 1
                nxt[s] += 1

    def drain(t_end):
        n = kf = 0
        while time.perf_counter() < t_end:
            push_all()
            outs = pipe.pop(timeout_ms=100)
            for o in outs:
                n += 1
                kf += o.is_keyframe
            pipe.release(outs)
        return n, kf
    drain(time.perf_counter() + 1.0)                   # warm-up (bootstraps, graph uploads, clocks)
    st0 = pipe.stats()
    t_a = time.perf_counter()
    n, kf = drain(t_a + seconds)
    t_b = time.perf_counter()
    st1 = pipe.stats()
    pipe.close()
    elem = 4
    share = kf / max(n, 1)
    res = {"case": name, "memory": memory, "front_end": "stereo" if stereo else "rgbd", "width": W, "height": Hh,
           "streams": n_streams, "frames": n, "seconds": round(t_b - t_a, 3), "frames_per_s": round(n / (t_b - t_a), 1),
           "keyframe_share": round(share, 4),
           "kernel_launches_per_frame": round((st1["kernel_launches"] - st0["kernel_launches"]) / max(n, 1), 2),
           "graph_launches_per_frame": round((st1["graph_launches"] - st0["graph_launches"]) / max(n, 1), 3),
           "staged_copies": st1["staged_copies"]}
    if stereo:
        res["host_link_bytes_per_frame"] = round(W * Hh * (1 + share), 1)
    else:
        res["depth_bytes_per_frame"] = round(W * Hh * elem * share, 1)
        res["host_link_bytes_per_frame"] = round(W * Hh * (1 + elem * share), 1)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=32)
    ap.add_argument("--seconds", type=float, default=2.0)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    build.build()
    line = {"bench": "rgbd_pipeline", **gpu_info()}
    checks = {}
    for name in ("kinect", "euroc"):
        p, cam, stream = case_setup(name)
        frames, order, rel = pool_frames(stream)
        checks[name] = oracle_check(p, cam, frames, order, rel)
    line["oracle_check"] = checks
    res = []
    for name in ("kinect", "euroc"):
        for memory in ("device", "pinned"):
            res.append(run_case(name, memory, a.streams, a.seconds))
    res.append(run_case("euroc", "pinned", a.streams, a.seconds, stereo=True))
    line["results"] = res
    line["ok"] = all(not c["mismatching_frames"] for c in checks.values())
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
