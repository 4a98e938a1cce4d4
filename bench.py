#!/usr/bin/env python
"""bench.py -- stereo front-end frame-pairs/s on synthetic Euroc-shaped input (BASELINE.json).

  python bench.py --gpus N --steps K --warmup W [--config c2|c3|c4]     (torchrun for N > 1, one rank per GPU)
  python bench.py --impl reference ...                                 (the reference's OpenCV CPU path: oracle/)

One PASS = the whole hot path over one batch of `batch` stereo frame-pairs, one per independent camera
stream.  One STEP = `--inner` consecutive passes (default 128), so that the timed region of the
driver's `--steps 20` lasts more than a second instead of 11 ms.  Every stream replays a synthetic
sequence forwards then backwards (continuous motion, any length).  Both measurements go through
kvfe_pipeline_* (include/kvfe.h), the queue-in / queue-out boundary of the reference's front-end module (split
step graphs: the keyframe kernels are launched only for the frames the on-device decision makes keyframes):

  value  images already resident in HBM (the pipeline reads them in place); outputs -- packets and the
         keyframes' rectified images -- are still delivered to pinned host memory;
  e2e    images in pinned HOST memory, pulled over the host link inside the timed region; the same
         outputs delivered to the host, every delivered byte read by the dispatcher (checksum).

Frames are queued ahead (rotation input mode 1: the front-end accumulates the frame-to-frame IMU
rotation itself, like the reference's front-end does with the IMU samples of its input packet), so
neither number assumes an a-priori keyframe schedule.  Streams shard across ranks with no data-path
collective (weak scaling: the per-GPU batch is fixed).
"""
from __future__ import annotations

import argparse
import ctypes as C
import dataclasses
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# one hardware work queue per camera stream (read by the driver when torch creates the CUDA context, i.e.
# before libkvfe.so -- which sets the same default at load -- is loaded): see csrc/api.cu kvfe_on_load
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

from kimera_vio_b200.hostprobe import sobel_cpu_tail_start  # noqa: E402
from kimera_vio_b200.params import CameraParams, FrontendParams  # noqa: E402
from kimera_vio_b200.rig import StereoRigSetup  # noqa: E402
from kimera_vio_b200.synth import SynthStream  # noqa: E402

DT_NS = 50_000_000
T0_NS = 1403715273262142976

# BASELINE.json configs[1..3]; B_alg of SURVEY 8(d) is computed from the measured keyframe ratio
CONFIGS = {
    "c2": dict(W=752, H=480, feats=300, batch=32, pool_streams=4, pool_frames=48, cpu_pairs=600,
               workload="Euroc stereo 752x480, 300 feats, 1xB200 batch=32 frame-pairs (BASELINE.json configs[1])"),
    "c3": dict(W=1280, H=720, feats=500, batch=16, pool_streams=2, pool_frames=24, cpu_pairs=200,
               workload="uHumans2-shaped 720p stereo 1280x720, 500 feats, 1xB200, 16 streams (BASELINE.json configs[2], without the Mesher)"),
    "c4": dict(W=1920, H=1080, feats=1000, batch=1, pool_streams=1, pool_frames=24, cpu_pairs=80,
               workload="Synthetic 1080p stereo 1920x1080, 1000 feats, one independent stream per B200 (BASELINE.json configs[3])"),
    "c5": dict(W=3840, H=2160, feats=2000, batch=1, pool_streams=1, pool_frames=10, cpu_pairs=24,
               workload="4K stereo 3840x2160, 2000 feats, one stream on ONE B200 (the single-GPU side of BASELINE.json configs[4])"),
}


def config_rig(cfg):
    left, right = CameraParams.euroc_left(), CameraParams.euroc_right()
    if (cfg["W"], cfg["H"]) != (left.width, left.height):
        left, right = left.scaled(cfg["W"], cfg["H"]), right.scaled(cfg["W"], cfg["H"])
    return left, right, StereoRigSetup(left, right)


def config_params(cfg):
    return dataclasses.replace(FrontendParams.euroc(), max_features_per_frame=cfg["feats"])


def _gen_stream(args):
    name, s, n_frames = args
    cfg = CONFIGS[name]
    left, right, rig = config_rig(cfg)
    st = SynthStream(left, right, rig.R1, seed=20240 + 1000 * s)
    L = np.zeros((n_frames, cfg["H"], cfg["W"]), np.uint8)
    R = np.zeros_like(L)
    for k in range(n_frames):
        f = st.frame(k)
        L[k], R[k] = f.left, f.right
    fwd = np.stack([st.kf_rotation(k, k + 1) for k in range(n_frames - 1)])
    bwd = np.stack([st.kf_rotation(k + 1, k) for k in range(n_frames - 1)])
    return L, R, fwd, bwd


def frame_pool(name: str):
    """pool_streams synthetic sequences of pool_frames pairs + the frame-to-frame rotations in both
    directions, cached in the temporary directory (generation is numpy, one process per sequence)."""
    cfg = CONFIGS[name]
    PS, NF = cfg["pool_streams"], cfg["pool_frames"]
    cache = os.path.join(tempfile.gettempdir(), "kvfe_bench_pool_v2_%s_%d_%d.npz" % (name, PS, NF))
    if os.path.exists(cache):
        try:
            z = np.load(cache)
            return z["left"], z["right"], z["fwd"], z["bwd"]
        except Exception:
            pass                                   # unreadable cache: regenerate (deterministic)
    import multiprocessing as mp
    with mp.get_context("fork").Pool(min(PS, 8)) as pool:
        res = pool.map(_gen_stream, [(name, s, NF) for s in range(PS)])
    left, right = np.stack([r[0] for r in res]), np.stack([r[1] for r in res])
    fwd, bwd = np.stack([r[2] for r in res]), np.stack([r[3] for r in res])
    try:
        # several ranks may build the cache at once: write privately, publish atomically
        tmp = "%s.%d.tmp" % (cache, os.getpid())
        with open(tmp, "wb") as fh:
            np.savez(fh, left=left, right=right, fwd=fwd, bwd=bwd)
        os.replace(tmp, cache)
    except Exception:
        pass
    return left, right, fwd, bwd


def pass_frame(t: int, NF: int) -> int:
    """frame of the pool replayed at pass t: 0, 1, ..., NF-1, NF-2, ..., 1, 0, 1, ..."""
    period = 2 * (NF - 1)
    u = t % period
    return u if u < NF else period - u


def pass_rotation(fwd, bwd, s: int, t: int, NF: int):
    """camLrectKm1_R_camLrectK of pass t (identity for the first pass)."""
    if t == 0:
        return np.eye(3)
    a, b = pass_frame(t - 1, NF), pass_frame(t, NF)
    return fwd[s, a] if b == a + 1 else bwd[s, b]


def slot_timestamp(b: int, t: int) -> int:
    # staggers the keyframe cadence across batch slots: slot b's first gap is (1 + b % 4) periods
    return T0_NS + (t + (b % 4 if t >= 1 else 0)) * DT_NS


def mat3(a, b):
    """3x3 product in the device's operation order (common.cuh matmul3: a0*b0 + (a1*b1 + a2*b2))."""
    a, b = np.asarray(a, np.float64).reshape(3, 3), np.asarray(b, np.float64).reshape(3, 3)
    c = np.zeros((3, 3))
    for i in range(3):
        for j in range(3):
            c[i, j] = float(a[i, 0]) * float(b[0, j]) + (float(a[i, 1]) * float(b[1, j]) + float(a[i, 2]) * float(b[2, j]))
    return c


class ClockSampler:
    def __init__(self, gpu_index: int):
        self.rows, self.stop = [], False
        self.idx = gpu_index
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([c.strip() for c in o.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


def pin_to_gpu_numa_node(local: int):
    """Restrict this rank (and the dispatcher threads it will create) to the CPUs next to its GPU."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        path = "/sys/bus/pci/devices/%s/local_cpulist" % bus.lower()[-12:]
        txt = open(path).read().strip()
        cpus = set()
        for part in txt.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"pci": bus, "cpus": len(cpus)}
    except Exception as e:                       # no sysfs / NVML: leave the affinity alone
        return {"error": str(e)[:80]}
    return None


# ------------------------------------------------------------------------------------------------
# the oracle front-end as the timed CPU baseline (cv2 == the reference's OpenCV code path)
# ------------------------------------------------------------------------------------------------
def _oracle_worker(args):
    name, slot, n_warm, n_timed, threads, collect = args
    import cv2
    from oracle import frontend as ofe
    from oracle.rig import StereoRig
    cv2.setNumThreads(threads)
    cfg = CONFIGS[name]
    lcam, rcam, _ = config_rig(cfg)
    rig = StereoRig(lcam, rcam)
    left, right, fwd, bwd = frame_pool(name)
    PS, NF = cfg["pool_streams"], cfg["pool_frames"]
    s = slot % PS
    fe = ofe.StereoFrontend(config_params(cfg), rig)
    acc = np.eye(3)
    t0, n_kf, rec = None, 0, []
    for t in range(n_warm + n_timed):
        if t == n_warm:
            t0 = time.perf_counter()
        f = pass_frame(t, NF)
        R = mat3(acc, pass_rotation(fwd, bwd, s, t, NF))
        sf = ofe.StereoFrame.make(t, slot_timestamp(slot, t), left[s, f], right[s, f], rig)
        o = fe.spin(sf, R)
        acc = np.eye(3) if o.is_keyframe else R
        n_kf += bool(o.is_keyframe) and t >= n_warm
        if collect and t < collect:
            lf = o.frame.left_frame
            rec.append((bool(o.is_keyframe), np.array(lf.keypoints, np.float32).reshape(-1, 2),
                        np.array(lf.landmarks, np.int64)))
    return time.perf_counter() - t0, n_timed, n_kf, rec


def cpu_baseline_single(name: str, n_warm: int, n_timed: int, collect: int):
    dt, n, n_kf, rec = _oracle_worker((name, 0, n_warm, n_timed, 1, collect))
    return {"value": n / dt, "unit": "frame-pairs/s", "cores": 1, "kind": "port",
            "sample": "oracle (cv2 4.13 + numpy RANSAC), stream of batch slot 0, %d timed pairs after %d warm-up, %d keyframes, "
                      "cv2.setNumThreads(1), %.1f s" % (n, n_warm, n_kf, dt)}, rec


REF_INNER = 8


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (the oracle: same OpenCV
    calls), one single-threaded process per host core, one camera stream each.  A step = REF_INNER
    passes (frames) of every process."""
    import multiprocessing as mp
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    ncores = len(os.sched_getaffinity(0))
    nproc = max(1, min(ncores, 32))     # 32 / 64 / 128 processes were tried on the 128-thread box: 32 is the fastest
    frame_pool(args.config)                                  # build the cache once
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(nproc) as pool:
        res = pool.map(_oracle_worker, [(args.config, i, args.warmup * REF_INNER, args.steps * REF_INNER, 1, 0) for i in range(nproc)])
    wall = max(r[0] for r in res)
    total = sum(r[1] for r in res)
    value = total / wall
    line = {
        "impl": "reference", "metric": "stereo front-end frame-pairs/sec @ %dx%d" % (cfg["W"], cfg["H"]), "value": value,
        "unit": "frame-pairs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8/int32/f32/f64 (OpenCV CPU)", "data": "synthetic",
        "config": {"workload": cfg["workload"], "inner_passes_per_step": REF_INNER,
                   "arm": "reference CPU front-end (oracle = the reference's OpenCV calls through cv2): %d independent "
                          "streams on %d host processes, 1 thread each" % (nproc, nproc)},
        "cpu_baseline": {"value": value, "unit": "frame-pairs/s", "cores": nproc, "kind": "port",
                         "sample": "%d streams x %d timed pairs, one single-threaded process per core" % (nproc, args.steps * REF_INNER)},
        "e2e": {"value": value, "unit": "frame-pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "host_cores_available": ncores, "wall_s_incl_setup": time.perf_counter() - t0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
DUMP_SEED = 0
DUMP_PACKET_BYTES = 24 << 20          # budget of the sampled packets' per-keypoint arrays
DUMP_RECT_BYTES = 32 << 20            # budget of the sampled keyframes' rectified pairs (float32)


def dump_plan(pass_count: int, B: int, cap: int, W: int, H: int):
    """Which outputs of the last timed step --dump-outputs writes in full: a seeded sample of (pass, stream)
    slots sized so that the whole dump stays under 64 MB (at most 38 float64 values per keypoint slot)."""
    n = max(1, min(256, pass_count * B, DUMP_PACKET_BYTES // (38 * 8 * max(cap, 1))))
    flat = np.sort(np.random.default_rng(DUMP_SEED).choice(pass_count * B, size=n, replace=False))
    return {"want": {(int(f) // B, int(f) % B) for f in flat}, "n_rect": min(8, DUMP_RECT_BYTES // (2 * 4 * W * H)),
            "got": {}}


def dump_outputs(d: str, chk, kf, nkp, plan):
    """Writes what the caller of kvfe_pipeline_* received in the last timed step as DIR/<name>.npy:
    step_*        (passes, streams) per output: keyframe flag, keypoint count, output checksum (two 32-bit halves);
    packet_*      the sampled packets (slots in packet_pass_stream): header values one row per packet, keypoint
                  arrays concatenated in slot order (row counts: packet_n, packet_n_smart, packet_n_mesh_triangles);
    rect_*        the rectified pairs of the first sampled keyframes (slots in rect_pass_stream).
    Arrays with no elements are not written: the bench runs with the 2D mesh off, so no mesh triangles.
    Every value written is finite: a non-finite entry (uR of a smart stereo measurement whose right keypoint is not
    valid is NaN) is stored as 0 and marked in <name>_nonfinite (0 finite, 1 NaN, 2 +inf, 3 -inf), which is written
    only for arrays holding such entries."""
    from kimera_vio_b200.lib import PACKET_FIELDS
    os.makedirs(d, exist_ok=True)

    def save(name, a):
        a = np.asarray(a)
        if a.size == 0:
            return
        a = a if a.dtype == np.float32 else a.astype(np.float64)
        bad = ~np.isfinite(a)
        if bad.any():
            code = np.where(np.isnan(a), 1, np.where(a > 0, 2, 3)) * bad
            np.save(os.path.join(d, name + "_nonfinite.npy"), code.astype(np.float32))
            a = np.where(bad, 0, a).astype(a.dtype)
        np.save(os.path.join(d, name + ".npy"), a)

    chk = chk.astype(np.uint64)
    save("step_is_keyframe", kf.astype(np.float32))
    save("step_n_keypoints", nkp.astype(np.float32))
    save("step_checksum_hi", chk >> np.uint64(32))
    save("step_checksum_lo", chk & np.uint64(0xFFFFFFFF))
    keys = sorted(plan["got"])
    pk = [plan["got"][k] for k in keys]
    save("packet_pass_stream", np.array(keys).reshape(-1, 2))
    per_kp = {name for name, _, _ in PACKET_FIELDS}
    for name in pk[0]:
        if name in ("left_rect", "right_rect", "stream", "tag"):
            continue
        vals = [p[name] for p in pk]
        if name == "checksum":
            v = np.array(vals, np.uint64)
            save("packet_checksum_hi", v >> np.uint64(32))
            save("packet_checksum_lo", v & np.uint64(0xFFFFFFFF))
        elif name == "timestamp":
            save("packet_timestamp_from_t0", np.array(vals, np.int64) - T0_NS)
        elif name in per_kp:
            save("packet_" + name, np.concatenate(vals))
        else:
            save("packet_" + name, np.stack([np.asarray(v) for v in vals]))
    rk = [k for k in keys if "left_rect" in plan["got"][k]][:plan["n_rect"]]
    save("rect_pass_stream", np.array(rk, np.int64).reshape(-1, 2))
    for side in ("left_rect", "right_rect"):
        if rk:
            save("rect_" + side.split("_")[0], np.stack([plan["got"][k][side] for k in rk]).astype(np.float32))


def run_gpu(args):
    name = args.config
    cfg = CONFIGS[name]
    W, H = cfg["W"], cfg["H"]
    B = args.batch or cfg["batch"]
    PS, NF = cfg["pool_streams"], cfg["pool_frames"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    left, right, fwd, bwd = frame_pool(name)            # before CUDA is initialised (forks)
    affinity = pin_to_gpu_numa_node(local) if not args.no_pin else None

    import torch
    import torch.distributed as dist
    from kimera_vio_b200 import lib as kl

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    K, Wm, R_in = args.steps, args.warmup, args.inner
    n_warm, n_timed = Wm * R_in, K * R_in
    n_pass = n_warm + n_timed
    lcam, rcam, rig = config_rig(cfg)
    p = config_params(cfg)
    tail = sobel_cpu_tail_start(W)
    kcfg = kl.make_config(p, W, H, batch=1, sobel_cpu_tail_start=tail)
    pipe = kl.Pipeline(kcfg, rig.to_c(), n_streams=B, n_workers=args.workers, queue_depth=n_pass + 8, output_slots=4,
                       want_rectified=True, rotation_mode=1, checksum_outputs=True, max_in_flight=args.in_flight)
    pkb = pipe.packet_bytes
    img = W * H

    # device-resident and pinned-host copies of the frame pool
    dL, dR = torch.from_numpy(left).cuda(), torch.from_numpy(right).cuda()
    pL, pR = torch.from_numpy(left).pin_memory(), torch.from_numpy(right).pin_memory()
    torch.cuda.synchronize()

    frame_of = np.array([pass_frame(t, NF) for t in range(n_pass)], np.int64)
    rot_tab = np.stack([np.stack([pass_rotation(fwd, bwd, s, t, NF).reshape(9) for t in range(n_pass)]) for s in range(PS)])
    gslot = rank * B + np.arange(B, dtype=np.int64)                     # global batch slot of every local stream

    def plan(base_l: int, base_r: int, t0: int, t1: int):
        n = (t1 - t0) * B
        streams = np.tile(np.arange(B, dtype=np.int32), t1 - t0)
        tt = np.repeat(np.arange(t0, t1, dtype=np.int64), B)
        ff = frame_of[tt]
        ss = streams.astype(np.int64) % PS
        off = (ss * NF + ff) * img
        lp = (base_l + off).astype(np.uint64)
        rp = (base_r + off).astype(np.uint64)
        stagger = np.where(tt >= 1, np.tile(gslot % 4, t1 - t0), 0)
        ts = (T0_NS + (tt + stagger) * DT_NS).astype(np.int64)
        Rm = np.ascontiguousarray(rot_tab[ss, tt])
        return n, streams, lp, rp, ts, Rm, tt.astype(np.uint64)

    out_dt = np.dtype([("stream", "<i4"), ("slot", "<i4"), ("tag", "<u8"), ("is_keyframe", "<i4"), ("n_keypoints", "<i4"),
                       ("checksum", "<u8"), ("packet", "<u8"), ("rect_left", "<u8"), ("rect_right", "<u8")])
    assert out_dt.itemsize == C.sizeof(kl.PipelineOutput)
    lib, ph = pipe.lib, pipe.h
    OUTS = (kl.PipelineOutput * 1024)()
    outs_np = np.frombuffer(OUTS, dtype=out_dt)

    def run(pl, keep_packets=0, dump=None):
        """Pushes a whole plan (queue-ahead) and pops until everything is done.  Returns per-(pass, slot)
        arrays of checksum / is_keyframe / n_keypoints (+ parsed packets of slot 0 for the first passes).
        dump: dump_plan() of the plan's last step, whose sampled packets are parsed into dump["got"]."""
        n, streams, lp, rp, ts, Rm, tags = pl
        t_first = int(tags[0])
        chk = np.zeros((n // B, B), np.uint64)
        kf = np.zeros((n // B, B), bool)
        nkp = np.zeros((n // B, B), np.int32)
        kept = {}
        acc = lib.kvfe_pipeline_push_many(ph, n, streams.ctypes.data, lp.ctypes.data, rp.ctypes.data, W, ts.ctypes.data,
                                          Rm.ctypes.data, tags.ctypes.data)
        assert acc == n, (acc, n, lib.kvfe_pipeline_last_error(ph))
        done = 0
        while done < n:
            m = lib.kvfe_pipeline_pop(ph, OUTS, 1024, 2000)
            assert m > 0, "pipeline stalled: %s" % lib.kvfe_pipeline_last_error(ph)
            o = outs_np[:m]
            ti = (o["tag"] - t_first).astype(np.int64)
            chk[ti, o["stream"]] = o["checksum"]
            kf[ti, o["stream"]] = o["is_keyframe"] != 0
            nkp[ti, o["stream"]] = o["n_keypoints"]
            if keep_packets:
                for i in np.nonzero((o["stream"] == 0) & (o["tag"] < keep_packets))[0]:
                    kept[int(o["tag"][i])] = pipe.parse(OUTS[int(i)], copy_rect=False)
            if dump is not None:
                for i in np.nonzero(o["tag"] >= dump["from"])[0]:
                    key = (int(o["tag"][i]) - dump["from"], int(o["stream"][i]))
                    if key in dump["want"]:
                        dump["got"][key] = pipe.parse(OUTS[int(i)], copy_rect=dump["n_rect"] > 0)
            lib.kvfe_pipeline_release(ph, OUTS, m)
            done += m
        return chk, kf, nkp, kept

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    N_PAR = 24            # passes of slot 0 compared with the oracle (parity self-check)
    dump = None
    if args.dump_outputs and rank == 0:       # sampled in the e2e run, the last timed one
        dump = dump_plan(R_in, B, pipe.cap, W, H)
        dump["from"] = n_pass - R_in
    res = {}
    for label, bl, br in (("value", dL.data_ptr(), dR.data_ptr()), ("e2e", pL.data_ptr(), pR.data_ptr())):
        pipe.reset()
        warm = run(plan(bl, br, 0, n_warm), keep_packets=N_PAR if (label == "e2e" and rank == 0) else 0)
        pl = plan(bl, br, n_warm, n_pass)
        barrier()
        st0 = pipe.stats()
        sampler = ClockSampler(local)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with sampler:
            ev0.record()
            t0 = time.perf_counter()
            timed = run(pl, dump=dump if label == "e2e" else None)
            ev1.record()
            barrier()
            wall = time.perf_counter() - t0
        st1 = pipe.stats()
        res[label] = dict(ms_events=ev0.elapsed_time(ev1), wall_s=wall, warm=warm, timed=timed, clocks=sampler.summary(),
                          graph_launches=st1["graph_launches"] - st0["graph_launches"],
                          kernel_launches=st1["kernel_launches"] - st0["kernel_launches"],
                          launch_cpu_s=st1["launch_seconds"] - st0["launch_seconds"], staged=st1["staged_copies"])
    # the two runs process the same frames: every output (packet + rectified images) must be byte-identical
    same_outputs = bool(np.array_equal(res["value"]["timed"][0], res["e2e"]["timed"][0]) and
                        np.array_equal(res["value"]["warm"][0], res["e2e"]["warm"][0]))
    if dump is not None:
        chk, kf, nkp, _ = res["e2e"]["timed"]
        dump_outputs(args.dump_outputs, chk[-R_in:], kf[-R_in:], nkp[-R_in:], dump)
    kf_all = np.concatenate([res["e2e"]["warm"][1], res["e2e"]["timed"][1]])
    rho = float(res["e2e"]["timed"][1].mean())
    n_kp_mean = float(res["e2e"]["timed"][2].mean())
    n_kf_timed = int(res["e2e"]["timed"][1].sum())

    # ---------------- dominant kernel (LK) launch duration, live CUDA events ----------------
    # one context holding the whole batch, the step run stage by stage with events on the library stream
    # (kvfe_frontend_step_dev_timed); keyframe_R_cur accumulated on the host from the schedule observed above
    lk_ms, stage_ms = None, None
    if rank == 0:
        T_LK = min(28, n_warm)
        big = kl.Context(kl.make_config(p, W, H, batch=B, sobel_cpu_tail_start=tail), rig.to_c())
        acc = [np.eye(3) for _ in range(B)]
        stages = []
        for t in range(T_LK):
            f = pass_frame(t, NF)
            idx = torch.tensor([(b % PS) for b in range(B)], device="cuda")
            bl, br = dL[idx, f].contiguous(), dR[idx, f].contiguous()
            Rk = np.zeros((B, 9))
            for b in range(B):
                Rb = mat3(acc[b], pass_rotation(fwd, bwd, b % PS, t, NF))
                Rk[b] = Rb.reshape(9)
                acc[b] = np.eye(3) if kf_all[t, b] else Rb
            tsk = np.array([slot_timestamp(rank * B + b, t) for b in range(B)], np.int64)
            ms = big.step_dev_timed(bl.data_ptr(), br.data_ptr(), W, tsk, np.ascontiguousarray(Rk))
            if t >= 4:
                stages.append(ms)
        stage_ms = np.mean(stages, axis=0)
        lk_ms = float(stage_ms[8])
        big.close()

    # ---------------- host link rate and single-stream latency ----------------
    link, latency = None, None
    if rank == 0:
        nb = min(2 * B * img, pL.numel())
        hbuf, dbuf = pL.reshape(-1)[:nb], dL.reshape(-1)[:nb].clone()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dbuf.copy_(hbuf, non_blocking=True)
        torch.cuda.synchronize()
        c0.record()
        for _ in range(8):
            dbuf.copy_(hbuf, non_blocking=True)
        c1.record()
        torch.cuda.synchronize()
        link = {"h2d_gbs_copy_engine": 8 * hbuf.numel() / (c0.elapsed_time(c1) * 1e-3) / 1e9, "copy_bytes": int(hbuf.numel())}
        one = kl.Pipeline(kcfg, rig.to_c(), n_streams=1, n_workers=1, queue_depth=2, output_slots=2, want_rectified=True,
                          rotation_mode=1, checksum_outputs=False)
        lat, lat_kf = [], []
        for t in range(64):
            f = pass_frame(t, NF)
            Rm = np.ascontiguousarray(pass_rotation(fwd, bwd, 0, t, NF))
            t1 = time.perf_counter()
            one.push(0, pL[0, f].data_ptr(), pR[0, f].data_ptr(), W, slot_timestamp(0, t), Rm, tag=t)
            outs = one.pop(timeout_ms=5000)
            dt = (time.perf_counter() - t1) * 1e3
            assert len(outs) == 1
            if t >= 8:
                (lat_kf if outs[0].is_keyframe else lat).append(dt)
            one.release(outs)
        one.close()
        allv = np.array(lat + lat_kf)
        latency = {"what": "kvfe_pipeline push -> pop, host buffers, one stream alone on the GPU [ms]",
                   "p50": float(np.percentile(allv, 50)), "p99": float(np.percentile(allv, 99)),
                   "non_keyframe_p50": float(np.median(lat)) if lat else None,
                   "keyframe_p50": float(np.median(lat_kf)) if lat_kf else None, "frames": int(allv.size)}

    times = torch.tensor([res["value"]["ms_events"], res["e2e"]["wall_s"] * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = float(times[0]), float(times[1])

    if rank == 0:
        pairs = world * B * n_timed
        value = pairs / (dev_ms * 1e-3)
        e2e_value = pairs / (e2e_ms * 1e-3)
        b_alg = (1 - rho) * img + rho * 4 * img + 112 * n_kp_mean             # SURVEY 8(d), measured rho
        peaks, which = measured_peaks()
        # LK launch: (i) the compulsory bytes of SURVEY 8(d) for the B frame-pairs one launch serves;
        # (ii) what the kernel itself must read: previous + current pyramids of every stream (DESIGN.md section 3)
        lk_alg = b_alg * B
        pyr_bytes = sum(((W + (1 << l) - 1) >> l) * ((H + (1 << l) - 1) >> l) for l in range(p.klt_max_level + 1))
        lk_kernel_bytes = 2 * pyr_bytes * B
        achieved = lk_alg / (lk_ms * 1e-3) / 1e9
        step_achieved = b_alg * (B * n_timed / (dev_ms * 1e-3)) / 1e9            # whole path, per GPU
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "lk_traffic.json")
        if os.path.exists(tp) and name == "c2":
            tj = json.load(open(tp))
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
        # parity self-check: the first passes of slot 0 against the oracle fed the same frames and rotations
        parity, cpu = None, None
        if world == 1 and not args.no_cpu_baseline:
            cpu, rec = cpu_baseline_single(name, 8, args.cpu_pairs or cfg["cpu_pairs"], N_PAR)
            kept = res["e2e"]["warm"][3]
            bad = []
            for t, (okf, okp, olm) in enumerate(rec):
                g = kept.get(t)
                if g is None or g["n"] != len(okp) or bool(g["is_keyframe"]) != okf or not np.array_equal(g["landmark"], olm):
                    bad.append(t)
                elif len(okp) and np.abs(np.stack([g["kp_x"], g["kp_y"]], 1) - okp).max() > 1e-3:
                    bad.append(t)
            parity = {"passes_compared": len(rec), "slot": 0, "mismatching_passes": bad,
                      "fields": "n, is_keyframe, landmark ids (exact), keypoints (1e-3 px)"}
        r_v, r_e = res["value"], res["e2e"]
        line = {
            "metric": "stereo front-end frame-pairs/sec @ %dx%d" % (W, H), "value": value, "unit": "frame-pairs/s",
            "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": dev_ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8/int32 images, f32 LK+response, f64 geometry",
            "data": "synthetic",
            "config": {"workload": cfg["workload"], "inner_passes_per_step": R_in, "ms_per_pass": dev_ms / n_timed,
                       "batch_per_gpu": B, "streams_in_flight": B, "dispatcher_threads": pipe.pc.n_workers,
                       "steps_in_flight_per_stream": pipe.pc.max_in_flight, "rotation_input": "frame-to-frame (mode 1), accumulated on the device",
                       "keyframe_ratio": rho, "mean_keypoints": n_kp_mean, "numa_affinity": affinity,
                       "timing": "value: CUDA events around the timed region (device idle on both sides), max over ranks; e2e: "
                                 "wall clock between barriers; every pass reads other frames of a %d MB frame pool (> L2), no L2 flush" %
                                 ((2 * left.nbytes) // 2 ** 20)},
            "e2e": {"value": e2e_value, "unit": "frame-pairs/s", "ms_per_step": e2e_ms / K, "ms_per_pass": e2e_ms / n_timed,
                    # left image + step inputs of every frame, right image of the keyframes only (fetched after the
                    # keyframe decision: the reference does not touch the right image on other frames, SURVEY 8(d))
                    "h2d_bytes_per_step": int((n_timed * B * (img + 80) + n_kf_timed * img) / K),
                    "d2h_bytes_per_step": int((n_timed * B * pkb + n_kf_timed * 2 * img) / K),
                    "what": "kvfe_pipeline push/pop, images in pinned host memory pulled over the link by the TMA unit inside the step "
                            "graph (left image of every frame, right image of the keyframes after the on-device decision); packets "
                            "+ keyframe rectified pairs stored into pinned host memory and checksummed by the dispatcher",
                    "outputs_identical_to_value_run": same_outputs},
            "gpu_launches": int(r_v["kernel_launches"]),
            "graph_launches": int(r_v["graph_launches"]),
            "host_enqueue_ms_per_pass": {"value": 1e3 * r_v["launch_cpu_s"] / n_timed, "e2e": 1e3 * r_e["launch_cpu_s"] / n_timed,
                                         "note": "CPU time inside the launch path summed over the dispatcher threads"},
            "device_ms_e2e_events": r_e["ms_events"], "staged_copies": int(r_e["staged"]),
            "host_link": link, "latency_ms": latency,
            "clocks": r_v["clocks"], "clocks_e2e": r_e["clocks"],
            "roofline": {"bound": "hbm", "kernel": "lk_kernel_tma<24> (pyramidal LK, patch boxes staged by TMA: ~67% of the path's warp instructions)",
                         "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": which + " (burst copy)",
                         "algorithmic_bytes_per_launch": lk_alg, "launch_ms": lk_ms,
                         "bytes_definition": "SURVEY 8(d) compulsory bytes per frame-pair x %d frame-pairs per launch" % B,
                         "kernel_input_bytes": {"bytes_per_launch": lk_kernel_bytes,
                                                "achieved": lk_kernel_bytes / (lk_ms * 1e-3) / 1e9,
                                                "frac": lk_kernel_bytes / (lk_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                                "what": "previous + current pyramids of every stream (what LK itself must read)"},
                         "whole_step": {"algorithmic_bytes_per_frame_pair": b_alg, "achieved": step_achieved,
                                        "frac": step_achieved / peaks["hbm_gbs"]},
                         "stage_ms": [float(v) for v in stage_ms],
                         "note": "latency/issue-bound: serial float chains imposed by bit-exactness, see DESIGN.md"},
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
            line["parity_check"] = parity
        print(json.dumps(line))
    pipe.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--inner", type=int, default=128, help="passes (batches of frame-pairs) per step")
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="streams per GPU (0: the config's)")
    ap.add_argument("--workers", type=int, default=0, help="dispatcher threads (0: library default)")
    ap.add_argument("--in-flight", type=int, default=0, help="steps in flight per stream, 1 or 2 (0: library default)")
    ap.add_argument("--cpu-pairs", type=int, default=0, help="timed frame-pairs of the CPU baseline sample (0: the config's, ~10-30 s of CPU work)")
    ap.add_argument("--impl", default="kvfe", choices=["kvfe", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pin", action="store_true", help="do not pin the rank to the GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step delivered (step-wide flags and checksums, a seeded sample of "
                         "packets and keyframe rectified pairs) as DIR/<name>.npy, float32/float64, under 64 MB")
    args = ap.parse_args()
    if args.steps < 1 or args.inner < 1:
        ap.error("--steps and --inner must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
