#!/usr/bin/env python
"""bench.py -- frames/s of the per-frame armor pipeline (preprocess -> YOLOv8n -> decode+NMS -> PnP).

Contract: `python bench.py --gpus N --steps K --warmup W` (N>1 under torch.distributed.run, one rank
per GPU).  One step = one pass of the hot path over one batch of synthetic frames per GPU.
Workload = BASELINE.json configs[3]: 1280x1024 8-bit Bayer camera frames, batch 256 per GPU, full
preprocess + YOLOv8n (nc=14, seeded random-init FP16) + decode/NMS + PnP; frames are independent,
so ranks share nothing (weak scaling, no data-path collective).  Rank 0 prints ONE JSON line.

`--impl reference` times the reference path's CPU form (cv2 flip/resize, OpenCV-DNN on the ONNX
export of the same weights, numpy NMS, cv2.solvePnP) on the box's host cores.

`--dump-outputs DIR` writes what the timed path returned for rank 0's frames in its last step as
DIR/<name>.npy (float32 / float64), so that two builds can be compared output for output: the inputs
(frames and weights) are seeded and identical from run to run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "frames/s (640^2 YOLOv8n+NMS+PnP)"
SRC_W, SRC_H = 1280, 1024
FLOPS_PER_FRAME = 8.0956416e9          # SURVEY.md section 8d, 63 convs
K_CAM = [957.669211, 0.0, 345.943891, 0.0, 969.127115, 284.057302, 0.0, 0.0, 1.0]
D_CAM = [-0.405274, 0.126058, -0.026939, -0.006503, 0.0]


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries (NCCL's version banner, cv2) write to fd 1; the contract is ONE JSON line on stdout,
    so everything but that line is sent to stderr."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------- inputs
def make_bayer_frames_device(n: int, seed: int, device):
    """n synthetic RGGB frames on the device (torch used as plumbing): rm_test.jpg with per-frame
    circular shift, gain and sensor noise (irmv_detection_b200.synth, vectorised)."""
    import torch
    from irmv_detection_b200 import synth
    base = torch.from_numpy(synth.load_base()[..., ::-1].copy()).to(device)        # RGB u8 [H,W,3]
    g = torch.Generator(device=device)
    g.manual_seed(1234 + seed)
    out = torch.empty((n, SRC_H, SRC_W), dtype=torch.uint8, device=device)
    yy = (torch.arange(SRC_H, device=device) & 1)[:, None]
    xx = (torch.arange(SRC_W, device=device) & 1)[None, :]
    chan = torch.where((yy == 0) & (xx == 0), 0, torch.where((yy == 1) & (xx == 1), 2, 1))      # RGGB
    rng = np.random.default_rng(seed)
    for i in range(n):
        dx, dy = rng.integers(-96, 97, 2)
        gain = float(rng.uniform(0.9, 1.2))
        f = torch.roll(base, (int(dy), int(dx)), (0, 1)).float() * gain
        f = f + torch.randn(f.shape, generator=g, device=device) * 3.0
        f = f.round().clamp_(0, 255).to(torch.uint8)
        out[i] = torch.gather(f, 2, chan[..., None]).squeeze(2)
    return out


_SCRATCH = None


def scratch_path(name: str) -> str:
    """A path in this process's temporary directory (removed at exit): weight files and the ONNX export go
    there, never into the source tree."""
    global _SCRATCH
    if _SCRATCH is None:
        _SCRATCH = tempfile.TemporaryDirectory(prefix="irmv_bench_")
    return os.path.join(_SCRATCH.name, name)


def weights_file(seed: int = 0) -> str:
    from irmv_detection_b200 import weights
    path = scratch_path(f"seed{seed}.irmw")
    weights.write_random(path, seed)
    return path


def dump_outputs(out_dir: str, eng, dets, n: int) -> None:
    """What a caller of the timed path receives for the step's n frames: detections per frame (source-pixel
    boxes, scores, class ids; zero past counts[f], max_det slots) and the fused PnP poses of those detections."""
    md = eng.max_det
    counts = np.array([len(d) for d in dets], np.float32)
    boxes, scores, classes = np.zeros((n, md, 4), np.float32), np.zeros((n, md), np.float32), np.zeros((n, md), np.float32)
    for f, frame in enumerate(dets):
        for i, d in enumerate(frame):
            boxes[f, i], scores[f, i], classes[f, i] = d.xyxy, d.score, int(d.class_id)
    rv, tv, ok = eng.fetch_poses(n)
    valid = np.arange(md)[None, :] < counts[:, None]
    arrays = {"counts": counts, "boxes": boxes, "scores": scores, "class_ids": classes,
              "rvecs": np.where(valid[..., None], rv, 0.0), "tvecs": np.where(valid[..., None], tv, 0.0),
              "pose_ok": (ok & valid).astype(np.float32)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ---------------------------------------------------------------------------------- CPU reference
class CpuReference:
    """The reference path's CPU form (BASELINE.md section 3), through the oracle modules."""

    def __init__(self, wpath: str, threads: int):
        import cv2
        import torch
        from oracle import export_onnx, yolov8n_ref as Y
        cv2.setNumThreads(threads)
        torch.set_num_threads(threads)
        self.threads = threads
        self.model = Y.build(wpath)
        self.kind_net = "torch-cpu"
        self.net = None
        try:
            onnx_path = wpath.replace(".irmw", ".onnx")
            export_onnx.export(self.model, onnx_path)
            self.net = cv2.dnn.readNetFromONNX(onnx_path)
            self.kind_net = "opencv-dnn"
        except Exception:
            self.net = None

    def frame(self, bayer: np.ndarray):
        import cv2
        import torch
        from oracle import nms_ref as N, pnp_ref as P
        rgb = cv2.cvtColor(bayer, cv2.COLOR_BayerRGGB2RGB)              # camera ISP step (mv_camera.cpp:96)
        img = cv2.flip(rgb, -1)
        r = cv2.resize(img, (640, 640), interpolation=cv2.INTER_LINEAR)
        x = np.ascontiguousarray((r.astype(np.float32) / 255.0).transpose(2, 0, 1))[None]
        if self.net is not None:
            self.net.setInput(x)
            out = self.net.forward()[0]
            boxes, scores = out[:, :4], out[:, 4:]
        else:
            with torch.no_grad():
                b, s = self.model(torch.from_numpy(x))
            boxes, scores = b[0].numpy(), s[0].numpy()
        # class-aware NMS in C++ (cv2.dnn.NMSBoxesBatched == the oracle's rule, tests/test_oracle_cpu.py)
        a, c = np.nonzero(scores > N.SCORE_THR)
        if a.size:
            sc = scores[a, c]
            top = np.argsort(-sc, kind="stable")[:N.MAX_CAND]
            a, c, sc = a[top], c[top], sc[top]
            bb = boxes[a]
            xywh = np.concatenate((bb[:, :2], bb[:, 2:] - bb[:, :2]), 1)
            sel = np.asarray(cv2.dnn.NMSBoxesBatched(xywh.tolist(), sc.tolist(), c.tolist(), N.SCORE_THR, N.IOU_THR)).ravel()
            sel = sel[np.argsort(-sc[sel], kind="stable")][:N.MAX_DET]
            kb, ks, kc = bb[sel], sc[sel], c[sel]
        else:
            kb, ks, kc = np.zeros((0, 4), np.float32), np.zeros(0, np.float32), np.zeros(0, np.int32)
        ob, _, _ = N.parse_output(kb, ks, kc, SRC_W, SRC_H)
        n = 0
        if len(ob):
            sx, sy = 640.0 / SRC_W, 480.0 / SRC_H
            pts = np.stack([np.stack([ob[:, 0] * sx, ob[:, 3] * sy], 1), np.stack([ob[:, 0] * sx, ob[:, 1] * sy], 1),
                            np.stack([ob[:, 2] * sx, ob[:, 1] * sy], 1), np.stack([ob[:, 2] * sx, ob[:, 3] * sy], 1)], 1)
            P.solve_cv2(pts.astype(np.float32))
            n = len(ob)
        return n

    def run(self, frames: np.ndarray, budget_s: float, min_frames: int = 4):
        self.frame(frames[0])                      # warm-up
        t0 = time.perf_counter()
        n = 0
        while n < len(frames) and (n < min_frames or time.perf_counter() - t0 < budget_s):
            self.frame(frames[n])
            n += 1
        dt = time.perf_counter() - t0
        return n / dt, n, dt


def replay_split(args):
    """(frames per replay, lanes) of the engine for this run.  Default: the whole 256-frame step in ONE replay on one
    lane -- every launch carries a fixed cost of ~7 us (pipeline fill, last epilogue, drain), 50 GEMM launches per
    replay, so one 256-frame replay beats two of 128 by 3 % (measured: 4.60 vs 4.75 ms per step; --sub-batch 128
    --lanes 2 is the round-1 split)."""
    sub = args.sub_batch or min(args.batch, 256)
    lanes = args.lanes or min(2, (args.batch + sub - 1) // sub)
    return sub, lanes


def workload_config(batch: int, sub_batch: int, lanes: int) -> dict:
    """`config` of the JSON line, identical for both arms (the driver compares them)."""
    return {"workload": "1280x1024 8-bit Bayer RGGB frames, batch 256/GPU, fused demosaic+rot180+resize -> "
                        "YOLOv8n nc=14 (seeded random-init, FP16 tcgen05) -> decode+NMS -> PnP "
                        "(BASELINE.json configs[3])",
            "frames_per_gpu_per_step": batch, "sub_batch": sub_batch, "lanes": lanes,
            "l2": "inputs larger than L2 (335 MB of frames per step per GPU, activations cycled per replay)",
            "timing": "CUDA events on the engine's streams, summed over steps, max over ranks"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from irmv_detection_b200 import synth
    threads = os.cpu_count() or 1
    wpath = weights_file(0)
    ref = CpuReference(wpath, threads)
    base = synth.load_base()
    # A step of the workload is 256 frames (9 s of CPU work on 16 cores); the arm times a bounded sample of
    # every step -- the first `ref_frames` frames of the step's batch -- and scales ms_per_step to the full step.
    per_step = args.ref_frames
    frames = synth.bayer_from_rgb(synth.frames_from_base(base, per_step, seed=0)[..., ::-1], "RGGB")
    for _ in range(args.warmup):
        for f in frames:
            ref.frame(f)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for f in frames:
            ref.frame(f)
    dt = time.perf_counter() - t0
    fps = args.steps * per_step / dt
    sample = (f"the first {per_step} of each step's {args.batch} frames x {args.steps} steps (+ {args.warmup} warm-up steps) of the same "
              f"1280x1024 Bayer workload; cv2 demosaic+flip+resize, {ref.kind_net} YOLOv8n FP32, cv2 NMSBoxesBatched, "
              f"cv2.solvePnP(IPPE); ms_per_step is scaled from the sample to the full {args.batch}-frame step")
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": args.batch / fps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.batch, *replay_split(args)),
        "note": "reference CPU path on host cores; TensorRT unavailable offline",
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ---------------------------------------------------------------------------------- ours
def source_hash() -> str:
    """Hash of the CUDA sources: ncu-derived figures under profiles/ are only quoted for the build they
    were captured from."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "irmv_detection_b200", "csrc")
    for name in sorted(os.listdir(d)):
        if name.endswith((".cu", ".cuh")):
            h.update(name.encode())
            h.update(open(os.path.join(d, name), "rb").read())
    return h.hexdigest()[:16]


def profile_json(name: str):
    """profiles/<name> if it was captured from the current sources, else (None, why)."""
    path = os.path.join(ROOT, "profiles", name)
    if not os.path.exists(path):
        return None, f"profiles/{name} missing"
    d = json.load(open(path))
    if d.get("src_hash") != source_hash():
        return None, f"profiles/{name} was captured from other sources (src_hash {d.get('src_hash')} != {source_hash()}): not quoted"
    return d, None


def h2d_ceiling(hosts, dev_buf, steps: int, world: int, local_rank: int, device: str):
    """Plain cudaMemcpyAsync of the step's pinned frame buffers to the device, no kernels, all ranks at the
    same time: the PCIe ceiling of the end-to-end path on this box.  One stream and two streams (each half
    of the buffer) are both timed and the faster one is the ceiling.  Returns (ms per batch, GB/s, streams),
    the time being the max over ranks."""
    import torch
    from irmv_detection_b200 import sharding
    src = [torch.from_numpy(h) for h in hosts]
    half = src[0].shape[0] // 2
    side = torch.cuda.Stream()
    best = None
    for nstreams in (1, 2):
        for s in src:                                    # warm
            dev_buf.copy_(s, non_blocking=True)
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier(device_ids=[local_rank])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            h = src[i % len(src)]
            if nstreams == 1:
                dev_buf.copy_(h, non_blocking=True)
            else:
                side.wait_stream(torch.cuda.current_stream())
                dev_buf[:half].copy_(h[:half], non_blocking=True)
                with torch.cuda.stream(side):
                    dev_buf[half:].copy_(h[half:], non_blocking=True)
                torch.cuda.current_stream().wait_stream(side)
        e1.record()
        torch.cuda.synchronize()
        ms, _ = sharding.reduce_max_sum(e0.elapsed_time(e1) / steps, 0.0, device=device)
        if best is None or ms < best[0]:
            best = (ms, hosts[0].nbytes / (ms * 1e-3) / 1e9, nstreams)
    return best


def pnp_stress(n: int = 1_000_000, cpu_budget_s: float = 8.0):
    """BASELINE.json configs[4]: 1 M armor quads through the IPPE kernel; cv2.solvePnP(IPPE) on all host
    cores over a bounded sample beside it."""
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    from concurrent.futures import ThreadPoolExecutor
    base = synth.armor_quads(20000, seed=0)
    rng = np.random.default_rng(1)
    reps = (n + len(base) - 1) // len(base)
    q = np.ascontiguousarray(np.tile(base, (reps, 1, 1))[:n] + rng.normal(0, 0.05, (n, 4, 2)).astype(np.float32), np.float32)
    s = irmv.PnPSolver(K_CAM, D_CAM)
    dev = torch.from_numpy(q).cuda()
    rv = np.empty((n, 3)); tv = np.empty((n, 3)); ok = np.empty(n, np.uint8)
    for _ in range(3):
        s.solve_batch_device(dev.data_ptr(), n, rv, tv, ok)
    k = float(np.median([s.solve_batch_device(dev.data_ptr(), n, rv, tv, ok) for _ in range(5)]))
    t0 = time.perf_counter()
    for _ in range(2):
        s.solve_batch(q)
    wall_host = (time.perf_counter() - t0) / 2
    s.close()
    peaks, kind = measured_peaks()
    out = {"workload": f"{n} armor quads, IPPE, FP64, one armor per thread (BASELINE.json configs[4])",
           "gpu_kernel_ms": k, "armors_per_s_kernel": n / (k * 1e-3), "armors_per_s_host_to_host": n / wall_host,
           "hbm_bytes_per_armor": 80, "hbm_gbs_achieved": 80.0 * n / (k * 1e-3) / 1e9,
           "hbm_frac": 80.0 * n / (k * 1e-3) / 1e9 / float(peaks.get("hbm_gbs", 6650.0)),
           "bound": "FP64 ALU / latency (2.5 kFLOP of dependent FP64 per armor), not HBM",
           "ok_fraction": float(ok.mean())}
    try:
        from oracle import pnp_ref as P                    # CPU baseline leg: the reference's own call
        cores = os.cpu_count() or 1
        sample = 4000 * cores
        chunks = np.array_split(np.arange(sample), cores)
        t0 = time.perf_counter()
        with ThreadPoolExecutor(cores) as ex:
            list(ex.map(lambda idx: P.solve_cv2(q[idx]), chunks))
        cpu_s = time.perf_counter() - t0
        out.update({"cpu_armors_per_s": sample / cpu_s, "cpu_cores": cores, "cpu_sample": sample,
                    "cpu_kind": "reference call (cv2.solvePnP SOLVEPNP_IPPE, src/pnp_solver.cpp:49-51)",
                    "speedup_kernel_vs_cpu": (n / (k * 1e-3)) / (sample / cpu_s)})
    except Exception as ex:
        out["cpu_error"] = str(ex)
    return out


def reference_protocol(wpath: str):
    """The reference's own benchmark protocol (test/yolo_test.cpp:68-106; README.md:9-20 quotes its result):
    100 warm-ups, 30 runs x 10 x {memcpy of the 3.9 MB RGB frame into the source buffer + detect()}, through
    the C++ drop-in YoloEngine class (tests/cpp/drop_in_test.cpp)."""
    import shutil
    import tempfile
    from irmv_detection_b200 import build as B, synth
    if not os.path.exists(B.DROP_IN_TEST):
        return {"error": "drop_in_test not built"}
    with tempfile.TemporaryDirectory() as d:
        shutil.copy(wpath, os.path.join(d, "yolov7.irmw"))
        synth.load_base().tofile(os.path.join(d, "frame.raw"))
        r = subprocess.run([B.DROP_IN_TEST, os.path.join(d, "yolov7.onnx"), os.path.join(d, "frame.raw"), "30", "protocol"],
                           capture_output=True, text=True, timeout=240)
    for l in r.stdout.splitlines():
        if l.startswith("protocol "):
            f = l.split()
            return {"avg_ms": float(f[4]), "min_ms": float(f[6]), "max_ms": float(f[8]), "runs": int(f[2]), "iters_per_run": 10,
                    "frame": "rm_test.jpg, packed 1280x1024x3 (3.9 MB memcpy per iteration), batch 1, C++ YoloEngine::detect()",
                    "reference_figure": "~5 ms on Jetson Orin Nano, 4-5 ms on RTX 3060 Laptop (reference README.md:9-14); bound < 30 ms (test/yolo_test.cpp:106)"}
    return {"error": f"rc {r.returncode}: {r.stdout[-300:]} {r.stderr[-300:]}"}


def full_node_path(wpath: str, local_rank: int, steps: int):
    """detect -> extract_armors -> solvePnP -> quaternion -> distance (the whole of message_callback,
    reference src/irm_detector.cpp:181-230) as one replay, on seeded light-bar scenes (the random-init
    network's boxes then contain real light bars): device-resident frames/s and the end-to-end rate with the
    per-armor payload read back."""
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    B, distinct = 128, 16
    scenes = np.stack([synth.armor_scene(12, 500 + i)[0][::-1, ::-1] for i in range(distinct)])     # camera view (un-rotated)
    raw = synth.bayer_from_rgb(scenes[..., ::-1], "RGGB")
    raw = np.ascontiguousarray(np.tile(raw, (B // distinct, 1, 1)))
    host = torch.empty(raw.shape, dtype=torch.uint8, pin_memory=True)
    host.numpy()[...] = raw
    dev = host.cuda()
    eng = irmv.YoloEngine(wpath, (SRC_W, SRC_H), chan_order=irmv.CH_BAYER_RGGB, max_batch=B, sub_batch=64, num_lanes=2,
                          device=local_rank)
    eng.enable_armors()
    eng.enable_pnp(K_CAM, D_CAM, (640.0 / SRC_W, 480.0 / SRC_H))
    for _ in range(3):
        eng.enqueue_batch_device(dev.data_ptr(), B)
        eng.sync()
    ms = 0.0
    for _ in range(steps):
        eng.enqueue_batch_device(dev.data_ptr(), B)
        ms += eng.sync()
    counts = sum(len(d) for d in eng.fetch(B))
    poses = eng.fetch_armor_poses(B)
    k, st = eng.profile_stages(dev.data_ptr(), 64)
    hn = host.numpy()
    pend = [eng.submit_batch(hn), eng.submit_batch(hn)]
    t0 = time.perf_counter()
    for _ in range(steps):
        pend.append(eng.submit_batch(hn))
        t = pend.pop(0)
        eng.collect_arrays(t, poses=True)
        eng.fetch_armor_poses(B, t)
    e2e_ms = (time.perf_counter() - t0) * 1e3 / steps
    while pend:
        eng.collect_arrays(pend.pop(0))
    out = {"workload": f"{B} Bayer frames of seeded light-bar scenes per step (12 armors each), sub_batch 64 x 2 lanes: "
                       "preprocess -> YOLOv8n -> NMS -> extract_armors -> IPPE -> tf2 quaternion + distance_to_image_center",
           "frames_per_s_device": B / (ms / steps * 1e-3), "frames_per_s_e2e": B / (e2e_ms * 1e-3),
           "detections_per_step": counts, "armors_with_pose_per_step": int(poses["ok"].sum()),
           "stage_ms_64_frames": st, "note": "stage_ms.pnp = extract_armors + quads + IPPE (+ quaternion/distance epilogue)"}
    eng.close()
    return out


def run_ours(args):
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import sharding
    rank, world, local_rank = sharding.env_rank_world()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback exists for the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        sharding.init_process_group("nccl")
    try:                                         # one disjoint core set per rank (8 ranks share the box's host cores)
        cores = sorted(os.sched_getaffinity(0))
        per = max(1, len(cores) // max(world, 1))
        mine = cores[local_rank * per:(local_rank + 1) * per] if world > 1 else cores
        if mine:
            os.sched_setaffinity(0, mine)
    except Exception:
        mine = []
    B = args.batch
    wpath = weights_file(0)
    frames_dev = make_bayer_frames_device(B, seed=rank, device=dev)
    torch.cuda.synchronize()
    sub_batch, lanes = replay_split(args)
    eng = irmv.YoloEngine(wpath, (SRC_W, SRC_H), chan_order=irmv.CH_BAYER_RGGB, max_batch=B,
                          sub_batch=sub_batch, num_lanes=lanes, device=local_rank)
    eng.enable_pnp(K_CAM, D_CAM, (640.0 / SRC_W, 480.0 / SRC_H))
    ptr = frames_dev.data_ptr()

    # ---- device-resident throughput (`value`) ------------------------------------------------
    # Phase 0 (untimed, reported as clock_warmup): bring the clocks and nvidia-smi up.  Then exactly
    # --warmup untimed steps, then exactly --steps timed steps.
    sampler = ClockSampler(local_rank)
    sampler.start()
    t_w = time.perf_counter()
    n_clock = 0
    while time.perf_counter() - t_w < args.clock_warmup_s:
        eng.enqueue_batch_device(ptr, B)
        eng.sync()
        n_clock += 1
    clock_warm = {"steps": n_clock, "seconds": time.perf_counter() - t_w,
                  "note": "untimed phase before the --warmup steps: lets the SM clocks ramp and nvidia-smi start sampling"}
    for _ in range(args.warmup):
        eng.enqueue_batch_device(ptr, B)
        eng.sync()
    if world > 1:
        torch.distributed.barrier(device_ids=[local_rank])
    torch.cuda.synchronize()
    dev_ms = 0.0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.enqueue_batch_device(ptr, B)
        dev_ms += eng.sync()                      # CUDA events on the engine's own streams
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop()
    dets = eng.fetch(B)
    n_dets = sum(len(d) for d in dets)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, dets, B)
    if world > 1:
        torch.distributed.barrier(device_ids=[local_rank])
    step_ms_local = dev_ms / args.steps
    step_ms, frames_per_step = sharding.reduce_max_sum(step_ms_local, float(B), device=str(dev))
    value = frames_per_step / (step_ms * 1e-3)

    # ---- end to end through the public API with host buffers (`e2e`) ---------------------------
    # submit_batch()/collect_arrays(): every step copies its own 256 frames from pinned host memory
    # (three rotating pinned buffers), runs the pipeline and reads detections + poses back; `inflight`
    # batches are queued ahead, so H2D copies run under the previous batch's kernels (what the
    # reference's TripleBuffer does between camera and detector threads).
    hosts = []
    for _ in range(3):
        h = torch.empty((B, SRC_H, SRC_W), dtype=torch.uint8, pin_memory=True)
        h.copy_(frames_dev)
        hosts.append(h.numpy())
    torch.cuda.synchronize()
    eng.detect_batch_arrays(hosts[0])
    e2e_steps = args.steps
    inflight = max(1, min(3, args.inflight))
    for _ in range(3):                            # warm the pipelined path (all three result sets, copy stream)
        eng.collect_arrays(eng.submit_batch(hosts[0]), poses=True)
    if world > 1:
        torch.distributed.barrier(device_ids=[local_rank])
    pending = [eng.submit_batch(hosts[i % 3]) for i in range(inflight - 1)]
    h2d_0, d2h_0 = eng.copy_bytes()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        pending.append(eng.submit_batch(hosts[(i + inflight - 1) % 3]))   # H2D + pipeline + D2H queued ahead ...
        eng.collect_arrays(pending.pop(0), poses=True)                    # ... while the oldest batch finishes and is parsed
    e2e_ms_local = (time.perf_counter() - t0) * 1e3 / e2e_steps
    h2d_1, d2h_1 = eng.copy_bytes()
    while pending:
        eng.collect_arrays(pending.pop(0), poses=True)
    # the synchronous call (one batch at a time, nothing overlapped) for comparison
    t0 = time.perf_counter()
    for _ in range(3):
        eng.detect_batch_arrays(hosts[0])
        eng.fetch_poses(B)
    sync_ms_local = (time.perf_counter() - t0) * 1e3 / 3
    e2e_ms, _ = sharding.reduce_max_sum(e2e_ms_local, 0.0, device=str(dev))
    sync_ms, _ = sharding.reduce_max_sum(sync_ms_local, 0.0, device=str(dev))
    e2e_value = frames_per_step / (e2e_ms * 1e-3)
    h2d = (h2d_1 - h2d_0) // e2e_steps            # counted by the engine from the copies it queued
    d2h = (d2h_1 - d2h_0) // e2e_steps
    # the PCIe ceiling of that path on this box: the same pinned buffers, plain copies, all ranks at once
    ceil_ms, ceil_gbs, ceil_streams = h2d_ceiling(hosts, frames_dev, max(4, min(e2e_steps, 10)), world, local_rank, str(dev))
    ceil_fps = frames_per_step / (ceil_ms * 1e-3)

    if rank != 0:
        eng.close()
        return

    # ---- roofline of the dominant kernel group (the tcgen05 convolutions) ---------------------
    peaks, peak_kind = measured_peaks()
    k, st = None, None
    conv_ms, pre_ms = [], []
    for _ in range(5):
        k, st = eng.profile_stages(ptr, B)
        conv_ms.append(st["conv"]); pre_ms.append(st["preprocess"])
    conv_t = statistics.median(conv_ms) * 1e-3
    st["conv"], st["preprocess"] = statistics.median(conv_ms), statistics.median(pre_ms)
    achieved = FLOPS_PER_FRAME * k / conv_t / 1e12
    peak = float(peaks.get("bf16_tflops", 1590.0))
    traffic, traffic_note = None, None
    tj, why = profile_json("r2_traffic.json")      # dram__bytes_read+write of the GEMM launches, ncu capture of THIS build
    if tj:
        traffic = tj["conv_group_dram_bytes_per_frame"] * k
    else:
        traffic_note = why
    # the single largest launch, timed live with CUDA events around it (eager replay, so the figure
    # carries a few us of launch latency): Detect P3 box.0|cls.0, 3x3 64->128 on the 80x80 grid
    top = None
    try:
        import ctypes as C
        from irmv_detection_b200 import _lib
        ms = np.zeros(80, np.float32)
        runs = []
        for _ in range(5):
            nops = _lib.lib().irmv_engine_profile_ops(eng._h, C.c_void_p(ptr), k, ms.ctypes.data, 80)
            runs.append(ms[:nops].copy())
        op_ms = np.median(np.stack(runs), axis=0)
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        from analyze_launches import name_ops
        i_top = [l[0] for l in name_ops(eng.describe_ops())].index("h0.01")     # conv0 lives in the stem
        fl = 2.0 * k * 80 * 80 * 9 * 64 * 128
        t_top = float(op_ms[i_top]) * 1e-3
        tk = None
        kj, _ = profile_json("r2_top_kernel.json")
        if kj:
            tk = kj["dram_bytes_per_launch"] * k / kj["frames"]
        top = {"kernel": "conv_raster_kernel Detect P3 box.0|cls.0 (3x3, 64->128, 80x80)", "flop_per_launch": fl,
               "ms_per_launch": t_top * 1e3, "achieved": fl / t_top / 1e12, "peak": peak, "unit": "TFLOP/s",
               "frac": fl / t_top / 1e12 / peak, "traffic": tk,
               "algorithmic_bytes_per_launch": k * 80 * 80 * (64 + 128) * 2}
    except Exception as ex:
        top = {"error": str(ex)}
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": traffic,
                "kernel": "conv_raster_kernel + conv_tc_kernel (the GEMM launches of one replay, timed as a group with CUDA "
                          "events: no single launch exceeds 5 % of the step)",
                "flop_per_launch_group": FLOPS_PER_FRAME * k, "top_launch": top,
                "frames_per_replay": k, "peak_source": f"{peak_kind} bf16_tflops (burst: stage timed alone)",
                "stage_ms": st,
                "preprocess": {"kernel": "stem_bayer2x_kernel (demosaic + rot180 + resize + /255 + conv0)", "bound": "hbm",
                               "algorithmic_bytes_per_frame": 1310720 + 16 * 320 * 320 * 2,
                               "achieved_gbs": (1310720 + 16 * 320 * 320 * 2) * k / (st["preprocess"] * 1e-3) / 1e9,
                               "frac": (1310720 + 16 * 320 * 320 * 2) * k / (st["preprocess"] * 1e-3) / 1e9 / hbm,
                               "peak_gbs": hbm},
                "hbm_frac_preprocess": (3768320.0 * k / (st["preprocess"] * 1e-3) / 1e9) / hbm if st["preprocess"] > 0 else None}
    if traffic_note:
        roofline["traffic_note"] = traffic_note

    # ---- batch-1 latency (BASELINE.json metric's second half) ----------------------------------
    lat = None
    try:
        e1 = irmv.YoloEngine(wpath, (SRC_W, SRC_H), chan_order=irmv.CH_BAYER_RGGB, max_batch=1, device=local_rank)
        e1.enable_pnp(K_CAM, D_CAM, (640.0 / SRC_W, 480.0 / SRC_H))
        e1.get_src_image_buffer(0)[...] = hosts[0][0]
        for _ in range(50):
            e1.detect(0)
        wall, devt = [], []
        for _ in range(1000):
            t0 = time.perf_counter()
            e1.detect(0)
            wall.append((time.perf_counter() - t0) * 1e6)
            devt.append(e1.last_device_ms() * 1e3)
        lat = {"p50_us_e2e_host_frame": statistics.median(wall), "p99_us_e2e_host_frame": sorted(wall)[989],
               "p50_us_device_graph": statistics.median(devt), "p99_us_device_graph": sorted(devt)[989], "iters": 1000,
               "note": "detect(): H2D of one 1.31 MB Bayer frame + CUDA graph + D2H + parse, single stream"}
        e1.close()
    except Exception as ex:                              # latency is a secondary key; never lose the line
        lat = {"error": str(ex)}

    # ---- CPU baseline on a bounded sample (rank 0, N=1 only) ------------------------------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            threads = os.cpu_count() or 1
            ref = CpuReference(wpath, threads)
            fps, n, dt = ref.run(hosts[0], budget_s=args.cpu_budget)
            cpu = {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                   "sample": f"{n} of the step's 256 Bayer frames in {dt:.1f} s; cv2 demosaic+flip+resize, "
                             f"{ref.kind_net} YOLOv8n FP32, cv2 NMSBoxesBatched, cv2.solvePnP(IPPE)"}
        except Exception as ex:
            cpu = {"value": None, "unit": "frames/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex}"}

    cfg = workload_config(B, sub_batch, lanes)
    cfg.update({"detections_per_step": n_dets, "wall_ms_per_step": wall_ms / args.steps, "host_cores_of_this_rank": len(mine) or None})
    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": cfg,
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": e2e_ms, "steps": e2e_steps, "batches_in_flight": inflight, "sync_call_ms_per_step": sync_ms,
                "h2d_ceiling": {"ms_per_step": ceil_ms, "gbs_per_gpu": ceil_gbs, "frames_per_s": ceil_fps,
                                "streams": ceil_streams,
                                "how": "cudaMemcpyAsync of the same pinned 256-frame buffers, no kernels, all ranks at once, max over "
                                       "ranks; the faster of one stream and two streams (half a buffer each)"},
                "frac_of_h2d_ceiling": e2e_value / ceil_fps,
                "note": "submit_batch()/collect_arrays() on pinned host frames: per step H2D of 256 frames + pipeline + D2H of "
                        "detections, poses, quaternions, distances + parse; bytes are counted by the engine from the copies it "
                        "queues; sync_call = detect_batch_arrays()"},
        "gpu_launches": eng.kernel_launches(B) * args.steps,
        "clock_warmup": clock_warm,
        "clocks": clocks, "roofline": roofline, "latency_batch1": lat,
    }
    if cpu is not None:
        line["cpu_baseline"] = cpu
    eng.close()
    extra = {}
    if world == 1 and not args.no_extras:
        for name, fn in (("pnp_stress", lambda: pnp_stress()),
                         ("reference_protocol_ms", lambda: reference_protocol(wpath)),
                         ("full_node_path", lambda: full_node_path(wpath, local_rank, 5)),
                         ("kpt_variant_batch64", lambda: kpt_variant(local_rank))):
            try:
                extra[name] = fn()
            except Exception as ex:
                extra[name] = {"error": str(ex)}
        # ---- light-bar / armor extraction stage (SURVEY.md section 8f row 1) on its own workload, the cv2 chain
        #      of the reference on the host cores beside it
        if not args.no_cpu_baseline:
            try:
                sys.path.insert(0, os.path.join(ROOT, "scripts"))
                import bench_armors
                extra["armor_stage"] = bench_armors.measure(32, 10)
            except Exception as ex:
                extra["armor_stage"] = {"error": str(ex)}
    line["extra_keys"] = extra
    emit(line)


def kpt_variant(local_rank: int):
    """BASELINE.json configs[2]: the keypoint variant at batch 64 on one B200 (one 64-frame replay per step,
    packed RGB frames, device resident)."""
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth, weights
    out = {}
    for arch in getattr(weights, "KPT_ARCHS", ("yolov8n-pose",)):
        path = scratch_path(f"{arch}.irmw")
        if arch == "yolov8n-pose":
            weights.write_random(path, 0, pose=True)
        else:
            weights.write_random(path, 0, arch=arch)
        fr = torch.from_numpy(synth.frames_from_base(synth.load_base(), 64, seed=2)).cuda()
        eng = irmv.YoloEngine(path, (SRC_W, SRC_H), max_batch=64, sub_batch=64, num_lanes=1, device=local_rank)
        eng.enable_pnp(K_CAM, D_CAM, (640.0 / SRC_W, 480.0 / SRC_H))
        for _ in range(5):
            eng.enqueue_batch_device(fr.data_ptr(), 64)
            eng.sync()
        ms = [0.0] * 20
        for i in range(20):
            eng.enqueue_batch_device(fr.data_ptr(), 64)
            ms[i] = eng.sync()
        k, st = eng.profile_stages(fr.data_ptr(), 64)
        out[arch] = {"frames_per_s": 64 / (statistics.median(ms) * 1e-3), "ms_per_64_frames": statistics.median(ms),
                     "stage_ms": st, "launches_per_replay": eng.kernel_launches(64), "keypoints": eng.has_keypoints()}
        eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--sub-batch", type=int, default=0)
    ap.add_argument("--lanes", type=int, default=0)
    ap.add_argument("--ref-frames", type=int, default=8, help="frames of each step the reference arm actually runs (bounded sample)")
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra_keys measurements (PnP stress, reference protocol, ...)")
    ap.add_argument("--clock-warmup-s", type=float, default=1.0, help="untimed clock ramp before the --warmup steps")
    ap.add_argument("--inflight", type=int, default=3, help="batches in flight in the end-to-end loop (1..3)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    quiet_stdout()
    try:
        if args.impl == "reference":
            run_reference(args)
        else:
            run_ours(args)
    finally:
        try:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                dist.destroy_process_group()
        except Exception:
            pass


if __name__ == "__main__":
    main()
