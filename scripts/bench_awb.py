"""Cost of automatic white balance (YoloEngine.set_auto_white_balance) on the bench workload.

`python scripts/bench_awb.py OUT_DIR [--rounds 5] [--steps 20] [--detects 300]` runs, in one process, four arms that
differ only in their colour stages and alternates them round by round:
  * off: no colour stage (bench.py's configuration);
  * matrix: a fixed colour-correction matrix (saturation 1.3) and a gamma 1/2.2 tone table;
  * awb: auto white balance with the default parameters;
  * awb_matrix: auto white balance composed with the same matrix and tone table.
For each arm:
  * the 256-frame device-resident step of bench.py's configuration (Bayer RGGB 1280x1024, one 256-frame replay,
    fused PnP): device ms per step from the engine's CUDA events;
  * the preprocess stage of profile_stages on the same frames (statistics kernel + camera-case stem);
and for the AWB arms the statistics kernel's own time (torch.profiler over profile_stages replays, in a separate
pass), with the bytes it must read (every 8-bit sample of every frame once) over that time as a share of the HBM
bandwidth of NVIDIA's B200 data sheet (7.7 TB/s).  Batch-1 detect() (host ms per call, p50) with AWB on and off.
Prints the GPU name and power limit read in the same run and writes OUT_DIR/bench_awb.json."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12


def gpu_info() -> dict:
    import torch
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(r.stdout.strip().splitlines()[0])
    except Exception as exc:                    # reported, not guessed
        info["power_limit_error"] = repr(exc)
    return info


def summary(v):
    return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v)), "n": len(v)}


def awb_kernel_us(eng, ptr, n, reps, trace_dir):
    """Device time of the statistics kernel (awb_kernel) per replay, from a torch.profiler trace of profile_stages."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    eng.profile_stages(ptr, n)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            eng.profile_stages(ptr, n)
        torch.cuda.synchronize()
    prof.export_chrome_trace(os.path.join(trace_dir, "bench_awb.pt.trace.json"))
    times = [e.device_time for e in prof.events() if "awb_kernel" in e.name]
    if len(times) != reps:
        raise RuntimeError(f"expected {reps} awb_kernel launches in the trace, found {len(times)}")
    return times


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--detects", type=int, default=300)
    args = ap.parse_args()
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import raw_lut
    import bench
    if not torch.cuda.is_available():
        raise SystemExit("bench_awb.py needs a CUDA device")
    os.makedirs(args.out_dir, exist_ok=True)
    info = gpu_info()
    print("GPU:", info, flush=True)
    ccm = np.array([[1.55, -0.35, -0.20], [-0.25, 1.45, -0.20], [-0.05, -0.45, 1.50]])
    m = raw_lut.color_matrix_q10(ccm, saturation=1.3)
    tone = raw_lut.make_raw_lut(0, (1, 1, 1), 1 / 2.2)
    wpath = bench.weights_file(0)
    B = 256
    W, H = bench.SRC_W, bench.SRC_H
    frames = bench.make_bayer_frames_device(B, seed=0, device=torch.device("cuda", 0))

    def configure(eng, arm):
        if arm in ("matrix", "awb_matrix"):
            eng.set_color_matrix(m, tone)
        if arm in ("awb", "awb_matrix"):
            eng.set_auto_white_balance({})

    arms = {}
    for arm in ("off", "matrix", "awb", "awb_matrix"):
        e = irmv.YoloEngine(wpath, (W, H), chan_order=irmv.CH_BAYER_RGGB, max_batch=B, sub_batch=B, num_lanes=1)
        e.enable_pnp(bench.K_CAM, bench.D_CAM, (640.0 / W, 480.0 / H))
        configure(e, arm)
        arms[arm] = e
    stem_ctas = {arm: e.stem_camera_ctas() for arm, e in arms.items()}
    print("camera-kernel CTAs per SM:", stem_ctas, flush=True)
    res = {arm: {"step_ms": [], "preprocess_ms": []} for arm in arms}
    for _ in range(args.rounds):
        for arm, e in arms.items():
            for _ in range(3):                   # warm: graphs, clocks
                e.enqueue_batch_device(frames.data_ptr(), B)
                e.sync()
            for _ in range(args.steps):
                e.enqueue_batch_device(frames.data_ptr(), B)
                res[arm]["step_ms"].append(e.sync())
            for _ in range(3):
                res[arm]["preprocess_ms"].append(e.profile_stages(frames.data_ptr(), B)[1]["preprocess"])
    kernel = {}
    for arm in ("awb", "awb_matrix"):
        us = awb_kernel_us(arms[arm], frames.data_ptr(), B, 10, args.out_dir)
        s = summary(us)
        nbytes = B * W * H
        s["bytes"] = nbytes
        s["share_of_hbm_peak_at_median"] = nbytes / (s["median"] * 1e-6) / HBM_BYTES_PER_S
        kernel[arm] = s
    gains = arms["awb"].fetch_white_balance(B)
    for e in arms.values():
        e.close()

    # batch-1 detect(): host ms per call
    host = bench.make_bayer_frames_device(1, seed=1, device=torch.device("cuda", 0)).cpu().numpy()[0]
    det = {}
    for arm in ("off", "awb"):
        e = irmv.YoloEngine(wpath, (W, H), chan_order=irmv.CH_BAYER_RGGB)
        configure(e, arm)
        e.get_src_image_buffer(0)[...] = host
        det[arm] = e
    lat = {arm: [] for arm in det}
    for _ in range(args.rounds):
        for arm, e in det.items():
            for _ in range(20):
                e.detect(0)
            for _ in range(args.detects // args.rounds):
                e.detect(0)
                lat[arm].append(e.get_profiling_time())
    for e in det.values():
        e.close()

    out = {
        "gpu": info,
        "arms": {"off": "no colour stage", "matrix": f"matrix {m.tolist()} (1/1024) + tone gamma 1/2.2",
                 "awb": "auto white balance, default parameters", "awb_matrix": "auto white balance + the same matrix and tone"},
        "stem_camera_ctas": stem_ctas,
        "workload": f"{B} device-resident {W}x{H} RGGB frames, one {B}-frame replay, fused PnP (bench.py)",
        "rounds": args.rounds, "steps_per_round": args.steps,
        **{arm: {k: summary(v) for k, v in res[arm].items()} for arm in arms},
        "awb_kernel_us": kernel,
        "awb_valid_frames": int(gains["valid"].sum()),
        "detect_batch1_host_ms": {arm: summary(v) | {"p50": float(np.percentile(v, 50))} for arm, v in lat.items()},
    }
    for arm in ("matrix", "awb", "awb_matrix"):
        out[f"{arm}_minus_off_median_ms"] = {k: out[arm][k]["median"] - out["off"][k]["median"] for k in res["off"]}
    with open(os.path.join(args.out_dir, "bench_awb.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
