"""Cost of 10/12-bit raw sources (raw_format RAW_12 and RAW_12_PACKED against RAW_8) on the bench workload.

`python scripts/bench_raw_bits.py OUT_DIR [--rounds 5] [--steps 20] [--e2e-steps 10]` builds, in one process, three
engines in bench.py's configuration (Bayer RGGB 1280x1024, one 256-frame replay, fused PnP) that differ only in
raw_format, and alternates them round by round:
  * the 256-frame device-resident step: device ms per step from the engine's CUDA events;
  * the preprocess stage of profile_stages (decode + camera-case stem for the 12-bit engines);
  * the pipelined host path with three batches in flight (submit_batch / collect_arrays on pinned frames):
    end-to-end frames/s and H2D bytes per step.
The 12-bit frames are (8-bit bench frames << 4) | seeded noise, so all three engines see the same picture.  A separate
torch.profiler pass (after the timed rounds) gives the decode kernel's own device time; its bytes (12-bit samples
read, 8-bit mosaic written) over that time are reported as a share of the HBM bandwidth bench.py uses
(MEASURED_PEAKS.json when present, else its fallback figure).  Prints the GPU name and power limit read in the same
run and writes OUT_DIR/bench_raw_bits.json."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))


def widen(frames8, fmt, seed):
    """u8 [n, H, W] device mosaics -> device frames of `fmt` (u8 bytes, the layout the engine takes)."""
    import torch
    import irmv_detection_b200 as irmv
    if fmt == irmv.RAW_8:
        return frames8
    g = torch.Generator(device=frames8.device)
    g.manual_seed(seed)
    raw = (frames8.to(torch.int32) << 4) | torch.randint(0, 16, frames8.shape, generator=g, device=frames8.device,
                                                         dtype=torch.int32)
    if fmt == irmv.RAW_12:
        return raw.to(torch.int16).contiguous().view(torch.uint8).view(raw.shape[0], raw.shape[1], -1)
    p0, p1 = raw[..., 0::2], raw[..., 1::2]
    packed = torch.stack([p0 >> 4, (p1 & 15) << 4 | (p0 & 15), p1 >> 4], -1).to(torch.uint8)
    return packed.reshape(raw.shape[0], raw.shape[1], -1).contiguous()


def kernel_device_us(prof, name):
    """Mean device time (us) of the kernels whose name contains `name` in a torch.profiler capture."""
    for evt in prof.key_averages():
        if name in evt.key:
            total = getattr(evt, "device_time_total", None)
            if total is None:
                total = evt.cuda_time_total
            return total / max(evt.count, 1), evt.count
    return None, 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--e2e-steps", type=int, default=10)
    args = ap.parse_args()
    import torch
    import irmv_detection_b200 as irmv
    import bench
    from bench_raw_lut import gpu_info, summary
    if not torch.cuda.is_available():
        raise SystemExit("bench_raw_bits.py needs a CUDA device")
    os.makedirs(args.out_dir, exist_ok=True)
    info = gpu_info()
    print("GPU:", info, flush=True)
    peaks, peak_kind = bench.measured_peaks()
    hbm_gbs = float(peaks.get("hbm_gbs", 6650.0))
    wpath = bench.weights_file(0)
    B, W, H = 256, bench.SRC_W, bench.SRC_H
    dev = torch.device("cuda", 0)
    frames8 = bench.make_bayer_frames_device(B, seed=0, device=dev)
    formats = {"raw8": irmv.RAW_8, "raw12": irmv.RAW_12, "raw12_packed": irmv.RAW_12_PACKED}
    arms = {}
    for name, fmt in formats.items():
        e = irmv.YoloEngine(wpath, (W, H), chan_order=irmv.CH_BAYER_RGGB, max_batch=B, sub_batch=B, num_lanes=1,
                            raw_format=fmt)
        e.enable_pnp(bench.K_CAM, bench.D_CAM, (640.0 / W, 480.0 / H))
        fr = widen(frames8, fmt, seed=7)
        hosts = []
        for _ in range(3):
            h = torch.empty(fr.shape, dtype=torch.uint8, pin_memory=True)
            h.copy_(fr)
            hn = h.numpy()
            hosts.append(hn.view(np.uint16) if fmt in (irmv.RAW_10, irmv.RAW_12) else hn)
        torch.cuda.synchronize()
        arms[name] = {"eng": e, "frames": fr, "hosts": hosts}
    # the three engines must agree on what they detect (the 12-bit frames decode to the 8-bit ones)
    ref = arms["raw8"]["eng"].detect_batch_device(arms["raw8"]["frames"].data_ptr(), B)
    same = {n: a["eng"].detect_batch_device(a["frames"].data_ptr(), B) == ref for n, a in arms.items()}
    print("same detections as RAW_8:", same, flush=True)
    res = {n: {"step_ms": [], "preprocess_ms": [], "e2e_frames_per_s": [], "h2d_bytes_per_step": []} for n in arms}
    for _ in range(args.rounds):
        for n, a in arms.items():
            e, fr, hosts = a["eng"], a["frames"], a["hosts"]
            for _ in range(3):                   # warm: graphs, clocks
                e.enqueue_batch_device(fr.data_ptr(), B)
                e.sync()
            for _ in range(args.steps):
                e.enqueue_batch_device(fr.data_ptr(), B)
                res[n]["step_ms"].append(e.sync())
            for _ in range(3):
                res[n]["preprocess_ms"].append(e.profile_stages(fr.data_ptr(), B)[1]["preprocess"])
            for _ in range(3):                   # warm the pipelined path (all three result sets)
                e.collect_arrays(e.submit_batch(hosts[0]), poses=True)
            pending = [e.submit_batch(hosts[i]) for i in range(2)]
            h0 = e.copy_bytes()[0]
            t0 = time.perf_counter()
            for i in range(args.e2e_steps):
                pending.append(e.submit_batch(hosts[(i + 2) % 3]))
                e.collect_arrays(pending.pop(0), poses=True)
            dt = time.perf_counter() - t0
            h1 = e.copy_bytes()[0]
            while pending:
                e.collect_arrays(pending.pop(0), poses=True)
            res[n]["e2e_frames_per_s"].append(B * args.e2e_steps / dt)
            res[n]["h2d_bytes_per_step"].append((h1 - h0) // args.e2e_steps)
    # decode kernel on its own: a profiler pass of its own, after the timed rounds
    decode = {}
    from torch.profiler import ProfilerActivity, profile
    for n in ("raw12", "raw12_packed"):
        e, fr = arms[n]["eng"], arms[n]["frames"]
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(10):
                e.enqueue_batch_device(fr.data_ptr(), B)
                e.sync()
        us, count = kernel_device_us(prof, "raw_decode_kernel")
        moved = B * W * H * ((2.0 if n == "raw12" else 1.5) + 1.0)
        decode[n] = {"kernel_us": us, "launches_seen": count, "bytes": moved,
                     "gbs": moved / (us * 1e-6) / 1e9 if us else None,
                     "hbm_frac": moved / (us * 1e-6) / 1e9 / hbm_gbs if us else None}
    out = {
        "gpu": info,
        "workload": f"{B} device-resident 1280x1024 RGGB frames, one {B}-frame replay, fused PnP (bench.py); "
                    "12-bit frames = (8-bit frames << 4) | noise; pipelined: submit_batch/collect_arrays, 3 in flight",
        "hbm_peak_gbs": hbm_gbs, "hbm_peak_source": peak_kind,
        "rounds": args.rounds, "steps_per_round": args.steps, "e2e_steps_per_round": args.e2e_steps,
        "same_detections_as_raw8": same,
        "arms": {n: {k: summary(v) for k, v in r.items()} for n, r in res.items()},
        "decode_kernel": decode,
    }
    base = out["arms"]["raw8"]
    out["over_raw8_median"] = {n: {k: out["arms"][n][k]["median"] / base[k]["median"] for k in base}
                               for n in ("raw12", "raw12_packed")}
    with open(os.path.join(args.out_dir, "bench_raw_bits.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))
    for a in arms.values():
        a["eng"].close()


if __name__ == "__main__":
    main()
