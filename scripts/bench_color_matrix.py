"""Cost of the colour-correction stage (YoloEngine.set_color_matrix) on the bench workload.

`python scripts/bench_color_matrix.py OUT_DIR [--rounds 5] [--steps 20]` runs, in one process, three arms that differ
only in their colour stages and alternates them round by round:
  * off: no table, no matrix (bench.py's configuration);
  * raw: the raw table alone (black level 8, gains 1.9 / 1.0 / 1.6, gamma 1/2.2);
  * colour: the ISP order -- raw table with gamma 1, then a colour-correction matrix at saturation 1.4, then the
    gamma 1/2.2 tone table.
For each arm:
  * the 256-frame device-resident step of bench.py's configuration (Bayer RGGB 1280x1024, one 256-frame replay,
    fused PnP): device ms per step from the engine's CUDA events;
  * the preprocess stage (camera-case stem) of profile_stages on the same frames;
  * the fused armor stage on seeded light-bar scenes (profile_stages' last stage: extract_armors + PnP on the
    armor corners, 64 frames).
Prints the GPU name and power limit read in the same run and writes OUT_DIR/bench_color_matrix.json."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import raw_lut, synth
    import bench
    if not torch.cuda.is_available():
        raise SystemExit("bench_color_matrix.py needs a CUDA device")
    os.makedirs(args.out_dir, exist_ok=True)
    info = gpu_info()
    print("GPU:", info, flush=True)
    lut = raw_lut.make_raw_lut(8, (1.9, 1.0, 1.6), 1 / 2.2)
    lut_lin = raw_lut.make_raw_lut(8, (1.9, 1.0, 1.6), 1.0)
    ccm = np.array([[1.55, -0.35, -0.20], [-0.25, 1.45, -0.20], [-0.05, -0.45, 1.50]])
    m = raw_lut.color_matrix_q10(ccm, saturation=1.4)
    tone = raw_lut.make_raw_lut(0, (1, 1, 1), 1 / 2.2)
    wpath = bench.weights_file(0)
    B = 256
    frames = bench.make_bayer_frames_device(B, seed=0, device=torch.device("cuda", 0))
    # light-bar scenes as an RGGB camera would write them (rotated view -> camera frame -> mosaic)
    NA = 64
    scenes = np.stack([synth.bayer_from_rgb(np.ascontiguousarray(synth.armor_scene(10, 1000 + f)[0][::-1, ::-1]), "RGGB")
                       for f in range(NA)])
    scenes_dev = torch.from_numpy(scenes).cuda()
    arms = {}
    for arm in ("off", "raw", "colour"):
        e = irmv.YoloEngine(wpath, (bench.SRC_W, bench.SRC_H), chan_order=irmv.CH_BAYER_RGGB, max_batch=B, sub_batch=B,
                            num_lanes=1)
        e.enable_pnp(bench.K_CAM, bench.D_CAM, (640.0 / bench.SRC_W, 480.0 / bench.SRC_H))
        a = irmv.YoloEngine(wpath, (bench.SRC_W, bench.SRC_H), chan_order=irmv.CH_BAYER_RGGB, max_batch=NA, sub_batch=NA,
                            num_lanes=1)
        a.enable_armors()
        a.enable_pnp(bench.K_CAM, bench.D_CAM, (640.0 / bench.SRC_W, 480.0 / bench.SRC_H))
        for eng in (e, a):
            if arm == "raw":
                eng.set_raw_lut(lut)
            elif arm == "colour":
                eng.set_raw_lut(lut_lin)
                eng.set_color_matrix(m, tone)
        arms[arm] = (e, a)
    stem_ctas = {arm: e.stem_camera_ctas() for arm, (e, a) in arms.items()}
    print("camera-kernel CTAs per SM:", stem_ctas, flush=True)
    res = {arm: {"step_ms": [], "preprocess_ms": [], "armor_stage_ms": []} for arm in arms}
    for _ in range(args.rounds):
        for arm, (e, a) in arms.items():
            for _ in range(3):                   # warm: graphs, clocks
                e.enqueue_batch_device(frames.data_ptr(), B)
                e.sync()
            for _ in range(args.steps):
                e.enqueue_batch_device(frames.data_ptr(), B)
                res[arm]["step_ms"].append(e.sync())
            for _ in range(3):
                res[arm]["preprocess_ms"].append(e.profile_stages(frames.data_ptr(), B)[1]["preprocess"])
                res[arm]["armor_stage_ms"].append(a.profile_stages(scenes_dev.data_ptr(), NA)[1]["pnp"])
    counts = {}
    for arm, (e, a) in arms.items():
        c, _ = a.detect_batch_arrays(scenes)
        counts[arm] = {"detections": int(c.sum()), "armors": int(a.fetch_armors(NA)["valid"].sum())}
    out = {
        "gpu": info,
        "arms": {"off": "no colour stage",
                 "raw": "raw table: black level 8, gains (1.9, 1.0, 1.6), gamma 1/2.2",
                 "colour": "raw table (black level 8, gains (1.9, 1.0, 1.6), gamma 1) + matrix "
                           f"{m.tolist()} (1/1024 units: CCM at saturation 1.4) + tone table gamma 1/2.2"},
        "stem_camera_ctas": stem_ctas,
        "workload": {"step": f"{B} device-resident 1280x1024 RGGB frames, one {B}-frame replay, fused PnP (bench.py)",
                     "armor_stage": f"{NA} seeded light-bar scenes (synth.armor_scene, RGGB), extract_armors + PnP"},
        "rounds": args.rounds, "steps_per_round": args.steps,
        **{arm: {k: summary(v) for k, v in res[arm].items()} for arm in arms},
        "armor_scene_counts": counts,
    }
    for arm in ("raw", "colour"):
        out[f"{arm}_over_off_median"] = {k: out[arm][k]["median"] / out["off"][k]["median"] for k in res["off"]}
    out["colour_over_raw_median"] = {k: out["colour"][k]["median"] / out["raw"][k]["median"] for k in res["off"]}
    with open(os.path.join(args.out_dir, "bench_color_matrix.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))
    for e, a in arms.values():
        e.close(); a.close()


if __name__ == "__main__":
    main()
