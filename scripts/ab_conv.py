"""A/B helper: conv-stage and total device time of one replay of the bench workload (1280x1024 Bayer frames, PnP on;
median of 7 eager stage profiles), for comparing two builds.  usage: python scripts/ab_conv.py [frames] [label]"""
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import irmv_detection_b200 as irmv
    import bench
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 256
    label = sys.argv[2] if len(sys.argv) > 2 else ""
    w = bench.weights_file(0)
    fr = bench.make_bayer_frames_device(n, seed=0, device=torch.device("cuda:0"))
    eng = irmv.YoloEngine(w, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB, max_batch=n, sub_batch=n, num_lanes=1)
    eng.enable_pnp(bench.K_CAM, bench.D_CAM, (0.5, 480 / 1024))
    for _ in range(30):                                   # clock ramp
        eng.enqueue_batch_device(fr.data_ptr(), n)
        eng.sync()
    conv, tot = [], []
    for _ in range(7):
        k, st = eng.profile_stages(fr.data_ptr(), n)
        conv.append(st["conv"]); tot.append(st["total"])
    print(f"{label:28s} frames {k}: conv {statistics.median(conv):.4f} ms  total {statistics.median(tot):.4f} ms")
    eng.close()


if __name__ == "__main__":
    main()
