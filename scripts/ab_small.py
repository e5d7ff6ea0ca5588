"""A/B helper for small replays: median device time of a graph replay of n frames of the bench workload (n = 1, 2, 3,
4, 8, or the list in AB_SIZES), for comparing two builds.  usage: python scripts/ab_small.py [label]"""
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import irmv_detection_b200 as irmv
    import bench
    label = sys.argv[1] if len(sys.argv) > 1 else ""
    w = bench.weights_file(0)
    out = []
    for n in [int(v) for v in os.environ.get("AB_SIZES", "1,2,3,4,8").split(",")]:
        fr = bench.make_bayer_frames_device(n, seed=0, device=torch.device("cuda:0"))
        eng = irmv.YoloEngine(w, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB, max_batch=n, sub_batch=n, num_lanes=1)
        eng.enable_pnp(bench.K_CAM, bench.D_CAM, (0.5, 480 / 1024))
        ms = []
        for i in range(300):
            eng.enqueue_batch_device(fr.data_ptr(), n)
            t = eng.sync()
            if i >= 100:
                ms.append(t)
        out.append(f"n={n}: {statistics.median(ms) * 1e3:.1f} us")
        eng.close()
    print(f"{label:16s}", "  ".join(out))


if __name__ == "__main__":
    main()
