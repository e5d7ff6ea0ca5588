"""Bring-up diagnostics on a B200: stage-by-stage and layer-by-layer errors of the CUDA path
against the CPU oracle, for both convolution kernels.  Writes gpurun_out/diag.log."""
import json
import os
import sys
import time
import traceback

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
LOG = open(os.path.join(ROOT, "gpurun_out", "diag.log"), "w")


def log(*a):
    s = " ".join(str(x) for x in a)
    print(s, flush=True)
    LOG.write(s + "\n")
    LOG.flush()


def section(name, fn):
    log(f"==== {name}")
    t0 = time.time()
    try:
        fn()
        log(f"---- {name} ok ({time.time() - t0:.1f}s)")
    except Exception:
        log(f"---- {name} FAILED\n{traceback.format_exc()}")


def main():
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth, weights
    from oracle import nms_ref as N, pnp_ref as P, preprocess_ref as PR, yolov8n_ref as Y
    log("cuda", torch.cuda.is_available(), torch.cuda.get_device_name(0) if torch.cuda.is_available() else "-")
    base = synth.load_base()
    fr = np.stack([base] + list(synth.frames_from_base(base, 2, seed=11)))
    wpath = "/tmp/diag_seed0.irmw"
    weights.write_random(wpath, 0)

    def pre():
        got = irmv.preprocess(fr[:2])
        for i in range(2):
            ref, _ = PR.preprocess_fp16(fr[i])
            d = got[i, :, :, :3].astype(np.float32) - ref.transpose(1, 2, 0).astype(np.float32)
            log("preprocess frame", i, "mismatching elements", int((d != 0).sum()), "max abs", float(np.abs(d).max()))
    section("preprocess", pre)

    def pnp():
        q = P.synth_quads(5000, seed=2)
        s = irmv.PnPSolver(P.K_DEFAULT, P.D_DEFAULT)
        rv, tv, ok = s.solve_batch(q)
        r1, t1 = P.solve_ippe(q)
        rel = np.linalg.norm(rv - r1, axis=1) / np.linalg.norm(r1, axis=1)
        log("pnp ok", bool(ok.all()), "median rel", float(np.median(rel)), "p99", float(np.quantile(rel, 0.99)), "max", float(rel.max()),
            "n>1e-4", int((rel > 1e-4).sum()), "kernel ms", s.last_device_ms())
    section("pnp", pnp)

    def nms():
        rng = np.random.default_rng(0)
        b = rng.uniform(0, 500, (8400, 4)).astype(np.float32)
        b[:, 2:] = b[:, :2] + rng.uniform(20, 200, (8400, 2)).astype(np.float32)
        s = (rng.random((8400, 14)) ** 8).astype(np.float32)
        (gi, gb, gs, gc), = irmv.nms(b[None], s[None])
        ri, rb, rs, rc = N.nms(b, s)
        log("nms cands", int((s > 0.25).sum()), "gpu kept", gi.size, "oracle kept", ri.size, "equal", bool(np.array_equal(gi, ri)))
    section("nms", nms)

    oracle = Y.build(wpath)

    def net(impl):
        eng = irmv.YoloEngine(wpath, (1280, 1024), max_batch=3, sub_batch=3, conv_impl=impl, use_graph=False)
        t0 = time.time()
        dets = eng.detect_batch(fr)
        log("impl", impl, "first batch wall", round(time.time() - t0, 3), "s; device ms", eng.last_device_ms(), "dets", [len(d) for d in dets])
        x = irmv.preprocess(fr)
        taps = {}
        with torch.no_grad():
            xin = torch.from_numpy(x[..., :3].astype(np.float32)).permute(0, 3, 1, 2).contiguous()
            outs = oracle.features(xin, taps)
            rboxes, rscores = Y.decode_heads(outs)
        for name, ref in taps.items():
            try:
                got = eng.read_tensor(name).astype(np.float32)
            except RuntimeError:
                log(f"  {name:4s} not materialised (fused into its consumer)")
                continue
            ref = ref.permute(0, 2, 3, 1).numpy()
            err = np.abs(got - ref)
            log(f"  {name:4s} max err {err.max():.4f} mean err {err.mean():.5f} ref absmax {np.abs(ref).max():.2f} nan {int(np.isnan(got).sum())}")
        for i in range(3):
            for nm, (rb, rc) in zip((f"box{i}", f"cls{i}"), [(outs[i][0], None), (None, outs[i][1])]):
                got = eng.read_tensor(nm).astype(np.float32)
                ref = (rb if rb is not None else rc).permute(0, 2, 3, 1).numpy()
                got = got[..., :ref.shape[-1]]
                log(f"  {nm} max err {np.abs(got - ref).max():.4f} ref absmax {np.abs(ref).max():.2f}")
        box = np.concatenate([eng.read_tensor(f"box{i}").reshape(3, -1, 64) for i in range(3)], 1)
        cls = np.concatenate([eng.read_tensor(f"cls{i}").reshape(3, -1, 16) for i in range(3)], 1)
        gb, gs = irmv.decode(box, cls)
        log("  decoded boxes max err px", float(np.abs(gb - rboxes.numpy()).max()), "scores max err", float(np.abs(gs - rscores.numpy()).max()))
        for f in range(3):
            ri, _, _, _ = N.nms(gb[f], gs[f])
            oi, _, _, _ = N.nms(rboxes[f].numpy(), rscores[f].numpy())
            ki = eng.kept_indices(f)
            log(f"  frame {f}: gpu kept {ki.size} oracle-on-gpu-inputs {ri.size} equal {bool(np.array_equal(ki, ri))}; fp32 oracle kept {oi.size} common {len(set(ki.tolist()) & set(oi.tolist()))}")
        # timing: a few more batches
        for _ in range(3):
            eng.detect_batch(fr)
        log("  steady device ms per 3 frames (no graph):", eng.last_device_ms())
        eng.close()
    section("network direct", lambda: net(irmv.CONV_DIRECT))
    section("network tcgen05", lambda: net(irmv.CONV_TCGEN05))


if __name__ == "__main__":
    main()
