"""plot_dgp's labelled video rendered in the estimate_pose pass (dgp_estimate_pose_stream_render): frames/s of the fused pass
against estimate_pose alone and against the reference's shape (estimate_pose, then a second pass that draws on the host),
plus the marker kernel's time per batch.  configs[1] (747x832, 4 joints, fp16), pinned cyclic source as bench.py's e2e arm.
Writes one JSON file (default profiles/r07_bench_render.json).

    python tools/bench_render.py [--out PATH] [--frames 10000] [--encode-frames 1500] [--rounds 3]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import make_frame_pool  # noqa: E402
from deepgraphpose_b200 import synthetic  # noqa: E402
from deepgraphpose_b200.engine import Engine, marker_colors, suggest_batch  # noqa: E402

H, W, NJ = 747, 832, 4


def gpu_info():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    name, power, clock = [v.strip() for v in out.stdout.strip().split(",")] if out.returncode == 0 else ("?", "?", "?")
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi_name": name, "power_limit": power, "max_sm_clock": clock}


def host_draw(frame, x, y, lik, dotsize, thr, colors):
    """One frame drawn with numpy on the host (the drawing contract, disc by disc over its bounding box)."""
    h, w, _ = frame.shape
    for j in range(x.shape[0]):
        if not lik[j] > thr or np.isnan(x[j]) or np.isnan(y[j]):
            continue
        xc, yc = int(min(np.trunc(x[j]), w - 1)), int(min(np.trunc(y[j]), h - 1))
        r0, r1, c0, c1 = max(yc - dotsize + 1, 0), min(yc + dotsize, h), max(xc - dotsize + 1, 0), min(xc + dotsize, w)
        if r0 >= r1 or c0 >= c1:
            continue
        rr, cc = np.ogrid[r0:r1, c0:c1]
        m = (rr - yc) ** 2 + (cc - xc) ** 2 < dotsize * dotsize
        frame[r0:r1, c0:c1][m] = colors[j]


def kernel_ms(nj, dotsize, B, launches):
    eng = Engine(nj, location_refinement=False)
    try:
        g = torch.Generator(device="cuda").manual_seed(nj)
        frames = torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8, device="cuda", generator=g)
        x = torch.rand((B, nj), dtype=torch.float64, device="cuda", generator=g) * (W - 1)
        y = torch.rand((B, nj), dtype=torch.float64, device="cuda", generator=g) * (H - 1)
        lik = torch.ones((B, nj), dtype=torch.float64, device="cuda")
        for _ in range(5):
            eng.draw_markers(frames, x, y, lik, dotsize, 0.1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # a ~50 ms spin ahead of the timed window lets the host enqueue every launch first, so the events bracket device
        # time only and not the Python cost of each draw_markers call
        torch.cuda._sleep(100_000_000)
        a.record()
        for _ in range(launches):
            eng.draw_markers(frames, x, y, lik, dotsize, 0.1)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / launches
    finally:
        eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_bench_render.json"))
    ap.add_argument("--frames", type=int, default=10000)
    ap.add_argument("--encode-frames", type=int, default=1500, help="frames of arm (c): the mp4v encoder is the bound")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--launches", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import cv2
    res = {"gpu": gpu_info()}
    B = suggest_batch(H, W, 24, 48)
    eng = Engine(NJ, location_refinement=False, precision="fp16")
    eng.load_weights(synthetic.make_weights(NJ, seed=0, location_refinement=False))
    pool = torch.from_numpy(make_frame_pool(4 * B, seed=1234, h=H, w=W, nj=NJ)).pin_memory()
    P = pool.shape[0]
    colors = marker_colors(NJ)
    dotsize, thr = 3, 0.1
    tmp = tempfile.mkdtemp(prefix="bench_render_")

    def arm_a(n):
        return eng.estimate_pose_stream(pool, H, W, n, batch=B)

    def arm_b(n):
        return eng.estimate_pose_render_stream(pool, H, W, n, lambda fr: None, dotsize, thr, batch=B)

    def arm_c(n):
        vw = cv2.VideoWriter(os.path.join(tmp, "labeled.mp4"), cv2.VideoWriter_fourcc(*"mp4v"), 30.0, (W, H))
        assert vw.isOpened()

        def write(fr):
            for f in fr:
                vw.write(np.ascontiguousarray(f[:, :, ::-1]))

        try:
            return eng.estimate_pose_render_stream(pool, H, W, n, write, dotsize, thr, batch=B)
        finally:
            vw.release()

    def arm_d(n):
        mu, peak, lik = arm_a(n)
        m = mu.numpy().astype(np.float64)
        x, y = m[:, :, 1] * eng.stride + 0.5 * eng.stride, m[:, :, 0] * eng.stride + 0.5 * eng.stride
        lk = lik.numpy().astype(np.float64)
        src = pool.numpy()
        for t in range(n):
            fr = src[t % P].copy()   # stands in for the second decode of the reference
            host_draw(fr, x[t], y[t], lk[t], dotsize, thr, colors)
        return mu, peak, lik

    arms = {"a_stream": (arm_a, args.frames), "b_render_discard": (arm_b, args.frames),
            "c_render_mp4v": (arm_c, args.encode_frames), "d_stream_then_host_draw": (arm_d, args.frames)}
    for name, (fn, _) in arms.items():  # warm-up: plans, rings, writer slots, encoder
        fn(4 * B)
    torch.cuda.synchronize()
    runs = {k: [] for k in arms}
    outputs = {}
    for r in range(args.rounds):
        for name, (fn, n) in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = fn(n)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            runs[name].append(n / dt)
            outputs[name] = out
    res["arms"] = {k: {"frames": arms[k][1], "fps_per_round": v, "fps_median": float(np.median(v))} for k, v in runs.items()}
    a_fps, b_fps = res["arms"]["a_stream"]["fps_median"], res["arms"]["b_render_discard"]["fps_median"]
    res["render_over_stream"] = b_fps / a_fps
    res["render_equals_stream"] = all(torch.equal(p, q) for p, q in zip(outputs["a_stream"], outputs["b_render_discard"]))
    res["d2h_bytes_per_frame"] = H * W * 3
    res["d2h_GB_per_s_at_b"] = b_fps * H * W * 3 / 1e9
    res["mp4v_bytes_per_frame"] = os.path.getsize(os.path.join(tmp, "labeled.mp4")) / args.encode_frames
    shutil.rmtree(tmp, ignore_errors=True)
    eng.close()
    res["marker_kernel"] = [{"nj": nj, "dotsize": d, "batch": B, "frame": [H, W], "launches": args.launches,
                             "ms_per_batch": kernel_ms(nj, d, B, args.launches)} for nj in (4, 20) for d in (3, 10)]
    res["config"] = {"frame": [H, W, 3], "num_joints": NJ, "precision": "fp16", "batch": B, "pool_frames": P,
                     "dotsize": dotsize, "mask_threshold": thr, "host_threads": torch.get_num_threads()}
    res["notes"] = ("arms run alternately, %d rounds, wall clock around each synchronous call. a: Engine.estimate_pose_stream "
                    "on a pinned cyclic source (frame t = pool[t %% %d]); b: Engine.estimate_pose_render_stream on the same "
                    "source with a writer that discards the frames (markers + D2H of every frame + writer hand-off); c: b with "
                    "a cv2.VideoWriter mp4v writer (single-threaded encoder) into a temporary directory, on %d frames; d: a, "
                    "then a host pass that copies each frame out of the pool (standing in for the second decode) and draws it "
                    "with numpy. marker kernel: CUDA events over %d back-to-back launches of dgp_draw_markers on one batch (queued "
                    "behind a device spin, so host enqueue time is excluded), centres inside the frame, every joint drawn." % (args.rounds, P, args.encode_frames, args.launches))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
