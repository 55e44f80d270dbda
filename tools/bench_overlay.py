"""Skeleton lines and joint trails of the labelled video (dgp_marker_style's edges / trailpoints): the marker kernel's device
time per 31-frame batch with and without the overlay, then frames/s of the fused Motion-JPEG render pass with markers only
against skeleton + 10-frame trails, arms alternated over rounds.  configs[1] (747x832, 4 joints, fp16), pinned cyclic source
as bench.py's e2e arm.  Writes one JSON file (default profiles/r10_bench_overlay.json).

    python tools/bench_overlay.py [--out PATH] [--frames 10000] [--rounds 3] [--launches 200]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import make_frame_pool  # noqa: E402
from deepgraphpose_b200 import synthetic  # noqa: E402
from deepgraphpose_b200.engine import Engine, suggest_batch  # noqa: E402
from tools.bench_render import gpu_info  # noqa: E402

H, W, NJ = 747, 832, 4
B_KERNEL = 31
L2_BYTES = 126 * 2 ** 20


def animal_labels(rng, T, nj):
    """(T, nj) x / y of an animal-sized pose wandering over the frame: joints 20-60 px apart along a chain, a few px of
    motion per frame (so that lines are limb-length and trails overlap, as in a real video)."""
    cx = np.cumsum(rng.uniform(-4, 4, T)) + W / 2
    cy = np.cumsum(rng.uniform(-4, 4, T)) + H / 2
    off = np.cumsum(rng.uniform(20, 60, nj) * rng.choice([-1, 1], nj))
    ang = rng.uniform(0, 2 * np.pi, nj)
    x = cx[:, None] + (off * np.cos(ang))[None, :] + rng.uniform(-2, 2, (T, nj))
    y = cy[:, None] + (off * np.sin(ang))[None, :] + rng.uniform(-2, 2, (T, nj))
    return np.clip(x, 0, W - 1), np.clip(y, 0, H - 1)


def kernel_ms(nj, K, launches, dotsize=3):
    """CUDA events around `launches` dgp_draw_markers calls on 31-frame batches (with K - 1 history rows), the frames rotated
    over enough distinct batches to exceed the L2 twice."""
    nb = max(2, -(-2 * L2_BYTES // (B_KERNEL * H * W * 3)))
    rng = np.random.default_rng(nj * 100 + K)
    frames = torch.from_numpy(rng.integers(0, 256, (nb * B_KERNEL, H, W, 3), dtype=np.uint8)).cuda()
    hist = max(K - 1, 0)
    x, y = animal_labels(rng, hist + nb * B_KERNEL, nj)
    xs, ys = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    lik = torch.ones_like(xs)
    edges = [(j, j + 1) for j in range(nj - 1)] if K else None   # K = 0: the markers-only arm
    eng = Engine(nj, location_refinement=False)
    try:
        def launch(k):
            b = k % nb
            r = slice(b * B_KERNEL, b * B_KERNEL + hist + B_KERNEL)
            eng.draw_markers(frames[b * B_KERNEL:(b + 1) * B_KERNEL], xs[r], ys[r], lik[r], dotsize, 0.1, None, edges,
                             (255, 255, 255), K, hist)

        for k in range(2 * nb):
            launch(k)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # the host enqueues every launch while the device spins, so the events bracket device time only
        torch.cuda._sleep(200_000_000)
        a.record()
        for k in range(launches):
            launch(k)
        b.record()
        torch.cuda.synchronize()
        return {"nj": nj, "edges": len(edges or ()), "trailpoints": K, "dotsize": dotsize, "batch": B_KERNEL,
                "distinct_batches": nb, "launches": launches, "us_per_batch": a.elapsed_time(b) / launches * 1e3}
    finally:
        eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_bench_overlay.json"))
    ap.add_argument("--frames", type=int, default=10000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--quality", type=int, default=90)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"gpu": gpu_info()}
    res["kernel"] = [kernel_ms(nj, K, args.launches) for nj in (4, 20) for K in (0, 5, 10)]
    B = suggest_batch(H, W, 24, 48)
    eng = Engine(NJ, location_refinement=False, precision="fp16")
    eng.load_weights(synthetic.make_weights(NJ, seed=0, location_refinement=False))
    pool = torch.from_numpy(make_frame_pool(4 * B, seed=1234, h=H, w=W, nj=NJ)).pin_memory()
    dotsize, thr, q = 3, 0.1, args.quality
    chain = [(j, j + 1) for j in range(NJ - 1)]

    def markers(n):
        return eng.estimate_pose_render_stream(pool, H, W, n, lambda d, s: None, dotsize, thr, batch=B, encoder="jpeg",
                                               quality=q)

    def overlay(n):
        return eng.estimate_pose_render_stream(pool, H, W, n, lambda d, s: None, dotsize, thr, batch=B, encoder="jpeg",
                                               quality=q, edges=chain, skeleton_color=(255, 255, 255), trailpoints=10)

    arms = {"jpeg_markers_only": markers, "jpeg_skeleton_trails10": overlay}
    for fn in arms.values():   # warm-up: plans, rings, writer slots, tables, encoder
        fn(4 * B)
    torch.cuda.synchronize()
    runs = {k: [] for k in arms}
    outputs = {}
    for _ in range(args.rounds):
        for name, fn in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            outputs[name] = fn(args.frames)
            torch.cuda.synchronize()
            runs[name].append(args.frames / (time.perf_counter() - t0))
    eng.close()
    res["fused_jpeg"] = {k: {"frames": args.frames, "fps_per_round": v, "fps_median": float(np.median(v))}
                         for k, v in runs.items()}
    med = [res["fused_jpeg"][k]["fps_median"] for k in arms]
    res["overlay_over_markers"] = med[1] / med[0]
    spread = [(max(v) - min(v)) / float(np.median(v)) for v in runs.values()]
    res["run_to_run_spread"] = {k: s for k, s in zip(arms, spread)}
    res["readouts_equal"] = all(torch.equal(p, q_) for p, q_ in zip(*outputs.values()))
    res["config"] = {"frame": [H, W, 3], "num_joints": NJ, "precision": "fp16", "batch": B, "pool_frames": pool.shape[0],
                     "dotsize": dotsize, "mask_threshold": thr, "quality": q, "skeleton": chain, "trailpoints": 10}
    res["notes"] = ("kernel: CUDA events over back-to-back dgp_draw_markers launches on 31-frame 747x832 batches queued "
                    "behind a device spin (host enqueue excluded), frames rotated over more than 2 x 126 MB of distinct "
                    "batches; labels are an animal-sized chain pose (joints 20-60 px apart, a few px of motion per frame), "
                    "all joints drawn; K = 0 is the markers-only kernel, K = 5 / 10 add the chain skeleton (nj - 1 edges) and "
                    "K - 1 trail frames. fused_jpeg: dgp_estimate_pose_stream_render_jpeg over a pinned cyclic source with a "
                    "packet writer that discards the packets, arms alternated over %d rounds, wall clock around each "
                    "synchronous call; run_to_run_spread = (max - min) / median of an arm's rounds." % args.rounds)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
