"""Motion-JPEG of the labelled video (dgp_encode_jpeg, dgp_estimate_pose_stream_render_jpeg): the encoder's device time per
batch, then frames/s of the fused render pass with each writer, arms alternated over rounds.  configs[1] (747x832, 4 joints,
fp16), pinned cyclic source as bench.py's e2e arm.  Writes one JSON file (default profiles/r08_bench_jpeg.json).

    python tools/bench_jpeg.py [--out PATH] [--frames 10000] [--encode-frames 1500] [--rounds 3] [--quality 90]
"""
import argparse
import ctypes as C
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import make_frame_pool  # noqa: E402
from deepgraphpose_b200 import synthetic  # noqa: E402
from deepgraphpose_b200.engine import Engine, jpeg_capacity, suggest_batch  # noqa: E402
from deepgraphpose_b200.mp4 import MJPEGWriter  # noqa: E402
from tools.bench_render import gpu_info  # noqa: E402

H, W, NJ = 747, 832, 4
L2_BYTES = 126 * 2 ** 20


def encode_kernel(eng, h, w, B, quality, launches):
    """CUDA events around `launches` back-to-back dgp_encode_jpeg calls on 31-frame batches, the input rotated over enough
    distinct batches to exceed the L2 (so frames are read from HBM)."""
    nb = max(2, -(-2 * L2_BYTES // (B * h * w * 3)))
    pool = torch.from_numpy(make_frame_pool(B * nb, seed=7, h=h, w=w, nj=NJ)).cuda()
    cap = jpeg_capacity(h, w) * B
    out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    meta = torch.empty((2, B), dtype=torch.int64, device="cuda")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def launch(k):
        x = pool[(k % nb) * B:(k % nb + 1) * B]
        rc = eng.lib.dgp_encode_jpeg(eng.h, C.c_void_p(x.data_ptr()), B, h, w, quality, C.c_void_p(out.data_ptr()), cap,
                                     C.c_void_p(meta[0].data_ptr()), C.c_void_p(meta[1].data_ptr()), stream)
        assert rc == 0

    for k in range(2 * nb):
        launch(k)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(100_000_000)   # the host enqueues every launch while the device spins: events bracket device time
    a.record()
    for k in range(launches):
        launch(k)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / launches
    sizes = []
    for k in range(nb):
        launch(k)
        torch.cuda.synchronize()
        sizes.append(meta[1].cpu().numpy().copy())
    sizes = np.concatenate(sizes)
    return {"frame": [h, w], "batch": B, "quality": quality, "distinct_batches": nb,
            "input_MB_rotated": nb * B * h * w * 3 / 1e6, "launches": launches, "ms_per_batch": ms,
            "frames_per_s": B / ms * 1e3, "input_GB_per_s": B * h * w * 3 / ms / 1e6,
            "bytes_out_per_frame_mean": float(sizes.mean()), "bytes_out_per_frame_max": int(sizes.max()),
            "capacity_per_frame": jpeg_capacity(h, w)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_bench_jpeg.json"))
    ap.add_argument("--frames", type=int, default=10000)
    ap.add_argument("--encode-frames", type=int, default=1500, help="frames of the mp4v arm: its encoder is the bound")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--quality", type=int, default=90)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import cv2
    res = {"gpu": gpu_info()}
    B = suggest_batch(H, W, 24, 48)
    eng = Engine(NJ, location_refinement=False, precision="fp16")
    eng.load_weights(synthetic.make_weights(NJ, seed=0, location_refinement=False))
    res["encode_kernel"] = [encode_kernel(eng, h, w, 31, args.quality, args.launches) for h, w in ((H, W), (1080, 1920))]
    pool = torch.from_numpy(make_frame_pool(4 * B, seed=1234, h=H, w=W, nj=NJ)).pin_memory()
    P = pool.shape[0]
    dotsize, thr, q = 3, 0.1, args.quality
    tmp = tempfile.mkdtemp(prefix="bench_jpeg_")
    written = {}

    def arm_a(n):
        return eng.estimate_pose_stream(pool, H, W, n, batch=B)

    def arm_b(n):
        return eng.estimate_pose_render_stream(pool, H, W, n, lambda fr: None, dotsize, thr, batch=B)

    def arm_c(n):
        return eng.estimate_pose_render_stream(pool, H, W, n, lambda d, s: None, dotsize, thr, batch=B, encoder="jpeg",
                                               quality=q)

    def arm_d(n):
        path = os.path.join(tmp, "labeled_mjpeg.mp4")
        with MJPEGWriter(path, 30.0, W, H) as vw:
            out = eng.estimate_pose_render_stream(pool, H, W, n, vw.write_packed, dotsize, thr, batch=B, encoder="jpeg",
                                                  quality=q)
        written["d"] = os.path.getsize(path) / n
        return out

    def arm_e(n):
        path = os.path.join(tmp, "labeled_mp4v.mp4")
        vw = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"mp4v"), 30.0, (W, H))
        assert vw.isOpened()

        def write(fr):
            for f in fr:
                vw.write(np.ascontiguousarray(f[:, :, ::-1]))

        try:
            return eng.estimate_pose_render_stream(pool, H, W, n, write, dotsize, thr, batch=B)
        finally:
            vw.release()
            written["e"] = os.path.getsize(path) / n

    arms = {"a_stream": (arm_a, args.frames), "b_render_raw_discard": (arm_b, args.frames),
            "c_render_jpeg_discard": (arm_c, args.frames), "d_render_jpeg_mp4_file": (arm_d, args.frames),
            "e_render_mp4v_cv2": (arm_e, args.encode_frames)}
    for name, (fn, _) in arms.items():  # warm-up: plans, rings, writer slots, tables, encoder
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
            runs[name].append(n / (time.perf_counter() - t0))
            outputs[name] = out
    res["arms"] = {k: {"frames": arms[k][1], "fps_per_round": v, "fps_median": float(np.median(v))} for k, v in runs.items()}
    med = {k: v["fps_median"] for k, v in res["arms"].items()}
    res["jpeg_discard_over_raw_discard"] = med["c_render_jpeg_discard"] / med["b_render_raw_discard"]
    res["jpeg_discard_over_stream"] = med["c_render_jpeg_discard"] / med["a_stream"]
    res["jpeg_file_over_mp4v"] = med["d_render_jpeg_mp4_file"] / med["e_render_mp4v_cv2"]
    res["readouts_equal_stream"] = all(all(torch.equal(p, q_) for p, q_ in zip(outputs["a_stream"], outputs[k]))
                                       for k in ("b_render_raw_discard", "c_render_jpeg_discard", "d_render_jpeg_mp4_file"))
    res["file_bytes_per_frame"] = {"d_mjpeg": written.get("d"), "e_mp4v": written.get("e")}
    res["d2h_bytes_per_frame"] = {"raw": H * W * 3, "jpeg": written.get("d")}
    shutil.rmtree(tmp, ignore_errors=True)
    eng.close()
    res["config"] = {"frame": [H, W, 3], "num_joints": NJ, "precision": "fp16", "batch": B, "pool_frames": P,
                     "dotsize": dotsize, "mask_threshold": thr, "quality": q, "host_threads": torch.get_num_threads()}
    res["notes"] = ("encode_kernel: CUDA events over back-to-back dgp_encode_jpeg launches (4 kernels each) on 31-frame "
                    "synthetic batches, queued behind a device spin so host enqueue time is excluded; input rotated over more "
                    "than 2 x 126 MB of distinct batches. Arms run alternately, %d rounds, wall clock around each synchronous "
                    "call, pinned cyclic source (frame t = pool[t %% %d]). a: estimate_pose_stream; b: raw fused render, writer "
                    "discards the frames; c: jpeg fused render, packet writer discards the packets; d: c writing the MJPEG mp4 "
                    "(deepgraphpose_b200.mp4) into a temporary directory; e: raw fused render into cv2.VideoWriter mp4v on %d "
                    "frames." % (args.rounds, P, args.encode_frames))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
