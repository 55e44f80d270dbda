"""Frame resize + crop on the device (dgp_resize_crop): kernel time, its share of an estimate_pose batch, and end-to-end
frames/s of estimate_pose with new_size against streaming frames that are already at the network's size and against the
host-PIL generator path it replaces.  Writes one JSON file (default profiles/r05_bench_resize.json).

    python tools/bench_resize.py [--out PATH] [--frames 10000] [--pil-frames 300]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from deepgraphpose_b200 import synthetic  # noqa: E402
from deepgraphpose_b200.engine import Engine, frame_transform, suggest_batch  # noqa: E402

SHAPES = [((1494, 1664), (747, 832)), ((1080, 1920), (540, 960)), ((480, 640), (747, 832))]
L2_BYTES = 126 * 2 ** 20


def gpu_info():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    name, power, clock = [v.strip() for v in out.stdout.strip().split(",")] if out.returncode == 0 else ("?", "?", "?")
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi_name": name, "power_limit": power, "max_sm_clock": clock}


def event_ms(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(n):
        fn(i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def resize_into(eng, src, out, t):
    """dgp_resize_crop into a preallocated output (Engine.resize_crop allocates its result)."""
    import ctypes as C
    N, H0, W0, _ = src.shape
    rc = eng.lib.dgp_resize_crop(eng.h, C.c_void_p(src.data_ptr()), N, H0, W0, C.byref(t), C.c_void_p(out.data_ptr()),
                                 C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, rc


def kernel_times(eng, B, launches):
    rows = []
    for (H0, W0), (h, w) in SHAPES:
        src_bytes = B * H0 * W0 * 3
        nbuf = max(2, -(-3 * L2_BYTES // src_bytes))  # inputs rotated over more than the L2
        g = torch.Generator(device="cuda").manual_seed(0)
        srcs = [torch.randint(0, 256, (B, H0, W0, 3), dtype=torch.uint8, device="cuda", generator=g) for _ in range(nbuf)]
        out = torch.empty((B, h, w, 3), dtype=torch.uint8, device="cuda")
        t = frame_transform((h, w), None)
        for i in range(nbuf):
            resize_into(eng, srcs[i], out, t)
        ms = event_ms(lambda i: resize_into(eng, srcs[i % nbuf], out, t), launches)
        moved = src_bytes + B * h * w * 3
        rows.append({"source": [H0, W0], "output": [h, w], "batch": B, "launches": launches, "input_buffers": nbuf,
                     "ms_per_batch": ms, "us_per_frame": 1e3 * ms / B, "algorithmic_bytes": moved,
                     "GB_per_s": moved / (ms * 1e-3) / 1e9})
    return rows


def forward_ms(eng, B, H, W, launches):
    frames = [torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8, device="cuda") for _ in range(4)]

    def step(i):
        logits, _ = eng.forward(frames[i % 4])
        eng.softargmax(logits, want=("mu", "peak", "lik"))

    for i in range(4):
        step(i)
    return event_ms(step, launches)


def e2e(eng, B, n_frames, pil_frames):
    (H0, W0), (h, w) = SHAPES[0]
    # 64 frames: at batch 31 every third batch is the 2-frame wrap of the cyclic source, which runs the full-batch plan
    # (dgp_estimate_pose_stream); both device arms pay it, so they compare, but their absolute rates are below bench.py's
    P = 64
    pool_src, _ = synthetic.make_video(P, H0, W0, eng.nj, seed=1)
    pool_src = torch.from_numpy(pool_src).pin_memory()
    pool_net = eng.resize_crop(pool_src.cuda(), (h, w)).cpu().pin_memory()

    def timed(fn):
        fn(min(n_frames, 4 * B))  # warm-up: ring, plans, tables
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n = fn(None)
        torch.cuda.synchronize()
        return n / (time.perf_counter() - t0)

    resized = timed(lambda n: eng.estimate_pose_stream(pool_src, H0, W0, n or n_frames, batch=B, new_size=(h, w))[0].shape[0])
    native = timed(lambda n: eng.estimate_pose_stream(pool_net, h, w, n or n_frames, batch=B)[0].shape[0])
    from PIL import Image

    def pil_gen(n):
        for t in range(n):
            yield np.asarray(Image.fromarray(pool_src[t % P].numpy()).resize(size=(w, h)))

    host_pil = timed(lambda n: eng.estimate_pose_stream(pil_gen(n or pil_frames), h, w, n or pil_frames, batch=B)[0].shape[0])
    return {"source": [H0, W0], "new_size": [h, w], "batch": B, "pool_frames": P,
            "device_resize_fps": resized, "device_resize_frames": n_frames,
            "native_size_fps": native, "native_size_frames": n_frames,
            "host_pil_fps": host_pil, "host_pil_frames": pil_frames, "host_threads": torch.get_num_threads()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_bench_resize.json"))
    ap.add_argument("--frames", type=int, default=10000)
    ap.add_argument("--pil-frames", type=int, default=300)
    ap.add_argument("--launches", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    nj = 4
    eng = Engine(nj, location_refinement=False)
    eng.load_weights(synthetic.make_weights(nj, seed=0, location_refinement=False))
    B = suggest_batch(747, 832, 24, 48)
    res = {"gpu": gpu_info(), "kernels": kernel_times(eng, B, args.launches)}
    fwd = forward_ms(eng, B, 747, 832, args.launches)
    k0 = res["kernels"][0]["ms_per_batch"]
    res["batch_share"] = {"shape": "1494x1664 -> 747x832", "batch": B, "resize_ms": k0, "forward_softargmax_ms": fwd,
                          "resize_share": k0 / (k0 + fwd)}
    res["e2e"] = e2e(eng, B, args.frames, args.pil_frames)
    res["notes"] = ("kernel time: CUDA events over %d launches of dgp_resize_crop (horizontal + vertical pass) per shape, "
                    "inputs rotated over buffers larger than the 126 MB L2; GB/s counts the source read once and the output "
                    "written once, the uint8 intermediate excluded. e2e: pinned cyclic source streamed through "
                    "Engine.estimate_pose_stream (H2D, transform, forward, soft-argmax, D2H); host_pil_fps decodes nothing "
                    "and resizes each frame with PIL in the generator, as eval.py did before the device path." % args.launches)
    eng.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
