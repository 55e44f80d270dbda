"""Augmentation of labelled training frames on the device (dgp_augment): kernel time with every op on, the fit-loop step time
with fitdgp_util.build_aug pipelines against no pipeline (arms alternated in the same run), and the host cost of the same
four ops per frame with cv2 on one core.  Writes one JSON file (default profiles/r06_bench_augment.json).

    python tools/bench_augment.py [--out PATH] [--calls 40] [--steps 30]
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
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
from bench_resize import L2_BYTES, gpu_info  # noqa: E402
from deepgraphpose_b200 import fitdgp, synthetic  # noqa: E402
from deepgraphpose_b200.engine import Engine, output_dims  # noqa: E402
from deepgraphpose_b200.fitdgp_util import build_aug, data_aug  # noqa: E402

H, W, NJ, NT = bench.H, bench.W, bench.NJ, 10   # configs[3]: 747x832, 4 bodyparts, 10-frame batches, 3 labelled frames
VIS = [0, 3, 6]


def kernel_times(calls):
    """dgp_augment over n frames of a 10-frame 747x832 batch, every op on (apply_prob 1); batches rotated over more than the
    L2.  Each call is timed by its own event pair behind a device sleep, so the host's enqueue is not in the window."""
    eng = Engine(NJ, location_refinement=False)
    nbuf = max(2, -(-3 * L2_BYTES // (NT * H * W * 3)))
    g = torch.Generator(device="cuda").manual_seed(0)
    bufs = [torch.randint(0, 256, (NT, H, W, 3), dtype=torch.uint8, device="cuda", generator=g) for _ in range(nbuf)]
    rows = []
    for n in (3, 10):
        pipe = build_aug(apply_prob=1.0, seed=n)
        params = [pipe.sample(n) for _ in range(calls + 3)]
        pos = list(range(n))
        jl = torch.zeros((n, NJ, 2), dtype=torch.float64, device="cuda")
        for i in range(3):
            eng.augment(bufs[i % nbuf], pos, jl, params[i])
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(calls)]
        l0 = eng.launch_count()
        for i in range(calls):
            torch.cuda._sleep(2_000_000)
            ev[i][0].record()
            eng.augment(bufs[(i + 3) % nbuf], pos, jl, params[i + 3])
            ev[i][1].record()
        torch.cuda.synchronize()
        ms = [a.elapsed_time(b) for a, b in ev]
        rows.append({"frames": n, "H": H, "W": W, "ms_median": float(np.median(ms)), "ms_min": float(np.min(ms)),
                     "ms_max": float(np.max(ms)), "calls": calls, "launches_per_call": (eng.launch_count() - l0) / calls,
                     "input_buffers": nbuf, "input_bytes_rotated": nbuf * NT * H * W * 3})
    eng.close()
    return rows


def step_times(steps, rounds):
    """Fit-loop step at configs[3] size as _fit_loop runs it with an aug_pipeline: the batch uploaded from pinned host
    memory, data_aug on the device, forward + loss + backward + optimizer, loss values read back.  The arms (no pipeline,
    apply_prob 0.5, apply_prob 1) are alternated round by round; host wall clock around synchronised steps."""
    _, (hs, ws_) = output_dims(H, W)
    labels, batch = synthetic.make_training_batch(NT, hs, ws_, NJ, VIS, ((0, 1),), seed=100)
    edges = synthetic.chain_skeleton(NJ)
    S0 = np.zeros((len(edges), NJ))
    for l, (a, b) in enumerate(edges):
        S0[l, a], S0[l, b] = 1.0, -1.0
    cfg = dict(gm2=1, gm3=3, wt=0.0, wt_max=0.0, wn_visible=5.0, wn_hidden=3.0, gamma=1.0, gauss_len=1.0, lengthscale=1.0,
               locref_loss_weight=0.05, stride=8.0)
    ws, ws_max = fitdgp.spatial_clique_params([labels], S0, 8.0, 1000.0, 1.2)
    eng = Engine(NJ, location_refinement=True)
    eng.load_weights(synthetic.make_weights(NJ, seed=0))
    frames_pinned = torch.from_numpy(bench.make_frame_pool(NT, seed=1234)).pin_memory()
    arms = {"none": None, "apply_prob_0.5": build_aug(apply_prob=0.5, seed=1), "apply_prob_1": build_aug(apply_prob=1.0, seed=2)}

    def step(pipe):
        fr = frames_pinned.to("cuda", non_blocking=True)
        feed = batch
        if pipe is not None:
            fr, jl = data_aug(fr, VIS, labels, pipe, cfg, engine=eng)
            feed = dict(batch, targets=jl)
        out = fitdgp.train_forward_backward(eng, fr, feed, cfg, edges, ws, ws_max, 1000, 100, sync=False)
        eng.optimizer_step(0.005, 0.9, 10.0, 1.0)
        return out.cpu()

    for pipe in arms.values():
        for _ in range(3):
            step(pipe)
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, pipe in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                step(pipe)
            torch.cuda.synchronize()
            times[k].append((time.perf_counter() - t0) * 1e3 / steps)
    eng.close()
    base = float(np.median(times["none"]))
    return {k: {"ms_per_step_median": float(np.median(v)), "ms_per_step_rounds": [float(x) for x in v],
                "vs_none": float(np.median(v)) / base - 1.0} for k, v in times.items()}


def host_cv2_ms(frames=5):
    """The same four ops on one 747x832 frame with cv2 on one host core (elastic: float32 noise, GaussianBlur, remap)."""
    import cv2
    cv2.setNumThreads(1)
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    M = cv2.getRotationMatrix2D((W / 2 - 0.5, H / 2 - 0.5), 17.0, 1.0)
    k = np.zeros((7, 7), np.float32)
    k[:, 3] = 1 / 7
    t = {"rotate": [], "motion_blur": [], "dropout": [], "elastic": []}
    for _ in range(frames):
        t0 = time.perf_counter()
        out = cv2.warpAffine(img, M, (W, H), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
        t1 = time.perf_counter()
        out = cv2.filter2D(out, -1, k)
        t2 = time.perf_counter()
        mask = (rng.random((30, 33)) >= 0.02).astype(np.uint8)
        out = out * cv2.resize(mask, (W, H), interpolation=cv2.INTER_NEAREST)[..., None]
        t3 = time.perf_counter()
        dx = cv2.GaussianBlur(rng.uniform(-1, 1, (H, W)).astype(np.float32), (41, 41), 5.0) * 40
        dy = cv2.GaussianBlur(rng.uniform(-1, 1, (H, W)).astype(np.float32), (41, 41), 5.0) * 40
        out = cv2.remap(out, xx + dx, yy + dy, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
        t4 = time.perf_counter()
        for name, a, b in (("rotate", t0, t1), ("motion_blur", t1, t2), ("dropout", t2, t3), ("elastic", t3, t4)):
            t[name].append((b - a) * 1e3)
    res = {k_: float(np.median(v)) for k_, v in t.items()}
    res["total"] = float(sum(res.values()))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_bench_augment.json"))
    ap.add_argument("--calls", type=int, default=40)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_augment needs a CUDA device")
    res = {"gpu": gpu_info(), "kernel": kernel_times(args.calls), "fit_step": step_times(args.steps, args.rounds),
           "host_cv2_ms_per_frame_one_core": host_cv2_ms()}
    res["note"] = ("kernel: dgp_augment with rotation, motion blur (k=7), dropout and elastic (sigma 5) on every frame; "
                   "fit_step: configs[3] (747x832, 10 frames, 3 labelled) step with the batch uploaded from pinned memory")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
