#!/usr/bin/env python
"""Inference and training speed of the ResNet-50 pose net at slim output_stride 16 and 8 on one GPU.

On BASELINE.json configs[1] (747x832, nj 4, part_pred head, chain skeleton, fp16 storage, batch from engine.suggest_batch
for that stride), the two strides alternate over --rounds rounds in one process, each with its own engine and its own
device-resident batches (4 batches, together larger than the 126 MB L2, rotated step by step):
  * device-resident frames/s of bench.py's step (forward + soft-argmax read-out + potentials);
  * the conv-GEMM roofline fraction as bench.py computes it (one event pair around each step's run of GEMM launches), with
    the algorithmic FLOPs of that stride's layer list (tools/bench_depths.conv_flops_per_frame);
  * the end-to-end stream of bench.py's `e2e` (eval.estimate_pose_sharded on one GPU: pinned host frames, H2D per batch,
    D2H of the read-outs).
Then the configs[3] training step (tools/bench_train.py: nt = 10, wt = 1) at both strides.  Card name and power limit are
read in the same run.  Prints one JSON document and writes it to --out.

  python tools/bench_output_stride.py --steps 20 --warmup 5 --out profiles/r09_bench_output_stride.json
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from bench_depths import card, conv_flops_per_frame  # noqa: E402

RESNET50_UNITS = (3, 4, 6, 3)


class StrideWorkload(bench.Workload):
    """bench.Workload (configs[1]) with the backbone at `output_stride`."""

    def __init__(self, output_stride, precision="fp16"):
        from deepgraphpose_b200 import synthetic
        from deepgraphpose_b200.engine import Engine, suggest_batch
        self.key = "stride%d" % output_stride
        self.H, self.W, self.nj, self.skeleton_kind, self.label = bench.CONFIGS["b"]
        self.dev = torch.device("cuda", 0)
        self.B = suggest_batch(self.H, self.W, 24, 48, output_stride=output_stride)
        self.eng = Engine(self.nj, location_refinement=False, device=0, precision=precision, output_stride=output_stride)
        self.eng.load_weights(synthetic.make_weights(self.nj, seed=0, location_refinement=False))
        self.edges = synthetic.chain_skeleton(self.nj)
        self.flops_frame, (self.hs, self.ws) = conv_flops_per_frame(self.H, self.W, self.nj, RESNET50_UNITS,
                                                                   output_stride=output_stride)
        assert (self.hs, self.ws) == self.eng.output_dims(self.H, self.W)[1]
        self.n_pool = 4
        self.pool_host = torch.from_numpy(bench.make_frame_pool(self.n_pool * self.B, seed=1234, h=self.H, w=self.W,
                                                                nj=self.nj)).pin_memory()
        self.pool = [self.pool_host[i * self.B:(i + 1) * self.B].to(self.dev) for i in range(self.n_pool)]
        self.ws_vec = np.full(len(self.edges), 1000.0 / 60.0, np.float32)
        self.ws_max = np.full(len(self.edges), 1.2 * 80.0, np.float32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--e2e-frames", type=int, default=10000)
    ap.add_argument("--train-steps", type=int, default=10)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import bench_train
    torch.cuda.set_device(0)
    assert conv_flops_per_frame(bench.H, bench.W, bench.NJ, RESNET50_UNITS) == bench.conv_flops_per_frame(bench.H, bench.W, bench.NJ)
    peaks, peak_src = bench.load_peaks()
    strides = (16, 8)
    wls = {s: StrideWorkload(s) for s in strides}
    doc = {"card": card(), "precision": "fp16", "workload": bench.WORKLOAD, "steps": args.steps, "warmup": args.warmup,
           "rounds": args.rounds,
           "timing": "as bench.py --gpus 1: CUDA events around K device-resident steps (forward + soft-argmax + potentials), "
                     "4 batches per stride rotated step by step; GEMM roofline from one event pair around each step's run of "
                     "conv_gemm launches; e2e = wall clock around eval.estimate_pose_sharded on one GPU from pinned host frames. "
                     "The strides alternate within each round.",
           "train": "tools/bench_train.py measure(): configs[3] DGP training step, 747x832, nt=10, wt=1, nj=4 + locref, "
                    "device-resident inputs, %d timed steps" % args.train_steps,
           "strides": {s: {"batch": wls[s].B, "scoremap": [wls[s].hs, wls[s].ws],
                           "gflop_per_frame": wls[s].flops_frame / 1e9, "rounds": []} for s in strides}}
    for r in range(args.rounds):
        for s in strides:
            wl = wls[s]
            m = bench.measure_device(wl, args.steps, args.warmup, 1, 0)
            roof = bench.roofline_of(wl, m, args.steps, peaks, peak_src)
            _, e2e = bench.measure_e2e(wl, args.e2e_frames, 1)
            entry = {"frames_per_s": m["value"], "ms_per_step": m["ms"] / args.steps, "gemm_tflops": roof["achieved"],
                     "gemm_roofline_frac": roof["frac"], "gemm_share_of_step": roof["share_of_step"],
                     "gemm_launches_per_step": roof["kernel"], "e2e_frames_per_s": e2e["value"], "clocks": m["clocks"]}
            doc["strides"][s]["rounds"].append(entry)
            print("round %d output_stride %d %s" % (r, s, json.dumps(entry)), file=sys.stderr, flush=True)
    for s in strides:
        rs = doc["strides"][s]["rounds"]
        for k in ("frames_per_s", "gemm_tflops", "gemm_roofline_frac", "e2e_frames_per_s"):
            v = [e[k] for e in rs]
            doc["strides"][s][k] = {"median": float(np.median(v)), "min": float(min(v)), "max": float(max(v))}
        doc["strides"][s]["gemm_peak_tflops"] = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
    for wl in wls.values():
        wl.close()
    del wls
    torch.cuda.empty_cache()
    for s in strides:
        line = bench_train.measure(0, 0, 1, args.train_steps, 3, 10, bench.H, bench.W, profile=False, wt=1.0, output_stride=s)
        doc["strides"][s]["train_ms_per_step"] = line["ms_per_step"]
        doc["strides"][s]["train_frames_per_s"] = line["value"]
        doc["strides"][s]["train_loss_after"] = line["loss_after"]
        torch.cuda.empty_cache()
    f16, f8 = (doc["strides"][s]["frames_per_s"]["median"] for s in strides)
    doc["os8_over_os16_frames_per_s"] = f8 / f16
    doc["peak_source"] = peak_src
    print(json.dumps(doc), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
