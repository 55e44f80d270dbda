#!/usr/bin/env python
"""Inference and training speed of the three DLC backbones (net_type resnet_50 / resnet_101 / resnet_152) on one GPU.

For each depth, on BASELINE.json configs[1] (747x832, nj 4, part_pred head, chain skeleton, fp16 storage, batch from
engine.suggest_batch for that depth's unit counts):
  * device-resident frames/s of bench.py's step (forward + soft-argmax read-out + potentials, inputs resident in HBM);
  * the conv-GEMM roofline fraction as bench.py computes it (one event pair around each step's run of GEMM launches, the
    algorithmic FLOPs of the depth, the same peaks file);
  * the configs[3] training step time (tools/bench_train.py: nt = 10, wt = 1) with that depth's weights.
Prints one JSON document (and writes it to --out): card name and power limit are read in the same run.

  python tools/bench_depths.py --steps 20 --warmup 5 --out profiles/r03_bench_depths.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402


def conv_flops_per_frame(h, w, nj, units, locref=False, output_stride=16):
    """bench.conv_flops_per_frame with the units per block of the backbone: algorithmic forward FLOPs (2*MACs) of the convs
    and the deconv heads at output stride 16, or 8 (block 2 keeps its resolution; atrous convs cost what dense ones do)."""
    c2 = lambda v: -(-v // 2)
    hh, ww = c2(h), c2(w)
    total = 2 * hh * ww * 147 * 64
    hh, ww = c2(hh), c2(ww)
    cin = 64
    strides = (2, 2, 1, 1) if output_stride == 16 else (2, 1, 1, 1)   # stride of each block as executed
    for base, n_units, bstride in zip((64, 128, 256, 512), units, strides):
        for u in range(n_units):
            s = bstride if u == n_units - 1 else 1
            depth = 4 * base
            ho, wo = (c2(hh), c2(ww)) if s == 2 else (hh, ww)
            if cin != depth:
                total += 2 * hh * ww * cin * depth
            total += 2 * hh * ww * cin * base
            total += 2 * ho * wo * 9 * base * base
            total += 2 * ho * wo * base * depth
            hh, ww, cin = ho, wo, depth
    total += 2 * hh * ww * 2048 * 9 * nj * (3 if locref else 1)
    return total, (2 * hh, 2 * ww)


class DepthWorkload(bench.Workload):
    """bench.Workload (configs[1]) on the synthetic weights of another backbone."""

    def __init__(self, net_type, precision="fp16"):
        from deepgraphpose_b200 import synthetic
        from deepgraphpose_b200.engine import Engine, suggest_batch
        self.key = "depth"
        self.H, self.W, self.nj, self.skeleton_kind, self.label = bench.CONFIGS["b"]
        self.dev = torch.device("cuda", 0)
        units = synthetic.BLOCK_UNITS[net_type]
        self.B = suggest_batch(self.H, self.W, 24, 48, units=units)
        self.eng = Engine(self.nj, location_refinement=False, device=0, precision=precision)
        self.eng.load_weights(synthetic.make_weights(self.nj, seed=0, location_refinement=False, net_type=net_type))
        assert self.eng.net_type == net_type
        self.edges = synthetic.chain_skeleton(self.nj)
        self.flops_frame, (self.hs, self.ws) = conv_flops_per_frame(self.H, self.W, self.nj, units)
        self.n_pool = 4
        self.pool_host = torch.from_numpy(bench.make_frame_pool(self.n_pool * self.B, seed=1234, h=self.H, w=self.W, nj=self.nj))
        self.pool = [self.pool_host[i * self.B:(i + 1) * self.B].to(self.dev) for i in range(self.n_pool)]
        self.ws_vec = np.full(len(self.edges), 1000.0 / 60.0, np.float32)
        self.ws_max = np.full(len(self.edges), 1.2 * 80.0, np.float32)


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip()
    name, power, clock = [s.strip() for s in out.split(",")]
    return {"name": name, "power_limit": power, "sm_max_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--train-steps", type=int, default=10)
    ap.add_argument("--depths", default="resnet_50,resnet_101,resnet_152")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    from deepgraphpose_b200 import synthetic
    import bench_train
    assert conv_flops_per_frame(bench.H, bench.W, bench.NJ, synthetic.BLOCK_UNITS["resnet_50"]) == \
        bench.conv_flops_per_frame(bench.H, bench.W, bench.NJ)
    peaks, peak_src = bench.load_peaks()
    doc = {"card": card(), "precision": "fp16", "workload": bench.WORKLOAD, "steps": args.steps, "warmup": args.warmup,
           "timing": "as bench.py --gpus 1: CUDA events around K device-resident steps (forward + soft-argmax + potentials); "
                     "GEMM roofline from one event pair around each step's run of conv_gemm launches",
           "train": "tools/bench_train.py measure(): configs[3] DGP training step, 747x832, nt=10, wt=1, nj=4 + locref, "
                    "device-resident inputs, %d timed steps" % args.train_steps,
           "depths": {}}
    for net_type in args.depths.split(","):
        wl = DepthWorkload(net_type)
        m = bench.measure_device(wl, args.steps, args.warmup, 1, 0)
        roof = bench.roofline_of(wl, m, args.steps, peaks, peak_src)
        convs = len(synthetic.conv_specs(net_type))
        entry = {"units": list(synthetic.BLOCK_UNITS[net_type]), "convs": convs, "batch": wl.B,
                 "frames_per_s": m["value"], "ms_per_step": m["ms"] / args.steps,
                 "gflop_per_frame": wl.flops_frame / 1e9, "gemm_roofline_frac": roof["frac"],
                 "gemm_tflops": roof["achieved"], "gemm_peak_tflops": roof["peak"], "gemm_share_of_step": roof["share_of_step"],
                 "gemm_launches_per_step": roof["kernel"], "clocks": m["clocks"]}
        wl.close()
        torch.cuda.empty_cache()
        line = bench_train.measure(0, 0, 1, args.train_steps, 3, 10, bench.H, bench.W, profile=False, wt=1.0, net_type=net_type)
        entry["train_ms_per_step"] = line["ms_per_step"]
        entry["train_frames_per_s"] = line["value"]
        entry["train_loss_after"] = line["loss_after"]
        torch.cuda.empty_cache()
        doc["depths"][net_type] = entry
        print(net_type, json.dumps(entry), file=sys.stderr, flush=True)
    doc["peak_source"] = peak_src
    print(json.dumps(doc), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
