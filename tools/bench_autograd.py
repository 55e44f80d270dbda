#!/usr/bin/env python
"""Cost of training through torch.autograd, BASELINE.json configs[3] (747x832, nt = 10, nj = 4 + locref, fp16 storage,
device-resident inputs, one GPU).  ms per training step of three paths on the same network kernels:

  fused    dgp_train_forward_backward (DGP loss inside the C ABI) + Engine.optimizer_step (Momentum + global-norm clip)
  module   autograd.TrainablePoseNet + fitdgp.dgp_loss_function (the same DGP loss as an autograd node) + optimizer_step
  torch    TrainablePoseNet + a loss written in PyTorch (sigmoid cross-entropy to disc targets + Huber locref) +
           torch.optim.SGD(momentum=0.9) on the parameter arena

Each path has its own engine; the paths are timed in alternating rounds of --steps steps (CUDA events, device-synchronised)
and the median round is reported.  Card name and power limit are read in the same run.

  python tools/bench_autograd.py --steps 20 --rounds 5 --out profiles/r04_bench_autograd.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip()
    name, power, clock = [s.strip() for s in out.split(",")]
    return {"name": name, "power_limit": power, "sm_max_clock": clock}


def torch_loss(logits, locref, tgt, lmap, lmask):
    return F.binary_cross_entropy_with_logits(logits, tgt) + 0.05 * F.huber_loss(locref * lmask, lmap * lmask, delta=1.0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--nt", type=int, default=10)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    from deepgraphpose_b200 import fitdgp, synthetic
    from deepgraphpose_b200.autograd import TrainablePoseNet
    from deepgraphpose_b200.engine import Engine, output_dims
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    H, W, NJ, nt, wt = bench.H, bench.W, bench.NJ, args.nt, 1.0
    _, (hs, ws_) = output_dims(H, W)
    vis = [0, 3, 6][: max(1, nt // 3)]
    # the feed of tools/bench_train.py (configs[3]): skeleton + temporal cliques, a device-resident flow-magnitude field
    labels, batch = synthetic.make_training_batch(nt, hs, ws_, NJ, vis, ((0, 1),), seed=100)
    edges = synthetic.chain_skeleton(NJ)
    S0 = np.zeros((len(edges), NJ))
    for l, (a, b) in enumerate(edges):
        S0[l, a], S0[l, b] = 1.0, -1.0
    cfg = dict(gm2=1, gm3=3, wt=wt, wt_max=0.0, wn_visible=5.0, wn_hidden=3.0, gamma=1.0, gauss_len=1.0, lengthscale=1.0,
               locref_loss_weight=0.05, stride=8.0)
    ws, ws_max = fitdgp.spatial_clique_params([labels], S0, 8.0, 1000.0, 1.2)
    yy, xx = np.meshgrid(np.arange(H, dtype=np.float32), np.arange(W, dtype=np.float32), indexing="ij")
    batch["vector_field_tf"] = torch.from_numpy(np.stack([0.9 + 0.8 * np.sin(yy / (37.0 + 3 * t)) * np.cos(xx / (41.0 + 5 * t))
                                                          for t in range(nt - 1)]).astype(np.float32)).to(dev)
    batch["wt_batch_pl"] = np.ones(nt - 1, np.float32) * wt
    batch["wt_batch_mask_pl"] = np.ones(nt - 1, np.float32)
    frames = torch.from_numpy(bench.make_frame_pool(nt, seed=1234)).to(dev)
    weights = synthetic.make_weights(NJ, seed=0)
    rng = np.random.default_rng(0)
    tgt = torch.from_numpy((rng.uniform(size=(nt, hs, ws_, NJ)) < 0.01).astype(np.float32)).to(dev)
    lmap = torch.from_numpy(rng.normal(0, 0.7, (nt, hs, ws_, 2 * NJ)).astype(np.float32)).to(dev)
    lmask = tgt.repeat_interleave(2, dim=3)

    def engine():
        e = Engine(NJ, location_refinement=True, device=0, precision="fp16")
        e.load_weights(weights)
        e.train_enable()
        return e

    e_fused, e_module, e_torch = engine(), engine(), engine()
    net_module, net_torch = TrainablePoseNet(e_module), TrainablePoseNet(e_torch)
    sgd = torch.optim.SGD(net_torch.parameters(), lr=0.005, momentum=0.9)

    def fused():
        out = fitdgp.train_forward_backward(e_fused, frames, batch, cfg, edges, ws, ws_max, 1000, 100, sync=False)
        e_fused.optimizer_step(0.005, 0.9, 10.0, 1.0)
        return out[5]

    def module():
        net_module.zero_grad()
        logits, locref = net_module(frames)
        loss = fitdgp.dgp_loss_function(logits, locref, batch, cfg, edges, ws, ws_max, 1000, 100, engine=e_module)["total_loss"]
        loss.backward()
        e_module.optimizer_step(0.005, 0.9, 10.0, 1.0)
        return loss.detach()

    def torch_path():
        sgd.zero_grad()
        loss = torch_loss(*net_torch(frames), tgt, lmap, lmask)
        loss.backward()
        sgd.step()
        return loss.detach()

    paths = {"fused": fused, "module_dgp_loss": module, "torch_loss_sgd": torch_path}
    losses = {k: [] for k in paths}
    for k, fn in paths.items():
        for _ in range(args.warmup):
            fn()
    torch.cuda.synchronize()
    rounds = {k: [] for k in paths}
    for _ in range(args.rounds):
        for k, fn in paths.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                last = fn()
            e1.record()
            torch.cuda.synchronize()
            rounds[k].append(e0.elapsed_time(e1) / args.steps)
            losses[k].append(float(last))
    head_mb = 4 * nt * hs * ws_ * 3 * NJ / 1e6
    doc = {"card": card(), "precision": "fp16",
           "workload": "configs[3]: DGP training step, %dx%d, nt=%d (%d visible), nj=%d + locref, gm2=1 gm3=3 ws=1000 wt=%g, "
                       "device-resident inputs, one GPU" % (H, W, nt, len(vis), NJ, wt),
           "timing": "CUDA events around %d steps per round, %d alternating rounds per path after %d warm-up steps each; "
                     "median round" % (args.steps, args.rounds, args.warmup),
           "head_tensor_mb": head_mb,
           "paths": {k: {"ms_per_step": float(np.median(v)), "ms_per_step_rounds": v, "loss_last": losses[k][-1]}
                     for k, v in rounds.items()}}
    f = doc["paths"]["fused"]["ms_per_step"]
    for k in ("module_dgp_loss", "torch_loss_sgd"):
        doc["paths"][k]["overhead_ms_vs_fused"] = doc["paths"][k]["ms_per_step"] - f
    print(json.dumps(doc), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(doc, fh, indent=1)
    for e in (e_fused, e_module, e_torch):
        e.close()


if __name__ == "__main__":
    main()
