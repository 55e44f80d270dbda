#!/usr/bin/env python
"""Training-step benchmark, BASELINE.json configs[3]: DGP semi-supervised step (visible + hidden frames, skeleton clique,
fwd + bwd + clip/Momentum) in the default 16-bit storage mode (fp16), data-parallel over the ranks torchrun starts (one per GPU, NCCL all-reduce of the flat
gradient buffer).  747x832 frames, nt frames per replica, nj = 4 with the locref head.  Prints one JSON line (rank 0).

  python tools/bench_train.py --steps 10 --warmup 3 [--nt 10]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P tools/bench_train.py
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def cpu_train_step_seconds(nt, H, W, NJ):
    """The reference's training step on the host cores: torch-CPU autograd through the oracle network + dgp_loss (the CPU
    restatement of sess.run([loss, train_op]); TF1.15 is not installable here).  Returns (seconds per step, cores)."""
    import time
    from deepgraphpose_b200 import synthetic
    from deepgraphpose_b200.engine import output_dims
    from oracle import dgp_loss as oracle_loss
    from oracle import dgp_ops, pose_net
    from oracle import feeders
    torch.set_num_threads(os.cpu_count())
    _, (hs, ws_) = output_dims(H, W)
    labels, batch = synthetic.make_training_batch(nt, hs, ws_, NJ, [0], (), seed=7)
    batch["locref_map"], batch["locref_mask"] = feeders.batch_locref_maps(labels, [0], nt, hs, ws_, NJ)
    xg, yg = np.meshgrid(np.linspace(0, hs - 1, hs), np.linspace(0, ws_ - 1, ws_))
    batch["alpha_tf"] = np.array([xg, yg]).swapaxes(1, 2)
    edges = synthetic.chain_skeleton(NJ)
    S0 = dgp_ops.skeleton_matrix(edges, NJ)
    cfg = oracle_loss.default_dgp_cfg(gm2=1, gm3=3, wt=0.0)
    ws, ws_max = oracle_loss.spatial_clique_params(labels, S0, cfg)
    Wn = synthetic.make_weights(NJ, seed=0)
    Wt = {k: torch.from_numpy(v).requires_grad_(k.endswith(("/weights", "/gamma", "/beta", "/biases"))) for k, v in Wn.items()}
    frames = synthetic.make_video(nt, H, W, NJ, seed=3)[0]
    t0 = time.perf_counter()
    heads = pose_net.get_net(torch.from_numpy(frames.astype(np.float32)), Wt, True)
    _, total, _ = oracle_loss.dgp_loss_from_heads(heads["part_pred"], heads["locref"], batch, cfg, S0, ws, ws_max, 1000, 100)
    total.backward()
    params = [t for t in Wt.values() if t.requires_grad]
    with torch.no_grad():
        oracle_loss.momentum_step(params, [p.grad for p in params], [torch.zeros_like(p) for p in params])
    return time.perf_counter() - t0, os.cpu_count()


def measure(rank, local_rank, world, steps, warmup, nt, height, width, profile=True, precision="fp16", wt=1.0,
            net_type="resnet_50", output_stride=16):
    """One data-parallel training benchmark on the already-initialised process group; returns the JSON dict (rank 0) or None.
    ``net_type`` picks the backbone of the synthetic weights (the FLOP figures of the line are ResNet-50's at output stride
    16); ``output_stride`` 8 trains on stride-4 scoremaps of twice the resolution."""
    import argparse as _a
    args = _a.Namespace(steps=steps, warmup=warmup, nt=nt, height=height, width=width)
    import torch.distributed as dist
    from deepgraphpose_b200 import dp, fitdgp, fitdgp_util, synthetic
    from deepgraphpose_b200.engine import Engine, output_dims
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    H, W, NJ, nt = args.height, args.width, bench.NJ, args.nt
    _, (hs, ws_) = output_dims(H, W, output_stride)
    stride = output_stride / 2.0
    vis = [0, 3, 6][: max(1, nt // 3)]
    # feed_dict contract of fit_dgp; the locref target / mask maps are generated on the device by the coord2map feeder
    # kernel (no 6 MB feed per step)
    labels, batch = synthetic.make_training_batch(nt, hs, ws_, NJ, vis, ((0, 1),), seed=100 + rank)
    edges = synthetic.chain_skeleton(NJ)
    S0 = np.zeros((len(edges), NJ))
    for l, (a, b) in enumerate(edges):
        S0[l, a], S0[l, b] = 1.0, -1.0
    cfg = dict(gm2=1, gm3=3, wt=float(wt), wt_max=0.0, wn_visible=5.0, wn_hidden=3.0, gamma=1.0, gauss_len=1.0, lengthscale=1.0,
               locref_loss_weight=0.05, stride=stride, output_stride=output_stride)
    ws, ws_max = fitdgp.spatial_clique_params([labels], S0, stride, 1000.0, 1.2)
    eng = Engine(NJ, location_refinement=True, device=local_rank, precision=precision, output_stride=output_stride)
    eng.load_weights(synthetic.make_weights(NJ, seed=0, net_type=net_type))
    frames_host = bench.make_frame_pool(nt, seed=1234 + rank) if (H, W) == (bench.H, bench.W) else \
        synthetic.make_video(nt, H, W, NJ, seed=1234 + rank)[0]
    frames = torch.from_numpy(frames_host).to(dev)
    import bench_depths
    flops_fwd, _ = bench_depths.conv_flops_per_frame(H, W, NJ, synthetic.BLOCK_UNITS["resnet_50"], True, output_stride)
    flow_pinned = None
    if wt > 0:
        # temporal clique (fitdgp.py:1079-1124): vector_field_tf = optical-flow magnitude per consecutive frame pair
        # (nt-1, Hin, Win).  A synthetic smooth field of the right shape and range stands in for learn_wt's Farneback output;
        # it is resident on the device for the kernel-level number and copied from pinned host memory every e2e step.
        yy, xx = np.meshgrid(np.arange(H, dtype=np.float32), np.arange(W, dtype=np.float32), indexing="ij")
        flow = np.stack([0.9 + 0.8 * np.sin(yy / (37.0 + 3 * t)) * np.cos(xx / (41.0 + 5 * t)) for t in range(nt - 1)]).astype(np.float32)
        flow_pinned = torch.from_numpy(flow).pin_memory()
        batch["vector_field_tf"] = flow_pinned.to(dev)
        batch["wt_batch_pl"] = np.ones(nt - 1, np.float32) * wt
        batch["wt_batch_mask_pl"] = np.ones(nt - 1, np.float32)

    def step():
        out = fitdgp.train_forward_backward(eng, frames, batch, cfg, edges, ws, ws_max, 1000, 100, sync=False)
        scale = dp.allreduce_gradients(eng)
        eng.optimizer_step(0.005, 0.9, 10.0, scale)
        return out

    sampler = bench.ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler.begin()
    l0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = step()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    launches = eng.launch_count() - l0
    clocks = sampler.stop()
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    # ---- end to end as fit_dgp runs it: frames from (pinned) host memory every step, loss values read back every step
    frames_pinned = torch.from_numpy(frames_host).pin_memory()
    e2e_steps = max(3, min(args.steps, 10))

    def e2e_step():
        fr = frames_pinned.to(dev, non_blocking=True)
        # wt > 0: the flow-magnitude field of THIS batch, computed on the device from the frames just copied (dgp_learn_wt: the
        # reference's learn_wt = cv2 Farneback on the host, 175 ms per frame pair)
        # -- on the engine's side stream, as fit_dgp does: it overlaps the forward pass, the loss waits for its event
        b2 = batch if flow_pinned is None else dict(batch, vector_field_tf=fitdgp_util.learn_wt(fr, engine=eng, overlap=True))
        out = fitdgp.train_forward_backward(eng, fr, b2, cfg, edges, ws, ws_max, 1000, 100, sync=False)
        scale = dp.allreduce_gradients(eng)
        eng.optimizer_step(0.005, 0.9, 10.0, scale)
        return out.cpu()      # [loss_eval, _] = sess.run([loss, train_op]) hands the losses to the host

    e2e_step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    import time
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_dt], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_dt = float(t.item())
    prof, ms_prof = None, 0.0
    if profile:
        eng.get_profile()
        eng.set_profiling(True)
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        for _ in range(args.steps):
            out = step()
        p1.record()
        torch.cuda.synchronize()
        ms_prof = p0.elapsed_time(p1)
        eng.set_profiling(False)
        prof = eng.get_profile()
    loss = float(out.cpu()[5])
    exposed_ms = eng.allreduce_exposed_ms() if world > 1 else None
    line = None
    if rank == 0:
        peaks, src = bench.load_peaks()
        peak_tf = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
        n = nt * args.steps
        fam = {k: v[0] / args.steps for k, v in prof.items()} if prof else None
        tf = lambda gf, ms_: (gf * n / (ms_ / 1e3) / 1e12) if ms_ > 0 else None
        if prof is None:
            prof = {k: (0.0, 0) for k in ("conv_gemm", "dgrad_gemm", "wgrad_gemm")}
        line = {
            "metric": "training frames/sec (DGP semi-supervised step: fwd + bwd + clip/Momentum)", "value": world * n / (ms / 1e3),
            "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "dtype": precision, "data": "synthetic",
            "config": {"workload": "configs[3]: DGP training step, %dx%d, nt=%d frames per replica (%d visible), nj=%d + locref, gm2=1 gm3=3 ws=1000 wt=%g (temporal + skeleton cliques)"
                                   % (H, W, nt, len(vis), NJ, wt), "parallelism": ("dp%d, dgp_allreduce_gradients: NCCL SUM all-reduce of the 94 MB fp32 gradient arena inside the C ABI, 4 buckets in backward order "
                                       "(block4+heads, block3, block2, rest) overlapped with the backward pass" % world) if world > 1 else "single GPU",
                       "feeds": "device-timed value: frames and a (nt-1,H,W) flow-magnitude field resident on the device; e2e: frames from the host, the field from dgp_learn_wt (Farneback on the GPU); labels and marker index vectors fed from the host every step; locref maps built by dgp_locref_targets"},
            "allreduce": {"exposed_ms_last_step": exposed_ms, "path": "C ABI (dgp_allreduce_gradients)" if world > 1 else "none",
                          "note": "time between the end of the backward pass and the end of the gradient all-reduce on rank 0"},
            "clocks": clocks, "gpu_launches": launches, "loss_after": loss, "finite": bool(np.isfinite(loss)),
            "e2e": {"value": world * nt * e2e_steps / e2e_dt, "unit": "frames/s", "ms_per_step": 1e3 * e2e_dt / e2e_steps,
                    "h2d_bytes_per_step": int(frames_pinned.numel())
                                          + int(sum(np.asarray(v).nbytes for v in batch.values() if not isinstance(v, (int, list, torch.Tensor)))),
                    "d2h_bytes_per_step": 24, "timing": "wall clock, frames copied from pinned host memory, the Farneback flow-magnitude field of the batch computed on the device (dgp_learn_wt on a side stream beside the forward pass; the loss waits for its event) and the 6 loss values read back every step, max over ranks"},
            "ms_per_step_by_family": fam, "ms_per_step_with_events": ms_prof / args.steps,
            "tflops": {"forward_gemm": tf(flops_fwd, prof["conv_gemm"][0]), "dgrad_gemm": tf(flops_fwd, prof["dgrad_gemm"][0]),
                       "wgrad_gemm": tf(flops_fwd, prof["wgrad_gemm"][0]),
                       "step_total_3x_fwd": 3 * flops_fwd * n / (ms / 1e3) / 1e12, "peak": peak_tf, "peak_source": src,
                       "note": "algorithmic FLOPs: dgrad ~ wgrad ~ forward (conv1 has no dgrad; the 2 stride-2 dgrads run 4x zero-inserted)"},
        }
    eng.close()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--nt", type=int, default=10)
    ap.add_argument("--wt", type=float, default=1.0, help="temporal clique weight (0 = off)")
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--height", type=int, default=bench.H)
    ap.add_argument("--width", type=int, default=bench.W)
    ap.add_argument("--cpu-frames", type=int, default=0, help="also time the CPU restatement of the step on this many frames")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    line = measure(rank, local_rank, world, args.steps, args.warmup, args.nt, args.height, args.width, precision=args.precision,
                   wt=args.wt)
    if rank == 0:
        if args.cpu_frames > 0 and world == 1:
            sec, cores = cpu_train_step_seconds(args.cpu_frames, args.height, args.width, bench.NJ)
            line["cpu_baseline"] = {"value": args.cpu_frames / sec, "unit": "frames/s", "cores": cores, "kind": "port",
                                    "sample": "one step of %d frame(s): torch-CPU autograd through the oracle network + dgp_loss + "
                                              "Momentum, %.1f s (TF1.15 not installable)" % (args.cpu_frames, sec)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
