#!/usr/bin/env python
"""bench.py -- frames/sec of the DGP scoremap-and-graph hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one rank per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port) on the host cores
  python bench.py --steps K --warmup W --dump-outputs DIR  # ... and write what the last timed step returned as DIR/*.npy

Headline (`value`, every N): BASELINE.json configs[1] -- synthetic 4-bodypart reaching video, 747x832, estimate_pose
inference.  A "step" is one pass of the hot path over one batch of frames: ResNet-50 OS16 scoremap net + part_pred deconv
head + fused soft-argmax / peak / likelihood + skeleton & temporal potentials (+ the one-frame halo exchange when N > 1),
inputs resident in HBM.  `e2e` is the same workload through the public API with HOST buffers: a 10 000-frame (per GPU)
video streamed from pinned host memory through eval.estimate_pose_sharded -- H2D of every batch, D2H of the read-outs, and at
N > 1 the halo exchange, the potentials and the all-gather of the per-frame results inside the timed region.
Extra objects on the same line: `configs2` (configs[2]: 1280x1024, 16 bodyparts, frame-sharded across the N GPUs, with an
in-run bit-exactness check of the sharded result against a single-GPU recomputation), `configs4` (configs[4]: 640x480 x 20
bodyparts, dense skeleton, batch sweep 1..256), `train_step` (configs[3]),
`aux_bf16` (the same step in the bf16 storage mode), `roofline`, `roofline_aux`, `cpu_baseline`.
Prints ONE JSON line (rank 0).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the source tree as it found it (no __pycache__ of the modules it imports)

H, W, NJ = 747, 832, 4
METRIC = "frames/sec (ResNet-50 scoremap + DGP soft-argmax/potentials)"
WORKLOAD = "configs[1]: synthetic 4-bodypart reaching video 747x832, estimate_pose inference (part_pred head, chain skeleton)"
PRECISION = "fp16"   # the storage mode whose GPU tests assert BASELINE.json's tolerances (tests/test_gpu_forward.py)

CONFIGS = {  # BASELINE.json configs -> (H, W, num_joints, skeleton, label)
    "b": (747, 832, 4, "chain", WORKLOAD),
    "c": (1024, 1280, 16, "chain", "configs[2]: synthetic 1280x1024 video, 16 bodyparts with chain skeleton, frame-sharded estimate_pose inference"),
    "e": (480, 640, 20, "dense", "configs[4]: synthetic 640x480 videos x 20 bodyparts with dense skeleton (190 edges), estimate_pose inference"),
}


def conv_flops_per_frame(h, w, nj, locref=False):
    """Algorithmic forward FLOPs (2*MACs) of the conv + deconv layers (SURVEY.md 8d / Appendix B closed form)."""
    c2 = lambda v: -(-v // 2)
    total = 0
    hh, ww = c2(h), c2(w)
    total += 2 * hh * ww * 147 * 64
    hh, ww = c2(hh), c2(ww)
    cin = 64
    blocks = ((64, 3, 2), (128, 4, 2), (256, 6, 1), (512, 3, 1))  # stride as executed at output_stride 16
    for base, units, bstride in blocks:
        for u in range(units):
            s = bstride if u == units - 1 else 1
            depth = 4 * base
            ho, wo = c2(hh) if s == 2 else hh, c2(ww) if s == 2 else ww
            if cin != depth:
                total += 2 * hh * ww * cin * depth
            total += 2 * hh * ww * cin * base
            total += 2 * ho * wo * 9 * base * base
            total += 2 * ho * wo * base * depth
            hh, ww, cin = ho, wo, depth
    heads = nj * (3 if locref else 1)
    total += 2 * hh * ww * 2048 * 9 * heads
    return total, (2 * hh, 2 * ww)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


def csrc_sha():
    """Hash of the kernel sources: ncu-derived numbers under profiles/ are only quoted while they describe THIS code."""
    d = os.path.join(ROOT, "deepgraphpose_b200", "csrc")
    hsh = hashlib.sha256()
    for fn in sorted(os.listdir(d)):
        with open(os.path.join(d, fn), "rb") as f:
            hsh.update(fn.encode() + b"\0" + f.read())
    return hsh.hexdigest()[:16]


class ClockSampler:
    """SM clocks / throttle reasons sampled DURING the timed region (NVML every 2 ms; nvidia-smi as fallback)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index = index
        self.sm, self.bits = [], 0
        self.stop_flag = False
        self.active = False     # samples are kept only while the timed region runs
        self.ready = threading.Event()
        self.th = None
        self.max_mhz = None

    def _loop(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.ready.set()
            while not self.stop_flag:
                if self.active:
                    self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                    try:
                        self.bits |= int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                    except Exception:
                        self.bits |= int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                time.sleep(0.002)
        except Exception:
            self.ready.set()
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
                a, b = [float(x) for x in out.strip().split(",")]
                self.sm.append(a)
                self.max_mhz = b
            except Exception:
                pass

    def begin(self):
        """Call right before the timed region (the thread was started earlier so that NVML is already initialised)."""
        self.ready.wait(timeout=10)
        self.active = True

    def start(self):
        self.th = threading.Thread(target=self._loop, daemon=True)
        self.th.start()

    def stop(self):
        self.active = False
        self.stop_flag = True
        if self.th:
            self.th.join(timeout=5)
        reasons = sorted(n for b, n in self.REASONS.items() if self.bits & b)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(self.sm)}


def make_frame_pool(n_frames, seed=1234, h=None, w=None, nj=None):
    """n_frames distinct synthetic frames (uint8, T,H,W,3): a short seeded clip, extended by cyclic shifts."""
    from deepgraphpose_b200 import synthetic
    h, w, nj = h or H, w or W, nj or NJ
    base_n = min(n_frames, 16)
    base, _ = synthetic.make_video(base_n, h, w, nj, seed=seed)
    out = np.empty((n_frames, h, w, 3), np.uint8)
    for i in range(n_frames):
        out[i] = np.roll(base[i % base_n], shift=(3 * (i // base_n), 5 * (i // base_n)), axis=(0, 1))
    return out


def cpu_reference_fps(n_frames, warmup=1, threads=None):
    """The reference's CPU path (oracle restatement; TF1.15 is not installable here) on the host cores, batch 1 like
    eval.py:328.  Returns (fps, cores, seconds)."""
    from deepgraphpose_b200 import synthetic
    from oracle import dgp_ops, pose_net
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    Wn = synthetic.make_weights(NJ, seed=0, location_refinement=False)
    Wt = {k: torch.from_numpy(v) for k, v in Wn.items()}
    frames = make_frame_pool(max(2, min(n_frames, 4)))
    edges = synthetic.chain_skeleton(NJ)
    S0 = dgp_ops.skeleton_matrix(edges, NJ)

    def one(i):
        x = torch.from_numpy(frames[i % len(frames)][None].astype(np.float32))
        with torch.no_grad():
            net = pose_net.extract_features(x, Wt)
            pred = pose_net.prediction_layer(net, Wt, "part_pred")
            mu, _ = dgp_ops.argmax_2d_from_cm(pred, NJ, 1, 1)
        dgp_ops.estimate_pose_readout(mu.numpy(), pred.numpy())
        dgp_ops.skeleton_distances(mu, S0)
        return mu

    for i in range(warmup):
        one(i)
    t0 = time.perf_counter()
    for i in range(n_frames):
        one(i)
    dt = time.perf_counter() - t0
    return n_frames / dt, threads, dt


def headline_config(B, skeleton_kind, precision, world):
    """The `config` object of the JSON line: printed identically by both arms (the reference arm times the CPU path on the
    workload this describes; what it sampled of it is in its `cpu_baseline.sample`)."""
    return {"workload": WORKLOAD, "frames_per_step_per_gpu": B, "frame": [H, W, 3], "num_joints": NJ,
            "skeleton": skeleton_kind,
            "precision": "%s operands on tcgen05 kind::f16, fp32 accumulate / BN epilogue / logits: the mode whose GPU tests assert BASELINE.json's tolerances "
                         "(sigmoid 1e-2, soft-argmax 0.5 px, loss 1e-3) on all four inference shapes and the training step" % precision,
            "l2": "4 rotating input batches (%d MB) and per-layer activations (>600 MB/step) exceed the 126 MB L2" % (4 * B * H * W * 3 // 2 ** 20),
            "batch_choice": "engine.suggest_batch: tile counts of the persistent GEMM grid land on multiples of the SM count",
            "parallelism": "frame shards x%d, 1-frame halo all_gather" % world if world > 1 else "single GPU"}


def run_reference(args, rank):
    if rank != 0:
        return
    per_step = 2
    from deepgraphpose_b200.engine import suggest_batch      # pure host arithmetic: the batch size the other arm reports
    B = args.batch if args.batch > 0 else suggest_batch(H, W, *((12, 24) if args.config == "c" else (24, 48)))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    for _ in range(max(args.warmup, 1)):
        cpu_reference_fps(1, warmup=0)
    fps, cores, dt = cpu_reference_fps(per_step * args.steps, warmup=0)
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": headline_config(B, CONFIGS[args.config][3], args.precision, world),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": "%d frames of that workload (%d per step), batch 1 as eval.py:328, fp32, CPU restatement of the "
                                   "reference TF1 path (TF1.15 not installable: py3.12, no network)" % (per_step * args.steps, per_step)},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


class Workload:
    """One inference configuration on this rank: engine, device-resident input batches, pinned host pool, skeleton."""

    def __init__(self, key, local_rank, rank, precision, batch=0):
        from deepgraphpose_b200 import synthetic
        from deepgraphpose_b200.engine import Engine, suggest_batch
        self.key = key
        self.H, self.W, self.nj, self.skeleton_kind, self.label = CONFIGS[key]
        self.dev = torch.device("cuda", local_rank)
        self.B = batch if batch > 0 else suggest_batch(self.H, self.W, *((12, 24) if key == "c" else (24, 48)))
        self.eng = Engine(self.nj, location_refinement=False, device=local_rank, precision=precision)
        self.eng.load_weights(synthetic.make_weights(self.nj, seed=0, location_refinement=False))
        self.edges = synthetic.dense_skeleton(self.nj) if self.skeleton_kind == "dense" else synthetic.chain_skeleton(self.nj)
        self.flops_frame, (self.hs, self.ws) = conv_flops_per_frame(self.H, self.W, self.nj, locref=False)
        self.n_pool = 4
        # ONE video for all ranks (frame t = pool[t % P]): every rank reads its own contiguous range of it
        self.pool_host = torch.from_numpy(make_frame_pool(self.n_pool * self.B, seed=1234, h=self.H, w=self.W, nj=self.nj)).pin_memory()
        # device-resident batches for the kernel-level number: distinct per rank, together larger than the 126 MB L2
        self.pool = [torch.roll(self.pool_host[i * self.B:(i + 1) * self.B], shifts=7 * rank, dims=2).to(self.dev)
                     for i in range(self.n_pool)]
        self.ws_vec = np.full(len(self.edges), 1000.0 / 60.0, np.float32)
        self.ws_max = np.full(len(self.edges), 1.2 * 80.0, np.float32)

    def step(self, i, world):
        from deepgraphpose_b200 import sharding
        logits, _ = self.eng.forward(self.pool[i % self.n_pool], want_locref=False)
        out = self.eng.softargmax(logits, None, 1.0, 1.0, want=("mu", "peak", "lik"))
        halo = sharding.exchange_halo(out["mu"][0]) if world > 1 else None
        pot = self.eng.potentials(out["mu"], self.edges, halo_next=halo, ws=self.ws_vec, ws_max=self.ws_max, wt_max=0.0)
        return out, pot

    def close(self):
        self.eng.close()


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()


def max_over_ranks(x, world, dev):
    if world == 1:
        return x
    import torch.distributed as dist
    t = torch.tensor([x], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def measure_device(wl, steps, warmup, world, local_rank, profile=True):
    """K device-timed steps with inputs resident in HBM; the handle's event pairs around the GEMM run give the roofline."""
    sampler = ClockSampler(local_rank)
    sampler.start()
    for i in range(warmup):
        wl.step(i, world)
    torch.cuda.synchronize()
    barrier(world)
    sampler.begin()
    launches0 = wl.eng.launch_count()
    if profile:
        # The handle records one CUDA-event pair around every run of same-kind launches on the launching stream, IN the timed
        # steps: the 54 conv_gemm layers of a step are one run (the pool is fused into conv1), so their total is measured with
        # the programmatic-dependent-launch chaining of the real step intact (an event record between two layers would
        # serialise them; tools/instep_layers.py does that on purpose for the per-layer table).  The roofline therefore
        # describes the very steps `value` is computed from (a separate second pass ran ~1 % slower: hotter GPU).
        wl.eng.get_profile()
        wl.eng.set_profiling(2)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(steps):
        outputs = wl.step(i, world)
    e1.record()
    torch.cuda.synchronize()
    barrier(world)
    ms_local = e0.elapsed_time(e1)
    ms = max_over_ranks(ms_local, world, wl.dev)
    launches = wl.eng.launch_count() - launches0
    clocks = sampler.stop()
    prof, ms_prof = None, None
    if profile:
        wl.eng.set_profiling(False)
        prof = wl.eng.get_profile()
        ms_prof = ms_local
    return {"ms": ms, "launches": launches, "clocks": clocks, "prof": prof, "ms_prof": ms_prof,
            "value": world * wl.B * steps / (ms / 1e3), "outputs": outputs}


def measure_e2e(wl, frames_per_gpu, world):
    """The public API with HOST buffers: eval.estimate_pose_sharded streams a (world * frames_per_gpu)-frame video from
    pinned host memory (frame t = pool[t % P]) -- every rank its contiguous shard -- H2D per batch, D2H of the read-outs,
    halo exchange + potentials + all-gather of the per-frame results.  Wall clock between barriers, max over ranks."""
    from deepgraphpose_b200.eval import estimate_pose_sharded
    T = world * frames_per_gpu
    run = lambda n: estimate_pose_sharded(wl.eng, wl.pool_host, n, wl.H, wl.W, wl.edges, wl.ws_vec, wl.ws_max, 0.0, batch=wl.B)
    run(world * 2 * wl.B)     # warm-up: plans, pinned ring, NCCL communicator
    if world > 1:
        run(T)                # ... and NCCL's first all_gather at the full result size (70 ms once, tools/e2e_phases.py)
    torch.cuda.synchronize()
    barrier(world)
    t0 = time.perf_counter()
    res = run(T)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    barrier(world)
    dt = max_over_ranks(dt, world, wl.dev)
    return res, {"value": T / dt, "unit": "frames/s", "frames": T, "seconds": dt,
                 "h2d_bytes_per_step": wl.B * wl.H * wl.W * 3, "d2h_bytes_per_step": wl.B * wl.nj * (8 + 8 + 4),
                 "timing": "wall clock around eval.estimate_pose_sharded (synchronous public API: pinned host frames -> "
                           "streamed H2D per %d-frame batch -> forward + soft-argmax -> D2H of mu / peak / likelihood%s), "
                           "max over ranks" % (wl.B, "; halo all_gather + potentials + all_gather of the per-frame results" if world > 1 else "; potentials")}


def check_sharded_equals_single(wl, res, world, rank, k=8):
    """Bit-exactness of the sharded run IN the run: rank 0 recomputes the k frames around the first shard boundary on its
    own GPU in ONE batch (different batch composition, no halo needed) and compares mu / peak / likelihood / skeleton and
    temporal potentials with the gathered result bit for bit."""
    if world == 1:
        return None
    from deepgraphpose_b200 import sharding
    T = res["markers"].shape[0]
    b0 = sharding.shard_range(T, 0, world)[1]
    lo, hi = max(0, b0 - k // 2), min(T, b0 + k // 2)
    ok = True
    if rank == 0:
        P = wl.pool_host.shape[0]
        idx = torch.tensor([t % P for t in range(lo, hi)])
        frames = wl.pool_host[idx].to(wl.dev)
        logits, _ = wl.eng.forward(frames, want_locref=False)
        out = wl.eng.softargmax(logits, None, 1.0, 1.0, want=("mu", "peak", "lik"))
        pot = wl.eng.potentials(out["mu"], wl.edges, ws=wl.ws_vec, ws_max=wl.ws_max, wt_max=0.0)
        ok = (np.array_equal(out["mu"].cpu().numpy().astype(np.float64), res["markers"][lo:hi])
              and np.array_equal(out["peak"].cpu().numpy(), res["mu_likelihoods"][lo:hi])
              and np.array_equal(out["lik"].cpu().numpy().astype(np.float64), res["likelihoods"][lo:hi])
              and np.array_equal(pot["temporal"].cpu().numpy(), res["temporal"][lo:hi - 1])
              and np.array_equal(pot["skel"].t().cpu().numpy(), res["skel"][lo:hi]))
    return {"equal": bool(ok), "frames_checked": [lo, hi], "shard_boundary": b0,
            "what": "mu, integer peaks, likelihoods, skeleton distances, temporal potentials across the shard edge; bit for bit"}


def dump_outputs(outputs, out_dir):
    """Write the arrays one step returned (soft-argmax read-out and potentials) as out_dir/<name>.npy: float32 arrays as
    they are, integer ones (the peaks) as float64, which holds them exactly."""
    out, pot = outputs
    arrays = dict(out)
    arrays.update({k: v for k, v in pot.items() if not k.startswith("_") and v is not None})
    os.makedirs(out_dir, exist_ok=True)
    for name, t in sorted(arrays.items()):
        a = t.cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def roofline_of(wl, m, steps, peaks, peak_src):
    prof = m["prof"]
    gemm_ms, gemm_n = prof["conv_gemm"]
    frames_timed = wl.B * steps
    achieved_tf = wl.flops_frame * frames_timed / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else None
    peak_tf = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
    traffic, traffic_note = None, "no ncu --set full capture of the current kernel sources under profiles/"
    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(tpath) and wl.key == "b":
        with open(tpath) as f:
            tj = json.load(f)
        if tj.get("csrc_sha") == csrc_sha():
            traffic = tj["traffic_bytes_per_frame"] * wl.B / tj["gemm_launches_per_step"]
            traffic_note = ("dram__bytes_read.sum + dram__bytes_write.sum per conv_gemm launch (mean over the %d GEMM launches of a step) "
                            "from the ncu capture %s of these kernel sources (csrc sha %s, B=%d there); algorithmic minimum %.0f MB/launch"
                            % (tj["gemm_launches_per_step"], tj.get("source", "profiles/r02_launches_dram.csv"), tj["csrc_sha"], tj["batch"],
                               tj["minimum_bytes_per_frame_16bit"] * wl.B / tj["gemm_launches_per_step"] / 1e6))
        else:
            traffic_note = "profiles/r02_traffic.json describes other kernel sources (csrc sha %s != %s): not quoted" % (tj.get("csrc_sha"), csrc_sha())
    return {"bound": "tensor", "kernel": "conv_gemm_kernel (tcgen05 implicit GEMM, %d launches)" % gemm_n,
            "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
            "frac": (achieved_tf / peak_tf) if achieved_tf else None, "traffic": traffic, "traffic_note": traffic_note,
            "peak_source": peak_src + ", 16-bit dense sustained (cuBLAS bf16; fp16 runs at the same tensor rate)",
            "share_of_step": gemm_ms / m["ms_prof"],
            "timing": "CUDA events on the launching stream around each step's run of %d consecutive conv_gemm launches, recorded "
                      "in the timed steps themselves (%.3f ms/step); achieved = algorithmic FLOPs of the timed launches / their "
                      "summed duration" % (gemm_n // steps, m["ms_prof"] / steps),
            "algorithmic_gflop_per_frame": wl.flops_frame / 1e9}


def softargmax_roofline(local_rank, peaks):
    """GPU-filling soft-argmax measurement (the in-step launch moves 5 MB and is latency bound): 2-16 k maps of each BASELINE
    shape, far larger than the L2, CUDA events around 10 back-to-back stream + finalize pairs, best of 3 after warm-up."""
    from deepgraphpose_b200.engine import Engine
    out = {}
    for tag, (hs, ws, nj) in {"nj4_94x104": (94, 104, 4), "nj16_128x160": (128, 160, 16), "nj20_60x80": (60, 80, 20)}.items():
        # ~2.5-3 GB per call (0.5-0.7 ms of GPU time): the 10 queued calls stay device-bound even when the host threads of
        # several ranks share cores
        nmaps = 16384 if nj <= 4 else (2048 if nj == 16 else 8192)
        eng = Engine(nj, location_refinement=False, device=local_rank)
        x = torch.randn((nmaps, hs, ws, nj), device="cuda:%d" % local_rank) * 3.0
        for _ in range(3):
            eng.softargmax(x, None, 1.0, 1.0, want=("mu", "peak", "lik"))
        best = None
        reps = 10   # back-to-back calls per event pair: the queue stays full, so host-side dispatch time is not in the figure
        for _ in range(3):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                eng.softargmax(x, None, 1.0, 1.0, want=("mu", "peak", "lik"))
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b) / reps
            best = ms if best is None else min(best, ms)
        gbs = x.numel() * 4 / (best / 1e3) / 1e9
        out[tag] = {"maps": nmaps, "bytes": x.numel() * 4, "ms": best, "achieved": gbs, "unit": "GB/s",
                    "frac": gbs / peaks.get("hbm_gbs"), "calls_per_timing": reps}
        eng.close()
        del x
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=0, help="frames per step per GPU (0 = engine.suggest_batch)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the auxiliary training-step measurement (configs[3])")
    ap.add_argument("--no-aux", action="store_true", help="skip configs[2], the bf16 line and the soft-argmax microbenchmark")
    ap.add_argument("--config", default="b", choices=sorted(CONFIGS),
                    help="BASELINE.json workload of the headline: b = configs[1] (default), c = configs[2], e = configs[4]")
    ap.add_argument("--precision", default=PRECISION, choices=["fp16", "bf16"])
    ap.add_argument("--e2e-frames", type=int, default=10000, help="frames per GPU of the end-to-end video (configs[1]: 10 k)")
    ap.add_argument("--cpu-frames", type=int, default=64, help="frames of the workload the CPU baseline times (about 10 s on 16 cores)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline returned as DIR/<name>.npy (rank 0's frames); "
                         "the same arguments give the same inputs, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    global H, W, NJ, WORKLOAD
    H, W, NJ, skeleton_kind, WORKLOAD = CONFIGS[args.config]
    if args.config != "b":
        args.no_train = True

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    peaks, peak_src = load_peaks()
    # The soft-argmax microbenchmark is a kernel timed alone against the BURST HBM figure of MEASURED_PEAKS.json (a best-of-10
    # copy on a cool GPU): it runs first, before the sustained phases pull the SM clock down (the kernel is issue-bound, its
    # throughput follows the SM clock: 0.90 here vs 0.69 after a minute of GEMMs at nj = 4).
    sa_fill = softargmax_roofline(local_rank, peaks) if (rank == 0 and not args.no_aux) else None
    wl = Workload(args.config, local_rank, rank, args.precision, args.batch)
    m = measure_device(wl, args.steps, args.warmup, world, local_rank)
    if args.dump_outputs and rank == 0:
        dump_outputs(m["outputs"], args.dump_outputs)
    res, e2e = measure_e2e(wl, args.e2e_frames, world)
    finite = bool(np.isfinite(res["x"]).all())
    roof = roofline_of(wl, m, args.steps, peaks, peak_src) if rank == 0 else None
    sa_ms, sa_n = m["prof"]["softargmax"]
    fam = {k: v[0] for k, v in m["prof"].items()}
    B = wl.B
    wl.close()
    del wl
    torch.cuda.empty_cache()

    aux = {}
    if not args.no_aux:
        # ---- configs[2] (the multi-GPU workload north_star names): device-timed step + sharded e2e + in-run exactness
        if args.config != "c":
            wc = Workload("c", local_rank, rank, args.precision)
            mc = measure_device(wc, max(5, args.steps // 2), 3, world, local_rank)
            resc, e2ec = measure_e2e(wc, 2000, world)
            chk = check_sharded_equals_single(wc, resc, world, rank)
            if rank == 0:
                rc = roofline_of(wc, mc, max(5, args.steps // 2), peaks, peak_src)
                aux["configs2"] = {"workload": wc.label, "value": mc["value"], "unit": "frames/s", "ms_per_step": mc["ms"] / max(5, args.steps // 2),
                                   "frames_per_step_per_gpu": wc.B, "frame": [wc.H, wc.W, 3], "num_joints": wc.nj, "n_gpus": world,
                                   "parallelism": ("contiguous frame shards x%d, 1-frame halo" % world) if world > 1 else "single GPU",
                                   "e2e": e2ec, "sharded_equals_single": chk, "roofline_frac": rc["frac"],
                                   "finite": bool(np.isfinite(resc["x"]).all())}
            wc.close()
            del wc
            torch.cuda.empty_cache()
        # ---- the other storage mode, same step
        other = "bf16" if args.precision == "fp16" else "fp16"
        wo = Workload(args.config, local_rank, rank, other, B)
        mo = measure_device(wo, max(5, args.steps // 2), 3, world, local_rank)
        if rank == 0:
            ro = roofline_of(wo, mo, max(5, args.steps // 2), peaks, peak_src)
            aux["aux_" + other] = {"value": mo["value"], "unit": "frames/s", "ms_per_step": mo["ms"] / max(5, args.steps // 2), "roofline_frac": ro["frac"],
                                   "note": "same kernels and step with %s storage; its GPU tests assert %s" % (
                                       other, "wider, documented bounds (sigmoid <= 5e-2), not BASELINE's" if other == "bf16" else "BASELINE's tolerances")}
        wo.close()
        del wo
        torch.cuda.empty_cache()
    # ---- configs[4]: 640x480 videos x 20 bodyparts with a dense (190-edge) skeleton, throughput sweep over the batch size
    if not args.no_aux and args.config == "b":
        sweep = []
        for bsz in (1, 8, 32, 64, 128, 256):
            we = Workload("e", local_rank, rank, args.precision, bsz)
            n_steps = max(4, min(40, 512 // bsz))
            me = measure_device(we, n_steps, 3, world, local_rank, profile=False)
            sweep.append({"batch": bsz, "value": me["value"], "ms_per_step": me["ms"] / n_steps})
            finite_e = bool(torch.isfinite(we.step(0, world)[0]["mu"]).all().item())
            we.close()
            del we
            torch.cuda.empty_cache()
        if rank == 0:
            aux["configs4"] = {"workload": CONFIGS["e"][4], "unit": "frames/s", "n_gpus": world, "frame": [480, 640, 3], "num_joints": 20,
                               "skeleton_edges": 190, "sweep": sweep, "finite": finite_e,
                               "note": "device-resident inputs, the same step as the headline (forward + soft-argmax + potentials), frames per step per GPU = batch"}

    # ---- configs[3] alongside: one data-parallel DGP training step per rank (fwd + bwd + all-reduce + clip/Momentum)
    train_line = None
    if not args.no_train:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_train
            train_line = bench_train.measure(rank, local_rank, world, 20, 3, 10, H, W, profile=False, precision=args.precision)
        except Exception as ex:  # the headline line must survive a failure of the auxiliary measurement
            train_line = {"error": repr(ex)}
    if rank == 0:
        sa_bytes = 4 * (2 * -(-H // 16)) * (2 * -(-W // 16)) * NJ * B * args.steps
        line = {
            "metric": METRIC, "value": m["value"], "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": m["ms"] / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "config": headline_config(B, skeleton_kind, args.precision, world),
            "clocks": m["clocks"],
            "e2e": e2e,
            "gpu_launches": m["launches"],
            "roofline": roof,
            "roofline_aux": {"softargmax_in_step": {"bound": "hbm", "achieved": sa_bytes / (sa_ms / 1e3) / 1e9 if sa_ms > 0 else None,
                                                    "peak": peaks.get("hbm_gbs"), "unit": "GB/s", "launches": sa_n,
                                                    "note": "stream + finalize pair inside the step: 4.9 MB per batch, latency bound"},
                             "softargmax": sa_fill,
                             "ms_by_kernel_family": fam},
            "finite": finite,
        }
        line.update(aux)
        if train_line is not None:
            keep = ("metric", "value", "unit", "ms_per_step", "config", "gpu_launches", "loss_after", "finite", "e2e", "error", "dtype",
                    "allreduce")
            line["train_step"] = {k: train_line[k] for k in keep if k in train_line}
        if world == 1 and not args.no_cpu_baseline and args.config == "b":
            fps, cores, cdt = cpu_reference_fps(args.cpu_frames, warmup=1)
            line["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                                    "sample": "%d frames of the same workload, batch 1 (eval.py:328), %.1f s; CPU restatement of "
                                              "the reference TF1 path (TF1.15 not installable)" % (args.cpu_frames, cdt)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
