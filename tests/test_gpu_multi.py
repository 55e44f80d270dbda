"""Frame-sharded inference on 2 GPUs (NCCL halo) == single-GPU inference, bit for bit (SURVEY.md 8e exactness test).
Skipped on boxes with fewer than 2 GPUs."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, T, H, W, nj, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from deepgraphpose_b200 import sharding, synthetic
    from deepgraphpose_b200.engine import Engine
    frames, _ = synthetic.make_video(T, H, W, nj, seed=21)
    eng = Engine(nj, location_refinement=False, device=rank)
    eng.load_weights(synthetic.make_weights(nj, seed=0, location_refinement=False))
    edges = synthetic.chain_skeleton(nj)
    a, b = sharding.shard_range(T, rank, world)
    logits, _ = eng.forward(torch.from_numpy(frames[a:b]).cuda(rank))
    out = eng.softargmax(logits)
    halo = sharding.exchange_halo(out["mu"][0])
    pot = eng.potentials(out["mu"], edges, halo_next=halo)
    temporal = pot["temporal"]
    if halo is None:  # last shard has no frame after its last one
        temporal = torch.cat([temporal, torch.zeros(1, nj, device=temporal.device)])
    full = {k: sharding.gather_frames(v, T) for k, v in
            dict(mu=out["mu"], peak=out["peak"], lik=out["lik"], temporal=temporal, skel=pot["skel"].t().contiguous()).items()}
    if rank == 0:
        np.savez(os.path.join(out_dir, "sharded.npz"), **{k: v.cpu().numpy() for k, v in full.items()})
    dist.barrier()
    dist.destroy_process_group()


def test_two_gpu_shards_match_single_gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from deepgraphpose_b200 import synthetic
    from deepgraphpose_b200.engine import Engine
    T, H, W, nj = 9, 96, 128, 4
    mp.spawn(_worker, args=(2, 29533, T, H, W, nj, str(tmp_path)), nprocs=2, join=True)
    got = np.load(os.path.join(str(tmp_path), "sharded.npz"))
    frames, _ = synthetic.make_video(T, H, W, nj, seed=21)
    eng = Engine(nj, location_refinement=False, device=0)
    eng.load_weights(synthetic.make_weights(nj, seed=0, location_refinement=False))
    logits, _ = eng.forward(torch.from_numpy(frames).cuda(0))
    out = eng.softargmax(logits)
    pot = eng.potentials(out["mu"], synthetic.chain_skeleton(nj))
    assert np.array_equal(got["mu"], out["mu"].cpu().numpy())
    assert np.array_equal(got["peak"], out["peak"].cpu().numpy())
    assert np.array_equal(got["lik"], out["lik"].cpu().numpy())
    assert np.array_equal(got["temporal"][: T - 1], pot["temporal"].cpu().numpy())
    assert np.array_equal(got["skel"], pot["skel"].t().cpu().numpy())
    eng.close()


def _sharded_worker(rank, world, port, T, H, W, nj, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from deepgraphpose_b200 import eval as dgp_eval
    from deepgraphpose_b200 import synthetic
    from deepgraphpose_b200.engine import Engine
    frames, _ = synthetic.make_video(T, H, W, nj, seed=22)
    eng = Engine(nj, location_refinement=False, device=rank)
    eng.load_weights(synthetic.make_weights(nj, seed=0, location_refinement=False))
    res = dgp_eval.estimate_pose_sharded(eng, torch.from_numpy(frames).pin_memory(), T, H, W, synthetic.chain_skeleton(nj),
                                         np.full(nj - 1, 9.0, np.float32), np.full(nj - 1, 70.0, np.float32), 0.0, batch=3)
    if rank == 0:
        np.savez(os.path.join(out_dir, "sharded_entry.npz"), **{k: v for k, v in res.items() if k != "shard"})
    dist.barrier()
    dist.destroy_process_group()
    eng.close()


def test_estimate_pose_sharded_entry_matches_single_gpu(tmp_path):
    """eval.estimate_pose_sharded on 2 ranks (streamed host frames -> halo -> potentials -> gather) == the same call on one."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from deepgraphpose_b200 import eval as dgp_eval
    from deepgraphpose_b200 import synthetic
    from deepgraphpose_b200.engine import Engine
    T, H, W, nj = 11, 96, 128, 4
    mp.spawn(_sharded_worker, args=(2, 29551, T, H, W, nj, str(tmp_path)), nprocs=2, join=True)
    got = np.load(os.path.join(str(tmp_path), "sharded_entry.npz"))
    frames, _ = synthetic.make_video(T, H, W, nj, seed=22)
    eng = Engine(nj, location_refinement=False, device=0)
    eng.load_weights(synthetic.make_weights(nj, seed=0, location_refinement=False))
    ref = dgp_eval.estimate_pose_sharded(eng, torch.from_numpy(frames).pin_memory(), T, H, W, synthetic.chain_skeleton(nj),
                                         np.full(nj - 1, 9.0, np.float32), np.full(nj - 1, 70.0, np.float32), 0.0, batch=4)
    for k in ("x", "y", "likelihoods", "mu_likelihoods", "markers", "temporal", "skel", "e_skel", "e_temp"):
        assert np.array_equal(got[k], ref[k]), k
    eng.close()


CHECK_VARS = ("resnet_v1_50/conv1/weights", "resnet_v1_50/block2/unit_1/bottleneck_v1/conv2/weights",
              "resnet_v1_50/block4/unit_3/bottleneck_v1/conv3/BatchNorm/gamma", "pose/part_pred/block4/weights",
              "pose/locref_pred/block4/biases")


def _train_setup(rank_seed):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import test_gpu_train as T
    W, frames, batch, edges, S0, cfg, ws, ws_max = T._setup(seed=3)
    from deepgraphpose_b200 import synthetic
    frames, _ = synthetic.make_video(T.NT, T.HIN, T.WIN, T.NJ, seed=50 + rank_seed)   # each replica draws its own batch
    return T, W, frames, batch, edges, cfg, ws, ws_max


def _train_worker(rank, world, port, out_dir, attach=True):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from deepgraphpose_b200 import dp, fitdgp
    from deepgraphpose_b200.engine import Engine
    T, W, frames, batch, edges, cfg, ws, ws_max = _train_setup(rank)
    eng = Engine(T.NJ, device=rank)
    eng.load_weights(W)
    if attach:
        assert dp.attach_comm(eng) == world      # the C handle owns the communicator and the bucketed all-reduce
    fr = torch.from_numpy(frames).cuda(rank)
    for _ in range(2):
        fitdgp.train_forward_backward(eng, fr, batch, cfg, edges, ws, ws_max, 200, 20)
        scale = dp.allreduce_gradients(eng)
        eng.optimizer_step(0.005, 0.9, 10.0, scale)
    assert eng.lib.dgp_comm_world_size(eng.h) == world      # without attach_comm: attached by the first allreduce_gradients
    same = dp.broadcast_check(eng, CHECK_VARS)
    if rank == 0:
        np.savez(os.path.join(out_dir, "dp.npz"), same=np.array(same), **{k.replace("/", "."): eng.get_variable(k) for k in CHECK_VARS})
    dist.barrier()
    dist.destroy_process_group()
    eng.close()


@pytest.mark.parametrize("attach", [True, False], ids=["c-abi-comm", "attach-on-first-use"])
def test_two_gpu_data_parallel_training_matches_mean_gradient(tmp_path, attach):
    """2 NCCL replicas with different batches, all-reduced gradients (dgp_allreduce_gradients inside the C ABI, with the
    communicator attached up front or, as fit_dgp does, by the first dp.allreduce_gradients), replicated clip + Momentum ==
    one process that averages the two batches' gradients itself (bit for bit: a two-rank sum is order independent)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from deepgraphpose_b200 import fitdgp
    from deepgraphpose_b200.engine import Engine
    mp.spawn(_train_worker, args=(2, 29541 + int(attach), str(tmp_path), attach), nprocs=2, join=True)
    got = np.load(os.path.join(str(tmp_path), "dp.npz"))
    assert bool(got["same"])
    engs, frs = [], []
    for r in range(2):
        T, W, frames, batch, edges, cfg, ws, ws_max = _train_setup(r)
        e = Engine(T.NJ, device=0)
        e.load_weights(W)
        engs.append(e)
        frs.append(torch.from_numpy(frames).cuda(0))
    for _ in range(2):
        for e, fr in zip(engs, frs):
            fitdgp.train_forward_backward(e, fr, batch, cfg, edges, ws, ws_max, 200, 20)
        total = engs[0].grad_buffer() + engs[1].grad_buffer()
        for e in engs:
            e.grad_buffer().copy_(total)
            e.optimizer_step(0.005, 0.9, 10.0, 0.5)
    for k in CHECK_VARS:
        assert np.array_equal(got[k.replace("/", ".")], engs[0].get_variable(k)), k
    for e in engs:
        e.close()
