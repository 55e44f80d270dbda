"""Every CUDA resource of libdgp_b200.so has one owner (csrc/owned.cuh): nothing else releases one, and a handle's whole
lifecycle -- plan eviction, training, estimate_pose, the entry points with temporary buffers -- gives back all it took."""
import ctypes as C
import gc
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RELEASE_CALLS = ("cudaFree(", "cudaFreeHost(", "cudaEventDestroy(", "cudaStreamDestroy(", "cudaGraphDestroy(",
                 "cudaGraphExecDestroy(")


def test_only_the_owner_types_release_cuda_resources():
    csrc = os.path.join(ROOT, "deepgraphpose_b200", "csrc")
    found = []
    for fn in sorted(os.listdir(csrc)):
        if fn == "owned.cuh":
            continue
        src = open(os.path.join(csrc, fn)).read()
        found += [(fn, call) for call in RELEASE_CALLS if call in src]
    assert found == []


def _live(lib):
    objects, device_bytes = C.c_int64(), C.c_int64()
    assert lib.dgp_debug_live_resources(C.byref(objects), C.byref(device_bytes)) == 0
    return objects.value, device_bytes.value


@pytest.mark.gpu
def test_handle_lifecycle_releases_every_resource():
    import torch

    from deepgraphpose_b200 import _lib, fitdgp, synthetic
    from deepgraphpose_b200.engine import Engine
    from oracle import dgp_loss as oracle_loss
    from oracle import dgp_ops
    from test_gpu_loss import make_batch

    nj = 4
    lib = _lib.load()
    gc.collect()
    gc.disable()  # an engine of another test finalized in the middle would move the process-wide counts
    try:
        base = _live(lib)
        eng = Engine(nj)
        eng.load_weights(synthetic.make_weights(nj, seed=3))
        assert _live(lib)[1] > base[1]

        def video(n, H, W, seed):
            return torch.from_numpy(synthetic.make_video(n, H, W, nj, seed=seed)[0]).cuda()

        # 7 shapes: the inference plan cache keeps 6, so the least recently used plan is evicted
        for k in range(7):
            eng.forward(video(2, 64 + 16 * k, 96, k))
        # fused and split training steps at 4 shapes: the training plan cache keeps 3; the second backward of a shape
        # replays a captured graph
        eng.train_enable()
        edges = synthetic.chain_skeleton(nj)
        S0 = dgp_ops.skeleton_matrix(edges, nj)
        cfg = oracle_loss.default_dgp_cfg(gm2=1, gm3=3, wt=0.0)
        rng = np.random.default_rng(0)
        for k in range(4):
            Hin, Win = 64 + 16 * k, 96
            fr = video(3, Hin, Win, 20 + k)
            labels, batch = make_batch(rng, 3, 2 * -(-Hin // 16), 2 * -(-Win // 16), nj, [0, 2], ((0, 1),))
            ws, ws_max = oracle_loss.spatial_clique_params(labels, S0, cfg)
            fitdgp.train_forward_backward(eng, fr, batch, cfg, edges, ws, ws_max, 200, 20)
            logits, locref, token = eng.train_forward(fr)
            eng.train_backward(token, torch.ones_like(logits), torch.zeros_like(locref))
            eng.optimizer_step()
        # estimate_pose from host frames with a transform, and streamed from a generator
        frames = synthetic.make_video(5, 120, 160, nj, seed=40)[0]
        eng.estimate_pose_host(torch.from_numpy(frames), batch=2, new_size=(96, 128))
        eng.estimate_pose_stream(iter(frames), 120, 160, 5, batch=2)
        # augment, learn_wt, softmax_map / soft_pose
        fr = video(3, 64, 96, 50)
        base_p = dict(rotate_deg=0.0, blur_k=0, blur_angle_deg=0.0, blur_direction=0.0, drop_p=0.0, drop_size_percent=0.0,
                      elastic_alpha=0.0, elastic_sigma=5.0, seed=0)
        eng.augment(fr, [0, 2], None, [dict(base_p, rotate_deg=10.0, elastic_alpha=30.0, seed=1),
                                       dict(base_p, blur_k=5, drop_p=0.1, drop_size_percent=0.2, seed=2)])
        eng.learn_wt(fr)
        logits, locref = eng.forward(fr)
        eng.softmax_map(logits)
        eng.soft_pose(logits, locref)
        torch.cuda.synchronize()

        # the entry points with temporary device buffers give all of them back before they return
        net = eng.extract_features(fr)
        rng = np.random.default_rng(1)
        x_deconv = torch.from_numpy(rng.standard_normal((2, 5, 7, 256)).astype(np.float32)).cuda()
        w_deconv = (rng.standard_normal((3, 3, 7, 256)) * 0.05).astype(np.float32)
        x_conv = torch.from_numpy(rng.standard_normal((2, 13, 17, 64)).astype(np.float32)).to(eng.act_dtype).cuda()
        w_conv = (rng.standard_normal((1, 1, 64, 64)) * 0.05).astype(np.float32)
        calls = {"prediction_layers": lambda: eng.prediction_layers(net),
                 "deconv2d": lambda: eng.deconv2d(x_deconv, w_deconv, np.ones(7, np.float32)),
                 "conv2d": lambda: eng.conv2d(x_conv, w_conv)}
        for name, call in calls.items():
            before = _live(lib)
            call()
            assert _live(lib) == before, name

        eng.close()
        assert _live(lib) == base
    finally:
        gc.enable()
