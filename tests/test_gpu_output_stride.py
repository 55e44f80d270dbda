"""Pose nets at slim output_stride 8 on the GPU (atrous blocks 3 and 4, stride-4 scoremaps) against the fp32 oracle at the
same geometry: inference parity at the north-star tolerances, every unit's shape, the consistency of the entry points,
training against oracle autograd, the fit_dgp drivers, checkpoints, the fused render / JPEG passes and 2-GPU runs."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import os8_oracle
from deepgraphpose_b200 import synthetic
from oracle import dgp_loss as oracle_loss
from oracle import dgp_ops

pytestmark = pytest.mark.gpu

SIGMOID_TOL = 1e-2     # BASELINE.json north_star, asserted in the fp16 storage mode
MU_TOL_PX = 0.5
OS = 8
SHAPES = [(2, 235, 301), (1, 470, 640), (3, 64, 96), (2, 101, 75), (1, 747, 832)]   # test_gpu_depths.SHAPES


def _engine(W, nj, locref=True, device=None, output_stride=OS):
    from deepgraphpose_b200.engine import Engine
    eng = Engine(nj, location_refinement=locref, device=device, output_stride=output_stride)
    eng.load_weights(W)
    return eng


@pytest.fixture(scope="module")
def sets50():
    nj = 4
    sets = {}
    for tl in (False, True):
        W = synthetic.make_weights(nj, seed=0, trained_like=tl)
        sets[tl] = (W, {k: torch.from_numpy(v) for k, v in W.items()}, _engine(W, nj))
    yield nj, sets
    for _, _, e in sets.values():
        e.close()


def _parity(eng, Wt, net_type, nj, shape, label):
    T, H, Wd = shape
    frames, _ = synthetic.make_video(T, H, Wd, nj, seed=H)
    ep = {}
    with torch.no_grad():
        pred, loc = os8_oracle.heads(torch.from_numpy(frames.astype(np.float32)), Wt, net_type, OS, True, ep)
    eng.keep_activations(True)
    logits, locref = eng.forward(torch.from_numpy(frames).cuda())
    torch.cuda.synchronize()
    eng.keep_activations(False)
    assert torch.equal(eng.forward(torch.from_numpy(frames).cuda())[0], logits)    # fused conv1+pool plan, same values
    worst = 0.0
    for name, ref in ep.items():
        got = torch.from_numpy(eng.get_activation(name))
        assert got.shape == ref.shape, name
        worst = max(worst, (got - ref).abs().max().item() / ref.abs().max().item())
    assert logits.shape == pred.shape and locref.shape == loc.shape
    assert logits.shape[1:3] == eng.output_dims(H, Wd)[1]
    sig = (torch.sigmoid(logits.cpu()) - torch.sigmoid(pred)).abs().max().item()
    out = eng.softargmax(logits, locref)
    mu_oracle, _ = dgp_ops.argmax_2d_from_cm(pred, nj, 1.0, 1.0)
    mu_err = (out["mu"].cpu() - mu_oracle).abs().max().item()
    print("output_stride 8 %s %s %s: activations max rel %.2e, sigmoid %.2e, soft-argmax %.4f px"
          % (net_type, shape, label, worst, sig, mu_err))
    assert len(ep) == 2 + sum(synthetic.BLOCK_UNITS[net_type])
    assert mu_err < MU_TOL_PX
    for t in range(T):   # integer peaks from the same fp32 maps: bit-exact
        _, pk, _ = dgp_ops.estimate_pose_readout(out["mu"][t:t + 1].cpu().numpy(), logits[t:t + 1].cpu().numpy())
        assert (pk == out["peak"][t].cpu().numpy()).all(), t
    return sig


@pytest.mark.parametrize("trained_like", [False, True], ids=["random-init", "trained-like"])
@pytest.mark.parametrize("shape", SHAPES)
def test_inference_parity_resnet_50(sets50, shape, trained_like):
    nj, sets = sets50
    W, Wt, eng = sets[trained_like]
    sig = _parity(eng, Wt, "resnet_50", nj, shape, "trained_like=%s" % trained_like)
    assert sig <= SIGMOID_TOL


def test_inference_parity_resnet_101():
    nj = 4
    W = synthetic.make_weights(nj, seed=0, net_type="resnet_101")
    eng = _engine(W, nj)
    sig = _parity(eng, {k: torch.from_numpy(v) for k, v in W.items()}, "resnet_101", nj, (2, 235, 301), "random-init")
    eng.close()
    assert sig <= SIGMOID_TOL


@pytest.mark.parametrize("net_type", ["resnet_50", "resnet_101", "resnet_152"])
def test_every_unit_has_the_oracle_shape(net_type):
    """Block 2 keeps block 1's resolution, and blocks 3 and 4 keep it too (rates 2 and 4)."""
    nj, T, H, W = 2, 1, 101, 75
    eng = _engine(synthetic.make_weights(nj, seed=1, location_refinement=False, net_type=net_type), nj, locref=False)
    frames, _ = synthetic.make_video(T, H, W, nj, seed=2)
    eng.keep_activations(True)
    eng.forward(torch.from_numpy(frames).cuda())
    torch.cuda.synchronize()
    want = os8_oracle.unit_shapes(H, W, net_type, OS)
    assert len(want) == sum(synthetic.BLOCK_UNITS[net_type])
    for scope, (h, w, c) in want.items():
        assert eng.get_activation(scope).shape == (T, h, w, c), scope
    eng.close()


def test_entry_points_agree(tmp_path, sets50):
    """extract_features + prediction_layers == forward bit for bit; a frame's outputs do not depend on its batch; an OS8 and an
    OS16 handle on the same weights give different scoremap shapes; estimate_pose (file and array) == estimate_pose_frames."""
    from deepgraphpose_b200 import eval as dgp_eval
    from deepgraphpose_b200.pose_net import PoseNet
    nj, sets = sets50
    W, _, eng = sets[True]
    frames, _ = synthetic.make_video(3, 235, 301, nj, seed=7)
    fr = torch.from_numpy(frames).cuda()
    logits, locref = eng.forward(fr)
    net = eng.extract_features(fr)
    assert net.shape == (3, 30, 38, 2048)
    l2, r2 = eng.prediction_layers(net)
    assert torch.equal(l2, logits) and torch.equal(r2, locref)
    for t in range(3):
        l1, r1 = eng.forward(fr[t:t + 1].contiguous())
        assert torch.equal(l1, logits[t:t + 1]) and torch.equal(r1, locref[t:t + 1]), t
    e16 = _engine(W, nj, output_stride=16)
    assert e16.forward(fr)[0].shape == (3, 30, 38, nj) and logits.shape == (3, 60, 76, nj)
    e16.close()
    pn = PoseNet({"num_joints": nj, "output_stride": 8, "stride": 4.0}, variables=W)
    assert pn.engine.output_stride == 8 and pn.engine.stride == 4.0
    assert torch.equal(pn.get_net(frames)["part_pred"], logits)
    pn.engine.close()
    cv2 = pytest.importorskip("cv2")
    T, H, Wd = 6, 96, 128
    Wv = synthetic.make_weights(nj, seed=4, location_refinement=False)
    vid, _ = synthetic.make_video(T, H, Wd, nj, seed=6)
    path = str(tmp_path / "reach.avi")
    vw = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 10.0, (Wd, H))
    if not vw.isOpened():
        pytest.skip("no MJPG encoder in this OpenCV build")
    for f in vid:
        vw.write(f[:, :, ::-1])
    vw.release()
    decoded = np.stack(list(dgp_eval._iter_video(path)))
    cfg = {"num_joints": nj, "all_joints_names": ["a", "b", "c", "d"], "stride": 4.0, "output_stride": 8}
    from_file = dgp_eval.estimate_pose(cfg, Wv, path, str(tmp_path), save_pose=False, batch=4)
    in_memory = dgp_eval.estimate_pose(cfg, Wv, decoded, str(tmp_path), save_pose=False, batch=4)
    for k in ("x", "y", "likelihoods"):
        assert np.array_equal(from_file[k], in_memory[k]), k
    e = _engine(Wv, nj, locref=False)
    ref = dgp_eval.estimate_pose_frames(e, decoded, batch=4)
    for k in ("x", "y", "likelihoods"):
        assert np.array_equal(ref[k], in_memory[k]), k
    assert np.array_equal(ref["x"], ref["markers"][:, :, 1] * 4.0 + 2.0)
    assert np.array_equal(ref["y"], ref["markers"][:, :, 0] * 4.0 + 2.0)
    lg, _ = e.forward(torch.from_numpy(decoded).cuda())
    mu = e.softargmax(lg, None, want=("mu",))["mu"].cpu().numpy().astype(np.float64)
    assert lg.shape[1:3] == (24, 32) and np.array_equal(mu, ref["markers"])
    e.close()


# ---------------------------------------------------------------- training at output stride 8
NJ, NT, HIN, WIN = 4, 3, 64, 96
HS, WS = 2 * -(-HIN // 8), 2 * -(-WIN // 8)
TRAINABLE = ("/weights", "/BatchNorm/gamma", "/BatchNorm/beta", "/biases")


def _train_setup(seed=3):
    from test_gpu_loss import make_batch
    rng = np.random.default_rng(seed)
    W = synthetic.make_weights(NJ, seed=seed)
    frames, _ = synthetic.make_video(NT, HIN, WIN, NJ, seed=11)
    labels, batch = make_batch(rng, NT, HS, WS, NJ, [0, 2], ((0, 1),))
    edges = synthetic.chain_skeleton(NJ)
    S0 = dgp_ops.skeleton_matrix(edges, NJ)
    cfg = oracle_loss.default_dgp_cfg(gm2=1, gm3=3, wt=0.0, stride=4.0)
    ws, ws_max = oracle_loss.spatial_clique_params(labels, S0, cfg)
    return W, frames, batch, edges, S0, cfg, ws, ws_max * 0.3


def _step(eng, fr, s):
    from deepgraphpose_b200 import fitdgp
    W, frames, batch, edges, S0, cfg, ws, ws_max = s
    return fitdgp.train_forward_backward(eng, fr, batch, cfg, edges, ws, ws_max, 200, 20)


def test_training_matches_oracle_autograd():
    s = _train_setup()
    W, frames, batch, edges, S0, cfg, ws, ws_max = s
    Wt = {k: torch.from_numpy(v.copy()).requires_grad_(k.endswith(TRAINABLE)) for k, v in W.items()}
    pred, loc = os8_oracle.heads(torch.from_numpy(frames.astype(np.float32)), Wt, "resnet_50", OS, True)
    assert pred.shape == (NT, HS, WS, NJ)
    loss, total, _ = oracle_loss.dgp_loss_from_heads(pred, loc, batch, cfg, S0, ws, ws_max, 200, 20)
    total.backward()
    eng = _engine(W, NJ)
    fr = torch.from_numpy(frames).cuda()
    got = _step(eng, fr, s)
    assert abs(float(got["total_loss"]) - float(total.detach())) <= 1e-3 * abs(float(total.detach())), (got, loss)
    rows, bad = [], []
    for name, t in sorted(Wt.items()):
        if not t.requires_grad:
            continue
        g, g_ref = eng.get_variable(name, "grad"), t.grad.numpy()
        assert g.shape == g_ref.shape, name
        nr = float(np.linalg.norm(g_ref))
        if nr == 0.0:
            assert float(np.abs(g).max()) == 0.0, name
            continue
        cos = float((g * g_ref).sum() / (np.linalg.norm(g) * nr + 1e-30))
        rel = float(np.linalg.norm(g - g_ref) / nr)
        rows.append((name, cos, rel))
        if not (cos > 0.995 and rel < 0.10):
            bad.append((name, cos, rel))
    print("output stride 8 gradients: median cosine %.5f, median rel-L2 %.4f, worst rel-L2 %.4f"
          % (np.median([r[1] for r in rows]), np.median([r[2] for r in rows]), max(r[2] for r in rows)))
    assert not bad, bad[:8]
    eng2 = _engine(W, NJ)    # bitwise reproducible: a second handle, same batch
    _step(eng2, fr, s)
    assert torch.equal(eng.grad_buffer(), eng2.grad_buffer())
    eng.close()
    eng2.close()


def test_tf_checkpoint_resume(tmp_path):
    """Two steps, save, a fresh OS8 handle restored from the bundle, one more step on both: bitwise identical."""
    from deepgraphpose_b200 import tf_checkpoint
    from deepgraphpose_b200.eval import load_variables
    s = _train_setup(seed=17)
    fr = torch.from_numpy(s[1]).cuda()
    a = _engine(s[0], NJ)
    for _ in range(2):
        _step(a, fr, s)
        a.optimizer_step(0.005, 0.9, 10.0, 1.0)
    prefix = str(tmp_path / "snapshot-step2-final--0")
    a.save_tf_checkpoint(prefix, global_step=2)
    full = tf_checkpoint.read_checkpoint(prefix, verify=True)
    b = _engine(load_variables(prefix, NJ, True), NJ)
    b.train_enable()
    for n in b.variable_names():
        b.set_variable(n, full[n + "/Momentum"], "momentum")
    for e in (a, b):
        _step(e, fr, s)
        e.optimizer_step(0.005, 0.9, 10.0, 1.0)
    for n in a.variable_names():
        assert np.array_equal(a.get_variable(n), b.get_variable(n)), n
    assert torch.equal(a.forward(fr)[0], b.forward(fr)[0])
    a.close()
    b.close()


def _os8_batcher(seed):
    import test_gpu_drivers as drv
    b = drv._Batcher(seed=seed)
    b.H, b.W = 2 * -(-drv.HIN // 8), 2 * -(-drv.WIN // 8)
    rng = np.random.default_rng(seed)
    b.labels = np.stack([rng.uniform(1, b.H - 2, (3, drv.NJ)), rng.uniform(1, b.W - 2, (3, drv.NJ))], axis=2)
    b.datasets = [drv._Dataset(b.labels, b.H, b.W)]
    return b


def test_fit_dgp_drivers_train():
    import test_gpu_drivers as drv
    from deepgraphpose_b200 import fitdgp
    cfg = drv._cfg(stride=4.0, output_stride=8)
    b = _os8_batcher(3)
    frame_lists = ([b.visible], [np.array([], dtype=np.int64)], [np.arange(drv.NT)])
    windows = [np.array([0, 1, 2, 3, 0], dtype=np.int32), np.array([4, 5, 6, 7, 0], dtype=np.int32)] * 3
    engines = []
    hist = fitdgp.fit_dgp("synthetic:0", "/nonexistent", batch_size=4, gm2=1, gm3=3, wt=0, saveiters=100, displayiters=100,
                          data_batcher=b, dgp_cfg=cfg, frame_lists=frame_lists, batch_ind_all=windows,
                          snapshot_fn=lambda eng, name, it: engines.append((eng.output_stride, eng.stride)), verbose=False)
    tot = [float(h["total_loss"]) for h in hist]
    assert len(hist) == 6 and all(np.isfinite(tot)) and tot[4] < tot[0] and tot[5] < tot[1]
    assert engines and set(engines) == {(8, 4.0)}
    b = _os8_batcher(4)
    hist = fitdgp.fit_dgp_labeledonly("synthetic:0", "/nonexistent", saveiters=100, data_batcher=b, dgp_cfg=cfg,
                                      frame_lists=frame_lists, batch_ind_all=[np.array([5, 0])] * 4, snapshot_fn=lambda *a: None,
                                      verbose=False)
    vis = [float(h["visible_loss_pred"]) + float(h["visible_loss_locref"]) for h in hist]
    assert len(hist) == 4 and vis[-1] < vis[0]


@pytest.mark.parametrize("hw", [(188, 208), (256, 320)], ids=["747x832", "1024x1280"])
def test_loss_at_stride_4_matches_oracle_autograd(hw):
    """The loss kernels on OS8 scoremaps (a 256x320 plane is 320 KB: past the shared-memory staging of the marker kernels, so
    their global-memory path runs) with the temporal clique on a (nt-1, 4H, 4W) flow field, against oracle autograd."""
    from test_gpu_loss import LOSS_REL_TOL, make_batch
    from deepgraphpose_b200 import fitdgp
    from deepgraphpose_b200.engine import Engine
    rng = np.random.default_rng(29)
    nt, nj = 3, 4
    H, W = hw
    labels, batch = make_batch(rng, nt, H, W, nj, [0, 2], ((0, 1),))
    pred = torch.from_numpy((rng.standard_normal((nt, H, W, nj)) * 2).astype(np.float32)).requires_grad_(True)
    loc = torch.from_numpy(rng.standard_normal((nt, H, W, 2 * nj)).astype(np.float32)).requires_grad_(True)
    edges = synthetic.chain_skeleton(nj)
    S0 = dgp_ops.skeleton_matrix(edges, nj)
    cfg = oracle_loss.default_dgp_cfg(gm2=1, gm3=3, wt=20.0, stride=4.0)
    yy, xx = np.meshgrid(np.arange(4 * H), np.arange(4 * W), indexing="ij")
    batch["vector_field_tf"] = np.stack([0.9 + 0.8 * np.sin(yy / (29.0 + t)) * np.cos(xx / (37.0 + 2 * t)) for t in range(nt - 1)])
    batch["wt_batch_pl"] = np.ones(nt - 1) * 20.0
    batch["wt_batch_mask_pl"] = np.array([1.0, 1.0])
    ws, ws_max = oracle_loss.spatial_clique_params(labels, S0, cfg)
    ws_max = ws_max * 0.3
    ref, ref_total, _ = oracle_loss.dgp_loss_from_heads(pred, loc, batch, cfg, S0, ws, ws_max, 200, 20)
    ref_total.backward()
    ref = {k: float(v.detach()) if isinstance(v, torch.Tensor) else float(v) for k, v in ref.items()}
    eng = Engine(nj, output_stride=8)
    assert eng.stride == 4.0
    got, (g_pred, g_loc) = fitdgp.loss_forward(eng, pred.detach().cuda(), loc.detach().cuda(), batch, cfg, edges, ws, ws_max,
                                               200, 20, backward=True)
    for k, v in ref.items():
        assert abs(float(got[k]) - float(v)) <= LOSS_REL_TOL * max(abs(float(v)), 1e-6), (k, float(got[k]), float(v))
    gp, gl = pred.grad, loc.grad
    assert (g_pred.cpu() - gp).abs().max().item() <= 2e-3 * gp.abs().max().item() + 1e-9, \
        ((g_pred.cpu() - gp).abs().max().item(), gp.abs().max().item())
    assert (g_loc.cpu() - gl).abs().max().item() <= 1e-4 * gl.abs().max().item() + 1e-12
    out = eng.softargmax(pred.detach().cuda(), None, want=("mu", "peak"))
    mu_ref, _ = dgp_ops.argmax_2d_from_cm(pred.detach(), nj, 1.0, 1.0)
    assert (out["mu"].cpu() - mu_ref).abs().max().item() < 1e-3
    eng.close()


# ---------------------------------------------------------------- rendering at stride 4
def test_fused_render_and_jpeg_passes():
    from deepgraphpose_b200.engine import Engine
    nj, B, T, H, W = 4, 4, 10, 96, 128
    frames, _ = synthetic.make_video(T, H, W, nj, seed=11)
    eng = Engine(nj, location_refinement=False, output_stride=8)
    try:
        eng.load_weights(synthetic.make_weights(nj, seed=0, trained_like=True, location_refinement=False))
        mu0, peak0, lik0 = eng.estimate_pose_stream(iter(frames), H, W, T, batch=B)
        thr = float(np.sort(lik0.numpy().ravel())[T * nj // 2])
        raw = []
        mu, peak, lik = eng.estimate_pose_render_stream(iter(frames), H, W, T, lambda fr: raw.append(fr.copy()), dotsize=3,
                                                        mask_threshold=thr, batch=B)
        assert torch.equal(mu, mu0) and torch.equal(peak, peak0) and torch.equal(lik, lik0)
        drawn = np.concatenate(raw)
        m = mu.numpy().astype(np.float64)
        dev = torch.from_numpy(frames).cuda()
        eng.draw_markers(dev, m[:, :, 1] * 4.0 + 2.0, m[:, :, 0] * 4.0 + 2.0, lik.numpy().astype(np.float64), 3, thr)
        ref = dev.cpu().numpy()
        assert (ref != frames).any() and np.array_equal(drawn, ref)
        packets = []

        def writer(data, sizes):
            o = 0
            for s in sizes:
                packets.append(bytes(data[o:o + s]))
                o += int(s)

        mu, _, _ = eng.estimate_pose_render_stream(iter(frames), H, W, T, writer, dotsize=3, mask_threshold=thr, batch=B,
                                                   encoder="jpeg", quality=80)
        assert torch.equal(mu, mu0)
        assert packets == eng.encode_jpeg(dev, 80)
    finally:
        eng.close()


# ---------------------------------------------------------------- 2 GPUs
def _two_gpu_worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from deepgraphpose_b200 import dp
    from deepgraphpose_b200 import eval as dgp_eval
    T, H, W, nj = 11, 96, 128, 4
    frames, _ = synthetic.make_video(T, H, W, nj, seed=22)
    eng = _engine(synthetic.make_weights(nj, seed=0, location_refinement=False), nj, False, rank)
    res = dgp_eval.estimate_pose_sharded(eng, torch.from_numpy(frames).pin_memory(), T, H, W, synthetic.chain_skeleton(nj),
                                         np.full(nj - 1, 9.0, np.float32), np.full(nj - 1, 70.0, np.float32), 0.0, batch=3)
    eng.close()
    s = _train_setup(seed=3)
    fr = torch.from_numpy(synthetic.make_video(NT, HIN, WIN, NJ, seed=50 + rank)[0]).cuda(rank)
    te = _engine(s[0], NJ, True, rank)
    assert dp.attach_comm(te) == world
    for _ in range(2):
        _step(te, fr, s)
        te.optimizer_step(0.005, 0.9, 10.0, dp.allreduce_gradients(te))
    names = ["resnet_v1_50/conv1/weights", "resnet_v1_50/block3/unit_6/bottleneck_v1/conv2/weights",
             "resnet_v1_50/block4/unit_3/bottleneck_v1/conv3/BatchNorm/gamma", "pose/part_pred/block4/weights"]
    same = dp.broadcast_check(te, names)
    if rank == 0:
        np.savez(os.path.join(out_dir, "two_gpu.npz"), same=np.array(same), **{k: v for k, v in res.items() if k != "shard"})
    dist.barrier()
    dist.destroy_process_group()
    te.close()


def test_two_gpu_sharded_inference_and_data_parallel_replicas(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from deepgraphpose_b200 import eval as dgp_eval
    mp.spawn(_two_gpu_worker, args=(2, 29573, str(tmp_path)), nprocs=2, join=True)
    got = np.load(os.path.join(str(tmp_path), "two_gpu.npz"))
    assert bool(got["same"])
    T, H, W, nj = 11, 96, 128, 4
    frames, _ = synthetic.make_video(T, H, W, nj, seed=22)
    eng = _engine(synthetic.make_weights(nj, seed=0, location_refinement=False), nj, False, 0)
    ref = dgp_eval.estimate_pose_sharded(eng, torch.from_numpy(frames).pin_memory(), T, H, W, synthetic.chain_skeleton(nj),
                                         np.full(nj - 1, 9.0, np.float32), np.full(nj - 1, 70.0, np.float32), 0.0, batch=4)
    for k in ("x", "y", "likelihoods", "mu_likelihoods", "markers", "temporal", "skel", "e_skel", "e_temp"):
        assert np.array_equal(got[k], ref[k]), k
    eng.close()
