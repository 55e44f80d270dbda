"""Training through torch.autograd (deepgraphpose_b200.autograd.TrainablePoseNet + fitdgp.dgp_loss_function): the split
entries dgp_train_forward / dgp_train_backward against the fused step, a loss the library does not have against oracle
autograd, gradient accumulation, stale tokens, torch optimizers on the parameter arena, and data-parallel replicas."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import depth_oracle
import test_gpu_train as T
from deepgraphpose_b200 import synthetic
from oracle import pose_net

pytestmark = pytest.mark.gpu

NJ, NT, HIN, WIN = T.NJ, T.NT, T.HIN, T.WIN


def _engine(W, device=None):
    from deepgraphpose_b200.engine import Engine
    e = Engine(NJ, device=device)
    e.load_weights(W)
    return e


def _targets(seed, nt=NT, Hin=HIN, Win=WIN):
    """Disc score-map targets (radius 2 px around one random point per joint and frame), locref regression targets and
    the disc mask -- what a DeepLabCut-style detection loss trains on."""
    rng = np.random.default_rng(seed)
    H, W = 2 * -(-Hin // 16), 2 * -(-Win // 16)
    yy, xx = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    tgt = np.zeros((nt, H, W, NJ), np.float32)
    for t in range(nt):
        for j in range(NJ):
            cy, cx = rng.uniform(1, H - 2), rng.uniform(1, W - 2)
            tgt[t, :, :, j] = ((yy - cy) ** 2 + (xx - cx) ** 2 <= 4.0)
    lmap = rng.normal(0, 0.7, (nt, H, W, 2 * NJ)).astype(np.float32)
    lmask = np.repeat(tgt, 2, axis=3)
    return [torch.from_numpy(a) for a in (tgt, lmap, lmask)]


def my_loss(logits, locref, tgt, lmap, lmask):
    """Sigmoid cross-entropy to the discs + 0.05 x Huber on the masked locref, per frame: not a loss of the library."""
    nt = logits.shape[0]
    ce = F.binary_cross_entropy_with_logits(logits, tgt, reduction="sum") / nt
    hub = F.huber_loss(locref * lmask, lmap * lmask, delta=1.0, reduction="sum") / nt
    return ce + 0.05 * hub


def _cuda(ts):
    return [t.cuda() for t in ts]


# ---------------------------------------------------------------------------------------------------- 1. fused parity
def test_module_with_dgp_loss_equals_fused_step():
    """Module forward + dgp_loss_function(...)["total_loss"].backward() == dgp_train_forward_backward on the same batch:
    equal losses and heads, and the arena == the fused arena / loss scale bit for bit, eagerly (step 1) and on graph replay
    (steps 2-3)."""
    from deepgraphpose_b200 import fitdgp
    from deepgraphpose_b200.autograd import TrainablePoseNet
    W, frames, batch, edges, S0, cfg, ws, ws_max = T._setup()
    fr = torch.from_numpy(frames).cuda()
    a, b = _engine(W), _engine(W)
    net = TrainablePoseNet(b)
    for step in range(3):
        la = fitdgp.train_forward_backward(a, fr, batch, cfg, edges, ws, ws_max, 200, 20)
        net.zero_grad()
        logits, locref = net(fr)
        out = fitdgp.dgp_loss_function(logits, locref, batch, cfg, edges, ws, ws_max, 200, 20, engine=b)
        out["total_loss"].backward()
        la_logits, la_locref = a.train_outputs(NT, HIN, WIN)
        assert torch.equal(logits, la_logits) and torch.equal(locref, la_locref), step
        for k in fitdgp.LOSS_KEYS:
            assert float(out[k].detach()) == float(la[k]), (step, k, float(out[k].detach()), la[k])
        assert net.flat.grad is not None and net.flat.grad.data_ptr() == b.grad_buffer().data_ptr()
        assert torch.equal(net.flat.grad, a.grad_buffer() / 1024.0), step
    # per-variable gradients read back through the recorded arena scale
    name = "resnet_v1_50/block3/unit_2/bottleneck_v1/conv2/weights"
    assert np.array_equal(a.get_variable(name, "grad"), b.get_variable(name, "grad"))
    # the loss-only default handle gives the same values
    logits, locref = net(fr)
    out2 = fitdgp.dgp_loss_function(logits, locref, batch, cfg, edges, ws, ws_max, 200, 20)
    assert float(out2["total_loss"].detach()) == float(out["total_loss"].detach())
    assert not out2["visible_loss_pred"].requires_grad and out2["total_loss"].requires_grad
    a.close()
    b.close()


# ---------------------------------------------------------------------------------------------------- 2. a new loss
@pytest.mark.parametrize("net_type", ["resnet_50", "resnet_101"])
def test_custom_loss_gradients_match_oracle_autograd(net_type):
    from deepgraphpose_b200.autograd import TrainablePoseNet
    W = synthetic.make_weights(NJ, seed=3, net_type=net_type)
    frames, _ = synthetic.make_video(NT, HIN, WIN, NJ, seed=11)
    tgt, lmap, lmask = _targets(5)
    Wt = {k: torch.from_numpy(v.copy()).requires_grad_(k.endswith(T.TRAINABLE)) for k, v in W.items()}
    x = torch.from_numpy(frames.astype(np.float32))
    if net_type == "resnet_50":
        heads = pose_net.get_net(x, Wt, True)
        pred, loc = heads["part_pred"], heads["locref"]
    else:
        pred, loc = depth_oracle.heads(x, Wt, net_type, True)
    ref_loss = my_loss(pred, loc, tgt, lmap, lmask)
    ref_loss.backward()
    eng = _engine(W)
    net = TrainablePoseNet(eng)
    logits, locref = net(torch.from_numpy(frames).cuda())
    loss = my_loss(logits, locref, *_cuda((tgt, lmap, lmask)))
    loss.backward()
    assert abs(float(loss) - float(ref_loss)) <= 1e-3 * abs(float(ref_loss)), (float(loss), float(ref_loss))
    rows, bad = [], []
    for name, t in sorted(Wt.items()):
        if not t.requires_grad:
            continue
        g, g_ref = eng.get_variable(name, "grad"), t.grad.numpy()
        nr = float(np.linalg.norm(g_ref))
        assert nr > 0, name
        cos = float((g * g_ref).sum() / (np.linalg.norm(g) * nr + 1e-30))
        rel = float(np.linalg.norm(g - g_ref) / nr)
        rows.append((name, cos, rel))
        if not (cos > 0.995 and rel < 0.10):
            bad.append((name, cos, rel))
    print("%s custom loss: median cosine %.5f, median rel-L2 %.4f, worst rel-L2 %.4f"
          % (net_type, np.median([r[1] for r in rows]), np.median([r[2] for r in rows]), max(r[2] for r in rows)))
    assert not bad, bad[:8]
    eng.close()


# ---------------------------------------------------------------------------------------------------- 3. accumulation
def test_gradient_accumulation_is_exact():
    from deepgraphpose_b200 import fitdgp
    from deepgraphpose_b200._lib import DgpError
    from deepgraphpose_b200.autograd import TrainablePoseNet
    W, frames, batch, edges, S0, cfg, ws, ws_max = T._setup(seed=5)
    fa = torch.from_numpy(frames).cuda()
    fb = torch.from_numpy(synthetic.make_video(NT, HIN, WIN, NJ, seed=60)[0]).cuda()
    ta, tb = _cuda(_targets(1)), _cuda(_targets(2))
    eng = _engine(W)
    # the same gradients twice through the C entry: exactly 2 g
    logits, locref, tok = eng.train_forward(fa)
    lg, lr = logits.requires_grad_(), locref.requires_grad_()
    my_loss(lg, lr, *ta).backward()
    eng.train_backward(tok, lg.grad, lr.grad)
    g1 = eng.grad_buffer().clone()
    eng.train_backward(tok, lg.grad, lr.grad, accumulate=True)
    assert torch.equal(eng.grad_buffer(), 2 * g1)
    # batches A then B through the module == gA + gB of separate runs
    net = TrainablePoseNet(eng)
    sep = []
    for fr, tg in ((fa, ta), (fb, tb)):
        net.zero_grad()
        my_loss(*net(fr), *tg).backward()
        sep.append(net.flat.grad.clone())
    assert torch.equal(sep[0], g1)
    net.zero_grad()
    for fr, tg in ((fa, ta), (fb, tb)):
        my_loss(*net(fr), *tg).backward()
    assert torch.equal(net.flat.grad, sep[0] + sep[1])
    net.zero_grad(set_to_none=False)        # zeroed in place: the next backward adds onto zeros
    my_loss(*net(fb), *tb).backward()
    assert torch.equal(net.flat.grad, sep[1])
    # a gradient tensor that is not the engine's buffer
    net.flat.grad = torch.zeros_like(net.flat)
    with pytest.raises(ValueError):
        my_loss(*net(fa), *ta).backward()
    # adding onto the loss-scaled arena of the fused step is refused
    fitdgp.train_forward_backward(eng, fa, batch, cfg, edges, ws, ws_max, 200, 20)
    _, _, tok = eng.train_forward(fa)
    with pytest.raises(DgpError) as ei:
        eng.train_backward(tok, lg.grad, lr.grad, accumulate=True)
    assert ei.value.status == -4
    eng.close()


# ---------------------------------------------------------------------------------------------------- 4. stale tokens
def test_stale_token_raises():
    from deepgraphpose_b200._lib import DgpError
    W, frames, *_ = T._setup(seed=7)
    fr = torch.from_numpy(frames).cuda()
    other = torch.from_numpy(synthetic.make_video(2, 80, 112, NJ, seed=3)[0]).cuda()
    eng = _engine(W)
    g = torch.ones((NT, 2 * -(-HIN // 16), 2 * -(-WIN // 16), NJ), device="cuda")

    def stale(tok):
        with pytest.raises(DgpError) as ei:
            eng.train_backward(tok, g)
        assert ei.value.status == -4 and "stale" in str(ei.value)

    _, _, t1 = eng.train_forward(fr)
    _, _, t2 = eng.train_forward(fr)
    stale(t1)
    eng.train_backward(t2, g)
    _, _, t3 = eng.train_forward(fr)
    _, _, t_other = eng.train_forward(other)          # another shape: t3 stays live
    eng.train_backward(t3, g)
    eng.train_backward(t_other, None)
    eng.optimizer_step(0.001, 0.9, 10.0, 1.0)          # a weight change
    stale(t3)
    _, _, t4 = eng.train_forward(fr)
    eng.params_changed()
    stale(t4)
    _, _, t5 = eng.train_forward(fr)
    eng.set_variable("pose/part_pred/block4/biases", np.zeros(NJ, np.float32))
    stale(t5)
    eng.close()


# ---------------------------------------------------------------------------------------------------- 5. torch.optim
def test_torch_optimizers_on_the_parameter_arena():
    from deepgraphpose_b200.autograd import TrainablePoseNet
    W, frames, *_ = T._setup(seed=9)
    fr = torch.from_numpy(frames).cuda()
    tg = _cuda(_targets(3))
    a, b = _engine(W), _engine(W)
    na, nb = TrainablePoseNet(a), TrainablePoseNet(b)
    for n in (na, nb):
        my_loss(*n(fr), *tg).backward()
    assert torch.equal(na.flat.grad, nb.flat.grad)
    lr = 0.002
    a.optimizer_step(lr, 0.9, 0.0, 1.0)                # Momentum, no clipping
    opt = torch.optim.SGD(nb.parameters(), lr=lr, momentum=0.9)
    opt.step()
    pa, pb = a.param_buffer(), nb.flat.detach()
    assert ((pa - pb).abs().max() <= 1e-6 * pa.abs().max()).item()
    # the next forward sees the in-place update: bitwise the forward of a fresh engine loaded from the exported variables
    exported = dict(b._frozen, **{n: b.get_variable(n) for n in b.variable_names()})
    fresh = _engine(exported)
    lg, lr_ = nb(fr)
    lf, rf = fresh.forward(fr)
    assert torch.equal(lg, lf) and torch.equal(lr_, rf)
    with torch.no_grad():
        li, ri = nb(fr)
    assert torch.equal(li, lf) and torch.equal(ri, rf)
    fresh.close()
    # Adam keeps every structural zero of the layouts (conv1's space-to-depth padding, padded head rows) exactly 0
    opt = torch.optim.Adam(na.parameters(), lr=1e-3)
    p0 = na.flat.detach().clone()
    na.zero_grad()
    my_loss(*na(fr), *tg).backward()
    zeros = (p0 == 0) & (na.flat.grad == 0)
    assert int(zeros.sum()) >= 64 * (256 - 7 * 7 * 3)
    moving = na.flat.grad != 0
    for _ in range(3):
        opt.step()
        opt.zero_grad()
        assert int((na.flat.detach()[zeros] != 0).sum()) == 0
        assert bool((na.flat.detach() != p0)[moving].all())     # every parameter with a gradient took its Adam step
        my_loss(*na(fr), *tg).backward()
    a.close()
    b.close()


# ---------------------------------------------------------------------------------------------------- 6. two GPUs
CHECK_VARS = ("resnet_v1_50/conv1/weights", "resnet_v1_50/block2/unit_1/bottleneck_v1/conv2/weights",
              "resnet_v1_50/block4/unit_3/bottleneck_v1/conv3/BatchNorm/gamma", "pose/part_pred/block4/weights",
              "pose/locref_pred/block4/biases")


def _replica_inputs(rank):
    W, *_ = T._setup(seed=3)
    frames, _ = synthetic.make_video(NT, HIN, WIN, NJ, seed=50 + rank)
    return W, frames, _targets(20 + rank)


def _dp_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from deepgraphpose_b200 import dp
    from deepgraphpose_b200.autograd import TrainablePoseNet
    W, frames, tg = _replica_inputs(rank)
    eng = _engine(W, device=rank)
    assert dp.attach_comm(eng) == world
    net = TrainablePoseNet(eng)
    fr = torch.from_numpy(frames).cuda(rank)
    tg = [t.cuda(rank) for t in tg]
    for _ in range(2):
        net.zero_grad()
        my_loss(*net(fr), *tg).backward()
        scale = dp.allreduce_gradients(eng)
        eng.optimizer_step(0.005, 0.9, 10.0, scale)
    same = dp.broadcast_check(eng, CHECK_VARS)
    if rank == 0:
        np.savez(os.path.join(out_dir, "dp.npz"), same=np.array(same), **{k.replace("/", "."): eng.get_variable(k) for k in CHECK_VARS})
    dist.barrier()
    dist.destroy_process_group()
    eng.close()


def test_two_gpu_replicas_with_a_custom_loss_match_mean_gradient(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from deepgraphpose_b200.autograd import TrainablePoseNet
    mp.spawn(_dp_worker, args=(2, 29561, str(tmp_path)), nprocs=2, join=True)
    got = np.load(os.path.join(str(tmp_path), "dp.npz"))
    assert bool(got["same"])
    nets, inputs = [], []
    for r in range(2):
        W, frames, tg = _replica_inputs(r)
        nets.append(TrainablePoseNet(_engine(W, device=0)))
        inputs.append((torch.from_numpy(frames).cuda(0), _cuda(tg)))
    for _ in range(2):
        for n, (fr, tg) in zip(nets, inputs):
            n.zero_grad()
            my_loss(*n(fr), *tg).backward()
        total = nets[0].flat.grad + nets[1].flat.grad
        for n in nets:
            n.flat.grad.copy_(total)
            n.engine.optimizer_step(0.005, 0.9, 10.0, 0.5)
    for k in CHECK_VARS:
        assert np.array_equal(got[k.replace("/", ".")], nets[0].engine.get_variable(k)), k
    for n in nets:
        n.engine.close()
