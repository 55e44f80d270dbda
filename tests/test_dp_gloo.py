"""world_size-2 gloo test of the data-parallel gradient exchange (host logic of SURVEY.md 8e training; runs on CPU):
bucketed SUM all-reduce of a flat buffer + 1/world scale + the oracle's clip/Momentum step == one replica stepping on the
mean gradient."""
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from deepgraphpose_b200 import dp
from oracle import dgp_loss as oracle_loss


def _worker(rank, world, port, n, q):
    import os
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    grads = [torch.randn(n, generator=torch.Generator().manual_seed(100 + r)) for r in range(world)]
    flat = grads[rank].clone()
    scale = dp.allreduce_flat_(flat, buckets=3)
    mean = sum(grads) / world
    ok = abs(scale - 1.0 / world) < 1e-12 and torch.allclose(flat * scale, mean, rtol=1e-6, atol=1e-6)
    # every replica applies the same update
    p0 = torch.ones(n)
    (p1,), _, gnorm = oracle_loss.momentum_step([p0], [flat * scale], [torch.zeros(n)], lr=0.005, momentum=0.9, clip_norm=10.0)
    (p2,), _, _ = oracle_loss.momentum_step([p0], [mean], [torch.zeros(n)], lr=0.005, momentum=0.9, clip_norm=10.0)
    ok = ok and torch.allclose(p1, p2, rtol=1e-6, atol=1e-7)
    vals = dp.allreduce_mean_scalars(torch.tensor([float(rank), 2.0]))
    ok = ok and torch.allclose(vals, torch.tensor([(world - 1) / 2.0, 2.0]))
    q.put((rank, bool(ok)))
    dist.barrier()
    dist.destroy_process_group()


def test_bucketed_allreduce_equals_mean_gradient():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    world = 2
    procs = [ctx.Process(target=_worker, args=(r, world, 29647, 10007, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]


class _FakeEngine:
    """The gradient buffer dp.allreduce_gradients reduces over gloo, on CPU tensors (the real Engine's buffer lives on the GPU)."""

    def __init__(self, grads):
        self._g = grads

    def grad_buffer(self):
        return self._g


def _engine_worker(rank, world, port, q):
    import os
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    grads = [torch.randn(10007, generator=torch.Generator().manual_seed(7 + r)) for r in range(world)]
    eng = _FakeEngine(grads[rank].clone())
    scale = dp.allreduce_gradients(eng)          # gloo group: the bucketed torch.distributed path, no C communicator
    ok = torch.allclose(eng.grad_buffer() * scale, sum(grads) / world, rtol=1e-6, atol=1e-6)
    q.put((rank, bool(ok)))
    dist.barrier()
    dist.destroy_process_group()


def test_allreduce_gradients_through_the_engine_interface():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_engine_worker, args=(r, 2, 29653, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in range(2)]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]


def test_single_process_is_identity():
    t = torch.arange(5.0)
    assert dp.allreduce_flat_(t) == 1.0 and torch.equal(t, torch.arange(5.0))
