"""Data-parallel training plumbing (SURVEY.md 8e, training): one process per GPU, replicas draw their own batches, and the
only exchange is a SUM all-reduce of the flat float32 gradient buffer, scaled by 1/world before clipping -- the tower
averaging of the reference's multi-GPU helper (src/deepgraphpose/helpers/utils_tf.py:4-39: average_gradients).  Frozen
BatchNorm means there is no other cross-replica state.  The backend of the process group picks the exchange: over NCCL the
engine's C handle owns a communicator and reduces its gradient arena itself (``dgp_allreduce_gradients``, overlapped with
the backward pass); over gloo (CPU tensors, tests) the buffer goes through ``allreduce_flat_``.
"""
import torch
import torch.distributed as dist

BUCKETS = 4  # launch-latency sized: ~24 MB each for the 94 MB ResNet-50 gradient


def allreduce_flat_(flat, group=None, buckets=BUCKETS):
    """In-place SUM all-reduce of a flat tensor in `buckets` contiguous chunks issued back to back (async), then waited.
    Returns the factor that turns the sum into the replica mean (1 / world)."""
    if not dist.is_available() or not dist.is_initialized():
        return 1.0
    world = dist.get_world_size(group)
    if world == 1:
        return 1.0
    n = flat.numel()
    step = -(-n // buckets)
    step += (-step) % 1024  # keep chunk boundaries 4 KB aligned
    works = [dist.all_reduce(flat[a:min(a + step, n)], op=dist.ReduceOp.SUM, group=group, async_op=True)
             for a in range(0, n, step)]
    for w in works:
        w.wait()
    return 1.0 / world


def attach_comm(engine, group=None):
    """Give the engine's C handle its own NCCL communicator over the ranks of ``group`` (dgp_comm_unique_id on rank 0, the
    128-byte id broadcast through torch.distributed -- plumbing only --, dgp_comm_init_rank everywhere).  From then on
    ``allreduce_gradients`` is one C call (dgp_allreduce_gradients): four buckets in backward order on the handle's
    communication stream, overlapped with the backward pass; torch.distributed is no longer on the data path.
    Returns the world size.  A no-op (returns 1) without an initialised process group or on CPU-only groups."""
    import ctypes as C
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return 1
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    engine.train_enable()
    ident = C.create_string_buffer(128)
    if rank == 0:
        from ._lib import check
        check(engine.lib.dgp_comm_unique_id(ident))
    box = [bytes(ident.raw)]
    dist.broadcast_object_list(box, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    engine._check(engine.lib.dgp_comm_init_rank(engine.h, box[0], world, rank))
    engine._c_comm = True
    return world


def _ensure_comm(engine, group):
    """attach_comm once per engine when the process group runs on NCCL; True when the C handle owns the all-reduce."""
    if getattr(engine, "_c_comm", None) is None:
        engine._c_comm = False
        if "nccl" in str(dist.get_backend(group)).lower():
            attach_comm(engine, group)
    return engine._c_comm


def allreduce_gradients(engine, group=None):
    """All-reduce the engine's gradient buffer across ranks; returns grad_scale for Engine.optimizer_step.

    Over NCCL this is ``dgp_allreduce_gradients`` (the communicator is attached on first use); over gloo it is
    ``allreduce_flat_`` of the buffer."""
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return 1.0
    if not _ensure_comm(engine, group):
        return allreduce_flat_(engine.grad_buffer(), group)
    import ctypes as C
    from .engine import _stream
    scale = C.c_float(1.0)
    engine._check(engine.lib.dgp_allreduce_gradients(engine.h, _stream(engine.device), C.byref(scale)))
    return float(scale.value)


def allreduce_mean_scalars(values, group=None):
    """Mean over ranks of a small float tensor (loss values for reporting)."""
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return values
    out = values.clone()
    dist.all_reduce(out, op=dist.ReduceOp.SUM, group=group)
    return out / dist.get_world_size(group)


def broadcast_check(engine, names, group=None):
    """True when every rank holds bit-identical values of the named variables (replicas must never drift)."""
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return True
    ok = True
    for n in names:
        v = torch.from_numpy(engine.get_variable(n)).to(engine.device)
        lo, hi = v.clone(), v.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=group)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=group)
        ok = ok and bool(torch.equal(lo, hi))
    return ok
