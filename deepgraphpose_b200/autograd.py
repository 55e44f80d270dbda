"""The pose network as a ``torch.nn.Module``: any loss written in PyTorch and any ``torch.optim`` optimizer train it on the
library's kernels (training forward, dgrad / wgrad on tcgen05, frozen-BN gradients, CUDA-graph backward).

``TrainablePoseNet(engine)`` exposes the engine's fp32 parameter arena as ONE parameter, ``flat`` (layout
``[weights | gamma | beta | head bias]`` as Engine.param_buffer); its gradient is the engine's gradient buffer::

    net = TrainablePoseNet(engine)
    opt = torch.optim.Adam(net.parameters(), lr=1e-4)
    logits, locref = net(frames)                  # uint8 CUDA (nt,H,W,3) -> float32 heads
    my_loss(logits, locref).backward()            # dgp_train_backward: flat.grad = the engine's gradient buffer
    opt.step(); opt.zero_grad()

Per-variable views in TF names and layouts stay available through ``engine.get_variable(name, "grad" / "value")``.
"""
import torch

from .engine import Engine


class _PoseNetFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, frames, flat, net):
        logits, locref, token = net.engine.train_forward(frames)
        ctx.net, ctx.token = net, token
        return logits, locref

    @staticmethod
    def backward(ctx, g_logits, g_locref):
        ctx.net._backward(ctx.token, g_logits, g_locref)
        # the gradient is already in flat.grad (the engine's buffer, written in place): nothing for autograd to accumulate
        return None, None, None


class TrainablePoseNet(torch.nn.Module):
    """PoseNet (backbone + part_pred / locref_pred heads) of an ``Engine`` with loaded weights, trainable through autograd.

    ``flat.grad`` follows the usual accumulation rules: ``None`` -> the backward overwrites the engine's gradient buffer and
    binds ``flat.grad`` to it; already bound -> the backward adds to it (micro-batches); any other tensor -> ValueError.
    An in-place change of ``flat`` (an optimizer step) is seen through its version counter: the next forward re-derives the
    16-bit operands first (Engine.params_changed).  ``Engine.optimizer_step`` and ``dp.allreduce_gradients`` work on the same
    buffers unchanged."""

    def __init__(self, engine):
        super().__init__()
        if not isinstance(engine, Engine) or not engine.weights_loaded:
            raise ValueError("TrainablePoseNet needs an Engine with loaded weights")
        self.engine = engine
        engine.train_enable()
        self.flat = torch.nn.Parameter(engine.param_buffer())
        self._grad_view = engine.grad_buffer()
        self._seen_version = self.flat._version

    def _sync_params(self):
        if self.flat._version != self._seen_version:
            self.engine.params_changed()
            self._seen_version = self.flat._version

    def _backward(self, token, g_logits, g_locref):
        g = self.flat.grad
        if g is None:
            accumulate = False
        elif g.data_ptr() == self._grad_view.data_ptr() and g.shape == self._grad_view.shape:
            accumulate = True
        else:
            raise ValueError("flat.grad must be None or the engine's gradient buffer (the tensor the previous backward bound)")
        self.engine.train_backward(token, g_logits, g_locref if self.engine.location_refinement else None, accumulate)
        if g is None:
            self.flat.grad = self._grad_view

    def forward(self, frames):
        """frames: uint8 CUDA (nt,H,W,3).  Returns (logits (nt,2h,2w,nj), locref (nt,2h,2w,2nj) | None), float32 tensors that
        own their memory.  With gradients enabled this is the training forward (one live forward per input shape: a second
        forward at the same shape before the first one's backward makes that backward raise); under torch.no_grad() it is
        the inference path (Engine.forward)."""
        self._sync_params()
        if not (torch.is_grad_enabled() and self.flat.requires_grad):
            return self.engine.forward(frames)
        return _PoseNetFunction.apply(frames, self.flat, self)
