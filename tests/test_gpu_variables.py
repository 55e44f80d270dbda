"""The handle's trainable variables against the parameter arena: after load_weights the arena equals one assembled here in
numpy from the TF dict (the layout the all-reduce buckets, param_buffer() users and the backward kernels rely on),
get_variable / set_variable invert each other for every variable, and a loaded variable of the wrong shape is refused."""
import numpy as np
import pytest

from deepgraphpose_b200 import synthetic
from test_gpu_backward_kernels import conv1_s2d_weights

pytestmark = pytest.mark.gpu

NJ = 3


def _engine(W, locref=True):
    from deepgraphpose_b200.engine import Engine
    eng = Engine(NJ, location_refinement=locref)
    eng.load_weights(W)
    return eng


def _cdiv(a, b):
    return -(-a // b)


def _head_rows(n):
    """Rows of the deconv heads' GEMM matrix: n = 9*ctot padded to a multiple of the widest UMMA N (multiple of 16, <= 256)
    that tiles it with the least padding."""
    bn = min(_cdiv(_cdiv(n, _cdiv(n, 256)), 16) * 16, 256)
    return _cdiv(n, bn) * bn


def arena_reference(W, net_type, locref):
    """[conv weights | gamma | beta | head bias] in kernel layouts, from the TF-layout dict W."""
    weights, gamma, beta = [], [], []
    for scope, kh, kw, cin, cout in synthetic.conv_specs(net_type):
        w = W[scope + "/weights"]
        weights.append(conv1_s2d_weights(w)[0] if (kh, cin) == (7, 3) else w.reshape(kh * kw * cin, cout).T)
        gamma.append(W[scope + "/BatchNorm/gamma"])
        beta.append(W[scope + "/BatchNorm/beta"])
    heads = [("part_pred", NJ)] + ([("locref_pred", 2 * NJ)] if locref else [])
    ctot = sum(cn for _, cn in heads)
    head = np.zeros((_head_rows(9 * ctot), 2048))
    bias = np.zeros(_cdiv(ctot, 8) * 8)
    c0 = 0
    for name, cn in heads:
        w = W["pose/%s/block4/weights" % name].reshape(9, cn, 2048)
        for t in range(9):
            head[t * ctot + c0:t * ctot + c0 + cn] = w[t]
        bias[c0:c0 + cn] = W["pose/%s/block4/biases" % name]
        c0 += cn
    weights.append(head)
    parts = [a.reshape(-1) for a in weights] + [np.concatenate(gamma), np.concatenate(beta), bias]
    return np.concatenate(parts).astype(np.float32)


@pytest.mark.parametrize("net_type,locref", [("resnet_50", True), ("resnet_50", False), ("resnet_101", True)])
def test_arena_matches_numpy_layout(net_type, locref):
    W = synthetic.make_weights(NJ, seed=3, location_refinement=locref, net_type=net_type)
    eng = _engine(W, locref)
    try:
        got = eng.param_buffer().cpu().numpy()
        ref = arena_reference(W, net_type, locref)
        assert got.shape == ref.shape
        assert np.array_equal(got, ref)
    finally:
        eng.close()


def test_get_set_round_trip():
    W = synthetic.make_weights(NJ, seed=4)
    eng = _engine(W)
    try:
        names = eng.variable_names()
        for n in names:
            got = eng.get_variable(n)
            assert got.shape == W[n].shape and np.array_equal(got, W[n]), n
        conv1 = "resnet_v1_50/conv1/weights"
        mask = conv1_s2d_weights(W[conv1])[1]
        rng = np.random.default_rng(5)
        new = {}
        for n in names:
            new[n], m = (rng.standard_normal(W[n].shape).astype(np.float32) for _ in range(2))
            eng.set_variable(n, new[n])
            eng.set_variable(n, m, "momentum")
            assert np.array_equal(eng.get_variable(n), new[n]), n
            assert np.array_equal(eng.get_variable(n, "momentum"), m), n
            if n == conv1:
                arena = eng.param_buffer()[:64 * 256].cpu().numpy().reshape(64, 256)
                assert not arena[mask == 0].any()
        # the two heads share one matrix and one bias vector: setting one leaves the other as it was
        for a, b in (("part_pred", "locref_pred"), ("locref_pred", "part_pred")):
            for leaf in ("weights", "biases"):
                na, nb = "pose/%s/block4/%s" % (a, leaf), "pose/%s/block4/%s" % (b, leaf)
                new[na] = rng.standard_normal(W[na].shape).astype(np.float32)
                eng.set_variable(na, new[na])
                assert np.array_equal(eng.get_variable(nb), new[nb]), (na, nb)
        # every set wrote its own elements and nothing else: the arena is the layout of the new values
        frozen = {k: v for k, v in W.items() if k not in new}
        assert np.array_equal(eng.param_buffer().cpu().numpy(), arena_reference(dict(frozen, **new), "resnet_50", True))
    finally:
        eng.close()


@pytest.mark.parametrize("name,shape", [
    ("resnet_v1_50/block2/unit_3/bottleneck_v1/conv2/BatchNorm/beta", (127,)),
    ("resnet_v1_50/block2/unit_3/bottleneck_v1/conv2/BatchNorm/gamma", (127,)),
    ("resnet_v1_50/block2/unit_3/bottleneck_v1/conv2/BatchNorm/moving_mean", (127,)),
    ("resnet_v1_50/conv1/BatchNorm/moving_variance", (63,)),
    ("pose/part_pred/block4/biases", (NJ - 1,)),
    ("pose/locref_pred/block4/weights", (1, 1, 2 * NJ, 2048)),
])
def test_malformed_variable_is_refused(name, shape):
    from deepgraphpose_b200._lib import DgpError
    from deepgraphpose_b200.engine import Engine
    W = synthetic.make_weights(NJ, seed=6)
    W[name] = np.resize(W[name], shape).astype(np.float32)
    eng = Engine(NJ)
    try:
        with pytest.raises(DgpError) as ei:
            eng.load_weights(W)
        assert ei.value.status == -1   # DGP_ERR_INVALID
        assert name in str(ei.value), str(ei.value)
    finally:
        eng.close()
