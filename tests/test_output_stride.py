"""Pose nets trained at slim output_stride 8: shape algebra, the unit plan and config validation.  CPU only."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest
from hypothesis import given, settings
from hypothesis import strategies as st

import depth_oracle
import os8_oracle
from deepgraphpose_b200 import _lib, synthetic
from oracle import resnet_v1, tf_ops

DGP_ERR_INVALID = -1


def _dims_os(H, W, os_):
    lib = _lib.load()
    a, b, c, d = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    rc = lib.dgp_output_dims_os(H, W, os_, C.byref(a), C.byref(b), C.byref(c), C.byref(d))
    return rc, (a.value, b.value, c.value, d.value)


@settings(max_examples=200, deadline=None)
@given(st.integers(32, 2000), st.integers(32, 2000))
def test_output_dims_os8_equals_the_layer_chain(lib_built, H, W):
    """dgp_output_dims_os(.., 8) == the SAME-padding chain conv1 (s2) -> pool (s2) -> block1 (s2) -> deconv (x2), and the
    features have the shape the oracle's unit plan gives block 4; at 16 it is dgp_output_dims."""
    rc, (fh, fw, oh, ow) = _dims_os(H, W, 8)
    assert rc == 0
    h, w = H, W
    for k, s in ((7, 2), (3, 2), (3, 2)):
        h, w = tf_ops.same_pad(h, k, s)[2], tf_ops.same_pad(w, k, s)[2]
    assert (fh, fw) == (h, w) and (oh, ow) == (2 * h, 2 * w)
    assert list(os8_oracle.unit_shapes(H, W, "resnet_50", 8).values())[-1] == (fh, fw, 2048)
    rc, (gh, gw, _, _) = _dims_os(H, W, 16)
    assert rc == 0 and (gh, gw) == resnet_v1.output_dims(H, W)[0]
    assert list(os8_oracle.unit_shapes(H, W, "resnet_50", 16).values())[-1] == (gh, gw, 2048)


def test_output_dims_at_both_strides(lib_built):
    from deepgraphpose_b200.engine import output_dims
    assert output_dims(747, 832, 8) == ((94, 104), (188, 208))
    assert output_dims(1024, 1280, 8) == ((128, 160), (256, 320))
    assert output_dims(480, 640, 8) == ((60, 80), (120, 160))
    for H, W in ((747, 832), (1024, 1280), (480, 640), (235, 301)):
        assert output_dims(H, W) == output_dims(H, W, 16) == resnet_v1.output_dims(H, W)
    for bad in (4, 32, 0, 12):
        assert _dims_os(747, 832, bad)[0] == DGP_ERR_INVALID
        with pytest.raises(ValueError):
            output_dims(747, 832, bad)


@pytest.mark.parametrize("net_type", ["resnet_50", "resnet_101", "resnet_152"])
def test_unit_plan_at_output_stride_8(net_type):
    """slim stack_blocks_dense at output_stride 8: block 1 as at 16 (its last unit keeps stride 2), every unit of block 2 at
    stride 1 / rate 1, block 3 at rate 2, block 4 at rate 4."""
    plan = depth_oracle.unit_plan(net_type, 8)
    units = synthetic.BLOCK_UNITS[net_type]
    assert len(plan) == sum(units)
    by_block = {}
    for scope, depth, dbn, stride, rate in plan:
        by_block.setdefault(scope.split("/")[1], []).append((stride, rate))
    assert by_block["block1"] == [(1, 1)] * (units[0] - 1) + [(2, 1)]
    assert by_block["block2"] == [(1, 1)] * units[1]
    assert by_block["block3"] == [(1, 2)] * units[2]
    assert by_block["block4"] == [(1, 4)] * units[3]
    # at 16 the same net runs block 2's last unit at stride 2 and block 4 at rate 2
    plan16 = depth_oracle.unit_plan(net_type, 16)
    assert [p[3:] for p in plan16 if "/block2/" in p[0]][-1] == (2, 1)
    assert {p[3:] for p in plan16 if "/block4/" in p[0]} == {(1, 2)}


def test_suggest_batch_follows_the_unit_strides():
    from deepgraphpose_b200.engine import suggest_batch
    b8 = suggest_batch(747, 832, output_stride=8)
    assert 24 <= b8 <= 48
    assert suggest_batch(747, 832) == suggest_batch(747, 832, output_stride=16)
    with pytest.raises(ValueError):
        suggest_batch(747, 832, output_stride=32)


BAD_GEOMETRY = [
    ({"output_stride": 4, "stride": 2.0}, "output_stride"),
    ({"output_stride": 32, "stride": 16.0}, "output_stride"),
    ({"output_stride": 8, "stride": 8.0}, "stride"),
    ({"output_stride": 8}, "stride"),              # DLC's default stride (8.0) cannot go with output_stride 8
    ({"output_stride": 16, "deconvolutionstride": 1}, "deconvolutionstride"),
    ({"output_stride": 8, "stride": 4.0, "deconvolutionstride": 4}, "deconvolutionstride"),
]


@pytest.mark.parametrize("geom,what", BAD_GEOMETRY)
def test_configs_outside_the_path_raise_value_error(lib_built, tmp_path, geom, what):
    """Every entry that builds a graph from a dlc_cfg / dgp_cfg refuses these before it creates an engine."""
    from deepgraphpose_b200 import eval as dgp_eval
    from deepgraphpose_b200 import fitdgp
    from deepgraphpose_b200.pose_net import PoseNet
    cfg = dict({"num_joints": 2, "net_type": "resnet_50"}, **geom)
    with pytest.raises(ValueError, match=what):
        dgp_eval.check_geometry(cfg)
    with pytest.raises(ValueError, match=what):
        PoseNet(cfg)
    with pytest.raises(ValueError, match=what):
        PoseNet(SimpleNamespace(**cfg))
    with pytest.raises(ValueError, match=what):
        dgp_eval.setup_dgp_eval_graph(cfg, "synthetic")
    with pytest.raises(ValueError, match=what):
        dgp_eval.estimate_pose(cfg, "synthetic", np.zeros((2, 64, 64, 3), np.uint8), str(tmp_path))
    proj = tmp_path / "config.yaml"
    proj.write_text("Task: t\ndate: d\nTrainingFraction: [0.95]\nscorer: s\nbodyparts: [a, b]\nproject_path: %s\n" % tmp_path)
    with pytest.raises(ValueError, match=what):
        dgp_eval.evaluate_dgp(str(proj), "synthetic", dlc_cfg=cfg)
    batcher = SimpleNamespace(S0=np.zeros((2, 2)), nj=2, datasets=[], n_frames_total=1, n_visible_frames_total=1)
    with pytest.raises(ValueError, match=what):
        fitdgp.dgp_loss(batcher, cfg, variables="synthetic")
    with pytest.raises(ValueError, match=what):
        fitdgp._loss_engine("cuda:0", 2, cfg)
    for fit in (fitdgp.fit_dgp, fitdgp.fit_dgp_labeledonly):
        with pytest.raises(ValueError, match=what):
            fit("snap", "proj", data_batcher=batcher, dgp_cfg=dict(cfg, batch_size=1), frame_lists=([[0]], [[]], [[0]]),
                variables="synthetic", verbose=False)


def test_engine_refuses_other_output_strides_before_any_device_work():
    from deepgraphpose_b200.engine import Engine
    for bad in (4, 32, 12, True):
        with pytest.raises(ValueError, match="output_stride"):
            Engine(2, output_stride=bad)


def test_good_geometries():
    from deepgraphpose_b200 import eval as dgp_eval
    assert dgp_eval.check_geometry({}) == (16, 8.0)
    assert dgp_eval.check_geometry({"output_stride": 16, "stride": 8.0, "deconvolutionstride": 2}) == (16, 8.0)
    assert dgp_eval.check_geometry({"output_stride": 8, "stride": 4.0}) == (8, 4.0)
    assert dgp_eval.check_geometry(SimpleNamespace(output_stride=8, stride=4)) == (8, 4.0)


def test_ctypes_symbols(lib_built):
    lib = _lib.load()
    for name in ("dgp_set_output_stride", "dgp_get_output_stride", "dgp_output_dims_os"):
        assert hasattr(lib, name) and name in _lib.SIGNATURES
    # no handle: invalid, not a crash
    v = C.c_int()
    assert lib.dgp_set_output_stride(None, 8) == DGP_ERR_INVALID
    assert lib.dgp_get_output_stride(None, C.byref(v)) == DGP_ERR_INVALID
