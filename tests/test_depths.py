"""ResNet-101 / ResNet-152 backbones (DLC net_type resnet_101 / resnet_152) on the CPU: layer tables, closed-form counts,
synthetic weights, checkpoint names and the net_type checks of the Python entry points."""
import hashlib
import importlib.util
import os

import numpy as np
import pytest
import torch

import depth_oracle
from deepgraphpose_b200 import synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# convs, conv params, BN channels, GFLOP/frame at 747x832 nj 4 and at 1024x1280 nj 16 (part_pred head only)
TABLE = {"resnet_50": (53, 23454912, 26560, 145.0, 306.1),
         "resnet_101": (104, 42394816, 52672, 237.6, 500.1),
         "resnet_152": (155, 57992384, 75712, 330.1, 694.0)}


def _load_tool(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "tools", name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _digest(W):
    h = hashlib.sha256()
    for k in sorted(W):
        h.update(k.encode())
        h.update(np.ascontiguousarray(W[k], np.float32).tobytes())
    return h.hexdigest()


@pytest.mark.parametrize("net_type", synthetic.NET_TYPES)
def test_layer_tables_match_the_closed_form(net_type):
    convs, params, bn, gf_b, gf_c = TABLE[net_type]
    specs = synthetic.conv_specs(net_type)
    assert len(specs) == convs
    assert sum(kh * kw * cin * cout for _, kh, kw, cin, cout in specs) == params
    assert sum(cout for *_, cout in specs) == bn
    plan = depth_oracle.unit_plan(net_type)
    assert len(plan) == sum(synthetic.BLOCK_UNITS[net_type])
    assert [u[0] for u in plan] == [s[:-len("/conv1")] for s, *_ in specs if s.endswith("/conv1") and "/unit_" in s]
    # output stride 16: blocks 3 and 4 run at stride 1, block 4 dilated by 2
    assert [u[3] for u in plan].count(2) == 2 and {u[4] for u in plan if "/block4/" in u[0]} == {2}
    bd = _load_tool("bench_depths")
    f_b, _ = bd.conv_flops_per_frame(747, 832, 4, synthetic.BLOCK_UNITS[net_type])
    f_c, _ = bd.conv_flops_per_frame(1024, 1280, 16, synthetic.BLOCK_UNITS[net_type])
    assert round(f_b / 1e9, 1) == gf_b and round(f_c / 1e9, 1) == gf_c


def test_depth_50_flops_equal_the_benchmark_formula():
    import bench
    bd = _load_tool("bench_depths")
    for h, w, nj in ((747, 832, 4), (1024, 1280, 16), (480, 640, 20)):
        assert bd.conv_flops_per_frame(h, w, nj, synthetic.BLOCK_UNITS["resnet_50"]) == bench.conv_flops_per_frame(h, w, nj)


def test_resnet50_weights_and_batch_choice_are_unchanged():
    """The ResNet-50 random stream every seeded test depends on, and suggest_batch's default, are those of the single-depth
    code (digests and batch sizes recorded from it)."""
    from deepgraphpose_b200.engine import suggest_batch
    assert _digest(synthetic.make_weights(4, seed=0)) == "78aee2330b19a974d522dd878aba4f43323c5c6a2bed4d71cc3307ad140837bf"
    assert _digest(synthetic.make_weights(4, seed=0, trained_like=True, location_refinement=False)) == \
        "5d0555826199460492c2903dade9d6c14b30f235f5dd837f2c4ed8cfa210ed53"
    assert synthetic.resnet50_conv_specs() == synthetic.conv_specs("resnet_50")
    assert (suggest_batch(747, 832), suggest_batch(1024, 1280, 12, 24), suggest_batch(480, 640)) == (31, 22, 47)
    assert suggest_batch(747, 832, units=synthetic.BLOCK_UNITS["resnet_50"]) == 31


@pytest.mark.parametrize("net_type", ["resnet_101", "resnet_152"])
@pytest.mark.parametrize("trained_like", [False, True], ids=["random-init", "trained-like"])
def test_deeper_weight_sets_give_non_degenerate_logits(net_type, trained_like):
    """Through the fp32 oracle the deeper sets keep the ResNet-50 set's logit spread (CONV3_GAMMA_SCALE): neither a
    saturated sigmoid nor a flat map."""
    frames, _ = synthetic.make_video(1, 235, 301, 4, seed=235)
    x = torch.from_numpy(frames.astype(np.float32))
    stats = {}
    for nt in ("resnet_50", net_type):
        W = synthetic.make_weights(4, seed=0, location_refinement=False, trained_like=trained_like, net_type=nt)
        assert all(k.startswith(("pose/", synthetic.net_scope(nt) + "/")) for k in W)
        with torch.no_grad():
            pred, _ = depth_oracle.heads(x, {k: torch.from_numpy(v) for k, v in W.items()}, nt, False)
        assert pred.shape == (1, 30, 38, 4) and torch.isfinite(pred).all()
        p = torch.sigmoid(pred)
        stats[nt] = (float(pred.std()), float(((p < 0.02) | (p > 0.98)).float().mean()))
    (s50, sat50), (s, sat) = stats["resnet_50"], stats[net_type]
    assert 0.6 * s50 < s < 1.6 * s50, stats
    assert sat < max(0.5, 1.5 * sat50), stats


def test_checkpoint_round_trip_with_resnet_v1_101_names(tmp_path):
    from deepgraphpose_b200 import tf_checkpoint
    from deepgraphpose_b200.eval import load_variables
    W = synthetic.make_weights(3, seed=1, net_type="resnet_101")
    assert sum(k.endswith("/weights") for k in W) == 104 + 2
    out = dict(W)
    out["resnet_v1_101/block3/unit_23/bottleneck_v1/conv3/weights/Momentum"] = np.ones((1, 1, 256, 1024), np.float32)
    out["global_step"] = np.array(7, dtype=np.int64)
    prefix = str(tmp_path / "snapshot-step2-final--0")
    tf_checkpoint.write_checkpoint(prefix, out)
    back = load_variables(prefix, 3, True)
    assert sorted(back) == sorted(W)
    assert all(np.array_equal(back[k], W[k]) for k in W)
    assert synthetic.net_type_of(back) == "resnet_101"


def test_net_type_checks():
    from deepgraphpose_b200.eval import check_net_type
    W50 = synthetic.make_weights(2, seed=0, location_refinement=False)
    W101 = synthetic.make_weights(2, seed=0, location_refinement=False, net_type="resnet_101")
    assert check_net_type(None, W101) == "resnet_101" and check_net_type("resnet_50", W50) == "resnet_50"
    with pytest.raises(ValueError, match="resnet_50.*resnet_101"):
        check_net_type("resnet_50", W101)
    with pytest.raises(ValueError, match="mobilenet"):
        check_net_type("mobilenet_v2_1.0", W50)
    mixed = dict(W50, **{"resnet_v1_101/conv1/weights": W101["resnet_v1_101/conv1/weights"]})
    with pytest.raises(ValueError, match="resnet_v1_101, resnet_v1_50"):
        synthetic.net_type_of(mixed)
    with pytest.raises(ValueError, match="none"):
        synthetic.net_type_of({k: v for k, v in W50.items() if k.startswith("pose/")})
    with pytest.raises(ValueError):
        synthetic.net_type_of({"resnet_v1_200/conv1/weights": np.zeros(1)})
