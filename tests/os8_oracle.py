"""fp32 oracle of the pose net at any slim output_stride, composed from oracle.resnet_v1's units (test helper).

slim's stack_blocks_dense turns the strides that would take the net past `output_stride` into atrous rates
(oracle.resnet_v1.unit_plan, tests.depth_oracle.unit_plan); everything else -- conv1, the pool, the bottleneck, the heads --
is the same at every stride.
"""
import torch

import depth_oracle
from deepgraphpose_b200 import synthetic
from oracle import pose_net, resnet_v1, tf_ops


def extract_features(inputs, W, net_type="resnet_50", output_stride=8, end_points=None):
    """PoseNet.extract_features on resnet_v1_<depth> at `output_stride`: inputs (N,H,W,3) float32 0..255 -> block4 output."""
    prefix = synthetic.net_scope(net_type)
    mean = torch.tensor(pose_net.MEAN_PIXEL, dtype=torch.float32).view(1, 1, 1, 3)
    x = resnet_v1._conv_bn(inputs - mean, W, prefix + "/conv1", stride=2, same_explicit=True)
    if end_points is not None:
        end_points[prefix + "/conv1"] = x
    x = tf_ops.max_pool2d_same(x, 3, 2)
    if end_points is not None:
        end_points[prefix + "/pool1"] = x
    for scope, depth, dbn, stride, rate in depth_oracle.unit_plan(net_type, output_stride):
        x = resnet_v1.bottleneck(x, W, scope, depth, dbn, stride, rate)
        if end_points is not None:
            end_points[scope] = x
    return x


def heads(inputs, W, net_type="resnet_50", output_stride=8, location_refinement=True, end_points=None):
    """(part_pred logits, locref | None) of the pose net on resnet_v1_<depth> at `output_stride`."""
    net = extract_features(inputs, W, net_type, output_stride, end_points)
    pred = pose_net.prediction_layer(net, W, "part_pred")
    loc = pose_net.prediction_layer(net, W, "locref_pred") if location_refinement else None
    return pred, loc


def unit_shapes(H, W, net_type, output_stride):
    """{end point: (h, w, c)} of every unit of resnet_v1_<depth> on an H x W frame, by the SAME-padding chain."""
    c2 = lambda v: -(-v // 2)
    h, w = c2(c2(H)), c2(c2(W))
    out = {}
    for scope, depth, _, stride, _ in depth_oracle.unit_plan(net_type, output_stride):
        if stride == 2:
            h, w = c2(h), c2(w)
        out[scope] = (h, w, depth)
    return out
