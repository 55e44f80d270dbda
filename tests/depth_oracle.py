"""fp32 oracle of slim resnet_v1_101 / resnet_v1_152, composed from oracle.resnet_v1's units (test helper).

slim's resnet_v1_101 and resnet_v1_152 are resnet_v1_50 with more units in blocks 2 and 3: the same bottleneck, the same
stack_blocks_dense bookkeeping (oracle.resnet_v1.unit_plan over another block table) under another variable scope.
"""
import torch

from deepgraphpose_b200 import synthetic
from oracle import pose_net, resnet_v1, tf_ops


def unit_plan(net_type, output_stride=16):
    """(scope, depth, depth_bottleneck, stride, rate) of every unit of slim resnet_v1_<depth>."""
    prefix = synthetic.net_scope(net_type)
    return [(scope.replace("resnet_v1_50/", prefix + "/", 1),) + tuple(rest)
            for scope, *rest in resnet_v1.unit_plan(output_stride, synthetic.net_blocks(net_type))]


def extract_features(inputs, W, net_type, end_points=None):
    """PoseNet.extract_features on resnet_v1_<depth>: inputs (N,H,W,3) float32 0..255 -> block4 output."""
    prefix = synthetic.net_scope(net_type)
    mean = torch.tensor(pose_net.MEAN_PIXEL, dtype=torch.float32).view(1, 1, 1, 3)
    x = resnet_v1._conv_bn(inputs - mean, W, prefix + "/conv1", stride=2, same_explicit=True)
    if end_points is not None:
        end_points[prefix + "/conv1"] = x
    x = tf_ops.max_pool2d_same(x, 3, 2)
    if end_points is not None:
        end_points[prefix + "/pool1"] = x
    for scope, depth, dbn, stride, rate in unit_plan(net_type):
        x = resnet_v1.bottleneck(x, W, scope, depth, dbn, stride, rate)
        if end_points is not None:
            end_points[scope] = x
    return x


def heads(inputs, W, net_type, location_refinement=True, end_points=None):
    """(part_pred logits, locref | None) of the pose net on resnet_v1_<depth>."""
    net = extract_features(inputs, W, net_type, end_points)
    pred = pose_net.prediction_layer(net, W, "part_pred")
    loc = pose_net.prediction_layer(net, W, "locref_pred") if location_refinement else None
    return pred, loc
