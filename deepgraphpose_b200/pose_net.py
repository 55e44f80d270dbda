"""Drop-in for deeplabcut.pose_estimation_tensorflow.nnet.pose_net on the DGP path
(reference: src/DeepLabCut/deeplabcut/pose_estimation_tensorflow/nnet/pose_net.py).

``PoseNet(cfg)`` keeps the reference's method names -- ``extract_features``, ``prediction_layers``, ``get_net``, ``test``,
``inference`` -- and the module-level ``prediction_layer``.  Where the reference returns TF graph nodes these return CUDA
tensors computed by the engine; ``inputs`` are uint8 frames (N,H,W,3) (the reference feeds uint8 pixel values into a float32
placeholder).  ``get_net`` runs the fused C-ABI call (``dgp_forward``); ``extract_features`` followed by
``prediction_layers`` gives bit-identical heads through ``dgp_extract_features`` / ``dgp_prediction_layers``.
"""
import ctypes as C

import numpy as np
import torch

from . import synthetic
from .engine import Engine, LOCREF_STDEV, MEAN_PIXEL, _ptr, _stream
from .eval import check_geometry, check_net_type


def _get(cfg, key, default=None):
    if isinstance(cfg, dict):
        return cfg.get(key, default)
    return getattr(cfg, key, default)


def _engine_of(obj):
    return obj.engine if isinstance(obj, PoseNet) else obj


class Features(torch.Tensor):
    """``net`` of extract_features: a float32 CUDA tensor (N,hf,wf,2048) that remembers the engine that produced it, so that
    the module-level ``prediction_layer(cfg, net, name, num_outputs)`` can find the variables of the graph, as the reference's
    TF variable scopes do."""
    engine = None


def prediction_layer(cfg, input, name, num_outputs, engine=None):
    """pose_net.py:18-26: ``slim.conv2d_transpose(input, num_outputs, [3,3], stride=2, SAME)`` under scope ``pose/<name>/block4``
    with the graph's variables.  ``input`` is the ``net`` returned by ``PoseNet.extract_features`` (or any float32 CUDA tensor
    (N,h,w,2048) together with ``engine=``); returns float32 (N,2h,2w,num_outputs)."""
    eng = _engine_of(engine) if engine is not None else getattr(input, "engine", None)
    if eng is None:
        raise ValueError("prediction_layer needs the net of PoseNet.extract_features (or engine=...): the head variables live in the engine")
    if _get(cfg, "deconvolutionstride", 2) != 2:
        raise ValueError("the B200 path implements deconvolutionstride=2")
    heads = {"part_pred": eng.nj, "locref_pred": 2 * eng.nj}
    if name not in heads or (name == "locref_pred" and not eng.location_refinement):
        raise ValueError("no prediction layer %r in this graph" % (name,))
    if int(num_outputs) != heads[name]:
        raise ValueError("%s has %d outputs in this graph, not %d" % (name, heads[name], num_outputs))
    logits, locref = eng.prediction_layers(input, want_locref=(name == "locref_pred"))
    return locref if name == "locref_pred" else logits


class PoseNet:
    def __init__(self, cfg, variables=None, device=None):
        """pose_net.py:28-34: output_stride 8 or 16 (the default), deconvolutionstride 2; at output_stride 8 the cfg's
        stride must be 4.0 (eval.check_geometry)."""
        self.cfg = cfg
        output_stride, stride = check_geometry(cfg)
        self.net_type = _get(cfg, "net_type", "resnet_50")
        synthetic.net_scope(self.net_type)   # resnet_50, resnet_101 or resnet_152 (pose_net.py:14-16)
        if _get(cfg, "intermediate_supervision", False):
            raise ValueError("intermediate_supervision is not on the B200 path (DGP never enables it)")
        self.num_joints = int(_get(cfg, "num_joints"))
        self.location_refinement = bool(_get(cfg, "location_refinement", True))
        self.engine = Engine(self.num_joints, self.location_refinement, device, stride,
                             float(_get(cfg, "locref_stdev", LOCREF_STDEV)), tuple(_get(cfg, "mean_pixel", MEAN_PIXEL)),
                             _get(cfg, "precision", "fp16"), output_stride)
        if variables is not None:
            self.restore(variables)

    def restore(self, variables):
        """Replaces Saver.restore: {tf_var_name: ndarray} with slim names (resnet_v1_<depth>/..., pose/...); the backbone they
        name must be the cfg's net_type (ValueError otherwise)."""
        check_net_type(self.net_type, variables)
        self.engine.load_weights(variables)

    def _frames(self, inputs):
        if isinstance(inputs, torch.Tensor):
            t = inputs
        else:
            t = torch.from_numpy(np.ascontiguousarray(inputs))
        if t.dtype != torch.uint8:
            t = t.to(torch.uint8)
        return t.to(self.engine.device)

    def extract_features(self, inputs):
        """pose_net.py:36-54 -> (net (N,hf,wf,2048) float32, end_points).  ``end_points`` holds the block outputs the
        reference's callers could read: only ``resnet_v1_<depth>/block4`` (= net) is materialised on this path."""
        net = self.engine.extract_features(self._frames(inputs)).as_subclass(Features)
        net.engine = self.engine
        return net, {synthetic.net_scope(self.net_type) + "/block4": net}

    def prediction_layers(self, features, end_points=None, reuse=None):
        """pose_net.py:56-78 -> {'part_pred': (N,2h,2w,nj)[, 'locref': (N,2h,2w,2nj)]}."""
        logits, locref = self.engine.prediction_layers(features, want_locref=self.location_refinement)
        out = {"part_pred": logits}
        if self.location_refinement:
            out["locref"] = locref
        return out

    def get_net(self, inputs):
        """pose_net.py:80-82 -> {'part_pred': logits (N,2h,2w,nj), 'locref': (N,2h,2w,2nj)}."""
        logits, locref = self.engine.forward(self._frames(inputs))
        out = {"part_pred": logits}
        if self.location_refinement:
            out["locref"] = locref
        return out

    def test(self, inputs):
        """pose_net.py:84-90."""
        heads = self.get_net(inputs)
        out = {"part_prob": self.engine.sigmoid(heads["part_pred"])}
        if self.location_refinement:
            out["locref"] = heads["locref"]
        return out

    def inference(self, inputs, reference_batched_locref=False):
        """pose_net.py:92-163: {'pose': (N*nj, 3)}, rows frame-major then joint, columns as the reference emits them:
        ``(row*stride + stride/2 + dy, col*stride + stride/2 + dx, likelihood)`` -- i.e. (y, x, likelihood); DLC's caller
        flips them afterwards.  The global arg-max, the locref gather and the sigmoid run in the fused soft-argmax kernel.

        For N > 1 the reference's batched branch (:129-163) reshapes the (N,H,W,2nj) locref tensor as (H,W,N,nj,2) WITHOUT
        transposing it first (:149), so its offsets come from scrambled positions.  By default every frame gets the offsets
        of its own peak (what the batch-size-1 branch computes); ``reference_batched_locref=True`` reproduces the reference's
        batched arithmetic literally (pinned by tests/golden/boundary.npz)."""
        heads = self.get_net(inputs)
        logits, locref = heads["part_pred"], heads.get("locref")
        r = self.engine.softargmax(logits, locref, want=("dlc_pose", "dlc_peak"))
        pose = r["dlc_pose"].reshape(-1, 3)[:, [1, 0, 2]].contiguous()
        N, H, W, nj = logits.shape
        if reference_batched_locref and locref is not None and N > 1:
            stride, sd = self.engine.stride, self.engine.locref_stdev
            peak = r["dlc_peak"].reshape(-1, 2).long()                      # (N*nj, 2) rows n = b*nj + j
            n = torch.arange(N * nj, device=peak.device)
            m = peak[:, 0] * W + peak[:, 1]                                 # maxloc of column n (pose_net.py:140)
            f = m * (N * nj) + n                                            # flat index into the (H*W, N*nj, 2) view (:153)
            # that view is the transpose [1,2,0,3,4] of the (H,W,N,nj,2) reshape: decode f -> (w, b', h, j')
            jq = f % nj
            hq = (f // nj) % H
            bq = (f // (nj * H)) % N
            wq = f // (nj * H * N)
            src = (((hq * W + wq) * N + bq) * nj + jq) * 2                  # element offset in the original memory
            flat = locref.reshape(-1)
            off = torch.stack([flat[src + 1], flat[src]], dim=1) * sd       # tf.gather(offset, [1, 0], axis=1)
            base = peak.float() * stride + 0.5 * stride
            pose = torch.cat([base + off, pose[:, 2:3]], dim=1)
        return {"pose": pose}
