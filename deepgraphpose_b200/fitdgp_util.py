"""Drop-in for the hot-path helpers of deepgraphpose.models.fitdgp_util
(reference: src/deepgraphpose/models/fitdgp_util.py).

``argmax_2d_from_cm`` keeps the reference signature (:342) and return pair; it takes the (N,H,W,nj) float32 logit
tensor as a CUDA tensor (or a numpy array, copied to the current device) instead of a tf.Tensor.
"""
import ctypes as C

import numpy as np
import torch

from .engine import Engine, _ptr, _stream

_ENGINES = {}


def _engine_for(nj, device):
    key = (int(nj), torch.device(device).index)
    if key not in _ENGINES:
        _ENGINES[key] = Engine(nj, location_refinement=False, device=key[1])
    return _ENGINES[key]


def argmax_2d_from_cm(tensor, nj, gamma=1, gauss_len=2, th=None):
    """fitdgp_util.py:342-402: spatial softmax -> Gaussian blur -> renormalise -> soft-argmax.

    Returns (spatial_soft_argmax (N,nj,2) [(row, col) in scoremap pixels], softmax_tensor0 (N,H,W,nj)).
    ``th`` (:379-389, no reference caller passes it): entries of the blurred map below ``th * max`` are zeroed and the map is
    renormalised before the expectation (``dgp_softmax_threshold``).
    """
    as_numpy = not isinstance(tensor, torch.Tensor)
    t = torch.from_numpy(np.ascontiguousarray(tensor, dtype=np.float32)).cuda() if as_numpy else tensor
    if t.dim() != 4 or t.shape[-1] != nj:
        raise ValueError("tensor must be (N, H, W, nj)")
    eng = _engine_for(nj, t.device)
    sm = eng.softmax_map(t, gamma, gauss_len)
    if th is None:
        mu = eng.softargmax(t, None, gamma, gauss_len, want=("mu",))["mu"]
    else:
        N, H, W, _ = sm.shape
        mu = torch.empty((N, nj, 2), dtype=torch.float32, device=sm.device)
        eng._check(eng.lib.dgp_softmax_threshold(eng.h, _ptr(sm), N, H, W, int(nj), float(th), _ptr(mu), _stream(sm.device)))
    if as_numpy:
        return mu.cpu().numpy(), sm.cpu().numpy()
    return mu, sm


def dgp_prediction_layer(weight_dlc, bias_dlc, dlc_cfg, inputs, name, num_outputs, init_flag, nc, train_flag, stride=2,
                         kernel_size=[3, 3], scope='block4', engine=None):
    """fitdgp_util.py:18-74: ``slim.conv2d_transpose(inputs, num_outputs, kernel_size, stride)`` under ``<name>/<scope>``,
    initialised from ``weight_dlc[:, :, :, :nc]`` / ``bias_dlc`` when ``init_flag``.  ``inputs`` is a float32 CUDA tensor
    (T,nx,ny,nc) (the ``net`` of ``PoseNet.extract_features``); returns float32 (T,2nx,2ny,num_outputs).

    With ``init_flag=False`` the reference creates fresh randomly initialised variables; here the layer then uses the
    variables of the graph ``inputs`` came from (``pose/<name>/block4`` of its engine), which is what its callers restore
    into them.  ``train_flag`` only marks the TF variables trainable and has no effect on the forward value."""
    if int(stride) != 2 or list(kernel_size) != [3, 3]:
        raise ValueError("the B200 path implements the 3x3 stride-2 transposed convolution of the DLC heads")
    t = inputs if isinstance(inputs, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(inputs, dtype=np.float32)).cuda()
    eng = engine if engine is not None else getattr(inputs, "engine", None)
    if init_flag:
        w = np.asarray(weight_dlc, dtype=np.float32)[:, :, :, :nc]
        if w.shape[:3] != (3, 3, int(num_outputs)) or w.shape[3] != t.shape[3]:
            raise ValueError("weight_dlc[:, :, :, :nc] must be [3, 3, %d, %d]" % (num_outputs, t.shape[3]))
        if eng is None:
            eng = _engine_for(int(num_outputs), t.device)
        return eng.deconv2d(t, w, np.asarray(bias_dlc, dtype=np.float32).reshape(-1))
    head = name.split("/")[-1]
    if eng is not None and head in ("part_pred", "locref_pred"):
        from .pose_net import prediction_layer
        return prediction_layer(dlc_cfg, t, head, num_outputs, engine=eng)
    # a scope the graph has no variables for (Dataset._compute_pred_dims builds a throw-away 'confidencemap' layer only to
    # read its output shape, dataset.py:348-371): fresh xavier-uniform weights and zero biases, as slim would create them
    if eng is None:
        eng = _engine_for(int(num_outputs), t.device)
    cin = int(t.shape[3])
    lim = np.sqrt(6.0 / (9 * cin + 9 * int(num_outputs)))
    w = np.random.default_rng(0).uniform(-lim, lim, (3, 3, int(num_outputs), cin)).astype(np.float32)
    return eng.deconv2d(t, w, np.zeros(int(num_outputs), np.float32))


def make_2Dgrids(H, W, device="cuda"):
    """fitdgp_util.py:318-339: (H, W, 1, 2) grid of (row, col)."""
    r = torch.arange(H, dtype=torch.float32, device=device).view(H, 1).expand(H, W)
    c = torch.arange(W, dtype=torch.float32, device=device).view(1, W).expand(H, W)
    return torch.stack([r, c], dim=2).unsqueeze(2)


class AsyncField:
    """A device tensor produced on a side stream plus the event recorded behind its producer (``learn_wt(..., overlap=True)``).
    Fed as ``vector_field_tf``, the loss waits for the event on its own stream (dgp_loss_batch.vector_field_ready_event), so the
    Farneback flow of the batch runs beside the forward pass instead of in front of it."""

    def __init__(self, tensor, event):
        self.tensor, self.event = tensor, event

    @property
    def shape(self):
        return self.tensor.shape


def learn_wt(all_data_batch, engine=None, overlap=False):
    """fitdgp_util.py:454-467: optical-flow magnitude per consecutive frame pair, the ``vector_field_tf`` feed of the
    temporal clique (nt-1, H, W): OpenCV Farneback flow (pyr_scale 0.5, 3 levels, window 15, 3 iterations, poly_n 5,
    poly_sigma 1.2) on the BGR2GRAY-converted frames, |u| + |v|.

    With ``engine`` the whole batch runs on its GPU (``dgp_learn_wt``: all pairs per launch, ~1 ms for 10 frames of 747x832
    where cv2 needs 175 ms per pair on the host) and a float32 CUDA tensor is returned -- ``TrainSession.run`` takes it as the
    ``vector_field_tf`` feed without a round trip; ``overlap=True`` runs it on the engine's side stream and returns an
    ``AsyncField`` (tensor + event) that the loss waits for, so the flow overlaps the forward pass of the training step.
    Without ``engine``: the reference's own cv2 loop on the host."""
    if engine is not None:
        fr = all_data_batch
        if not isinstance(fr, torch.Tensor):
            fr = np.asarray(fr)
            if fr.dtype != np.uint8:
                fr = fr.astype(np.uint8)        # the reference casts every frame with .astype(np.uint8)
            fr = torch.from_numpy(np.ascontiguousarray(fr))
        elif fr.dtype != torch.uint8:
            fr = fr.to(torch.uint8)
        fr = fr.to(engine.device)
        if not overlap:
            return engine.learn_wt(fr)
        main = torch.cuda.current_stream(engine.device)
        side = engine.side_stream()
        side.wait_stream(main)                 # the frames were produced (copied) on the caller's stream
        with torch.cuda.stream(side):
            field = engine.learn_wt(fr)
            ev = torch.cuda.Event()
            ev.record(side)
        field.record_stream(main)              # allocated under the side stream, consumed on the caller's
        fr.record_stream(side)
        return AsyncField(field, ev)
    import cv2
    frames = np.asarray(all_data_batch)
    gray = [cv2.cvtColor(f.astype(np.uint8), cv2.COLOR_BGR2GRAY) for f in frames]
    fields = [np.abs(cv2.calcOpticalFlowFarneback(a, b, None, 0.5, 3, 15, 3, 5, 1.2, 0)).sum(2) for a, b in zip(gray[:-1], gray[1:])]
    return np.array(fields)


class AugPipeline:
    """The pipeline of ``build_aug``: per frame, rotation, motion blur, coarse dropout and elastic deformation (in that order),
    each switched on with probability ``apply_prob`` (imgaug's ``Sometimes``), their parameters drawn from the pipeline's own
    ``np.random.Generator``.  ``sample(n)`` gives the n ``dgp_augment_params`` dicts of the next n frames; every frame
    consumes the same number of draws whichever ops it switches on."""

    def __init__(self, apply_prob, rotation, motion_blur_k, motion_blur_angle, dropout_p, dropout_size_percent, elastic_alpha,
                 elastic_sigma, seed):
        self.apply_prob = float(apply_prob)
        self.rotation = float(rotation)
        self.motion_blur_k = int(motion_blur_k)
        self.motion_blur_angle = tuple(float(v) for v in motion_blur_angle)
        self.dropout_p = tuple(float(v) for v in dropout_p)
        self.dropout_size_percent = tuple(float(v) for v in dropout_size_percent)
        self.elastic_alpha = tuple(float(v) for v in elastic_alpha)
        self.elastic_sigma = float(elastic_sigma)
        if self.motion_blur_k and (self.motion_blur_k < 3 or self.motion_blur_k % 2 == 0):
            raise ValueError("motion_blur_k must be 0 (off) or odd >= 3")
        self.rng = np.random.default_rng(seed)

    def sample(self, n):
        out = []
        for _ in range(int(n)):
            on = self.rng.random(4) < self.apply_prob
            rot = self.rng.uniform(-self.rotation, self.rotation)
            angle = self.rng.uniform(*self.motion_blur_angle)
            direction = self.rng.uniform(-1.0, 1.0)
            p = self.rng.uniform(*self.dropout_p)
            sp = self.rng.uniform(*self.dropout_size_percent)
            alpha = self.rng.uniform(*self.elastic_alpha)
            seed = int(self.rng.integers(0, 2 ** 63))
            out.append(dict(rotate_deg=rot if on[0] else 0.0, blur_k=self.motion_blur_k if on[1] else 0,
                            blur_angle_deg=angle, blur_direction=direction, drop_p=p if on[2] else 0.0,
                            drop_size_percent=sp if on[2] else 0.0, elastic_alpha=alpha if on[3] else 0.0,
                            elastic_sigma=self.elastic_sigma, seed=seed))
        return out


def build_aug(apply_prob=0.5, rotation=25, motion_blur_k=7, motion_blur_angle=(-90, 90), dropout_p=(0, 0.02),
              dropout_size_percent=(0.01, 0.05), elastic_alpha=(0, 40), elastic_sigma=5, seed=None):
    """fitdgp_util.py:412-451: the augmenters DeepLabCut's imgaug pipeline builds by default, each under
    ``iaa.Sometimes(apply_prob)``: ``Affine(rotate=(-rotation, rotation))``, ``MotionBlur(k=motion_blur_k,
    angle=motion_blur_angle)``, ``CoarseDropout(dropout_p, size_percent=dropout_size_percent)`` and
    ``ElasticTransformation(alpha=elastic_alpha, sigma=elastic_sigma)``.  Returns the sampler ``data_aug`` takes; the
    transforms run on the device (``dgp_augment``, bilinear elastic sampling -- see DESIGN.md)."""
    return AugPipeline(apply_prob, rotation, motion_blur_k, motion_blur_angle, dropout_p, dropout_size_percent, elastic_alpha,
                       elastic_sigma, seed)


def data_aug(all_data_batch, visible_frame_within_batch, joint_loc, pipeline, dlc_cfg, engine=None):
    """fitdgp_util.py data_aug, as called at fitdgp.py:773-779: augments the frames of the batch at the positions
    ``visible_frame_within_batch`` and moves their labels ``joint_loc`` ((n_vis, nj, 2) scoremap (row, col), stride
    ``dlc_cfg.stride``) with them.  ``all_data_batch``: (nt,H,W,3) frames on the host (non-uint8 values are rounded and
    clipped as ``TrainSession.run`` does) or a CUDA tensor; neither is modified.  Returns (uint8 CUDA frames, float64 CUDA
    joint_loc), ready to feed as ``inputs`` / ``targets``."""
    from .fitdgp import _get
    fr = all_data_batch
    dev = engine.device if engine is not None else (fr.device if isinstance(fr, torch.Tensor) and fr.is_cuda
                                                    else torch.device("cuda", torch.cuda.current_device()))
    if isinstance(fr, torch.Tensor):
        if fr.dtype != torch.uint8:
            raise ValueError("a tensor batch must hold uint8 frames")
        fr = fr.to(dev).clone(memory_format=torch.contiguous_format)
    else:
        fr = np.asarray(fr)
        if fr.dtype != np.uint8:
            fr = np.clip(np.round(fr), 0, 255).astype(np.uint8)
        fr = torch.from_numpy(np.ascontiguousarray(fr)).to(dev)
    if isinstance(joint_loc, torch.Tensor):
        jl = joint_loc.to(device=dev, dtype=torch.float64).clone(memory_format=torch.contiguous_format)
    else:
        jl = torch.from_numpy(np.ascontiguousarray(np.asarray(joint_loc, dtype=np.float64))).to(dev)
    pos = np.asarray(visible_frame_within_batch, dtype=np.int64).reshape(-1)
    if jl.dim() != 3 or jl.shape[0] != pos.shape[0] or jl.shape[2] != 2:
        raise ValueError("joint_loc must be (n_vis, nj, 2) with one label set per visible frame")
    if pos.shape[0] == 0:
        return fr, jl
    eng = engine if engine is not None else _engine_for(jl.shape[1], dev)
    eng.augment(fr, pos, jl, pipeline.sample(pos.shape[0]), stride=float(_get(dlc_cfg, "stride", 8.0)))
    return fr, jl
