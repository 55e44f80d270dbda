"""Drop-in for the hot-path part of deepgraphpose.models.fitdgp (reference: src/deepgraphpose/models/fitdgp.py).

``dgp_loss(data_batcher, dgp_cfg)`` keeps the reference's signature and 4-tuple return
``(loss, total_loss, total_loss_visible, placeholders)`` (:848-1144); the handles are evaluated by ``TrainSession.run``
with the reference's feed_dict keys.  ``momentum_train_op`` stands in for fitdgp.py:706-713 (MomentumOptimizer + global-norm
clipping); fetching it from ``TrainSession.run`` runs the whole training step on the GPU (network forward, fused loss
kernels, dgrad/wgrad of every conv on tcgen05, optimizer) and, when ``torch.distributed`` is initialised, averages the
gradients over the ranks with one NCCL all-reduce of the flat gradient buffer (``dp.allreduce_gradients``).
"""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import torch

from . import _lib
from .engine import Engine, _ptr, _stream
from .session import Handle

LOSS_KEYS = ("visible_loss_pred", "hidden_loss_pred", "visible_loss_locref", "ws_loss", "wt_loss", "total_loss")
PLACEHOLDER_KEYS = ("inputs", "targets", "locref_map", "locref_mask", "visible_marker_pl", "hidden_marker_pl",
                    "visible_marker_in_targets_pl", "wt_batch_mask_pl", "vector_field_tf", "nt_batch_pl", "wt_batch_pl",
                    "alpha_tf")
# One placeholder beyond the reference's twelve: feeding the batch positions of the visible frames (fit_dgp's own
# `visible_frame_within_batch`, fitdgp.py:763) INSTEAD of locref_map / locref_mask makes the device build the two maps
# (coord2map feeder kernel) rather than copying 2 x (nt,H,W,2nj) float64 arrays from the host every step.
EXTRA_PLACEHOLDER_KEYS = ("visible_frame_within_batch",)


def _get(cfg, key, default=None):
    if isinstance(cfg, dict):
        return cfg.get(key, default)
    return getattr(cfg, key, default)


def skeleton_edges(S0):
    """Rows of the reference's S0 incidence matrix (fitdgp.py:607-617) -> (+1 joint, -1 joint) pairs."""
    S0 = np.asarray(S0)
    edges = []
    for row in S0:
        a, b = np.where(row > 0)[0], np.where(row < 0)[0]
        if len(a) != 1 or len(b) != 1:
            raise ValueError("S0 rows must hold exactly one +1 and one -1")
        edges.append((int(a[0]), int(b[0])))
    return edges


def spatial_clique_params(joint_locs, S0, stride, ws, ws_max):
    """Host precompute of dgp_loss (fitdgp.py:874-892): per limb l = (a, b) of the skeleton and over every labelled frame t,
    ``L[t, l] = |label[t, a] - label[t, b]| * stride + stride / 2`` in image pixels, then the clique's upper bound
    ``ws_max_l = ws_max * max_t L`` and weight ``ws_l = ws / mean_t L``.  A coordinate difference with an unlabelled (NaN) end
    counts as 0, so a limb missing from a frame enters the mean with length stride/2 -- the reference's behaviour (its
    ``!= 0`` mask never excludes anything because stride/2 was already added), kept for parity.
    joint_locs: one (n_vis_i, nj, 2) array of scoremap (row, col) labels per dataset."""
    edges = skeleton_edges(S0)
    labelled = [np.asarray(j, dtype=np.float64) for j in joint_locs if len(j) > 0]
    if not labelled:
        raise ValueError("spatial_clique_params needs at least one labelled frame (the reference takes max over frames)")
    lab = np.concatenate(labelled, axis=0)
    head = np.array([e[0] for e in edges], dtype=np.int64)
    tail = np.array([e[1] for e in edges], dtype=np.int64)
    diff = lab[:, head, :] - lab[:, tail, :]                 # (T, nl, 2); NaN wherever an end point is unlabelled
    diff = np.where(np.isnan(diff), 0.0, diff)
    length_px = np.hypot(diff[..., 0], diff[..., 1]) * stride + 0.5 * stride
    upper = ws_max * length_px.max(axis=0) if len(edges) else np.zeros(0)
    weight = ws / (length_px.mean(axis=0) + 1e-20) if len(edges) else np.zeros(0)
    return weight.astype(np.float32), upper.astype(np.float32)


def _loss_args(dev, feed, cfg, edges, ws, ws_max, n_frames_total, n_visible_frames_total, nt, H, W, nj, pred=None,
               locref=None, with_locref=None, engine=None):
    """(dgp_loss_cfg, dgp_loss_batch, keep-alive list) from the reference's feed_dict values (fitdgp.py:797-815).
    When the feed carries ``visible_frame_within_batch`` instead of ``locref_map`` / ``locref_mask``, the two maps are
    generated on the device (Engine.locref_targets, the coord2map feeder) instead of being copied from the host."""
    def f32(a):   # host arrays are uploaded; CUDA tensors (feeds produced on the device) are used in place
        if isinstance(a, torch.Tensor):
            return a.to(device=dev, dtype=torch.float32).contiguous()
        return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32), device=dev)

    def i32(a):
        if isinstance(a, torch.Tensor):
            return a.to(device=dev, dtype=torch.int32).contiguous()
        return torch.as_tensor(np.ascontiguousarray(a, dtype=np.int32), device=dev)
    tg = feed["targets"]
    targets = f32(tg if isinstance(tg, torch.Tensor) else np.asarray(tg)).reshape(-1, nj, 2)
    vis, hid, vit = i32(feed["visible_marker_pl"]), i32(feed["hidden_marker_pl"]), i32(feed["visible_marker_in_targets_pl"])
    keep = [targets, vis, hid, vit]
    b = _lib.DgpLossBatch()
    b.nt, b.H, b.W = nt, H, W
    if pred is not None:
        b.pred_dev = pred.data_ptr()
    b.targets_dev, b.nv = targets.data_ptr(), targets.shape[0]
    if with_locref is None:
        with_locref = locref is not None
    if with_locref:
        if "locref_map" in feed:
            lm, lk = f32(feed["locref_map"]), f32(feed["locref_mask"])
        else:
            lm, lk = engine.locref_targets(feed["targets"], feed["visible_frame_within_batch"], nt, H, W,
                                           float(_get(cfg, "pos_dist_thresh", 17.0)), float(_get(cfg, "locref_stdev", 7.2801)))
        keep += [lm, lk]
        b.locref_map_dev, b.locref_mask_dev = lm.data_ptr(), lk.data_ptr()
        if locref is not None:
            b.locref_dev = locref.data_ptr()
    b.visible_marker_dev, b.nbv = vis.data_ptr(), vis.numel()
    b.hidden_marker_dev, b.nbh = hid.data_ptr(), hid.numel()
    b.visible_marker_in_targets_dev = vit.data_ptr()
    if len(edges) > 0:
        e, w1, w2 = i32(np.asarray(edges).reshape(-1, 2)), f32(ws), f32(ws_max)
        keep += [e, w1, w2]
        b.edges_dev, b.nl, b.ws_dev, b.ws_max_dev = e.data_ptr(), len(edges), w1.data_ptr(), w2.data_ptr()
    wt = float(_get(cfg, "wt", 0.0))
    if wt > 0:
        vfeed = feed["vector_field_tf"]
        ready = None
        if hasattr(vfeed, "event") and hasattr(vfeed, "tensor"):     # fitdgp_util.AsyncField: produced on a side stream
            vfeed, ready = vfeed.tensor, vfeed.event
        vf = f32(vfeed)
        if ready is not None:
            keep.append(ready)
            b.vector_field_ready_event = ready.cuda_event
        if vf.dim() != 3 or vf.shape[0] != nt - 1:
            raise ValueError("vector_field_tf must be (nt-1, Hin, Win) = (%d, ., .), got %s" % (nt - 1, tuple(vf.shape)))
        wb = f32(np.asarray(feed["wt_batch_pl"], dtype=np.float32) * np.asarray(feed["wt_batch_mask_pl"], dtype=np.float32))
        keep += [vf, wb]
        b.vector_field_dev, b.Hin, b.Win, b.wt_batch_dev = vf.data_ptr(), vf.shape[1], vf.shape[2], wb.data_ptr()
    c = _lib.DgpLossCfg(float(_get(cfg, "gamma", 1)), float(_get(cfg, "gauss_len", 1)), float(_get(cfg, "lengthscale", 1)),
                        wt, float(_get(cfg, "wt_max", 0)), float(_get(cfg, "wn_visible", 5)), float(_get(cfg, "wn_hidden", 3)),
                        float(_get(cfg, "locref_loss_weight", 0.05)), float(n_frames_total), float(n_visible_frames_total),
                        int(_get(cfg, "gm2", 1)), int(_get(cfg, "gm3", 3)),
                        0 if bool(_get(cfg, "locref_huber_loss", True)) else 1)
    return c, b, keep


def loss_forward(engine, pred, locref, feed, cfg, edges, ws, ws_max, n_frames_total, n_visible_frames_total,
                 backward=False, visible_only=False):
    """One call into dgp_loss_forward (or dgp_loss_backward).  pred/locref: CUDA tensors from Engine.forward; feed:
    reference feed_dict values.  With backward=True returns (losses, (grad_pred, grad_locref))."""
    dev = pred.device
    nt, H, W, nj = pred.shape
    c, b, keep = _loss_args(dev, feed, cfg, edges, ws, ws_max, n_frames_total, n_visible_frames_total, nt, H, W, nj, pred,
                            locref)
    out = torch.empty(6, dtype=torch.float32, device=dev)
    if backward:
        g_pred = torch.empty_like(pred)
        g_loc = torch.empty_like(locref) if locref is not None else None
        engine._check(engine.lib.dgp_loss_backward(engine.h, C.byref(c), C.byref(b), _ptr(out), _ptr(g_pred), _ptr(g_loc),
                                                   int(visible_only), _stream(dev)))
        vals = out.cpu().numpy()
        del keep
        return dict(zip(LOSS_KEYS, [np.float32(v) for v in vals])), (g_pred, g_loc)
    all_markers = torch.empty((nt * nj, 2), dtype=torch.float32, device=dev)
    engine._check(engine.lib.dgp_loss_forward(engine.h, C.byref(c), C.byref(b), _ptr(out), _ptr(all_markers), _stream(dev)))
    vals = out.cpu().numpy()
    del keep
    return dict(zip(LOSS_KEYS, [np.float32(v) for v in vals])), all_markers


class _DgpLossFunction(torch.autograd.Function):
    """dgp_loss_backward as an autograd node: the forward computes the six losses and the gradients of the differentiated
    total w.r.t. the heads in one call; the backward scales those gradients by grad_output."""

    @staticmethod
    def forward(ctx, pred, locref, engine, feed, cfg, edges, ws, ws_max, n_frames_total, n_visible_frames_total, visible_only):
        dev = pred.device
        nt, H, W, nj = pred.shape
        pred = pred.detach().contiguous()
        locref = locref.detach().contiguous() if locref is not None else None
        c, b, keep = _loss_args(dev, feed, cfg, edges, ws, ws_max, n_frames_total, n_visible_frames_total, nt, H, W, nj, pred,
                                locref, engine=engine)
        out = torch.empty(6, dtype=torch.float32, device=dev)
        g_pred = torch.empty_like(pred)
        g_loc = torch.empty_like(locref) if locref is not None else None
        engine._check(engine.lib.dgp_loss_backward(engine.h, C.byref(c), C.byref(b), _ptr(out), _ptr(g_pred), _ptr(g_loc),
                                                   int(visible_only), _stream(dev)))
        ctx.keep = keep   # feed tensors (some produced on a side stream) outlive the asynchronous loss kernels
        ctx.grads = (g_pred, g_loc)
        vals = torch.cat([out, (out[0] + out[2]).view(1)])   # + total_loss_visible
        ctx.mark_non_differentiable(vals)
        return vals[6 if visible_only else 5].clone(), vals

    @staticmethod
    def backward(ctx, g_total, g_vals):
        g_pred, g_loc = ctx.grads
        return (g_pred * g_total, g_loc * g_total if g_loc is not None else None) + (None,) * 9


def _loss_engine(dev, nj, cfg):
    """A weight-less handle that runs the loss kernels, one per (device, joints, stride, locref_stdev, output_stride)."""
    from .eval import check_geometry
    output_stride, stride = check_geometry(cfg)
    key = (str(dev), int(nj), stride, float(_get(cfg, "locref_stdev", 7.2801)), output_stride)
    eng = _LOSS_ENGINES.get(key)
    if eng is None:
        eng = _LOSS_ENGINES[key] = Engine(nj, device=dev, stride=key[2], locref_stdev=key[3], output_stride=output_stride)
    return eng


_LOSS_ENGINES = {}


def dgp_loss_function(pred, locref, feed, cfg, edges, ws, ws_max, n_frames_total, n_visible_frames_total, visible_only=False,
                      engine=None):
    """dgp_loss (fitdgp.py:934-1128) as a differentiable PyTorch function of the heads: pred float32 CUDA (nt,H,W,nj) and
    locref (nt,H,W,2nj) or None, e.g. from ``autograd.TrainablePoseNet``; the other arguments as in ``loss_forward``.
    Returns {LOSS_KEYS..., "total_loss_visible"} as 0-d tensors; ``total_loss`` (``total_loss_visible`` when visible_only)
    is differentiable, the others are values only.  ``dgp_total + my_term`` then trains on the sum.  ``engine``: the handle
    whose loss kernels run (default: a weight-less one per device and joint count)."""
    if engine is None:
        engine = _loss_engine(pred.device, pred.shape[-1], cfg)
    total, vals = _DgpLossFunction.apply(pred, locref, engine, feed, cfg, edges, ws, ws_max, n_frames_total,
                                         n_visible_frames_total, bool(visible_only))
    out = {k: vals[i] for i, k in enumerate(LOSS_KEYS + ("total_loss_visible",))}
    out["total_loss_visible" if visible_only else "total_loss"] = total
    return out


def train_forward_backward(engine, frames, feed, cfg, edges, ws, ws_max, n_frames_total, n_visible_frames_total,
                           visible_only=False, sync=True):
    """Forward + loss + full backward of one fit_dgp batch (fitdgp.py:817-818 without the apply step): fills the
    engine's gradient buffer.  frames: uint8 CUDA tensor (nt,H,W,3).  Returns the loss dict (or the device tensor of the 6
    loss values when sync=False)."""
    dev = frames.device
    nt, Hin, Win, _ = frames.shape
    _, (H, W) = engine.output_dims(Hin, Win)
    engine.train_enable()
    c, b, keep = _loss_args(dev, feed, cfg, edges, ws, ws_max, n_frames_total, n_visible_frames_total, nt, H, W, engine.nj,
                            with_locref=engine.location_refinement, engine=engine)
    out = torch.empty(6, dtype=torch.float32, device=dev)
    engine._check(engine.lib.dgp_train_forward_backward(engine.h, _ptr(frames.contiguous()), nt, Hin, Win, C.byref(c), C.byref(b),
                                                        int(visible_only), _ptr(out), _stream(dev)))
    if not sync:
        engine._keep = keep  # device buffers must outlive the asynchronous launches
        return out
    vals = out.cpu().numpy()
    del keep
    return dict(zip(LOSS_KEYS, [np.float32(v) for v in vals]))


def dgp_loss(data_batcher, dgp_cfg, variables=None, device=None):
    """fitdgp.py:848-1144.  Returns (loss, total_loss, total_loss_visible, placeholders) of handles; evaluate them with
    ``TrainSession(...)``.run(fetches, feed_dict) using the reference's placeholder keys.

    The reference builds the graph here and restores ``init_weights`` into it afterwards (``restorer.restore``,
    fitdgp.py:689-720).  The engine needs its variables at construction, so they come from ``variables`` (a
    ``{tf_var_name: ndarray}`` dict, an ``.npz``, a TensorFlow checkpoint prefix, or ``'synthetic[:seed]'`` spelled out) or,
    when that is None, from ``dgp_cfg.init_weights`` -- the snapshot the reference would restore.  There is no default: a
    drop-in call never trains from random weights silently."""
    from .eval import check_geometry, load_variables
    output_stride, stride = check_geometry(dgp_cfg)
    S0 = np.asarray(data_batcher.S0)
    nj = int(data_batcher.nj)
    gm2, gm3 = int(_get(dgp_cfg, "gm2", 1)), int(_get(dgp_cfg, "gm3", 3))
    if gm2 not in (0, 1, 2) or gm3 not in (0, 3):
        raise Exception("Not implemented")  # fitdgp.py:1021, 1037
    if gm3 == 3 and gm2 == 0:
        # the reference dies here with NameError: pred_h_scaled1 is only defined for gm2 in {1, 2} (fitdgp.py:994-1033)
        raise NameError("name 'pred_h_scaled1' is not defined (gm3=3 needs gm2 in {1, 2}, fitdgp.py:1027)")
    if variables is None:
        variables = _get(dgp_cfg, "init_weights", None)
        if variables is None:
            raise ValueError("dgp_loss needs the network variables: pass variables=... or set dgp_cfg.init_weights to the "
                             "snapshot fit_dgp would restore (fitdgp.py:592, 720)")
    ws, ws_max = spatial_clique_params([d.labels for d in data_batcher.datasets], S0, stride,
                                       float(_get(dgp_cfg, "ws", 1000.0)), float(_get(dgp_cfg, "ws_max", 1.2)))
    eng = Engine(nj, location_refinement=True, device=device, stride=stride,
                 locref_stdev=float(_get(dgp_cfg, "locref_stdev", 7.2801)),
                 mean_pixel=tuple(_get(dgp_cfg, "mean_pixel", (123.68, 116.779, 103.939))),
                 precision=_get(dgp_cfg, "precision", "fp16"), output_stride=output_stride)
    eng.load_weights(load_variables(variables, nj, True, _get(dgp_cfg, "net_type", "resnet_50")))
    graph = SimpleNamespace(engine=eng, cfg=dgp_cfg, edges=skeleton_edges(S0) if S0.shape[0] else [], ws=ws, ws_max=ws_max,
                            n_frames_total=float(data_batcher.n_frames_total),
                            n_visible_frames_total=float(data_batcher.n_visible_frames_total))
    keys = [k for k in LOSS_KEYS if (k != "wt_loss" or float(_get(dgp_cfg, "wt", 0)) > 0) and (k != "ws_loss" or S0.shape[0] > 0)]
    loss = {k: Handle(k, k) for k in keys}
    for hd in loss.values():
        hd.graph = graph
    total_loss_visible = Handle("total_loss_visible", "total_loss_visible")
    total_loss_visible.graph = graph
    placeholders = {k: Handle(k, k) for k in PLACEHOLDER_KEYS + EXTRA_PLACEHOLDER_KEYS}
    return loss, loss["total_loss"], total_loss_visible, placeholders


def momentum_train_op(total_loss, learning_rate=None, momentum=0.9, clip_norm=10.0, group=None):
    """fitdgp.py:706-713: ``optimizer = MomentumOptimizer(learning_rate, 0.9); grads = compute_gradients(total_loss,
    trainable_variables()); grads, _ = clip_by_global_norm(grads, 10.0); train_op = apply_gradients(...)``.
    ``total_loss`` is the handle to differentiate (``total_loss`` or ``total_loss_visible``); ``learning_rate`` a float or
    the placeholder handle returned by ``learning_rate_placeholder()``.  Returns the train_op handle."""
    op = Handle("train_op", "train_op")
    op.graph = total_loss.graph
    op.visible_only = total_loss.kind == "total_loss_visible"
    op.learning_rate, op.momentum, op.clip_norm, op.group = learning_rate, float(momentum), float(clip_norm), group
    return op


def learning_rate_placeholder():
    """``learning_rate = TF.placeholder(tf.float32, shape=[])`` (fitdgp.py:686)."""
    return Handle("learning_rate", "learning_rate")


class TrainSession:
    """``sess.run([loss, train_op], feed_dict)`` for the handles of ``dgp_loss`` / ``momentum_train_op``."""

    def __init__(self, placeholders):
        self.ph = placeholders

    def variables(self, graph, names):
        """Current values of trainable variables by TF name (what ``saver.save`` would write, fitdgp.py:830-839)."""
        return {n: graph.engine.get_variable(n) for n in names}

    def run(self, fetches, feed_dict):
        from . import dp
        feed = {}
        for k, v in feed_dict.items():
            if isinstance(k, str) and k in self.ph:     # plain placeholder names are accepted as keys too
                feed[k] = v
                continue
            for name, hd in self.ph.items():
                if k is hd:
                    feed[name] = v
        flat = []
        def collect(f):
            if isinstance(f, dict):
                for v in f.values():
                    collect(v)
            elif isinstance(f, (list, tuple)):
                for v in f:
                    collect(v)
            else:
                flat.append(f)
        collect(fetches)
        g = flat[0].graph
        frames = feed["inputs"]
        if isinstance(frames, torch.Tensor):           # frames already on the device (fitdgp_util.data_aug)
            if frames.dtype != torch.uint8:
                raise ValueError("a tensor fed as inputs must hold uint8 frames")
            frames = frames.to(g.engine.device).contiguous()
        else:
            frames = np.asarray(frames)
            if frames.dtype != np.uint8:
                frames = np.clip(np.round(frames), 0, 255).astype(np.uint8)
            frames = torch.from_numpy(np.ascontiguousarray(frames)).to(g.engine.device)
        train_ops = [f for f in flat if f.kind == "train_op"]
        if train_ops:
            op = train_ops[0]
            lr = op.learning_rate
            if isinstance(lr, Handle):
                lr = [v for k, v in feed_dict.items() if k is lr]
                if not lr:
                    raise ValueError("feed_dict must provide the learning_rate placeholder")
                lr = lr[0]
            # nothing blocks the host between the backward, the gradient all-reduce (whose first buckets overlap the rest of
            # the backward on the handle's communication stream) and the optimizer: the six loss values are read only after
            # all three are enqueued
            out = train_forward_backward(g.engine, frames, feed, g.cfg, g.edges, g.ws, g.ws_max, g.n_frames_total,
                                         g.n_visible_frames_total, visible_only=op.visible_only, sync=False)
            scale = dp.allreduce_gradients(g.engine, op.group)
            g.engine.optimizer_step(float(lr), op.momentum, op.clip_norm, scale)
            vals = dict(zip(LOSS_KEYS, [np.float32(v) for v in out.cpu().numpy()]))
        else:
            pred, locref = g.engine.forward(frames)
            vals, _ = loss_forward(g.engine, pred, locref, feed, g.cfg, g.edges, g.ws, g.ws_max, g.n_frames_total,
                                   g.n_visible_frames_total)
        vals["total_loss_visible"] = np.float32(vals["visible_loss_pred"] + vals["visible_loss_locref"])
        vals["train_op"] = None
        def build(f):
            if isinstance(f, dict):
                return {k: build(v) for k, v in f.items()}
            if isinstance(f, (list, tuple)):
                return type(f)(build(v) for v in f)
            return vals[f.kind]
        return build(fetches)


# ----------------------------------------------------------------------------------------------------------------------
# fit_dgp / fit_dgp_labeledonly step loops (fitdgp.py:549-845, 257-546)
# ----------------------------------------------------------------------------------------------------------------------
def gen_batch(visible_frame_total, hidden_frame_total, all_frame_total, dgp_cfg, maxiters):
    """Pre-computed batch list of fit_dgp (fitdgp_util.py:146-202): per dataset, windows of ``batch_size`` consecutive entries
    of its sorted frame pool starting at random offsets (single frames when the pool is smaller than a batch), each tagged
    with the dataset index as its last element; all windows shuffled.  Draws from ``np.random`` / ``random`` in the
    reference's order, so the same seeds give the same list (pinned by tests/golden/feeders.npz)."""
    import random
    batch_size = int(_get(dgp_cfg, "batch_size"))
    n_frames_total = int(np.sum([len(v) for v in all_frame_total]))
    nepoch = int(min(int(n_frames_total * _get(dgp_cfg, "n_times_all_frames") / batch_size), maxiters))
    windows = []
    for i in range(len(all_frame_total)):
        pool = np.unique(list(visible_frame_total[i]) + list(all_frame_total[i]) + list(hidden_frame_total[i]))
        n_win = max(1, int(nepoch / n_frames_total * len(pool)))
        if len(pool) < batch_size:
            width = 1
            starts = np.random.randint(0, len(pool), size=n_win)
        else:
            width = batch_size
            starts = np.random.randint(0, len(pool) - batch_size, size=n_win)
        picks = pool[(starts[:, None] + np.arange(width)[None, :]).astype(np.int64)]
        tagged = np.hstack([picks, np.full((n_win, 1), i)])
        windows += [w.astype(np.int32) for w in tagged]
    return random.sample(windows, len(windows))


def _fit_loop(data_batcher, dgp_cfg, variables, visible_frame_total, hidden_frame_total, all_frame_total, maxiters, step,
              saveiters, displayiters, debug, labeled_only, device, batch_ind_all=None, snapshot_fn=None, verbose=True,
              aug_pipeline=None):
    """The training loop both drivers share (fitdgp.py:727-845 / 431-546): batch schedule, per-batch feeds (learn_wt flow field
    when wt > 0, coord2map locref targets -- built on the device --, 2-D grids), ``sess.run([loss, train_op])`` and snapshots.
    With ``aug_pipeline`` (fitdgp_util.build_aug) the batch is uploaded once and its labelled frames and their labels are
    augmented on the device (fitdgp_util.data_aug, fitdgp.py:773-779) before they are fed.
    Returns the list of per-iteration loss dicts (the reference only prints them)."""
    import time
    from random import randint
    from .fitdgp_util import data_aug, learn_wt
    loss, total_loss, total_loss_visible, placeholders = dgp_loss(data_batcher, dgp_cfg, variables=variables, device=device)
    learning_rate = learning_rate_placeholder()
    train_op = momentum_train_op(total_loss_visible if labeled_only else total_loss, learning_rate)   # fitdgp.py:706-713
    sess = TrainSession(placeholders)
    engine = total_loss.graph.engine
    if batch_ind_all is None:
        if labeled_only:
            # fitdgp.py:431-439: one labelled frame per iteration, drawn uniformly over the (dataset, frame) pairs
            pairs = np.array([(v, i) for i, vis in enumerate(visible_frame_total) for v in vis]).reshape(-1, 2)
            n_vis = float(_get(dgp_cfg, "n_visible_frames_total", None) or data_batcher.n_visible_frames_total)
            nepoch = int(min(int(n_vis * _get(dgp_cfg, "n_times_all_frames")), maxiters))
            batch_ind_all = [pairs[k] for k in np.random.randint(0, pairs.shape[0], size=nepoch)]
        else:
            batch_ind_all = gen_batch(visible_frame_total, hidden_frame_total, all_frame_total, dgp_cfg, maxiters)
    save_iters = max(1, int(saveiters) if labeled_only else int(saveiters / int(_get(dgp_cfg, "batch_size"))))
    maxiters = len(batch_ind_all)
    data_batcher.reset()
    wt = float(_get(dgp_cfg, "wt", 0))
    prefix = str(_get(dgp_cfg, "snapshot_prefix", "snapshot"))
    history = []
    t_start = time.time()
    for it in range(maxiters):
        batch_ind = batch_ind_all[it]
        dataset_i = int(batch_ind[-1])
        all_frame_batch = batch_ind[:-1]
        visible_frame_i = visible_frame_total[dataset_i]
        all_frame_i = list(all_frame_total[dataset_i]) + list(hidden_frame_total[dataset_i])
        visible_frame_batch_i = np.sort(np.array([i for i in all_frame_batch if i in visible_frame_i]))
        if len(visible_frame_batch_i) == 0 and len(visible_frame_i) > 0:
            visible_frame_batch_i = np.array([visible_frame_i[randint(0, len(visible_frame_i) - 1)]])
        if labeled_only:
            hidden_frame_batch_i = np.array([], dtype=np.int64)
        else:
            hidden_frame_batch_i = np.sort(np.array([i for i in all_frame_batch if (i in all_frame_i) and (i not in visible_frame_i)]))
        (visible_frame, hidden_frame, _, all_data_batch, joint_loc, wt_batch_mask, all_marker_batch, addn_batch_info), d = \
            data_batcher.next_batch(0, dataset_i, visible_frame_batch_i, hidden_frame_batch_i)
        nt_batch = len(visible_frame) + len(hidden_frame)
        visible_marker, hidden_marker, visible_marker_in_targets = addn_batch_info
        all_frame = np.sort(list(visible_frame) + list(hidden_frame))
        visible_frame_within_batch = [int(np.where(all_frame == i)[0][0]) for i in visible_frame]
        if aug_pipeline is not None:
            all_data_batch, joint_loc = data_aug(all_data_batch, visible_frame_within_batch, joint_loc, aug_pipeline, dgp_cfg,
                                                 engine=engine)
        # Farneback flow on the GPU, on a side stream: it overlaps the forward pass of this step (the loss waits for its event)
        vector_field = learn_wt(all_data_batch, engine=engine, overlap=True) if wt > 0 else np.zeros((1, 1, 1))
        feed = {
            placeholders["inputs"]: all_data_batch,
            placeholders["targets"]: joint_loc,
            # coord2map (dataset.py:242-331) runs on the device from `targets` + the batch positions of the visible frames
            placeholders["visible_frame_within_batch"]: visible_frame_within_batch,
            placeholders["visible_marker_pl"]: visible_marker,
            placeholders["hidden_marker_pl"]: hidden_marker,
            placeholders["visible_marker_in_targets_pl"]: visible_marker_in_targets,
            placeholders["wt_batch_mask_pl"]: wt_batch_mask,
            placeholders["vector_field_tf"]: vector_field,
            placeholders["nt_batch_pl"]: nt_batch,
            placeholders["wt_batch_pl"]: np.ones(nt_batch - 1) * wt,
            learning_rate: float(_get(dgp_cfg, "lr", 0.005)),
        }
        t0 = time.time()
        loss_eval, _ = sess.run([loss, train_op], feed)
        history.append(loss_eval)
        if verbose and it % displayiters == 0 and it > 0:
            print("\nIteration {}/{}".format(it, maxiters))
            print("dataset_i: ", dataset_i, flush=True)
            print("\n running time: ", time.time() - t0, flush=True)
            print("\n loss: ", loss_eval, flush=True)
        if (it % save_iters == 0) or (it + 1) == maxiters:
            names = [prefix + "-step" + str(step) + "{}".format(debug) + "-"]
            if (it + 1) == maxiters:
                names.append(prefix + "-step" + str(step) + "{}".format(debug) + "-final-")
            for model_name in names:
                if snapshot_fn is not None:
                    snapshot_fn(engine, model_name, it)
                else:   # saver.save(sess, model_name, global_step=...): TensorFlow checkpoint bundles
                    engine.save_tf_checkpoint(model_name + "-0")
                    if model_name.endswith("-") and not model_name.endswith("-final-"):
                        engine.save_tf_checkpoint(model_name + "-%d" % it)
    if verbose:
        print("Finished {} iterations\n".format(maxiters), flush=True)
        print("\n\n TOTAL TIME ELAPSED: ", time.time() - t_start)
    engine.close()
    return history


_PROJECT_READER_MSG = (
    "%s(snapshot, dlcpath, ...): reading the DLC project (config.yaml, labelled frames, videos_dgp/*) into a MultiDataset is the "
    "reference's host-side data pipeline (dataset.py, moviepy decode) and is outside this library's scope (SURVEY.md 8: the "
    "path starts at the feed_dict).  Pass data_batcher= (any object with the MultiDataset interface: .datasets[i].nx_out / "
    ".ny_out / .labels, .S0, .nj, .n_frames_total, .n_visible_frames_total, .reset(), .next_batch(...)), dgp_cfg= and the frame "
    "index lists; the step loop, feeders, loss, backward and optimizer then run here.")


def fit_dgp(snapshot, dlcpath, batch_size=10, shuffle=1, step=2, saveiters=1000, displayiters=5, maxiters=200000, ns=10,
            nc=2048, n_max_frames=2000, gm2=0, gm3=0, nepoch=100, wt=0, aug=True, debug="", trainingsetindex=0, *,
            data_batcher=None, dgp_cfg=None, frame_lists=None, variables=None, device=None, batch_ind_all=None,
            snapshot_fn=None, verbose=True, aug_pipeline=None):
    """fitdgp.py:549-845 with the reference's argument list.  The keyword-only arguments carry what the reference derives from
    the DLC project on the host: ``data_batcher`` (MultiDataset interface), ``dgp_cfg`` (the merged training config; gm2 / gm3 /
    wt / batch_size given here override it like fitdgp.py:640-660), ``frame_lists`` = (visible_frame_total, hidden_frame_total,
    all_frame_total) and ``variables`` (what ``restorer.restore(sess, init_weights)`` would load; defaults to
    dgp_cfg.init_weights or ``snapshot``).  ``aug_pipeline`` (``fitdgp_util.build_aug(...)``): where the reference augments
    (``aug`` and ``wt == 0``, fitdgp.py:773-779) the labelled frames of every batch are augmented on the device with it;
    None trains on the frames as they are."""
    if data_batcher is None or dgp_cfg is None or frame_lists is None:
        raise NotImplementedError(_PROJECT_READER_MSG % "fit_dgp")
    cfg = SimpleNamespace(**(dict(dgp_cfg) if isinstance(dgp_cfg, dict) else vars(dgp_cfg)))
    cfg.batch_size, cfg.gm2, cfg.gm3, cfg.wt = batch_size, gm2, gm3, wt
    if aug and wt == 0 and verbose and aug_pipeline is None:
        print("note: imgaug augmentation of visible frames (fitdgp.py:773-775) is a host feeder outside this library")
    if variables is None:
        variables = _get(cfg, "init_weights", None) or snapshot
    vis, hid, allf = frame_lists
    return _fit_loop(data_batcher, cfg, variables, vis, hid, allf, maxiters, step, saveiters, displayiters, debug, False, device,
                     batch_ind_all, snapshot_fn, verbose, aug_pipeline if aug and wt == 0 else None)


def fit_dgp_labeledonly(snapshot, dlcpath, shuffle=1, step=1, saveiters=1000, displayiters=5, maxiters=50000, ns=10, nc=2048,
                        n_max_frames=2000, aug=True, trainingsetindex=0, *, data_batcher=None, dgp_cfg=None,
                        frame_lists=None, variables=None, device=None, batch_ind_all=None, snapshot_fn=None, verbose=True,
                        aug_pipeline=None):
    """fitdgp.py:257-546: the same loop on the labelled frames only -- no hidden frames in a batch, and the optimizer follows
    ``total_loss_visible`` (visible cross-entropy + locref Huber), fitdgp.py:406-414.  ``aug_pipeline`` as in ``fit_dgp``
    (used when ``aug``)."""
    if data_batcher is None or dgp_cfg is None or frame_lists is None:
        raise NotImplementedError(_PROJECT_READER_MSG % "fit_dgp_labeledonly")
    cfg = SimpleNamespace(**(dict(dgp_cfg) if isinstance(dgp_cfg, dict) else vars(dgp_cfg)))
    cfg.wt = 0
    cfg.batch_size = int(_get(cfg, "batch_size", 1))
    cfg.gm2, cfg.gm3 = int(_get(cfg, "gm2", 1)) or 1, int(_get(cfg, "gm3", 3))
    if variables is None:
        variables = _get(cfg, "init_weights", None) or snapshot
    vis, hid, allf = frame_lists
    return _fit_loop(data_batcher, cfg, variables, vis, hid, allf, maxiters, step, saveiters, displayiters, "", True, device,
                     batch_ind_all, snapshot_fn, verbose, aug_pipeline if aug else None)
