"""Drop-in for the hot-path part of deepgraphpose.models.eval (reference: src/deepgraphpose/models/eval.py).

``setup_dgp_eval_graph`` :147-214 and ``estimate_pose`` :217-372 keep their names, argument meaning and return
values; the TF graph/session are replaced by the sm_100a engine behind the C ABI.  Video decode (moviepy in the
reference) and the csv/h5 export are outside the path (SURVEY.md 8f): ``estimate_pose`` takes a video path (decoded
with OpenCV when present) or an in-memory uint8 array of frames.
"""
import os

import numpy as np
import torch

from . import synthetic
from .engine import OUTPUT_STRIDES, STRIDE, Engine, check_jpeg_quality, marker_colors, marker_style  # noqa: F401  (marker_colors: eval's public name)
from .mp4 import MJPEGWriter
from .session import Handle, Session


def _cfg_get(cfg, key, default=None):
    if isinstance(cfg, dict):
        return cfg.get(key, default)
    return getattr(cfg, key, default)


def load_variables(dgp_model_file, num_joints, location_refinement, net_type="resnet_50"):
    """Weights for the graph.  Accepts a ``{tf_var_name: ndarray}`` dict, a ``.npz`` of such arrays, or
    ``"synthetic"`` / ``"synthetic:<seed>"`` (random-init weights of ``net_type``, BASELINE.json configs), or the prefix of a
    TensorFlow checkpoint bundle (``snapshot-step2-final--0`` -> ``.index`` + ``.data-0000N-of-0000M``, read by
    tf_checkpoint.py)."""
    if isinstance(dgp_model_file, dict):
        return dgp_model_file
    name = str(dgp_model_file)
    if name.startswith("synthetic"):
        seed = int(name.split(":")[1]) if ":" in name else 0
        return synthetic.make_weights(num_joints, seed=seed, location_refinement=location_refinement, net_type=net_type)
    if name.endswith(".npz") and os.path.exists(name):
        with np.load(name) as z:
            return {k: z[k] for k in z.files}
    prefix = name[:-6] if name.endswith(".index") else name
    if os.path.exists(prefix + ".index"):
        # a TensorFlow checkpoint bundle (DLC / DGP snapshot, resnet_v1_{50,101,152}.ckpt): restorer.restore without TensorFlow
        from . import tf_checkpoint
        return tf_checkpoint.model_variables(tf_checkpoint.read_checkpoint(prefix))
    raise FileNotFoundError("no weights at %r: pass a {tf_var_name: ndarray} dict, an .npz of it, 'synthetic[:seed]', or the "
                            "prefix of a TensorFlow checkpoint (<prefix>.index + <prefix>.data-*)" % (name,))


def check_net_type(net_type, variables):
    """The backbone of ``variables`` (from their slim scope); ValueError if ``net_type`` (a dlc_cfg's, None = follow the
    weights) names another one or is not resnet_50 / resnet_101 / resnet_152."""
    if net_type is not None:
        synthetic.net_scope(net_type)
    found = synthetic.net_type_of(variables)
    if net_type is not None and found != net_type:
        raise ValueError("dlc_cfg net_type is %r but the weights hold %r (%s/...)" % (net_type, found, synthetic.net_scope(found)))
    return found


def check_geometry(cfg):
    """(output_stride, stride) of a dlc_cfg / pose_cfg (pose_cfg.yaml keys ``output_stride``, default 16, ``stride``,
    default 8.0, and ``deconvolutionstride``, default 2; pose_net.py:31-34).  ValueError for an output_stride other than 8 or
    16, a deconvolutionstride other than 2, or output_stride 8 with a stride other than 4.0: DLC cannot have trained such a
    model (its targets and predictions disagree in shape), and reading it out would put every joint at twice its distance."""
    output_stride = _cfg_get(cfg, "output_stride", 16)
    if isinstance(output_stride, bool) or output_stride not in OUTPUT_STRIDES:
        raise ValueError("the B200 path implements output_stride 8 or 16 (pose_net.py:31-34), got %r" % (output_stride,))
    if _cfg_get(cfg, "deconvolutionstride", 2) != 2:
        raise ValueError("the B200 path implements deconvolutionstride=2 (pose_net.py:31-34)")
    stride = float(_cfg_get(cfg, "stride", STRIDE))
    if output_stride == 8 and stride != 4.0:
        raise ValueError("output_stride 8 makes scoremaps of stride 4.0, but the config's stride is %r" % (stride,))
    return int(output_stride), stride


def setup_dgp_eval_graph(dlc_cfg, dgp_model_file, loc_ref=False, gauss_len=1, gamma=1, device=None):
    """eval.py:147-214.  Returns (sess, mu_n, softmax_tensor, scmap, locref, inputs).  ``dlc_cfg.net_type`` (resnet_50,
    resnet_101 or resnet_152) must match the backbone the weights name; without it the weights decide."""
    return _setup_eval_graph(dlc_cfg, dgp_model_file, _cfg_get(dlc_cfg, "net_type"), loc_ref, gauss_len, gamma, device)


def _setup_eval_graph(dlc_cfg, dgp_model_file, net_type, loc_ref=False, gauss_len=1, gamma=1, device=None):
    output_stride, stride = check_geometry(dlc_cfg)
    nj = int(_cfg_get(dlc_cfg, "num_joints"))
    variables = load_variables(dgp_model_file, nj, bool(loc_ref), net_type or "resnet_50")
    check_net_type(net_type, variables)
    eng = Engine(nj, location_refinement=bool(loc_ref), device=device, stride=stride,
                 locref_stdev=float(_cfg_get(dlc_cfg, "locref_stdev", 7.2801)),
                 mean_pixel=tuple(_cfg_get(dlc_cfg, "mean_pixel", (123.68, 116.779, 103.939))),
                 precision=_cfg_get(dlc_cfg, "precision", "fp16"), output_stride=output_stride)
    eng.load_weights(variables)
    handles = {
        "inputs": Handle("Placeholder:0", "inputs"),
        "mu_n": Handle("Sum:0", "mu_n"),
        "softmax_tensor": Handle("truediv:0", "softmax_tensor"),
        "scmap": Handle("pose/part_pred/block4/BiasAdd:0", "scmap"),
        "locref": Handle("pose/locref_pred/block4/BiasAdd:0", "locref") if loc_ref else None,
    }
    sess = Session(eng, handles, gamma=gamma, gauss_len=gauss_len)
    return sess, handles["mu_n"], handles["softmax_tensor"], handles["scmap"], handles["locref"], handles["inputs"]


def _iter_video(video_file):
    import cv2
    cap = cv2.VideoCapture(str(video_file))
    if not cap.isOpened():
        raise IOError("cannot open video %s" % video_file)
    while True:
        ok, frame = cap.read()
        if not ok:
            break
        yield frame[:, :, ::-1]  # BGR -> RGB, as moviepy delivers
    cap.release()


def estimate_pose_frames(engine, frames, batch=16, gamma=1.0, gauss_len=1.0, stride=None, new_size=None, crop_size=None):
    """The estimate_pose frame loop (eval.py:306-357) on in-memory frames: uint8 (T,H,W,3), numpy or CPU tensor.

    Host buffers in, host arrays out; the H2D copy of every batch and the D2H copy of its results happen inside.
    ``new_size`` (height, width) / ``crop_size`` (x0, y0, x1, y1) resize / crop every frame on the device exactly as the
    reference's PIL calls do (eval.py:319-322); the coordinates returned are those of the transformed frames.
    Returns dict(x, y, likelihoods, mu_likelihoods, markers) with the reference's shapes.
    """
    ft = frames if isinstance(frames, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(frames))
    mu, peak, lik = engine.estimate_pose_host(ft, batch=batch, gamma=gamma, gauss_len=gauss_len, new_size=new_size,
                                              crop_size=crop_size)
    stride = engine.stride if stride is None else stride
    markers = mu.numpy().astype(np.float64)
    xr = markers[:, :, 1] * stride + 0.5 * stride
    yr = markers[:, :, 0] * stride + 0.5 * stride
    return {"x": xr, "y": yr, "likelihoods": lik.numpy().astype(np.float64),
            "mu_likelihoods": peak.numpy().astype("int"), "markers": markers}


def _readout_dict(mu, peak, lik, stride):
    markers = mu.numpy().astype(np.float64)
    return {"x": markers[:, :, 1] * stride + 0.5 * stride, "y": markers[:, :, 0] * stride + 0.5 * stride,
            "likelihoods": lik.numpy().astype(np.float64), "mu_likelihoods": peak.numpy().astype("int"), "markers": markers}


def estimate_pose_stream(engine, source, H, W, n_frames=None, batch=16, gamma=1.0, gauss_len=1.0, chunk=65536, new_size=None,
                         crop_size=None):
    """The estimate_pose frame loop (eval.py:306-357) over a frame SOURCE instead of an in-memory array: an iterator of uint8
    (H,W,3) RGB frames (video decoder) or a pinned uint8 tensor (P,H,W,3) cycled for ``n_frames`` frames.  Frames stream
    through a pinned ring of 3 x ``batch`` frames (Engine.estimate_pose_stream): host memory does not grow with the video.
    ``n_frames`` may be None for iterators of unknown length (results are collected ``chunk`` frames at a time).
    ``H``, ``W`` are the source frame size; ``new_size`` / ``crop_size`` transform each frame on the device as in
    ``estimate_pose_frames``."""
    parts = []
    kw = dict(new_size=new_size, crop_size=crop_size)
    if isinstance(source, torch.Tensor):
        if n_frames is None:
            n_frames = source.shape[0]
        parts.append(engine.estimate_pose_stream(source, H, W, n_frames, batch, gamma, gauss_len, **kw))
    else:
        it = iter(source)
        left = None if n_frames is None else int(n_frames)
        while left is None or left > 0:
            want = chunk if left is None else min(chunk, left)
            mu, peak, lik = engine.estimate_pose_stream(it, H, W, want, batch, gamma, gauss_len, **kw)
            parts.append((mu, peak, lik))
            if left is not None:
                left -= mu.shape[0]
            if mu.shape[0] < want:
                break
    mu, peak, lik = (torch.cat([p[i] for p in parts]) for i in range(3))
    return _readout_dict(mu, peak, lik, engine.stride)


def estimate_pose_sharded(engine, source, T, H, W, edges=(), ws=None, ws_max=None, wt_max=0.0, batch=16, gamma=1.0,
                          gauss_len=1.0, group=None, gather=True, timings=None, new_size=None, crop_size=None):
    """estimate_pose over a T-frame video sharded contiguously by frame over the ranks of ``group`` (SURVEY.md 8e; one process
    per GPU): rank r streams frames [a_r, b_r) (``sharding.shard_range``) through its own engine, the ranks exchange the
    soft-argmax of their first frame (one all_gather of nj*8 bytes per rank) so that the temporal potential at every shard
    edge uses the exact neighbour, the skeleton / temporal potentials of the shard are evaluated on the device, and the
    per-frame results are all-gathered back into video order.  The reference has no multi-GPU inference; the per-frame
    arithmetic is that of estimate_pose (eval.py:306-357) and of the clique terms of dgp_loss (fitdgp.py:1063-1083).

    ``source``: a pinned uint8 tensor (P,H,W,3) cycled as the video (frame t = source[t % P]), or a callable
    ``(start, stop) -> iterator of frames`` that opens the rank's own range of a real video.
    Returns the estimate_pose dict plus 'skel' (T,nl), 'temporal' (T,nj; last row 0), 'e_skel', 'e_temp' (T) -- for the
    whole video on every rank when ``gather`` (else for the rank's shard) -- and 'shard' = (a_r, b_r).
    ``timings``: an optional dict that receives the wall-clock seconds of the phases ('stream', 'potentials', 'gather').
    ``H``, ``W`` are the source frame size; ``new_size`` / ``crop_size`` transform each frame on the device as in
    ``estimate_pose_frames``."""
    import time
    import torch.distributed as dist
    from . import sharding
    on = dist.is_available() and dist.is_initialized()
    world = dist.get_world_size(group) if on else 1
    rank = dist.get_rank(group) if on else 0
    if T < world:
        raise ValueError("a %d-frame video cannot be sharded over %d ranks" % (T, world))
    a, b = sharding.shard_range(T, rank, world)
    t_start = time.perf_counter()
    if isinstance(source, torch.Tensor):
        mu, peak, lik = engine.estimate_pose_stream(source, H, W, b - a, batch, gamma, gauss_len, start=a, new_size=new_size,
                                                    crop_size=crop_size)
    else:
        mu, peak, lik = engine.estimate_pose_stream(source(a, b), H, W, b - a, batch, gamma, gauss_len, new_size=new_size,
                                                    crop_size=crop_size)
    if mu.shape[0] != b - a:
        raise RuntimeError("rank %d: the source delivered %d of its %d frames" % (rank, mu.shape[0], b - a))
    dev = engine.device
    t_stream = time.perf_counter()
    mu_d = mu.to(dev, non_blocking=True)
    halo = sharding.exchange_halo(mu_d[0].contiguous(), group) if world > 1 else None
    edges = [tuple(e) for e in edges]
    pot = engine.potentials(mu_d, edges, halo_next=halo, ws=ws, ws_max=ws_max, wt_max=wt_max)
    temporal = pot["temporal"]
    if temporal.shape[0] < b - a:       # the video's last frame has no successor
        temporal = torch.cat([temporal, torch.zeros((1, engine.nj), dtype=temporal.dtype, device=dev)])
    local = {"mu": mu_d, "peak": peak.to(dev, non_blocking=True), "lik": lik.to(dev, non_blocking=True),
             "temporal": temporal, "skel": pot["skel"].t().contiguous(), "e_temp": pot["e_temp"]}
    if pot["e_skel"] is not None:
        local["e_skel"] = pot["e_skel"]
    if timings is not None:
        torch.cuda.synchronize(dev)
    t_pot = time.perf_counter()
    full = {k: (sharding.gather_frames(v, T, group) if gather else v) for k, v in local.items()}
    out = _readout_dict(full["mu"].cpu(), full["peak"].cpu(), full["lik"].cpu(), engine.stride)
    for k in ("temporal", "skel", "e_temp", "e_skel"):
        if k in full:
            out[k] = full[k].cpu().numpy()
    out["shard"] = (a, b)
    if timings is not None:
        timings.update(stream=t_stream - t_start, potentials=t_pot - t_stream, gather=time.perf_counter() - t_pot)
    return out


def _video_source(video_file, new_size=None):
    """(frame iterator, H0, W0, frame count or None, scale_x, scale_y) for a video file: frames are decoded one at a time
    (OpenCV) at their source size and never held beyond the ring; the reference's per-frame resize / crop (eval.py:309-326)
    runs on the device.  The scales map coordinates of the resized frame back to the video (eval.py:312-313)."""
    import cv2
    cap = cv2.VideoCapture(str(video_file))
    if not cap.isOpened():
        raise IOError("cannot open video %s" % video_file)
    w0, h0 = int(cap.get(cv2.CAP_PROP_FRAME_WIDTH)), int(cap.get(cv2.CAP_PROP_FRAME_HEIGHT))
    count = int(cap.get(cv2.CAP_PROP_FRAME_COUNT))
    cap.release()
    scale_x = scale_y = 1.0
    if new_size is not None:
        scale_x, scale_y = w0 / new_size[1], h0 / new_size[0]
    return _iter_video(video_file), h0, w0, (count if count > 0 else None), scale_x, scale_y


def estimate_pose(proj_cfg_file, dgp_model_file, video_file, output_dir, shuffle=1, save_pose=True, save_str="",
                  new_size=None, crop_size=None, batch=16):
    """eval.py:217-372.  ``proj_cfg_file`` may be a dict-like dlc_cfg (num_joints, stride, ...) or a DLC project yaml with
    ``bodyparts``; ``video_file`` a path or a uint8 array (T,H,W,3).  Returns {'x','y','likelihoods'} (T,nj) each.
    A video file is STREAMED: decoded frame by frame (as the reference's ``clip.iter_frames()``, eval.py:306) into a pinned
    ring that the GPU drains batch by batch, so a 100 k-frame clip needs no more host memory than a 100-frame one.
    ``new_size`` (height, width) and ``crop_size`` (x0, y0, x1, y1) resize and crop every frame on the device, bit-exact to
    the reference's ``PIL.Image.resize`` (Pillow's default filter, BICUBIC) and ``crop``.
    The backbone (ResNet-50, -101 or -152) is the one the weights' names describe, as the reference's estimate_pose tries
    each snapshot scope (eval.py:271-276)."""
    dlc_cfg = _load_dlc_cfg(proj_cfg_file)
    save_file = None
    scale_x = scale_y = 1.0
    if isinstance(video_file, (str, os.PathLike)):
        f = os.path.basename(str(video_file)).rsplit(".", 1)
        save_file = os.path.join(str(output_dir), f[0] + "_labeled%s" % save_str)
        if os.path.exists(save_file + ".csv"):
            print("labels already exist! video at %s will not be processed" % video_file)
            return save_file + ".csv"
        source, H0, W0, n_frames, scale_x, scale_y = _video_source(video_file, new_size)
        sess, mu_n, _, scmap, _, inputs = _setup_eval_graph(dlc_cfg, dgp_model_file, None)
        # the container's frame count is a hint only (it can be off by a few frames): read until the decoder runs dry
        res = estimate_pose_stream(sess.engine, source, H0, W0, None, batch=batch, new_size=new_size, crop_size=crop_size)
    else:
        frames = np.asarray(video_file)
        if new_size is not None:
            scale_x, scale_y = frames.shape[2] / new_size[1], frames.shape[1] / new_size[0]
        sess, mu_n, _, scmap, _, inputs = _setup_eval_graph(dlc_cfg, dgp_model_file, None)
        res = estimate_pose_frames(sess.engine, frames, batch=batch, new_size=new_size, crop_size=crop_size)
    sess.close()
    labels = {"x": res["x"] * scale_x, "y": res["y"] * scale_y, "likelihoods": res["likelihoods"]}
    if save_pose and save_file is not None:
        _save_labels(labels, dlc_cfg, dgp_model_file, save_file)
    return labels


def _load_dlc_cfg(proj_cfg_file):
    """A dict-like dlc_cfg as given, or the one of a DLC project yaml (its bodyparts)."""
    if isinstance(proj_cfg_file, (dict,)) or hasattr(proj_cfg_file, "num_joints"):
        return proj_cfg_file
    import yaml
    with open(proj_cfg_file, "r") as stream:
        proj = yaml.safe_load(stream)
    return {"num_joints": len(proj["bodyparts"]), "all_joints_names": list(proj["bodyparts"]), "stride": 8.0,
            "skeleton": proj.get("skeleton") or []}


def skeleton_from_cfg(dlc_cfg):
    """The (n, 2) joint index pairs of a dlc_cfg's ``skeleton``: pairs of bodypart names (a DLC project's config.yaml,
    mapped through ``all_joints_names``, its ``bodyparts``) or of joint indices.  ValueError for no skeleton, an unknown
    name or a malformed pair."""
    skel = _cfg_get(dlc_cfg, "skeleton") if dlc_cfg is not None else None
    if not skel:
        raise ValueError("draw_skeleton needs a 'skeleton' in the project config (pairs of bodypart names)")
    names = list(_cfg_get(dlc_cfg, "all_joints_names") or [])
    edges = []
    for pair in skel:
        if isinstance(pair, (str, bytes)) or len(pair) != 2:
            raise ValueError("skeleton entries must be pairs, got %r" % (pair,))
        e = []
        for v in pair:
            if isinstance(v, str):
                if v not in names:
                    raise ValueError("skeleton bodypart %r is not one of the bodyparts %s" % (v, names))
                e.append(names.index(v))
            elif isinstance(v, (int, np.integer)) and not isinstance(v, bool):
                e.append(int(v))
            else:
                raise ValueError("skeleton entries must be bodypart names or joint indices, got %r" % (pair,))
        edges.append(e)
    return np.asarray(edges, dtype=np.int64).reshape(-1, 2)


def _save_labels(labels, dlc_cfg, dgp_model_file, save_file):
    os.makedirs(os.path.dirname(save_file) or ".", exist_ok=True)
    names = _cfg_get(dlc_cfg, "all_joints_names", ["joint%d" % i for i in range(labels["x"].shape[1])])
    scorer = os.path.basename(str(dgp_model_file)) if isinstance(dgp_model_file, (str, os.PathLike)) else "dgp_b200"
    export_pose_like_dlc(labels, scorer, list(names), save_file)


def export_pose_like_dlc(labels, scorer, joints_names, save_file):
    """eval.py:621-645: the DeepLabCut table layout -- columns (scorer, bodypart, x | y | likelihood), one row per frame --
    written as ``save_file + '.csv'`` (three header rows + frame index column, what DLC / ``plot_dgp`` /
    ``load_pose_from_dlc_to_dict`` read) and, when pytables is installed, as ``save_file + '.h5'`` (key df_with_missing)."""
    import pandas as pd
    x = np.asarray(labels["x"])
    table = np.empty((x.shape[0], 3 * x.shape[1]), dtype=x.dtype)
    table[:, 0::3], table[:, 1::3], table[:, 2::3] = x, labels["y"], labels["likelihoods"]
    columns = pd.MultiIndex.from_product([[scorer], list(joints_names), ["x", "y", "likelihood"]],
                                         names=["scorer", "bodyparts", "coords"])
    frame = pd.DataFrame(table, columns=columns, index=np.arange(x.shape[0]))
    try:
        frame.to_hdf(save_file + ".h5", key="df_with_missing", format="table", mode="w")
    except ImportError:   # pytables is optional here; the csv carries the same table
        pass
    frame.to_csv(save_file + ".csv")


def load_pose_from_dlc_to_dict(filename):
    """eval.py:648-653: read a DLC csv back into {'x', 'y', 'likelihoods'} (T, nj) arrays."""
    body = np.genfromtxt(filename, delimiter=",", skip_header=3)[:, 1:]   # missing values (empty cells) become NaN
    return {"x": body[:, 0::3], "y": body[:, 1::3], "likelihoods": body[:, 2::3]}


def _video_writer(filename, fourcc, fps, H, W):
    import cv2
    os.makedirs(os.path.dirname(str(filename)) or ".", exist_ok=True)
    vw = cv2.VideoWriter(str(filename), cv2.VideoWriter_fourcc(*fourcc), float(fps), (int(W), int(H)))
    if not vw.isOpened():
        raise IOError("cannot open a %r video writer for %s" % (fourcc, filename))
    return vw


def _write_rgb(vw, frames):
    for fr in frames:
        vw.write(np.ascontiguousarray(fr[:, :, ::-1]))  # RGB -> BGR, what OpenCV encodes


def _check_fourcc(fourcc):
    if not isinstance(fourcc, str) or len(fourcc) != 4:
        raise ValueError("fourcc must be a four-character code such as 'mp4v' or 'FFV1', got %r" % (fourcc,))


def _check_encoder(encoder, fourcc, quality):
    """'cv2' (cv2.VideoWriter with ``fourcc``) or 'jpeg' (Motion-JPEG encoded on the device at ``quality``)."""
    if encoder == "cv2":
        _check_fourcc(fourcc)
    elif encoder == "jpeg":
        check_jpeg_quality(quality)
    else:
        raise ValueError("encoder must be 'cv2' or 'jpeg', got %r" % (encoder,))


def _mjpeg_writer(filename, fps, H, W):
    os.makedirs(os.path.dirname(str(filename)) or ".", exist_ok=True)
    return MJPEGWriter(str(filename), fps, W, H)


def create_annotated_movie(clip, df_x, df_y, mask_array=None, dotsize=3, colormap="cool", filename="movie.mp4", fps=None,
                           fourcc="mp4v", batch=16, engine=None, encoder="cv2", quality=90, skeleton=None,
                           skeleton_color=(0, 0, 0), trailpoints=0):
    """plot_dgp's renderer (src/deepgraphpose/models/eval.py): a video of ``clip`` with joint j of frame t marked by a disc
    of radius ``dotsize`` at (``df_x[t, j]``, ``df_y[t, j]``) (video pixels) where ``mask_array[t, j]`` (None: every joint),
    coloured by ``colormap`` (the name 'cool' or an (nj, 3) uint8 RGB table) -- the drawing contract of dgp_draw_markers.
    ``clip``: a video path (decoded with OpenCV) or a uint8 (T,H,W,3) RGB array.  Frames are drawn on the device in batches
    of ``batch`` (``engine``: an Engine with nj joints, else one is created for the call) and written with
    ``cv2.VideoWriter(filename, fourcc, fps)``; ``fps`` None = the video's own rate (required for an array).  Every frame
    the decoder yields is written, one label row per frame.  The reference writes ``int(duration * fps)`` frames with
    moviepy (libx264) and draws with matplotlib / skimage on the host; bitstream and anti-aliasing parity are not goals.
    ``encoder="jpeg"`` encodes the drawn frames on the device instead (Engine.encode_jpeg at ``quality``) and writes them
    to ``filename`` as Motion-JPEG (deepgraphpose_b200.mp4); ``fourcc`` is then unused.
    ``skeleton`` (joint index pairs) joins the joints of each pair by a line in ``skeleton_color`` (RGB) where both are
    marked; ``trailpoints`` K >= 2 also marks each joint in the K - 1 previous frames, counted from the first label row."""
    x = np.asarray(df_x, dtype=np.float64)
    y = np.asarray(df_y, dtype=np.float64)
    if x.ndim != 2 or y.shape != x.shape:
        raise ValueError("df_x and df_y must be (T, nj) arrays of one shape")
    nj = x.shape[1]
    mask = np.ones(x.shape, np.float64) if mask_array is None else np.asarray(mask_array, dtype=bool).astype(np.float64)
    if mask.shape != x.shape:
        raise ValueError("mask_array must be (T, nj) like df_x")
    # validates the style before any decode or device work
    marker_style(nj, dotsize, 0.5, colormap, edges=skeleton, skeleton_color=skeleton_color, trailpoints=trailpoints)
    trail = max(int(trailpoints) - 1, 0)
    _check_encoder(encoder, fourcc, quality)
    if isinstance(clip, (str, os.PathLike)):
        if fps is None:
            import cv2
            cap = cv2.VideoCapture(str(clip))
            fps = cap.get(cv2.CAP_PROP_FPS)
            cap.release()
        frames_iter = _iter_video(clip)
    else:
        arr = np.asarray(clip)
        if arr.dtype != np.uint8 or arr.ndim != 4 or arr.shape[-1] != 3:
            raise ValueError("clip must be a video path or a uint8 (T,H,W,3) array")
        if fps is None:
            raise ValueError("fps is required when clip is an array")
        frames_iter = iter(arr)
    own = engine is None
    eng = Engine(nj) if own else engine
    vw = None
    try:
        t0 = 0
        while True:
            chunk = []
            for fr in frames_iter:
                chunk.append(fr)
                if len(chunk) == batch:
                    break
            if not chunk:
                break
            n = len(chunk)
            if t0 + n > x.shape[0]:
                raise ValueError("the clip has more frames than the %d label rows" % x.shape[0])
            host = torch.from_numpy(np.ascontiguousarray(np.stack(chunk)))
            if vw is None:
                vw = (_mjpeg_writer(filename, fps, host.shape[1], host.shape[2]) if encoder == "jpeg"
                      else _video_writer(filename, fourcc, fps, host.shape[1], host.shape[2]))
            dev = host.to(eng.device)
            hist = min(trail, t0)   # the previous batches' last rows, for the trails
            eng.draw_markers(dev, x[t0 - hist:t0 + n], y[t0 - hist:t0 + n], mask[t0 - hist:t0 + n], dotsize, 0.5, colormap,
                             skeleton, skeleton_color, trailpoints, hist)
            if encoder == "jpeg":
                for packet in eng.encode_jpeg(dev, quality):
                    vw.write(packet)
            else:
                _write_rgb(vw, dev.cpu().numpy())
            t0 += n
    finally:
        if vw is not None:
            vw.close() if encoder == "jpeg" else vw.release()
        if own:
            eng.close()
    return filename


def plot_dgp(video_file, output_dir="", label_dir=None, proj_cfg_file=None, dgp_model_file=None, shuffle=1, dotsize=3,
             colormap="cool", save_str="", mask_threshold=0.1, new_size=None, crop_size=None, batch=16, fourcc="mp4v",
             encoder="cv2", quality=90, draw_skeleton=False, skeleton_color=(0, 0, 0), trailpoints=0):
    """plot_dgp (src/deepgraphpose/models/eval.py; step 3 of the reference demo): labels a video and renders the labelled
    movie ``<output_dir>/<video>_labeled<save_str>.mp4`` (cv2.VideoWriter with ``fourcc`` at the source fps) in which joint j
    is a disc of radius ``dotsize`` in ``colormap``'s colour j wherever its likelihood exceeds ``mask_threshold``.

    * An existing movie is left alone (nothing is computed).
    * No label csv ``<label_dir>/<video>_labeled<save_str>.csv`` (label_dir None = output_dir): ONE streamed pass
      (Engine.estimate_pose_render_stream) decodes the video once, estimates the pose as ``estimate_pose`` does (same csv)
      and draws the markers into the source frames on the device before they are written.
    * With the csv: the labels are read with ``load_pose_from_dlc_to_dict`` and drawn by ``create_annotated_movie``.

    ``proj_cfg_file`` / ``dgp_model_file`` / ``new_size`` / ``crop_size`` / ``batch`` as in estimate_pose; ``shuffle`` is
    accepted for the reference's signature.  ``fourcc='FFV1'`` writes lossless video (used by the tests).  Every frame the
    decoder yields is written; the reference writes ``int(duration * fps)`` frames with moviepy.  The defaults are the
    reference's as recorded in this project (dotsize 3, 'cool', mask_threshold 0.1); they have not been checked against a
    reference checkout.  Returns the movie's path.
    ``encoder="jpeg"`` writes the same path as Motion-JPEG at ``quality`` (Pillow's JPEG quality), encoded on the device
    in both branches, so that only the encoded bytes reach the host; the csv is the same.
    ``draw_skeleton`` joins the joints of each ``skeleton`` edge of the project config (pairs of bodypart names, or of
    joint indices in a dict-like dlc_cfg) by a line in ``skeleton_color`` (RGB); ``trailpoints`` K >= 2 also marks each
    joint in the K - 1 previous frames.  Both branches draw the same frames."""
    if not isinstance(video_file, (str, os.PathLike)):
        raise ValueError("video_file must be a path")
    _check_encoder(encoder, fourcc, quality)
    name = os.path.basename(str(video_file)).rsplit(".", 1)[0] + "_labeled%s" % save_str
    label_dir = output_dir if label_dir is None else label_dir
    movie = os.path.join(str(output_dir), name + ".mp4")
    csv = os.path.join(str(label_dir), name + ".csv")
    if os.path.exists(movie):
        print("labeled video already exists: %s" % movie)
        return movie
    dlc_cfg = _load_dlc_cfg(proj_cfg_file) if proj_cfg_file is not None else None
    skeleton = skeleton_from_cfg(dlc_cfg) if draw_skeleton else None
    overlay = {"skeleton_color": skeleton_color, "trailpoints": trailpoints}
    if os.path.exists(csv):
        labels = load_pose_from_dlc_to_dict(csv)
        marker_style(labels["x"].shape[1], dotsize, mask_threshold, colormap, edges=skeleton, **overlay)
        return create_annotated_movie(video_file, labels["x"], labels["y"], labels["likelihoods"] > mask_threshold,
                                      dotsize=dotsize, colormap=colormap, filename=movie, fourcc=fourcc, batch=batch,
                                      encoder=encoder, quality=quality, skeleton=skeleton, **overlay)
    if dlc_cfg is None:
        raise ValueError("no labels at %s: proj_cfg_file and dgp_model_file are needed to estimate them" % csv)
    marker_style(int(_cfg_get(dlc_cfg, "num_joints")), dotsize, mask_threshold, colormap, edges=skeleton, **overlay)
    import cv2
    cap = cv2.VideoCapture(str(video_file))
    fps = cap.get(cv2.CAP_PROP_FPS)
    cap.release()
    source, H0, W0, count, scale_x, scale_y = _video_source(video_file, new_size)
    sess = _setup_eval_graph(dlc_cfg, dgp_model_file, None)[0]
    eng = sess.engine
    if encoder == "jpeg":
        vw = _mjpeg_writer(movie, fps, H0, W0)
        write, close = vw.write_packed, vw.close
    else:
        vw = _video_writer(movie, fourcc, fps, H0, W0)
        write, close = (lambda fr: _write_rgb(vw, fr)), vw.release
    # one call covers the whole video unless the container under-reports its frame count by more than the margin; trails
    # restart at a call boundary
    parts, chunk = [], max(65536, (count or 0) + 4096)
    try:
        it = iter(source)
        while True:
            mu, peak, lik = eng.estimate_pose_render_stream(it, H0, W0, chunk, write, dotsize, mask_threshold, colormap,
                                                            new_size, crop_size, batch,
                                                            encoder="raw" if encoder == "cv2" else "jpeg", quality=quality,
                                                            edges=skeleton, **overlay)
            parts.append((mu, peak, lik))
            if mu.shape[0] < chunk:
                break
    finally:
        close()
        sess.close()
    res = _readout_dict(*(torch.cat([p[i] for p in parts]) for i in range(3)), eng.stride)
    labels = {"x": res["x"] * scale_x, "y": res["y"] * scale_y, "likelihoods": res["likelihoods"]}
    _save_labels(labels, dlc_cfg, dgp_model_file, os.path.join(str(label_dir), name))
    return movie


def evaluate_dgp_frames(engine, frames, loc_ref=True, loc_ref_calc="dlc", batch=16, gamma=1.0, gauss_len=1.0):
    """The per-image pose read-out of ``evaluate_dgp`` (eval.py:744-790) for a uint8 (T,H,W,3) array: returns (T, nj*3)
    rows of (x, y, likelihood) like ``PredicteData``.  Branches as in the reference: loc_ref with ``loc_ref_calc='dlc'`` ->
    argmax_pose_predict (global peak + locref offset, likelihood = sigmoid at the peak); ``'dgp'`` -> soft-argmax + softmax
    weighted locref offset (likelihood column 1); no loc_ref -> soft-argmax only."""
    frames = np.asarray(frames)
    T = frames.shape[0]
    out = np.empty((T, engine.nj * 3), np.float64)
    for t0 in range(0, T, batch):
        fr = torch.from_numpy(np.ascontiguousarray(frames[t0:t0 + batch])).to(engine.device)
        logits, locref = engine.forward(fr, want_locref=bool(loc_ref))
        if loc_ref and loc_ref_calc.lower() == "dlc":
            pose = engine.softargmax(logits, locref, gamma, gauss_len, want=("dlc_pose",))["dlc_pose"]
        elif loc_ref:
            pose = engine.soft_pose(logits, locref, gamma, gauss_len)
        else:
            mu = engine.softargmax(logits, None, gamma, gauss_len, want=("mu",))["mu"]
            pose = torch.cat([mu.flip(2) * engine.stride + 0.5 * engine.stride, torch.ones_like(mu[:, :, :1])], dim=2)
        out[t0:t0 + fr.shape[0]] = pose.reshape(fr.shape[0], -1).double().cpu().numpy()
    return out


def pairwisedistances(DataCombined, scorer1, scorer2, pcutoff=-1, bodyparts=None):
    """DeepLabCut's evaluate.pairwisedistances (called at eval.py:803-804) on the (scorer, bodypart, coord) column index:
    per frame and bodypart the Euclidean distance between the two scorers' (x, y), and the same masked to predictions of
    ``scorer2`` with likelihood >= pcutoff.  Returns (RMSE, RMSEpcutoff) DataFrames."""
    import pandas as pd
    mask = DataCombined[scorer2].xs("likelihood", level=1, axis=1) >= pcutoff
    if bodyparts is None:
        pointwise = (DataCombined[scorer1] - DataCombined[scorer2]) ** 2
    else:
        pointwise = (DataCombined[scorer1][bodyparts] - DataCombined[scorer2][bodyparts]) ** 2
        mask = mask[bodyparts]
    rmse = np.sqrt(pointwise.xs("x", level=1, axis=1) + pointwise.xs("y", level=1, axis=1))
    return rmse, rmse[mask]


def _read_collected_data(project_path, trainingset_folder, scorer):
    """Human labels of a DLC project: ``CollectedData_<scorer>.h5`` (key df_with_missing) as the reference reads it
    (eval.py:724-725), or the ``.csv`` DLC writes next to it when pytables is not installed."""
    import pandas as pd
    base = os.path.join(project_path, trainingset_folder, "CollectedData_" + scorer)
    try:
        return pd.read_hdf(base + ".h5", "df_with_missing")
    except (ImportError, FileNotFoundError, OSError):
        return pd.read_csv(base + ".csv", header=[0, 1, 2], index_col=0)


def evaluate_dgp(proj_cfg_file, dgp_model_file, shuffle=1, loc_ref=None, loc_ref_calc="dlc", *, dlc_cfg=None, batch=8,
                 device=None):
    """eval.py:656-813: RMSE per labelled frame / joint of a DLC project, train and test errors printed, the RMSE DataFrame
    returned.  ``proj_cfg_file`` is the project's config.yaml; the training-set folder, the train / test split
    (Documentation_data-*.pickle) and the pose config follow DeepLabCut's layout (auxiliaryfunctions.GetTrainingSetFolder /
    GetDataandMetaDataFilenames / LoadMetadata, restated here because deeplabcut is not a dependency).  ``dlc_cfg`` may supply
    the pose config (num_joints, all_joints_names, stride, location_refinement, locref_stdev) instead of the project's
    train/pose_cfg.yaml.  Frames are read with PIL and evaluated in batches of equal size through ``evaluate_dgp_frames``."""
    import pickle
    import pandas as pd
    import yaml
    from PIL import Image
    with open(proj_cfg_file, "r") as stream:
        proj_config = yaml.safe_load(stream)
    project_path = proj_config.get("project_path") or os.path.dirname(os.path.abspath(str(proj_cfg_file)))
    task, date = proj_config["Task"], proj_config["date"]
    iteration = proj_config.get("iteration", 0)
    trainingset_folder = os.path.join("training-datasets", "iteration-" + str(iteration), "UnaugmentedDataSet_" + task + date)
    train_fraction = proj_config["TrainingFraction"][0]
    if dlc_cfg is None:
        model_folder = os.path.join("dlc-models", "iteration-" + str(iteration),
                                    task + date + "-trainset" + str(int(train_fraction * 100)) + "shuffle" + str(shuffle))
        with open(os.path.join(project_path, model_folder, "train", "pose_cfg.yaml"), "r") as stream:
            dlc_cfg = yaml.safe_load(stream)
    dlc_cfg = dict(dlc_cfg) if isinstance(dlc_cfg, dict) else dict(vars(dlc_cfg))
    loc_ref = bool(dlc_cfg.get("location_refinement", True)) if loc_ref is None else bool(loc_ref)
    dlc_cfg["location_refinement"] = loc_ref
    dlc_cfg.setdefault("stride", 8.0)
    sess, mu_n, softmax_tensor, scmap_tf, locref_tf, inputs = setup_dgp_eval_graph(dlc_cfg, dgp_model_file, loc_ref=loc_ref,
                                                                                   device=device)
    Data = _read_collected_data(project_path, trainingset_folder, proj_config["scorer"])
    comparisonbodyparts = list(proj_config["bodyparts"])
    meta = os.path.join(project_path, trainingset_folder,
                        "Documentation_data-" + task + "_" + str(int(train_fraction * 100)) + "shuffle" + str(shuffle) + ".pickle")
    with open(meta, "rb") as f:
        _, trainIndices, testIndices, _ = pickle.load(f)
    names = dlc_cfg.get("all_joints_names") or comparisonbodyparts
    nj = len(names)
    PredicteData = np.ones((len(Data.index), 3 * nj))
    print("Analyzing data...")
    # images of one size go through the engine together (the reference runs them one by one, eval.py:741-742)
    by_shape = {}
    for imageindex, imagename in enumerate(Data.index):
        name = imagename if isinstance(imagename, str) else os.path.join(*imagename)
        image = np.asarray(Image.open(os.path.join(project_path, name)).convert("RGB"))
        by_shape.setdefault(image.shape, []).append((imageindex, image))
    for shape, items in by_shape.items():
        frames = np.stack([im for _, im in items])
        pose = evaluate_dgp_frames(sess.engine, frames, loc_ref, loc_ref_calc, batch=batch)
        for (imageindex, _), row in zip(items, pose):
            PredicteData[imageindex, :] = row
    sess.close()
    DLCscorer = "DGP"
    index = pd.MultiIndex.from_product([[DLCscorer], list(names), ["x", "y", "likelihood"]], names=["scorer", "bodyparts", "coords"])
    DataMachine = pd.DataFrame(PredicteData, columns=index, index=Data.index.values)
    DataCombined = pd.concat([Data.T, DataMachine.T], axis=0).T
    RMSE, _ = pairwisedistances(DataCombined, proj_config["scorer"], DLCscorer, proj_config.get("pcutoff", 0.1), comparisonbodyparts)
    testerror = np.nanmean(RMSE.iloc[testIndices].values.flatten())
    trainerror = np.nanmean(RMSE.iloc[trainIndices].values.flatten())
    print("Train error:", np.round(trainerror, 2), " pixels")
    print("Test error:", np.round(testerror, 2), " pixels")
    return RMSE
