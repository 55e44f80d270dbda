"""Thin host-side wrapper of the C ABI: PyTorch supplies device memory and streams, nothing else.

``Engine`` is the object behind the reference-shaped shims (``pose_net.PoseNet``, ``fitdgp_util.argmax_2d_from_cm``,
``eval.setup_dgp_eval_graph`` / ``estimate_pose``).  Every method ends in a call into libdgp_b200.so.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import DgpConfig, DgpError, check

MEAN_PIXEL = (123.68, 116.779, 103.939)  # PTF/default_config.py:23
STRIDE = 8.0                             # PTF/default_config.py:18
LOCREF_STDEV = 7.2801                    # PTF/default_config.py:29


OUTPUT_STRIDES = (8, 16)                 # slim resnet_v1 output_stride values of the B200 path (pose_net.py:31-34)


def check_output_stride(output_stride):
    """``output_stride`` as an int in OUTPUT_STRIDES; ValueError otherwise."""
    if isinstance(output_stride, bool) or not isinstance(output_stride, (int, np.integer, float)) \
            or output_stride not in OUTPUT_STRIDES:
        raise ValueError("output_stride must be 8 or 16, got %r" % (output_stride,))
    return int(output_stride)


def output_dims(H, W, output_stride=16):
    """(h_feat, w_feat), (h_out, w_out) -- closed form of Dataset._compute_pred_dims (dataset.py:348-371) for a backbone at
    ``output_stride`` 8 or 16."""
    lib = _lib.load()
    a, b, c, d = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    check(lib.dgp_output_dims_os(int(H), int(W), check_output_stride(output_stride), C.byref(a), C.byref(b), C.byref(c),
                                 C.byref(d)))
    return (a.value, b.value), (c.value, d.value)


def frame_transform(new_size=None, crop_size=None):
    """The dgp_frame_transform of estimate_pose's options, or None for neither: ``new_size`` = (height, width) of
    PIL's ``resize(size=(new_size[1], new_size[0]))`` (eval.py:319), ``crop_size`` = the PIL box (x0, y0, x1, y1) of
    ``crop(crop_size)`` taken on the resized frame (eval.py:322)."""
    if new_size is None and crop_size is None:
        return None
    t = _lib.DgpFrameTransform()
    if new_size is not None:
        t.resize_h, t.resize_w = int(new_size[0]), int(new_size[1])
        if t.resize_h < 1 or t.resize_w < 1:
            raise ValueError("new_size must be two positive sizes (height, width), got %r" % (tuple(new_size),))
    if crop_size is not None:
        x0, y0, x1, y1 = (int(v) for v in crop_size)
        if x1 <= x0 or y1 <= y0:
            raise ValueError("crop_size must be a box (x0, y0, x1, y1) with x1 > x0 and y1 > y0, got %r" % (tuple(crop_size),))
        t.crop_x0, t.crop_y0, t.crop_x1, t.crop_y1 = x0, y0, x1, y1
    return t


def transform_dims(H0, W0, new_size=None, crop_size=None):
    """(H, W) of an H0 x W0 frame after estimate_pose's resize / crop (dgp_transform_dims); ValueError if invalid."""
    lib = _lib.load()
    t = frame_transform(new_size, crop_size)
    H, W = C.c_int(), C.c_int()
    if lib.dgp_transform_dims(int(H0), int(W0), C.byref(t) if t is not None else None, C.byref(H), C.byref(W)) != 0:
        raise ValueError("invalid frame size %dx%d or transform new_size=%r crop_size=%r" % (H0, W0, new_size, crop_size))
    return H.value, W.value


MAX_DOTSIZE = 64  # kMaxDotsize of csrc/handle.cuh
MAX_EDGES = 256  # kMaxEdges
MAX_TRAILPOINTS = 64  # kMaxTrailpoints


def marker_colors(nj, colormap="cool"):
    """The (nj, 3) uint8 RGB marker colours of plot_dgp's default colormap, sampled as matplotlib's
    ``ScalarMappable(cmap='cool').to_rgba(linspace(0, 1, nj))`` does: idx_j = min(255, floor(256 j / (nj - 1))) (0 when
    nj == 1), colour (idx_j, 255 - idx_j, 255).  'cool' is the only colormap name; anything else is a ValueError."""
    if not isinstance(colormap, str) or colormap != "cool":
        raise ValueError("unknown colormap %r: 'cool' is the only named colormap (or pass an (nj, 3) uint8 table)" % (colormap,))
    nj = int(nj)
    if nj < 1:
        raise ValueError("nj must be positive")
    j = np.arange(nj, dtype=np.int64)
    idx = np.zeros(nj, np.int64) if nj == 1 else np.minimum(255, (256 * j) // (nj - 1))
    return np.stack([idx, 255 - idx, np.full(nj, 255)], axis=1).astype(np.uint8)


def _check_int(name, value, lo, hi):
    if isinstance(value, bool) or not isinstance(value, (int, np.integer)) or not lo <= int(value) <= hi:
        raise ValueError("%s must be an integer in [%d, %d], got %r" % (name, lo, hi, value))
    return int(value)


def skeleton_edges(nj, edges):
    """``edges`` (pairs of joint indices, or None) as a contiguous int32 (n, 2) table; ValueError for more than 256 pairs,
    a shape other than (n, 2) or an index outside [0, nj)."""
    if edges is None:
        return np.zeros((0, 2), np.int32)
    arr = np.asarray(edges)
    if arr.size == 0:
        return np.zeros((0, 2), np.int32)
    if arr.ndim != 2 or arr.shape[1] != 2 or not np.issubdtype(arr.dtype, np.integer):
        raise ValueError("edges must be (n, 2) pairs of joint indices, got %s %s" % (arr.dtype, arr.shape))
    if arr.shape[0] > MAX_EDGES:
        raise ValueError("at most %d skeleton edges, got %d" % (MAX_EDGES, arr.shape[0]))
    if arr.min() < 0 or arr.max() >= int(nj):
        raise ValueError("skeleton edge joints must lie in [0, %d), got %s" % (nj, arr.tolist()))
    return np.ascontiguousarray(arr, dtype=np.int32)


def marker_style(nj, dotsize=3, mask_threshold=0.1, colors=None, scale_x=1.0, scale_y=1.0, edges=None,
                 skeleton_color=(0, 0, 0), trailpoints=0, history=0):
    """(dgp_marker_style, tables) of a drawing call; the tables must stay alive while the style is in use.  ``colors``:
    None (the 'cool' table), a colormap name, or an (nj, 3) table of values in [0, 255].  ``edges``: joint index pairs
    joined by a line in ``skeleton_color`` (an RGB triple); ``trailpoints`` K >= 2 also paints each joint's discs of the
    K - 1 previous frames; ``history``: rows before the first frame in the coordinate tables (dgp_draw_markers), at most
    K - 1.  ValueError for a dotsize outside [0, 64], a table of another shape, a bad edge, K outside [0, 64] or a bad
    history."""
    _check_int("dotsize", dotsize, 0, MAX_DOTSIZE)
    if colors is None or isinstance(colors, str):
        table = marker_colors(nj, "cool" if colors is None else colors)
    else:
        arr = np.asarray(colors)
        if arr.shape != (int(nj), 3) or not (np.issubdtype(arr.dtype, np.integer) and arr.min() >= 0 and arr.max() <= 255):
            raise ValueError("colors must be an (%d, 3) table of RGB values in [0, 255], got %s %s" % (nj, arr.dtype, arr.shape))
        table = np.ascontiguousarray(arr, dtype=np.uint8)
    edge_table = skeleton_edges(nj, edges)
    sk = np.asarray(skeleton_color)
    if sk.shape != (3,) or not (np.issubdtype(sk.dtype, np.integer) and sk.min() >= 0 and sk.max() <= 255):
        raise ValueError("skeleton_color must be an RGB triple of integers in [0, 255], got %r" % (skeleton_color,))
    K = _check_int("trailpoints", trailpoints, 0, MAX_TRAILPOINTS)
    hist = _check_int("history", history, 0, max(K - 1, 0))
    st = _lib.DgpMarkerStyle(int(dotsize), float(mask_threshold), float(scale_x), float(scale_y), table.ctypes.data,
                             edge_table.ctypes.data if len(edge_table) else None, len(edge_table),
                             (C.c_uint8 * 3)(*(int(v) for v in sk)), K, hist)
    return st, (table, edge_table)


def check_jpeg_quality(quality):
    """``quality`` as an int in 1..100 (Pillow's JPEG quality); ValueError otherwise."""
    if isinstance(quality, bool) or not isinstance(quality, (int, np.integer)) or not 1 <= int(quality) <= 100:
        raise ValueError("quality must be an integer in [1, 100], got %r" % (quality,))
    return int(quality)


def jpeg_capacity(H, W):
    """Bytes one (H, W) frame's JPEG file can take at most (dgp_jpeg_capacity); ValueError outside 1..16383."""
    cap = _lib.load().dgp_jpeg_capacity(int(H), int(W))
    if cap < 0:
        raise ValueError("JPEG frames must be 1..16383 pixels on each side, got %dx%d" % (H, W))
    return int(cap)


def suggest_batch(H, W, lo=24, hi=48, num_sms=148, units=(3, 4, 6, 3), output_stride=16):
    """Frames per batch that minimise wave quantisation of the persistent conv-GEMM grid (one CTA per SM).

    Every GEMM layer runs ceil(B*pixels/tile_rows) * n_blocks tiles on `num_sms` CTAs; a batch size for which the
    dominant layers' tile counts are (just under) a multiple of the SM count avoids a nearly empty last wave.  Layers are
    weighted by their roofline bound (max of bf16 tensor time and HBM time), tile shapes follow csrc/capi.cu.  ``units``: the
    bottleneck units per block of the backbone (ResNet-50 by default; synthetic.BLOCK_UNITS for the others).  At
    ``output_stride`` 8 block 2 keeps its resolution (stride as executed: (2, 1, 1, 1))."""
    c2 = lambda v: -(-v // 2)
    layers = []  # (pixels per frame, tile rows, n_blocks, weight)
    hh, ww = c2(H), c2(W)
    def add(px, cin_k, cout, bytes_per_px):
        bn = min(cout, 256)
        rows = 256 if bn <= 128 else 128
        wgt = max(2.0 * px * cin_k * cout / 1414e12, px * bytes_per_px / 6464e9)
        layers.append((px, rows, -(-cout // bn), wgt))
    add(hh * ww, 256, 64, 32 + 128)
    hh, ww = c2(hh), c2(ww)
    cin = 64
    strides = (2, 2, 1, 1) if check_output_stride(output_stride) == 16 else (2, 1, 1, 1)
    for base, n_units, bstride in zip((64, 128, 256, 512), units, strides):
        for u in range(n_units):
            s_ = bstride if u == n_units - 1 else 1
            depth = 4 * base
            ho, wo = (c2(hh), c2(ww)) if s_ == 2 else (hh, ww)
            if cin != depth:
                add(hh * ww, cin, depth, 2 * (cin + depth))
            add(hh * ww, cin, base, 2 * (cin + base))
            add(ho * wo, 9 * base, base, 4 * base)
            add(ho * wo, base, depth, 2 * (base + 2 * depth))
            hh, ww, cin = ho, wo, depth
    best, best_b = None, lo
    for B in range(lo, hi + 1):
        t = 0.0
        for px, rows, nb, wgt in layers:
            tiles = -(-(px * B) // rows) * nb
            waves = -(-tiles // num_sms)
            t += wgt * waves * num_sms / tiles
        t /= B ** 0.0  # weights are per frame already
        if best is None or t < best - 1e-12:
            best, best_b = t, B
    return best_b


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class _Raw:
    """__cuda_array_interface__ carrier for memory owned by the handle."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"data": (int(ptr), False), "shape": tuple(shape), "typestr": typestr, "version": 2}


def _device_view(ptr, shape, typestr, device):
    with torch.cuda.device(device):
        return torch.as_tensor(_Raw(ptr, shape, typestr), device=device)


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class Engine:
    def __init__(self, num_joints, location_refinement=True, device=None, stride=None, locref_stdev=LOCREF_STDEV,
                 mean_pixel=MEAN_PIXEL, precision="fp16", output_stride=16):
        """``output_stride``: slim's output_stride of the backbone, 8 or 16 (pose_cfg.yaml ``output_stride``).  At 8 the
        scoremaps have twice the resolution on each axis.  ``stride``: input pixels per scoremap pixel (pose_cfg.yaml
        ``stride``); None = output_stride / 2, the value DLC's configs pair with it (8.0 at 16, 4.0 at 8)."""
        output_stride = check_output_stride(output_stride)
        if stride is None:
            stride = output_stride / 2.0
        if not torch.cuda.is_available():
            raise DgpError(-2, "no CUDA device: deepgraphpose_b200 has no CPU fallback")
        self.lib = _lib.load()
        if device is None:
            device = torch.cuda.current_device()
        self.device = torch.device("cuda", device if isinstance(device, int) else torch.device(device).index or 0)
        self.nj = int(num_joints)
        self.location_refinement = bool(location_refinement)
        cfg = DgpConfig()
        cfg.num_joints = self.nj
        cfg.location_refinement = int(self.location_refinement)
        cfg.device = self.device.index
        cfg.stride = stride
        cfg.locref_stdev = locref_stdev
        cfg.mean_pixel = (C.c_float * 3)(*mean_pixel)
        cfg.bn_epsilon = 1e-5
        if precision not in ("bf16", "fp16"):
            raise ValueError("precision must be 'bf16' or 'fp16'")
        cfg.precision = 1 if precision == "fp16" else 0
        self.precision = precision
        self.act_dtype = torch.float16 if precision == "fp16" else torch.bfloat16
        self.stride = float(stride)
        self.locref_stdev = float(locref_stdev)
        h = C.c_void_p()
        check(self.lib.dgp_create(C.byref(cfg), C.byref(h)))
        self.h = h
        self._check(self.lib.dgp_set_output_stride(self.h, output_stride))
        self.output_stride = output_stride
        self.weights_loaded = False
        self.net_type = None  # "resnet_50" / "resnet_101" / "resnet_152": the backbone the loaded weights name

    def close(self):
        if getattr(self, "h", None):
            self.lib.dgp_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, status):
        check(status, self.h)

    # ------------------------------------------------------------------ weights (Saver.restore replacement)
    def load_weights(self, variables):
        """variables: {tf_var_name: float32 ndarray in TF layout}."""
        for name, arr in variables.items():
            a = np.ascontiguousarray(arr, dtype=np.float32)
            shape = (C.c_int64 * a.ndim)(*a.shape)
            self._check(self.lib.dgp_load_weights(self.h, name.encode(), a.ctypes.data_as(C.c_void_p), shape, a.ndim, 0))
        self._check(self.lib.dgp_finalize_weights(self.h))
        self.weights_loaded = True
        depth = C.c_int()
        self._check(self.lib.dgp_net_depth(self.h, C.byref(depth)))
        self.net_type = "resnet_%d" % depth.value
        # the frozen moving statistics are not trainable state of the handle; keep them for checkpoint export
        self._frozen = {k: np.array(v, dtype=np.float32) for k, v in variables.items()
                        if k.endswith("/moving_mean") or k.endswith("/moving_variance")}

    def output_dims(self, H, W):
        """(h_feat, w_feat), (h_out, w_out) of an H x W frame through this engine's backbone (its output_stride)."""
        return output_dims(H, W, self.output_stride)

    # ------------------------------------------------------------------ forward
    def forward(self, frames, want_locref=None):
        """frames: uint8 cuda tensor (B,H,W,3). Returns (logits (B,2h,2w,nj) f32, locref (B,2h,2w,2nj) f32 | None)."""
        if frames.dtype != torch.uint8 or frames.dim() != 4 or frames.shape[-1] != 3 or not frames.is_cuda:
            raise ValueError("frames must be a uint8 CUDA tensor of shape (B,H,W,3)")
        frames = frames.contiguous()
        B, H, W, _ = frames.shape
        _, (ho, wo) = self.output_dims(H, W)
        if want_locref is None:
            want_locref = self.location_refinement
        logits = torch.empty((B, ho, wo, self.nj), dtype=torch.float32, device=frames.device)
        locref = torch.empty((B, ho, wo, 2 * self.nj), dtype=torch.float32, device=frames.device) if want_locref else None
        self._check(self.lib.dgp_forward(self.h, _ptr(frames), B, H, W, _ptr(logits), _ptr(locref), _stream(frames.device)))
        return logits, locref

    def extract_features(self, frames):
        """PoseNet.extract_features (pose_net.py:36-54): uint8 cuda frames (B,H,W,3) -> net (B,hf,wf,2048) float32."""
        if frames.dtype != torch.uint8 or frames.dim() != 4 or frames.shape[-1] != 3 or not frames.is_cuda:
            raise ValueError("frames must be a uint8 CUDA tensor of shape (B,H,W,3)")
        frames = frames.contiguous()
        B, H, W, _ = frames.shape
        (hf, wf), _ = self.output_dims(H, W)
        net = torch.empty((B, hf, wf, 2048), dtype=torch.float32, device=frames.device)
        self._check(self.lib.dgp_extract_features(self.h, _ptr(frames), B, H, W, _ptr(net), _stream(frames.device)))
        return net

    def prediction_layers(self, net, want_locref=None):
        """PoseNet.prediction_layers (pose_net.py:56-78) on a float32 cuda ``net`` (B,hf,wf,2048) -> (logits, locref | None)."""
        if net.dtype != torch.float32 or net.dim() != 4 or net.shape[-1] != 2048 or not net.is_cuda:
            raise ValueError("net must be a float32 CUDA tensor (B,hf,wf,2048)")
        net = net.contiguous()
        B, hf, wf, _ = net.shape
        if want_locref is None:
            want_locref = self.location_refinement
        logits = torch.empty((B, 2 * hf, 2 * wf, self.nj), dtype=torch.float32, device=net.device)
        locref = torch.empty((B, 2 * hf, 2 * wf, 2 * self.nj), dtype=torch.float32, device=net.device) if want_locref else None
        self._check(self.lib.dgp_prediction_layers(self.h, _ptr(net), B, hf, wf, _ptr(logits), _ptr(locref), _stream(net.device)))
        return logits, locref

    def deconv2d(self, x, w, bias=None):
        """slim.conv2d_transpose(x, Cout, [3,3], stride=2, 'SAME') + bias: x float32 cuda (N,H,W,Cin), Cin % 64 == 0;
        w float32 ndarray in the TF layout [3,3,Cout,Cin]; returns float32 (N,2H,2W,Cout)."""
        if x.dtype != torch.float32 or x.dim() != 4 or not x.is_cuda:
            raise ValueError("x must be a float32 CUDA tensor (N,H,W,Cin)")
        x = x.contiguous()
        w = np.ascontiguousarray(w, dtype=np.float32)
        if w.ndim != 4 or w.shape[0] != 3 or w.shape[1] != 3 or w.shape[3] != x.shape[3]:
            raise ValueError("w must be [3,3,Cout,Cin] with Cin = %d" % x.shape[3])
        N, H, W, Cin = x.shape
        Cout = w.shape[2]
        b = np.ascontiguousarray(bias, dtype=np.float32).reshape(-1) if bias is not None else None
        if b is not None and b.size != Cout:
            raise ValueError("bias must have %d entries" % Cout)
        out = torch.empty((N, 2 * H, 2 * W, Cout), dtype=torch.float32, device=x.device)
        self._check(self.lib.dgp_deconv2d(self.h, _ptr(x), N, H, W, Cin, w.ctypes.data_as(C.c_void_p),
                                          b.ctypes.data_as(C.c_void_p) if b is not None else None, Cout, _ptr(out),
                                          _stream(x.device)))
        return out

    def softargmax(self, logits, locref=None, gamma=1.0, gauss_len=1.0, want=("mu", "peak", "lik", "dlc_peak", "dlc_pose")):
        """Fused argmax_2d_from_cm + estimate_pose read-out + DLC argmax pose. Returns a dict of cuda tensors."""
        if logits.dtype != torch.float32 or logits.dim() != 4 or not logits.is_cuda:
            raise ValueError("logits must be a float32 CUDA tensor (B,H,W,nj)")
        logits = logits.contiguous()
        B, H, W, nj = logits.shape
        dev = logits.device
        out = {}
        out["mu"] = torch.empty((B, nj, 2), dtype=torch.float32, device=dev) if "mu" in want else None
        out["peak"] = torch.empty((B, nj, 2), dtype=torch.int32, device=dev) if "peak" in want else None
        out["lik"] = torch.empty((B, nj), dtype=torch.float32, device=dev) if "lik" in want else None
        out["dlc_peak"] = torch.empty((B, nj, 2), dtype=torch.int32, device=dev) if "dlc_peak" in want else None
        out["dlc_pose"] = torch.empty((B, nj, 3), dtype=torch.float32, device=dev) if "dlc_pose" in want else None
        if locref is not None:
            locref = locref.contiguous()
            if locref.shape != (B, H, W, 2 * nj) or locref.dtype != torch.float32:
                raise ValueError("locref must be float32 (B,H,W,2*nj)")
        self._check(self.lib.dgp_softargmax(self.h, _ptr(logits), _ptr(locref), B, H, W, nj, float(gamma), float(gauss_len),
                                            _ptr(out["mu"]), _ptr(out["peak"]), _ptr(out["lik"]), _ptr(out["dlc_peak"]),
                                            _ptr(out["dlc_pose"]), _stream(dev)))
        return {k: v for k, v in out.items() if v is not None}

    def softmax_map(self, logits, gamma=1.0, gauss_len=1.0):
        """Second output of argmax_2d_from_cm: blurred, renormalised spatial softmax (B,H,W,nj)."""
        logits = logits.contiguous()
        B, H, W, nj = logits.shape
        out = torch.empty_like(logits)
        self._check(self.lib.dgp_softmax_map(self.h, _ptr(logits), B, H, W, nj, float(gamma), float(gauss_len), _ptr(out),
                                             _stream(logits.device)))
        return out

    def soft_pose(self, logits, locref, gamma=1.0, gauss_len=1.0, swap_offsets=False):
        """evaluate_dgp's 'dgp' locref branch (eval.py:751-785) on the device: (B,nj,3) = (x, y, 1)."""
        logits, locref = logits.contiguous(), locref.contiguous()
        B, H, W, nj = logits.shape
        if locref.shape != (B, H, W, 2 * nj) or locref.dtype != torch.float32 or logits.dtype != torch.float32:
            raise ValueError("logits (B,H,W,nj) and locref (B,H,W,2*nj) must be float32")
        ws = torch.empty_like(logits)
        pose = torch.empty((B, nj, 3), dtype=torch.float32, device=logits.device)
        self._check(self.lib.dgp_soft_pose(self.h, _ptr(logits), _ptr(locref), B, H, W, nj, float(gamma), float(gauss_len),
                                           int(swap_offsets), _ptr(ws), _ptr(pose), _stream(logits.device)))
        return pose

    def sigmoid(self, logits):
        logits = logits.contiguous()
        out = torch.empty_like(logits)
        self._check(self.lib.dgp_sigmoid(self.h, _ptr(logits), _ptr(out), logits.numel(), _stream(logits.device)))
        return out

    def potentials(self, mu, edges, halo_next=None, ws=None, ws_max=None, wt_max=0.0, out=None):
        """mu (T,nj,2) f32 cuda; edges int32 (nl,2). Returns dict(skel (nl,T), temporal (T or T-1, nj), e_skel (T), e_temp (T)).
        ``out`` may carry the dict of a previous call to reuse its buffers (steady-state loops allocate nothing)."""
        mu = mu.contiguous()
        T, nj, _ = mu.shape
        dev = mu.device
        key = (tuple(map(tuple, np.asarray(edges, dtype=np.int64).reshape(-1, 2).tolist())), str(dev))
        cache = self.__dict__.setdefault("_edge_cache", {})
        if key not in cache:
            cache[key] = torch.as_tensor(np.asarray(edges, dtype=np.int32).reshape(-1, 2), device=dev)
        edges_t = cache[key]
        nl = edges_t.shape[0]
        if out is not None and out["_T"] == T and out["_nl"] == nl:
            skel, temporal, e_skel, e_temp = out["skel"], out["_temporal_full"], out["e_skel"], out["e_temp"]
        else:
            skel = torch.empty((nl, T), dtype=torch.float32, device=dev)
            temporal = torch.empty((T, nj), dtype=torch.float32, device=dev)
            e_skel = torch.empty((T,), dtype=torch.float32, device=dev) if ws is not None else None
            e_temp = torch.empty((T,), dtype=torch.float32, device=dev)
        wkey = ("ws", None if ws is None else tuple(np.asarray(ws, dtype=np.float32).tolist()),
                None if ws_max is None else tuple(np.asarray(ws_max, dtype=np.float32).tolist()), str(dev))
        if wkey not in cache:
            cache[wkey] = (torch.as_tensor(np.asarray(ws, dtype=np.float32), device=dev) if ws is not None else None,
                           torch.as_tensor(np.asarray(ws_max, dtype=np.float32), device=dev) if ws_max is not None else None)
        ws_t, wsm_t = cache[wkey]
        if halo_next is not None:
            halo_next = halo_next.contiguous()
        self._check(self.lib.dgp_potentials(self.h, _ptr(mu), _ptr(halo_next), T, nj, _ptr(edges_t), nl, _ptr(ws_t), _ptr(wsm_t),
                                            float(wt_max), _ptr(skel), _ptr(temporal), _ptr(e_skel), _ptr(e_temp), _stream(dev)))
        n_t = T if halo_next is not None else T - 1
        return {"skel": skel, "temporal": temporal[:n_t], "e_skel": e_skel, "e_temp": e_temp, "_temporal_full": temporal,
                "_T": T, "_nl": nl}

    def resize_crop(self, frames_dev, new_size=None, crop_size=None):
        """estimate_pose's per-frame ``PIL.Image.resize(size=(new_size[1], new_size[0]))`` + ``.crop(crop_size)`` on the
        device, bit-exact (dgp_resize_crop): uint8 cuda (N,H0,W0,3) -> new uint8 cuda (N,H,W,3)."""
        if frames_dev.dtype != torch.uint8 or frames_dev.dim() != 4 or frames_dev.shape[-1] != 3 or not frames_dev.is_cuda:
            raise ValueError("frames must be a uint8 CUDA tensor of shape (N,H,W,3)")
        frames_dev = frames_dev.contiguous()
        N, H0, W0, _ = frames_dev.shape
        H, W = transform_dims(H0, W0, new_size, crop_size)
        t = frame_transform(new_size, crop_size)
        out = torch.empty((N, H, W, 3), dtype=torch.uint8, device=frames_dev.device)
        self._check(self.lib.dgp_resize_crop(self.h, _ptr(frames_dev), N, H0, W0, C.byref(t) if t is not None else None,
                                             _ptr(out), _stream(frames_dev.device)))
        return out

    def augment(self, frames_dev, positions, joint_loc, params, stride=None):
        """fit_dgp's augmentation of labelled frames on the device (dgp_augment): rotation, motion blur, coarse dropout and
        elastic deformation of ``frames_dev`` (uint8 contiguous CUDA (nt,H,W,3), modified in place) at the batch
        ``positions``, frame ``positions[k]`` with ``params[k]`` (a dict of dgp_augment_params fields, missing ones 0, or a
        ``_lib.DgpAugmentParams``).  ``joint_loc``: the (n, nj, 2) scoremap (row, col) labels of those frames, a float64
        contiguous CUDA tensor moved in place (or a host array, uploaded), or None; ``stride``: scoremap stride of the labels
        (default: the engine's).  Returns the device labels (or None)."""
        if frames_dev.dtype != torch.uint8 or frames_dev.dim() != 4 or frames_dev.shape[-1] != 3 or not frames_dev.is_cuda:
            raise ValueError("frames must be a uint8 CUDA tensor of shape (nt,H,W,3)")
        if not frames_dev.is_contiguous():
            raise ValueError("frames must be contiguous: they are augmented in place")
        nt, H, W, _ = frames_dev.shape
        idx = np.ascontiguousarray(np.asarray(positions, dtype=np.int32).reshape(-1))
        n = idx.shape[0]
        if len(params) != n:
            raise ValueError("one parameter set per augmented frame is required")
        par = (_lib.DgpAugmentParams * max(n, 1))()
        for k, p in enumerate(params):
            par[k] = p if isinstance(p, _lib.DgpAugmentParams) else _lib.DgpAugmentParams(**p)
        jl = None
        if joint_loc is not None:
            jl = joint_loc
            if not isinstance(jl, torch.Tensor):
                jl = torch.from_numpy(np.ascontiguousarray(np.asarray(joint_loc, dtype=np.float64))).to(frames_dev.device)
            if jl.dtype != torch.float64 or not jl.is_cuda or not jl.is_contiguous() or tuple(jl.shape) != (n, self.nj, 2):
                raise ValueError("joint_loc must be a contiguous float64 CUDA tensor (%d, %d, 2)" % (n, self.nj))
        self._check(self.lib.dgp_augment(self.h, _ptr(frames_dev), nt, H, W, idx.ctypes.data_as(C.c_void_p), n, par,
                                          _ptr(jl) if jl is not None and jl.numel() else None,
                                          float(self.stride if stride is None else stride),
                                          _stream(frames_dev.device)))
        return jl

    def elastic_field(self, H, W, alpha, sigma, seed):
        """The elastic displacement fields dgp_augment samples with (dgp_elastic_field): float32 CUDA (dx, dy), each (H, W)."""
        dx = torch.empty((H, W), dtype=torch.float32, device=self.device)
        dy = torch.empty_like(dx)
        self._check(self.lib.dgp_elastic_field(self.h, int(H), int(W), float(alpha), float(sigma), int(seed), _ptr(dx), _ptr(dy),
                                               _stream(self.device)))
        return dx, dy

    def estimate_pose_host(self, frames_host, batch=16, gamma=1.0, gauss_len=1.0, new_size=None, crop_size=None):
        """End-to-end with HOST buffers (H2D + forward + soft-argmax + D2H inside). frames_host: uint8 (T,H0,W0,3) CPU tensor.
        ``new_size`` / ``crop_size`` (estimate_pose's options, see ``frame_transform``) resize / crop every frame on the
        device after the H2D copy, which carries the frames at their source size."""
        if frames_host.is_cuda or frames_host.dtype != torch.uint8 or frames_host.dim() != 4 or frames_host.shape[-1] != 3:
            raise ValueError("frames_host must be a uint8 CPU tensor (T,H,W,3) (pinned for async copies)")
        frames_host = frames_host.contiguous()
        T, H0, W0, _ = frames_host.shape
        transform_dims(H0, W0, new_size, crop_size)
        t = frame_transform(new_size, crop_size)
        mu = torch.empty((T, self.nj, 2), dtype=torch.float32).pin_memory()
        peak = torch.empty((T, self.nj, 2), dtype=torch.int32).pin_memory()
        lik = torch.empty((T, self.nj), dtype=torch.float32).pin_memory()
        self._check(self.lib.dgp_estimate_pose_host_transform(self.h, _ptr(frames_host), T, H0, W0,
                                                              C.byref(t) if t is not None else None, int(batch), float(gamma),
                                                              float(gauss_len), _ptr(mu), _ptr(peak), _ptr(lik)))
        return mu, peak, lik

    def draw_markers(self, frames_dev, x, y, lik, dotsize=3, mask_threshold=0.1, colors=None, edges=None,
                     skeleton_color=(0, 0, 0), trailpoints=0, history=0):
        """plot_dgp's markers drawn into ``frames_dev`` (uint8 contiguous CUDA (N,H,W,3) RGB, modified in place;
        dgp_draw_markers): joint j of frame t where ``lik[t, j] > mask_threshold``, a disc of radius ``dotsize`` at the
        video-pixel coordinates ``x[t, j]``, ``y[t, j]`` in ``colors[j]`` (see ``marker_style``); with ``edges`` a line
        in ``skeleton_color`` per edge under the discs, with ``trailpoints`` K >= 2 the discs of the K - 1 previous frames
        under both (the contract is in include/dgp_b200.h).  ``x``, ``y``, ``lik``: (history + N, nj) float64 CUDA
        tensors, or host arrays (uploaded), whose first ``history`` rows are the frames before ``frames_dev[0]``.
        Asynchronous on the current stream."""
        if frames_dev.dtype != torch.uint8 or frames_dev.dim() != 4 or frames_dev.shape[-1] != 3 or not frames_dev.is_cuda:
            raise ValueError("frames must be a uint8 CUDA tensor of shape (N,H,W,3)")
        if not frames_dev.is_contiguous():
            raise ValueError("frames must be contiguous: markers are drawn in place")
        N, H, W, _ = frames_dev.shape
        st, table = marker_style(self.nj, dotsize, mask_threshold, colors, edges=edges, skeleton_color=skeleton_color,
                                 trailpoints=trailpoints, history=history)
        cols = []
        for v in (x, y, lik):
            if not isinstance(v, torch.Tensor):
                v = torch.from_numpy(np.ascontiguousarray(np.asarray(v, dtype=np.float64)))
            v = v.to(device=frames_dev.device, dtype=torch.float64).contiguous()
            if tuple(v.shape) != (int(history) + N, self.nj):
                raise ValueError("x, y and lik must be (%d, %d)" % (int(history) + N, self.nj))
            cols.append(v)
        self._check(self.lib.dgp_draw_markers(self.h, _ptr(frames_dev), N, H, W, _ptr(cols[0]), _ptr(cols[1]), _ptr(cols[2]),
                                              C.byref(st), _stream(frames_dev.device)))
        return frames_dev

    def encode_jpeg(self, frames_dev, quality=90):
        """The JPEG file of every frame of ``frames_dev`` (uint8 contiguous CUDA (N,H,W,3) RGB), encoded on the device
        (dgp_encode_jpeg): exactly the bytes of ``PIL.Image.fromarray(frame).save(buf, format="JPEG", quality=quality,
        subsampling=2, restart_marker_rows=1)``.  Returns a list of N ``bytes``; synchronises with the current stream."""
        q = check_jpeg_quality(quality)
        if frames_dev.dtype != torch.uint8 or frames_dev.dim() != 4 or frames_dev.shape[-1] != 3 or not frames_dev.is_cuda:
            raise ValueError("frames must be a uint8 CUDA tensor of shape (N,H,W,3)")
        frames_dev = frames_dev.contiguous()
        N, H, W, _ = frames_dev.shape
        cap = jpeg_capacity(H, W) * N
        out = torch.empty(max(cap, 1), dtype=torch.uint8, device=frames_dev.device)
        meta = torch.empty((2, max(N, 1)), dtype=torch.int64, device=frames_dev.device)
        self._check(self.lib.dgp_encode_jpeg(self.h, _ptr(frames_dev), N, H, W, q, _ptr(out), cap, _ptr(meta[0]),
                                             _ptr(meta[1]), _stream(frames_dev.device)))
        if N == 0:
            return []
        offsets, sizes = meta.cpu().numpy()
        if (sizes < 0).any():
            raise DgpError(-1, "dgp_encode_jpeg: a frame exceeded dgp_jpeg_capacity")
        data = out[:int(offsets[-1] + sizes[-1])].cpu().numpy()
        return [data[o:o + n].tobytes() for o, n in zip(offsets, sizes)]

    def _frame_reader(self, source, H, W, T, start):
        """(reader, user, keep, state) of a stream source (see estimate_pose_stream); state["error"] holds an exception the
        source raised."""
        frame_bytes = int(H) * int(W) * 3
        state = {"error": None}
        if isinstance(source, torch.Tensor):
            if source.is_cuda or source.dtype != torch.uint8 or source.dim() != 4 or tuple(source.shape[1:]) != (H, W, 3):
                raise ValueError("a tensor source must be a uint8 CPU tensor (P,%d,%d,3)" % (H, W))
            pool = source.contiguous()
            src = _lib.DgpCyclicSource(pool.data_ptr(), pool.shape[0], int(start) + T, int(start), frame_bytes)
            return C.cast(self.lib.dgp_cyclic_reader, C.c_void_p), C.cast(C.pointer(src), C.c_void_p), (pool, src), state
        it = iter(source)

        def _read(user_, slot, want, direct):
            try:
                dst = np.ctypeslib.as_array(C.cast(slot, C.POINTER(C.c_uint8)), shape=(want, H, W, 3))
                n = 0
                for n in range(1, want + 1):
                    try:
                        fr = next(it)
                    except StopIteration:
                        n -= 1
                        break
                    fr = np.asarray(fr)
                    if fr.shape != (H, W, 3) or fr.dtype != np.uint8:
                        raise ValueError("the source must yield uint8 frames of shape (%d, %d, 3), got %s %s"
                                         % (H, W, fr.dtype, fr.shape))
                    dst[n - 1] = fr
                return n
            except Exception as ex:  # never unwind through the C frame
                state["error"] = ex
                return -1

        cb = _lib.FRAME_READER(_read)
        return C.cast(cb, C.c_void_p), C.c_void_p(0), cb, state

    def estimate_pose_stream(self, source, H, W, max_frames, batch=16, gamma=1.0, gauss_len=1.0, start=0, new_size=None,
                             crop_size=None):
        """Streaming estimate_pose (dgp_estimate_pose_stream): host memory is bounded by a ring of 3 pinned slots of `batch`
        frames, whatever the length of the video.  ``source`` is either

        * an iterator / generator yielding uint8 (H,W,3) RGB frames (a video decoder): frames are written into the pinned
          slot by a reader thread while the GPU works on the previous slots, or
        * a uint8 CPU tensor (P,H,W,3) (pinned for asynchronous copies): a video of ``max_frames`` frames that cycles over
          these P frames, served zero-copy by the library's own ``dgp_cyclic_reader`` (synthetic videos, bench.py);
          ``start`` is the index of the first frame to serve (frame t of the video is ``source[t % P]``), which lets every
          rank of a sharded run read its own contiguous range of the same video.

        ``H``, ``W`` are the size of the source frames.  ``new_size`` / ``crop_size`` (estimate_pose's options, see
        ``frame_transform``) resize / crop every frame on the device: the ring and the H2D copy carry source-size frames.

        Returns (mu (T,nj,2) f32, peak (T,nj,2) i32, lik (T,nj) f32) as CPU tensors, T = frames actually delivered."""
        T = int(max_frames)
        transform_dims(H, W, new_size, crop_size)
        tf = frame_transform(new_size, crop_size)
        mu = torch.empty((T, self.nj, 2), dtype=torch.float32).pin_memory()
        peak = torch.empty((T, self.nj, 2), dtype=torch.int32).pin_memory()
        lik = torch.empty((T, self.nj), dtype=torch.float32).pin_memory()
        done = C.c_int64(0)
        reader, user, keep, state = self._frame_reader(source, H, W, T, start)
        status = self.lib.dgp_estimate_pose_stream_transform(self.h, reader, user, int(H), int(W),
                                                             C.byref(tf) if tf is not None else None, int(batch),
                                                             float(gamma), float(gauss_len), T, _ptr(mu), _ptr(peak),
                                                             _ptr(lik), C.byref(done))
        if state["error"] is not None:
            raise state["error"]
        self._check(status)
        n = int(done.value)
        return mu[:n], peak[:n], lik[:n]

    def estimate_pose_render_stream(self, source, H, W, max_frames, writer, dotsize=3, mask_threshold=0.1, colors=None,
                                    new_size=None, crop_size=None, batch=16, gamma=1.0, gauss_len=1.0, start=0, encoder="raw",
                                    quality=90, edges=None, skeleton_color=(0, 0, 0), trailpoints=0):
        """estimate_pose_stream that renders plot_dgp's labelled video in the same pass (dgp_estimate_pose_stream_render):
        after each batch's soft-argmax the markers are drawn on the device into the batch's source frames (coordinates
        converted to video pixels as eval.estimate_pose does, scale W / new_size[1], H / new_size[0] under ``new_size``) and
        the annotated frames are handed to ``writer(frames)`` -- a uint8 (n,H,W,3) RGB array valid only during the call --
        from a writer thread, in video order.  An exception the writer raises aborts the pass and is re-raised here; a
        negative integer it returns aborts it with DgpError, as in the C ABI.
        ``encoder="jpeg"`` (dgp_estimate_pose_stream_render_jpeg) encodes the annotated frames on the device instead, as
        encode_jpeg does at ``quality``, and calls ``writer(data, sizes)``: a uint8 array holding the batch's JPEG files back
        to back in video order and an int64 array of their sizes, both valid only during the call.
        Sources and return value as in estimate_pose_stream; style arguments as in draw_markers.  Trails reach back to the
        first frame of the call across batches, so the frames do not depend on ``batch``."""
        if encoder not in ("raw", "jpeg"):
            raise ValueError("encoder must be 'raw' or 'jpeg', got %r" % (encoder,))
        q = check_jpeg_quality(quality)
        if encoder == "jpeg":
            jpeg_capacity(H, W)
        T = int(max_frames)
        transform_dims(H, W, new_size, crop_size)
        tf = frame_transform(new_size, crop_size)
        sx, sy = (1.0, 1.0) if new_size is None else (W / new_size[1], H / new_size[0])
        st, table = marker_style(self.nj, dotsize, mask_threshold, colors, sx, sy, edges, skeleton_color, trailpoints)
        if not callable(writer):
            raise ValueError("writer must be callable")
        mu = torch.empty((T, self.nj, 2), dtype=torch.float32).pin_memory()
        peak = torch.empty((T, self.nj, 2), dtype=torch.int32).pin_memory()
        lik = torch.empty((T, self.nj), dtype=torch.float32).pin_memory()
        done = C.c_int64(0)
        reader, user, keep, state = self._frame_reader(source, H, W, T, start)
        werr = {"error": None}

        def _write(user_, frames, n):
            try:
                rc = writer(np.ctypeslib.as_array(C.cast(frames, C.POINTER(C.c_uint8)), shape=(n, H, W, 3)))
                return int(rc) if isinstance(rc, (int, np.integer)) and rc < 0 else 0
            except Exception as ex:  # never unwind through the C frame
                werr["error"] = ex
                return -1

        def _write_packets(user_, data, sizes, n):
            try:
                sz = np.ctypeslib.as_array(C.cast(sizes, C.POINTER(C.c_int64)), shape=(n,))
                buf = np.ctypeslib.as_array(C.cast(data, C.POINTER(C.c_uint8)), shape=(int(sz.sum()),))
                rc = writer(buf, sz)
                return int(rc) if isinstance(rc, (int, np.integer)) and rc < 0 else 0
            except Exception as ex:  # never unwind through the C frame
                werr["error"] = ex
                return -1

        args = (self.h, reader, user, int(H), int(W), C.byref(tf) if tf is not None else None, int(batch), float(gamma),
                float(gauss_len), T, _ptr(mu), _ptr(peak), _ptr(lik), C.byref(done), C.byref(st))
        if encoder == "jpeg":
            wcb = _lib.PACKET_WRITER(_write_packets)
            status = self.lib.dgp_estimate_pose_stream_render_jpeg(*args, q, C.cast(wcb, C.c_void_p), None)
        else:
            wcb = _lib.FRAME_WRITER(_write)
            status = self.lib.dgp_estimate_pose_stream_render(*args, C.cast(wcb, C.c_void_p), None)
        for err in (state["error"], werr["error"]):
            if err is not None:
                raise err
        self._check(status)
        n = int(done.value)
        return mu[:n], peak[:n], lik[:n]

    # ------------------------------------------------------------------ training (fit_dgp's train_op)
    def train_enable(self):
        if not getattr(self, "_train", False):
            self._check(self.lib.dgp_train_enable(self.h))
            self._train = True
            if self.precision == "fp16":
                # keeps the smallest activation gradients out of fp16's subnormal range; a power of two, divided out again by
                # dgp_optimizer_step, so the update is unchanged wherever nothing underflowed
                self._check(self.lib.dgp_train_set_loss_scale(self.h, 1024.0))

    def optimizer_step(self, lr=0.005, momentum=0.9, clip_norm=10.0, grad_scale=1.0):
        """clip_by_global_norm(clip_norm) + MomentumOptimizer(lr, momentum) (fitdgp.py:706-713) on the gradient buffer."""
        self._check(self.lib.dgp_optimizer_step(self.h, float(lr), float(momentum), float(clip_norm), float(grad_scale),
                                                _stream(self.device)))

    def grad_buffer(self):
        """The flat float32 gradient buffer as a CUDA tensor VIEW (what a data-parallel caller all-reduces)."""
        self.train_enable()
        p, n = C.c_void_p(), C.c_size_t()
        self._check(self.lib.dgp_get_grad_buffer(self.h, C.byref(p), C.byref(n)))
        return _device_view(p.value, (n.value // 4,), "<f4", self.device)

    def param_buffer(self):
        """The flat float32 parameter arena (fp32 master copy, same layout as grad_buffer) as a CUDA tensor VIEW.  After
        changing it in place, call params_changed() before the next forward."""
        p, n = C.c_void_p(), C.c_size_t()
        self._check(self.lib.dgp_get_param_buffer(self.h, C.byref(p), C.byref(n)))
        return _device_view(p.value, (n.value // 4,), "<f4", self.device)

    def params_changed(self):
        """Re-derive the 16-bit weights, BatchNorm scale / shift and dgrad operands from param_buffer() (dgp_params_changed)."""
        self._check(self.lib.dgp_params_changed(self.h, _stream(self.device)))

    def train_forward(self, frames, want_locref=None):
        """Training forward (dgp_train_forward): frames uint8 cuda (nt,H,W,3) -> (logits, locref | None, token).  The outputs
        are new float32 tensors; the token names the kept activations for train_backward."""
        if frames.dtype != torch.uint8 or frames.dim() != 4 or frames.shape[-1] != 3 or not frames.is_cuda:
            raise ValueError("frames must be a uint8 CUDA tensor of shape (B,H,W,3)")
        self.train_enable()
        frames = frames.contiguous()
        B, H, W, _ = frames.shape
        _, (ho, wo) = self.output_dims(H, W)
        if want_locref is None:
            want_locref = self.location_refinement
        logits = torch.empty((B, ho, wo, self.nj), dtype=torch.float32, device=frames.device)
        locref = torch.empty((B, ho, wo, 2 * self.nj), dtype=torch.float32, device=frames.device) if want_locref else None
        token = C.c_uint64()
        self._check(self.lib.dgp_train_forward(self.h, _ptr(frames), B, H, W, _ptr(logits), _ptr(locref), C.byref(token),
                                               _stream(frames.device)))
        # head shapes of the live token of each input shape (at most one: a new forward at a shape makes the old token stale)
        live = self.__dict__.setdefault("_live_tokens", {})
        for t in [t for t, v in live.items() if v[0] == tuple(frames.shape)]:
            del live[t]
        live[int(token.value)] = (tuple(frames.shape), tuple(logits.shape))
        return logits, locref, int(token.value)

    def train_backward(self, token, g_logits, g_locref=None, accumulate=False):
        """Network backward of the train_forward named by ``token`` from the loss gradients w.r.t. its head outputs (float32
        cuda, None = zeros) into grad_buffer(): overwrite, or add with ``accumulate``.  The buffer then holds the true
        (unscaled) gradient.  A stale token raises DgpError (DGP_ERR_STATE)."""
        for g in (g_logits, g_locref):
            if g is not None and (g.dtype != torch.float32 or not g.is_cuda):
                raise ValueError("head gradients must be float32 CUDA tensors")
        live = self.__dict__.get("_live_tokens", {})
        if token in live:   # the C side checks the token; the sizes of the caller's buffers can only be checked here
            shp = live[token][1]
            if g_logits is not None and tuple(g_logits.shape) != shp:
                raise ValueError("g_logits must have the logits' shape %s" % (shp,))
            if g_locref is not None and tuple(g_locref.shape) != shp[:3] + (2 * self.nj,):
                raise ValueError("g_locref must have the locref shape %s" % (shp[:3] + (2 * self.nj,),))
        g_logits = g_logits.contiguous() if g_logits is not None else None
        g_locref = g_locref.contiguous() if g_locref is not None else None
        self._check(self.lib.dgp_train_backward(self.h, C.c_uint64(token), _ptr(g_logits), _ptr(g_locref), int(bool(accumulate)),
                                                _stream(self.device)))

    def set_loss_scale(self, loss_scale):
        """Loss scaling for fp16-storage training (no effect on the update; see dgp_train_set_loss_scale)."""
        self.train_enable()
        self._check(self.lib.dgp_train_set_loss_scale(self.h, float(loss_scale)))

    def allreduce_exposed_ms(self):
        """Milliseconds between the end of the last backward pass and the end of its C-side gradient all-reduce."""
        v = C.c_float()
        self._check(self.lib.dgp_allreduce_exposed_ms(self.h, C.byref(v)))
        return float(v.value)

    def grad_norm(self):
        v = C.c_float()
        self._check(self.lib.dgp_get_grad_norm(self.h, C.byref(v)))
        return float(v.value)

    def train_outputs(self, nt, H, W):
        """Views of the head outputs (logits, locref) the last training step at this input shape produced."""
        a, b = C.c_void_p(), C.c_void_p()
        self._check(self.lib.dgp_train_outputs(self.h, int(nt), int(H), int(W), C.byref(a), C.byref(b)))
        _, (ho, wo) = self.output_dims(H, W)
        logits = _device_view(a.value, (nt, ho, wo, self.nj), "<f4", self.device)
        locref = _device_view(b.value, (nt, ho, wo, 2 * self.nj), "<f4", self.device) if b.value else None
        return logits, locref

    def get_variable(self, name, what="value"):
        """A trainable variable (or its gradient / momentum accumulator) under its TF name, in TF layout (float32 ndarray)."""
        code = {"value": 0, "grad": 1, "momentum": 2}[what]
        shape = (C.c_int64 * 4)()
        nd = C.c_int()
        self._check(self.lib.dgp_get_variable(self.h, name.encode(), code, None, 0, shape, C.byref(nd)))
        shp = tuple(int(shape[i]) for i in range(nd.value))
        out = np.empty(shp, np.float32)
        self._check(self.lib.dgp_get_variable(self.h, name.encode(), code, out.ctypes.data_as(C.c_void_p), out.size, shape,
                                              C.byref(nd)))
        return out

    def locref_targets(self, joint_loc, visible_frame_within_batch, nt, H, W, pos_dist_thresh=17.0, locref_stdev=7.2801):
        """Device-side coord2map + batch scatter (dataset.py:246-271, fitdgp.py:781-795): joint_loc (n_vis,nj,2) float64
        scoremap (row,col) labels (NaN = missing).  Returns float32 CUDA tensors (locref_map, locref_mask) (nt,H,W,2nj)."""
        dev = self.device
        if isinstance(joint_loc, torch.Tensor):     # labels already on the device (fitdgp_util.data_aug) are read in place
            jl_d = joint_loc.to(device=dev, dtype=torch.float64).reshape(-1, self.nj, 2).contiguous()
        else:
            jl_d = torch.from_numpy(np.ascontiguousarray(np.asarray(joint_loc, dtype=np.float64).reshape(-1, self.nj, 2))).to(dev)
        idx = np.ascontiguousarray(np.asarray(visible_frame_within_batch, dtype=np.int32).reshape(-1))
        if jl_d.shape[0] != idx.shape[0]:
            raise ValueError("one batch position per labelled frame is required")
        if not jl_d.numel():
            jl_d = None
        idx_d = torch.from_numpy(idx).to(dev) if idx.size else None
        lmap = torch.empty((nt, H, W, 2 * self.nj), dtype=torch.float32, device=dev)
        lmask = torch.empty_like(lmap)
        self._check(self.lib.dgp_locref_targets(self.h, _ptr(jl_d), _ptr(idx_d), int(idx.shape[0]), int(nt), int(H), int(W),
                                                float(pos_dist_thresh), float(locref_stdev), _ptr(lmap), _ptr(lmask),
                                                _stream(dev)))
        return lmap, lmask

    def set_variable(self, name, array, what="value"):
        """Overwrite a trainable variable ("value") or its Momentum accumulator ("momentum") from a TF-layout array."""
        code = {"value": 0, "momentum": 2}[what]
        if code == 2:
            self.train_enable()
        a = np.ascontiguousarray(array, dtype=np.float32)
        self._check(self.lib.dgp_set_variable(self.h, name.encode(), code, a.ctypes.data_as(C.c_void_p), a.size))

    def variable_names(self):
        """TF names of every trainable variable of the graph (slim resnet_v1_<depth> of the loaded weights + the deconv heads)."""
        from .synthetic import conv_specs
        names = []
        for scope, *_ in conv_specs(self.net_type):
            names += [scope + "/weights", scope + "/BatchNorm/gamma", scope + "/BatchNorm/beta"]
        for head in ["part_pred"] + (["locref_pred"] if self.location_refinement else []):
            names += ["pose/%s/block4/weights" % head, "pose/%s/block4/biases" % head]
        return names

    def save_checkpoint(self, path):
        """All trainable variables and their Momentum accumulators under TF names -> .npz (Saver.save, fitdgp.py:830-839)."""
        out = {}
        for n in self.variable_names():
            out[n] = self.get_variable(n)
            if getattr(self, "_train", False):
                out["momentum::" + n] = self.get_variable(n, "momentum")
        np.savez(path, **out)

    def save_tf_checkpoint(self, prefix, with_momentum=True, global_step=None):
        """``saver.save(sess, prefix)`` (fitdgp.py:830-839) as a TensorFlow checkpoint bundle: every trainable variable, the
        frozen moving statistics and (like the reference's full Saver) the MomentumOptimizer slots ``<var>/Momentum``."""
        from . import tf_checkpoint
        out = dict(getattr(self, "_frozen", {}))
        for n in self.variable_names():
            out[n] = self.get_variable(n)
            if with_momentum and getattr(self, "_train", False):
                out[n + "/Momentum"] = self.get_variable(n, "momentum")
        if global_step is not None:
            out["global_step"] = np.array(int(global_step), dtype=np.int64)
        tf_checkpoint.write_checkpoint(prefix, out)

    def load_checkpoint(self, path):
        """Resume from save_checkpoint (the frozen moving statistics stay as loaded by load_weights)."""
        with np.load(path) as z:
            for k in z.files:
                if k.startswith("momentum::"):
                    self.set_variable(k[len("momentum::"):], z[k], "momentum")
                else:
                    self.set_variable(k, z[k], "value")

    # ------------------------------------------------------------------ test hooks
    def keep_activations(self, enable=True):
        self._check(self.lib.dgp_debug_keep_activations(self.h, int(enable)))

    def get_activation(self, end_point):
        shape = (C.c_int64 * 4)()
        self._check(self.lib.dgp_debug_get_activation(self.h, end_point.encode(), None, 0, shape))
        n = int(np.prod(list(shape)))
        out = np.empty(n, np.float32)
        self._check(self.lib.dgp_debug_get_activation(self.h, end_point.encode(), out.ctypes.data_as(C.c_void_p), n, shape))
        return out.reshape(tuple(shape))

    def conv2d(self, x, w_hwio, stride=1, dilation=1, pad_mode=0, scale=None, shift=None, residual=None, res_sub=1,
               relu=False, out_f32=False, block_n=0):
        """One conv through the tcgen05 implicit-GEMM kernel. x: bf16 cuda NHWC; w_hwio: float32 ndarray HWIO."""
        x = x.contiguous()
        N, H, W, Cin = x.shape
        w = np.ascontiguousarray(w_hwio, dtype=np.float32)
        R, S, _, Cout = w.shape
        if pad_mode == 2:
            Ho = (H - ((R - 1) * dilation + 1)) // stride + 1
            Wo = (W - ((S - 1) * dilation + 1)) // stride + 1
        else:
            Ho, Wo = -(-H // stride), -(-W // stride)
        if x.dtype != self.act_dtype:
            raise ValueError("x must be %s for this engine" % self.act_dtype)
        out = torch.empty((N, Ho, Wo, Cout), dtype=torch.float32 if out_f32 else self.act_dtype, device=x.device)
        sc = np.ascontiguousarray(scale, dtype=np.float32) if scale is not None else None
        sh = np.ascontiguousarray(shift, dtype=np.float32) if shift is not None else None
        res_H = res_W = 0
        if residual is not None:
            residual = residual.contiguous()
            res_H, res_W = residual.shape[1], residual.shape[2]
        self._check(self.lib.dgp_conv2d(
            self.h, _ptr(x), N, H, W, Cin, w.ctypes.data_as(C.c_void_p), R, S, Cout, stride, dilation, pad_mode,
            sc.ctypes.data_as(C.c_void_p) if sc is not None else None,
            sh.ctypes.data_as(C.c_void_p) if sh is not None else None,
            _ptr(residual), res_sub, res_H, res_W, int(relu), _ptr(out), int(out_f32), int(block_n), _stream(x.device)))
        return out

    def conv2d_wgrad(self, x, dy, R, stride=1, dilation=1, pad_mode=0, dbg=None):
        """Weight gradient of one conv through the tcgen05 wgrad GEMM: x (N,H,W,Cin), dy (N,P,Q,Cout) 16-bit NHWC ->
        float32 (Cout, R*R*Cin) in the kernel's weight layout (tap-major, then input channel)."""
        x = x.contiguous()
        dy = dy.contiguous()
        N, H, W, Cin = x.shape
        Cout = dy.shape[-1]
        if x.dtype != self.act_dtype or dy.dtype != self.act_dtype:
            raise ValueError("x and dy must be %s for this engine" % self.act_dtype)
        dw = torch.empty((Cout, R * R * Cin), dtype=torch.float32, device=x.device)
        d3 = (C.c_int32 * 3)(*[int(v) for v in dbg]) if dbg is not None else None
        self._check(self.lib.dgp_conv2d_wgrad(self.h, _ptr(x), N, H, W, Cin, _ptr(dy), R, R, Cout, stride, dilation, pad_mode,
                                              _ptr(dw), d3, _stream(x.device)))
        return dw

    def marker_indices(self, visible_frames, hidden_frames, joint_loc, nt):
        """gen_idx_chunk on the device (dgp_marker_indices).  Returns int32 CUDA tensors (visible_marker, hidden_marker,
        visible_marker_in_targets), already cut to their lengths (one 8-byte read-back of the two counts)."""
        dev = self.device
        vf = torch.as_tensor(np.asarray(visible_frames, dtype=np.int32)).to(dev)
        hf = torch.as_tensor(np.asarray(hidden_frames, dtype=np.int32)).to(dev)
        jl = torch.as_tensor(np.ascontiguousarray(np.asarray(joint_loc, dtype=np.float64).reshape(-1, self.nj, 2))).to(dev)
        cap = max(int(nt) * self.nj, 1)
        vm = torch.empty(cap, dtype=torch.int32, device=dev)
        hm = torch.empty(cap, dtype=torch.int32, device=dev)
        vit = torch.empty(cap, dtype=torch.int32, device=dev)
        cnt = torch.zeros(2, dtype=torch.int32, device=dev)
        self._check(self.lib.dgp_marker_indices(self.h, _ptr(vf) if vf.numel() else None, vf.numel(), _ptr(hf) if hf.numel() else None,
                                                hf.numel(), _ptr(jl) if jl.numel() else None, int(nt), _ptr(vm), _ptr(hm), _ptr(vit),
                                                _ptr(cnt), _stream(dev)))
        nv, nh = [int(x) for x in cnt.cpu().tolist()]
        return vm[:nv], hm[:nh], vit[:nv]

    def side_stream(self):
        """A second stream on the engine's device for feeders that may run beside the training step (learn_wt)."""
        if getattr(self, "_side_stream", None) is None:
            self._side_stream = torch.cuda.Stream(device=self.device)
        return self._side_stream

    def learn_wt(self, frames):
        """Farneback flow magnitude |u| + |v| per consecutive frame pair (dgp_learn_wt): frames uint8 cuda (T,H,W,3) ->
        float32 cuda (T-1,H,W), the `vector_field_tf` feed of the temporal clique."""
        if frames.dtype != torch.uint8 or not frames.is_cuda or frames.dim() != 4 or frames.shape[-1] != 3:
            raise ValueError("frames must be a uint8 CUDA tensor (T,H,W,3)")
        frames = frames.contiguous()
        T, H, W, _ = frames.shape
        out = torch.empty((max(T - 1, 0), H, W), dtype=torch.float32, device=frames.device)
        if T > 1:
            self._check(self.lib.dgp_learn_wt(self.h, _ptr(frames), T, H, W, _ptr(out), _stream(frames.device)))
        return out

    def motion_energy_sums(self, frames):
        """Exact byte sums of (frames[t] - frames[t-1]) mod 256 per frame (dgp_motion_energy): frames uint8 cuda (T,...)."""
        if frames.dtype != torch.uint8 or not frames.is_cuda:
            raise ValueError("frames must be a uint8 CUDA tensor")
        frames = frames.contiguous()
        T = frames.shape[0]
        sums = torch.zeros((T,), dtype=torch.int64, device=frames.device)
        if T:
            self._check(self.lib.dgp_motion_energy(self.h, _ptr(frames), T, frames[0].numel(), _ptr(sums), _stream(frames.device)))
        return sums

    PROFILE_KINDS = ("prep_s2d", "conv_gemm", "maxpool", "deconv_col2im", "softargmax", "dgrad_gemm", "wgrad_gemm",
                     "bwd_bandwidth")

    def set_profiling(self, enable=True):
        """True / 1: CUDA events around every launch; 2: one event pair around every run of same-kind launches."""
        self._check(self.lib.dgp_set_profiling(self.h, int(enable)))

    def get_profile(self):
        """{kind: (total_ms, launches)} since the last call (synchronises the device)."""
        n = len(self.PROFILE_KINDS)
        ms = (C.c_double * n)()
        cnt = (C.c_int64 * n)()
        self._check(self.lib.dgp_get_profile(self.h, ms, cnt, n))
        return {k: (ms[i], int(cnt[i])) for i, k in enumerate(self.PROFILE_KINDS)}

    def get_profile_records(self, max_records=65536):
        """[(kind, ms)] per launch, in launch order, since the last call (synchronises the device)."""
        ms = (C.c_float * max_records)()
        kind = (C.c_int32 * max_records)()
        n = C.c_int(0)
        self._check(self.lib.dgp_get_profile_records(self.h, ms, kind, max_records, C.byref(n)))
        return [(self.PROFILE_KINDS[kind[i]] if 0 <= kind[i] < len(self.PROFILE_KINDS) else str(kind[i]), ms[i]) for i in range(n.value)]

    def launch_count(self):
        return int(self.lib.dgp_launch_count(self.h))

    def num_sms(self):
        return int(self.lib.dgp_num_sms(self.h))
