"""ctypes binding of libdgp_b200.so (C ABI: include/dgp_b200.h).

There is no fallback: if the shared library is missing or the device is not sm_100 every entry point raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DGP_B200_LIB") or os.path.join(_HERE, "libdgp_b200.so")  # env: alternate build

DGP_OK = 0
STATUS_NAMES = {0: "DGP_OK", -1: "DGP_ERR_INVALID", -2: "DGP_ERR_CUDA", -3: "DGP_ERR_UNSUPPORTED",
                -4: "DGP_ERR_STATE", -5: "DGP_ERR_NOMEM"}


class DgpError(RuntimeError):
    def __init__(self, status, message):
        self.status = status
        super().__init__("%s: %s" % (STATUS_NAMES.get(status, status), message))


class DgpConfig(C.Structure):
    _fields_ = [
        ("num_joints", C.c_int32),
        ("location_refinement", C.c_int32),
        ("device", C.c_int32),
        ("stride", C.c_float),
        ("locref_stdev", C.c_float),
        ("mean_pixel", C.c_float * 3),
        ("bn_epsilon", C.c_float),
        ("precision", C.c_int32),
    ]


class DgpLossCfg(C.Structure):
    _fields_ = [("gamma", C.c_float), ("gauss_len", C.c_float), ("lengthscale", C.c_float), ("wt", C.c_float),
                ("wt_max", C.c_float), ("wn_visible", C.c_float), ("wn_hidden", C.c_float),
                ("locref_loss_weight", C.c_float), ("n_frames_total", C.c_float), ("n_visible_frames_total", C.c_float),
                ("gm2", C.c_int32), ("gm3", C.c_int32), ("locref_mse", C.c_int32)]


class DgpLossBatch(C.Structure):
    _fields_ = [("pred_dev", C.c_void_p), ("locref_dev", C.c_void_p), ("nt", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
                ("targets_dev", C.c_void_p), ("nv", C.c_int32), ("locref_map_dev", C.c_void_p),
                ("locref_mask_dev", C.c_void_p), ("visible_marker_dev", C.c_void_p), ("nbv", C.c_int32),
                ("hidden_marker_dev", C.c_void_p), ("nbh", C.c_int32), ("visible_marker_in_targets_dev", C.c_void_p),
                ("edges_dev", C.c_void_p), ("nl", C.c_int32), ("ws_dev", C.c_void_p), ("ws_max_dev", C.c_void_p),
                ("vector_field_dev", C.c_void_p), ("Hin", C.c_int32), ("Win", C.c_int32), ("wt_batch_dev", C.c_void_p),
                ("vector_field_ready_event", C.c_void_p)]


class DgpCyclicSource(C.Structure):
    _fields_ = [("pool", C.c_void_p), ("pool_frames", C.c_int64), ("total_frames", C.c_int64), ("position", C.c_int64),
                ("frame_bytes", C.c_size_t)]


class DgpFrameTransform(C.Structure):
    _fields_ = [("resize_h", C.c_int32), ("resize_w", C.c_int32), ("crop_x0", C.c_int32), ("crop_y0", C.c_int32),
                ("crop_x1", C.c_int32), ("crop_y1", C.c_int32)]


class DgpAugmentParams(C.Structure):
    _fields_ = [("rotate_deg", C.c_double), ("blur_k", C.c_int32), ("blur_angle_deg", C.c_double),
                ("blur_direction", C.c_double), ("drop_p", C.c_double), ("drop_size_percent", C.c_double),
                ("elastic_alpha", C.c_double), ("elastic_sigma", C.c_double), ("seed", C.c_uint64)]


class DgpMarkerStyle(C.Structure):
    _fields_ = [("dotsize", C.c_int32), ("mask_threshold", C.c_double), ("scale_x", C.c_double), ("scale_y", C.c_double),
                ("colors", C.c_void_p), ("edges", C.c_void_p), ("n_edges", C.c_int32), ("skeleton_color", C.c_uint8 * 3),
                ("trailpoints", C.c_int32), ("history", C.c_int32)]


# reader(user, slot, max_frames, &direct) -> frames delivered (0 = end of video, < 0 = error)
FRAME_READER = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_void_p))
# writer(user, frames, n) -> < 0 aborts
FRAME_WRITER = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int)
# packet writer(user, data, sizes, n) -> < 0 aborts
PACKET_WRITER = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int)


# name -> (restype, argtypes); kept in one table so the CPU test-suite can check every exported symbol.
_vp, _i, _f, _sz, _i64p = C.c_void_p, C.c_int, C.c_float, C.c_size_t, C.POINTER(C.c_int64)
SIGNATURES = {
    "dgp_create": (_i, [C.POINTER(DgpConfig), C.POINTER(_vp)]),
    "dgp_destroy": (None, [_vp]),
    "dgp_last_error": (C.c_char_p, [_vp]),
    "dgp_load_weights": (_i, [_vp, C.c_char_p, _vp, _i64p, _i, _i]),
    "dgp_finalize_weights": (_i, [_vp]),
    "dgp_net_depth": (_i, [_vp, C.POINTER(_i)]),
    "dgp_output_dims": (_i, [_i, _i, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "dgp_output_dims_os": (_i, [_i, _i, _i, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "dgp_set_output_stride": (_i, [_vp, _i]),
    "dgp_get_output_stride": (_i, [_vp, C.POINTER(_i)]),
    "dgp_forward": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "dgp_extract_features": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "dgp_prediction_layers": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "dgp_deconv2d": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "dgp_softargmax": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _f, _f, _vp, _vp, _vp, _vp, _vp, _vp]),
    "dgp_softmax_threshold": (_i, [_vp, _vp, _i, _i, _i, _i, _f, _vp, _vp]),
    "dgp_softmax_map": (_i, [_vp, _vp, _i, _i, _i, _i, _f, _f, _vp, _vp]),
    "dgp_loss_forward": (_i, [_vp, C.POINTER(DgpLossCfg), C.POINTER(DgpLossBatch), _vp, _vp, _vp]),
    "dgp_loss_backward": (_i, [_vp, C.POINTER(DgpLossCfg), C.POINTER(DgpLossBatch), _vp, _vp, _vp, _i, _vp]),
    "dgp_soft_pose": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _f, _f, _i, _vp, _vp, _vp]),
    "dgp_locref_targets": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, C.c_double, C.c_double, _vp, _vp, _vp]),
    "dgp_sigmoid": (_i, [_vp, _vp, _vp, _sz, _vp]),
    "dgp_potentials": (_i, [_vp, _vp, _vp, _i, _i, _vp, _i, _vp, _vp, _f, _vp, _vp, _vp, _vp, _vp]),
    "dgp_estimate_pose_host": (_i, [_vp, _vp, _i, _i, _i, _i, _f, _f, _vp, _vp, _vp]),
    "dgp_estimate_pose_stream": (_i, [_vp, _vp, _vp, _i, _i, _i, _f, _f, C.c_int64, _vp, _vp, _vp, _i64p]),
    "dgp_cyclic_reader": (_i, [_vp, _vp, _i, C.POINTER(_vp)]),
    "dgp_transform_dims": (_i, [_i, _i, C.POINTER(DgpFrameTransform), C.POINTER(_i), C.POINTER(_i)]),
    "dgp_resize_coefficients": (_i, [_i, _i, _i, _vp, _vp, _vp]),
    "dgp_resize_crop": (_i, [_vp, _vp, _i, _i, _i, C.POINTER(DgpFrameTransform), _vp, _vp]),
    "dgp_estimate_pose_host_transform": (_i, [_vp, _vp, _i, _i, _i, C.POINTER(DgpFrameTransform), _i, _f, _f, _vp, _vp,
                                              _vp]),
    "dgp_estimate_pose_stream_transform": (_i, [_vp, _vp, _vp, _i, _i, C.POINTER(DgpFrameTransform), _i, _f, _f, C.c_int64,
                                                _vp, _vp, _vp, _i64p]),
    "dgp_draw_markers": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, C.POINTER(DgpMarkerStyle), _vp]),
    "dgp_estimate_pose_stream_render": (_i, [_vp, _vp, _vp, _i, _i, C.POINTER(DgpFrameTransform), _i, _f, _f, C.c_int64,
                                             _vp, _vp, _vp, _i64p, C.POINTER(DgpMarkerStyle), _vp, _vp]),
    "dgp_jpeg_capacity": (C.c_int64, [_i, _i]),
    "dgp_encode_jpeg": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, C.c_int64, _vp, _vp, _vp]),
    "dgp_estimate_pose_stream_render_jpeg": (_i, [_vp, _vp, _vp, _i, _i, C.POINTER(DgpFrameTransform), _i, _f, _f,
                                                  C.c_int64, _vp, _vp, _vp, _i64p, C.POINTER(DgpMarkerStyle), _i, _vp,
                                                  _vp]),
    "dgp_motion_blur_kernel": (_i, [_i, C.c_double, C.c_double, _vp]),
    "dgp_elastic_field": (_i, [_vp, _i, _i, C.c_double, C.c_double, C.c_uint64, _vp, _vp, _vp]),
    "dgp_augment": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, C.POINTER(DgpAugmentParams), _vp, C.c_double, _vp]),
    "dgp_debug_keep_activations": (_i, [_vp, _i]),
    "dgp_debug_get_activation": (_i, [_vp, C.c_char_p, _vp, _sz, _i64p]),
    "dgp_debug_live_resources": (_i, [_i64p, _i64p]),
    "dgp_conv2d": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _i, _i, _i, _i, _vp,
                        _i, _i, _vp]),
    "dgp_conv2d_wgrad": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "dgp_train_enable": (_i, [_vp]),
    "dgp_train_forward_backward": (_i, [_vp, _vp, _i, _i, _i, C.POINTER(DgpLossCfg), C.POINTER(DgpLossBatch), _i, _vp, _vp]),
    "dgp_train_forward": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, C.POINTER(C.c_uint64), _vp]),
    "dgp_train_backward": (_i, [_vp, C.c_uint64, _vp, _vp, _i, _vp]),
    "dgp_optimizer_step": (_i, [_vp, _f, _f, _f, _f, _vp]),
    "dgp_get_param_buffer": (_i, [_vp, C.POINTER(_vp), C.POINTER(_sz)]),
    "dgp_params_changed": (_i, [_vp, _vp]),
    "dgp_get_grad_buffer": (_i, [_vp, C.POINTER(_vp), C.POINTER(_sz)]),
    "dgp_train_set_loss_scale": (_i, [_vp, _f]),
    "dgp_comm_unique_id": (_i, [C.c_char_p]),
    "dgp_comm_init_rank": (_i, [_vp, C.c_char_p, _i, _i]),
    "dgp_attach_comm": (_i, [_vp, _vp]),
    "dgp_comm_world_size": (_i, [_vp]),
    "dgp_allreduce_gradients": (_i, [_vp, _vp, C.POINTER(_f)]),
    "dgp_allreduce_exposed_ms": (_i, [_vp, C.POINTER(_f)]),
    "dgp_get_grad_norm": (_i, [_vp, C.POINTER(_f)]),
    "dgp_train_outputs": (_i, [_vp, _i, _i, _i, C.POINTER(_vp), C.POINTER(_vp)]),
    "dgp_get_variable": (_i, [_vp, C.c_char_p, _i, _vp, _sz, _i64p, C.POINTER(_i)]),
    "dgp_set_variable": (_i, [_vp, C.c_char_p, _i, _vp, _sz]),
    "dgp_set_profiling": (_i, [_vp, _i]),
    "dgp_marker_indices": (_i, [_vp, _vp, _i, _vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "dgp_learn_wt": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "dgp_motion_energy": (_i, [_vp, _vp, _i, C.c_size_t, _vp, _vp]),
    "dgp_get_profile": (_i, [_vp, C.POINTER(C.c_double), _i64p, _i]),
    "dgp_get_profile_records": (_i, [_vp, C.POINTER(C.c_float), C.POINTER(C.c_int32), _i, C.POINTER(C.c_int)]),
    "dgp_crc32c": (C.c_uint32, [_vp, _sz]),
    "dgp_launch_count": (C.c_int64, [_vp]),
    "dgp_num_sms": (_i, [_vp]),
}

_lib = None


def load():
    """dlopen libdgp_b200.so (built by deepgraphpose_b200/build.py or __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libdgp_b200.so is not built (%s). Run `python -m deepgraphpose_b200.build`; "
            "deepgraphpose_b200 has no CPU or PyTorch fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status, handle=None):
    if status != DGP_OK:
        msg = load().dgp_last_error(handle)
        raise DgpError(status, msg.decode() if msg else "")
