"""ctypes binding of libavh_b200.so (C ABI: include/avh_b200.h).  No torch types cross this boundary.

The product path has no CPU fallback: if the shared library is missing or does not load, importing code
gets a RuntimeError naming the build command.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libavh_b200.so")

AVH_F32, AVH_F16, AVH_BF16, AVH_U8 = 0, 1, 2, 3
AVH_COMPUTE_BF16, AVH_COMPUTE_FP32 = 0, 1
AVH_FUSE_CONCAT, AVH_FUSE_ADD = 0, 1

EXPORTS = [
    "avh_abi_version", "avh_last_error", "avh_create", "avh_destroy", "avh_load_tensor", "avh_finalize_weights",
    "avh_forward", "avh_forward_host", "avh_forward_host_async", "avh_read_stage", "avh_fbank", "avh_add_noise", "avh_gemm_bf16",
    "avh_launch_count", "avh_reset_launch_count", "avh_set_profiling", "avh_profile_json",
    "avh_gemm_set_trace", "avh_set_video_preprocess", "avh_video_preprocess", "avh_drop_host_weights",
    "avh_release_stream", "avh_attention_bf16", "avh_forward_ragged", "avh_encoder_forward", "avh_forward_train", "avh_bn_stats_count", "avh_read_bn_stats", "avh_dropout", "avh_interp_linear", "avh_graph_launch_count",
    "avh_mask_substitute", "avh_compute_logits", "avh_sum_squares", "avh_qformer_forward",
    "avh_encoder_grad_count", "avh_encoder_train_forward", "avh_encoder_backward",
    "avh_encoder_backward_buckets", "avh_grad_bucket_count", "avh_grad_bucket_range", "avh_grad_bucket_wait",
    "avh_refresh_weights_device",
    "avh_tail_grad_count", "avh_tail_train_forward", "avh_full_grad_count", "avh_full_train_forward",
    "avh_set_train_args",
]


class AvhConfig(ctypes.Structure):
    _fields_ = [
        ("encoder_layers", ctypes.c_int32),
        ("encoder_embed_dim", ctypes.c_int32),
        ("encoder_ffn_embed_dim", ctypes.c_int32),
        ("encoder_attention_heads", ctypes.c_int32),
        ("audio_feat_dim", ctypes.c_int32),
        ("modality_fuse", ctypes.c_int32),
        ("layer_norm_first", ctypes.c_int32),
        ("conv_pos", ctypes.c_int32),
        ("conv_pos_groups", ctypes.c_int32),
        ("compute_mode", ctypes.c_int32),
        ("frontend_chunk_frames", ctypes.c_int32),
        ("capture_stages", ctypes.c_int32),
        ("reserved", ctypes.c_int32 * 4),
    ]


class AvhTrainArgs(ctypes.Structure):
    _fields_ = [
        ("dropout_input", ctypes.c_float),
        ("dropout", ctypes.c_float),
        ("activation_dropout", ctypes.c_float),
        ("attention_dropout", ctypes.c_float),
        ("bn_momentum", ctypes.c_float),
        ("seed", ctypes.c_uint64),
        ("layer_skip", ctypes.c_void_p),
    ]


_lib = None


def load():
    """Load (once) and type the shared library."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: the CUDA extension is not built. Run `python -m multimodalvc_b200.build` "
            "(needs nvcc; there is no CPU fallback for this path).")
    lib = ctypes.CDLL(LIB_PATH)
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64
    lib.avh_abi_version.restype = i32
    lib.avh_last_error.restype = ctypes.c_char_p
    lib.avh_create.argtypes = [ctypes.POINTER(AvhConfig), i32, ctypes.POINTER(vp)]
    lib.avh_destroy.argtypes = [vp]
    lib.avh_load_tensor.argtypes = [vp, ctypes.c_char_p, vp, i32, ctypes.POINTER(i64), i32]
    lib.avh_finalize_weights.argtypes = [vp]
    lib.avh_drop_host_weights.argtypes = [vp]
    lib.avh_release_stream.argtypes = [vp, vp]
    lib.avh_forward.argtypes = [vp, vp, i32, vp, i32, ctypes.POINTER(i64), vp, i32, i32, i32, vp, i32, vp]
    lib.avh_forward_ragged.argtypes = [vp, vp, i32, vp, i32, ctypes.POINTER(i64), ctypes.POINTER(ctypes.c_int32), i32, i32, i32, vp,
                                       i32, vp]
    lib.avh_forward_train.argtypes = [vp, vp, i32, vp, i32, ctypes.POINTER(i64), vp, i32, i32, i32, ctypes.POINTER(AvhTrainArgs),
                                      vp, i32, vp]
    lib.avh_set_train_args.argtypes = [vp, ctypes.POINTER(AvhTrainArgs)]
    lib.avh_interp_linear.argtypes = [vp, i32, i32, i32, i32, vp, vp, i32, vp, vp, vp]
    lib.avh_encoder_grad_count.argtypes = [vp, ctypes.POINTER(i64)]
    lib.avh_tail_grad_count.argtypes = [vp, ctypes.POINTER(i64)]
    lib.avh_full_grad_count.argtypes = [vp, i32, i32, ctypes.POINTER(i64)]
    lib.avh_full_train_forward.argtypes = [vp, vp, i32, vp, i32, ctypes.POINTER(i64), vp, i32, i32, ctypes.c_float, ctypes.c_float,
                                           vp, i32, vp]
    lib.avh_tail_train_forward.argtypes = [vp, vp, i32, vp, i32, i32, vp, i32, vp]
    lib.avh_encoder_train_forward.argtypes = [vp, vp, i32, vp, i32, i32, vp, i32, vp]
    lib.avh_encoder_backward.argtypes = [vp, vp, i32, vp, i32, vp, i64, vp]
    lib.avh_encoder_backward_buckets.argtypes = [vp, vp, i32, vp, i32, vp, i32, i64, vp]
    lib.avh_grad_bucket_count.argtypes = [vp, ctypes.POINTER(ctypes.c_int32)]
    lib.avh_grad_bucket_range.argtypes = [vp, i32, ctypes.POINTER(i64), ctypes.POINTER(i64)]
    lib.avh_grad_bucket_wait.argtypes = [vp, i32, vp]
    lib.avh_refresh_weights_device.argtypes = [vp, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_int32),
                                               ctypes.POINTER(i64), i32, vp]
    lib.avh_qformer_forward.argtypes = [vp, vp, i32, vp, ctypes.POINTER(ctypes.c_int32), i32, i32, i32, vp, i32, vp]
    lib.avh_mask_substitute.argtypes = [vp, i32, i32, ctypes.POINTER(i64), i32, i32, i32, vp, vp, i32, vp, vp, i32, vp]
    lib.avh_compute_logits.argtypes = [vp, i32, i64, vp, i32, i64, vp, i64, i32, i32, i32, ctypes.c_float, vp, i64, vp]
    lib.avh_sum_squares.argtypes = [vp, i32, i64, vp, vp]
    lib.avh_dropout.argtypes = [vp, i32, i64, ctypes.c_float, ctypes.c_uint64, ctypes.c_uint32, vp]
    lib.avh_bn_stats_count.argtypes = [vp, ctypes.POINTER(i64)]
    lib.avh_read_bn_stats.argtypes = [vp, vp, i64, vp]
    lib.avh_encoder_forward.argtypes = [vp, vp, i32, vp, i32, i32, i32, vp, i32, vp]
    lib.avh_forward_host.argtypes = [vp, vp, i32, vp, i32, vp, i32, i32, i32, vp, i32, vp]
    lib.avh_forward_host_async.argtypes = [vp, vp, i32, vp, i32, vp, i32, i32, i32, vp, i32, vp]
    lib.avh_read_stage.argtypes = [vp, ctypes.c_char_p, vp, i64, vp]
    lib.avh_fbank.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp, vp]
    lib.avh_add_noise.argtypes = [vp, vp, i32, vp, i64, ctypes.c_float, vp, vp, vp]
    lib.avh_gemm_bf16.argtypes = [vp, vp, i64, i32, i32, vp, i32, vp, i32, vp, i32, i32, i32, i32, vp]
    lib.avh_attention_bf16.argtypes = [vp, vp, vp, i64, i32, i32, i32, i32, i32, vp, vp]
    lib.avh_gemm_set_trace.argtypes = [vp]
    lib.avh_set_video_preprocess.argtypes = [vp, i32, i32, ctypes.c_double, ctypes.c_double]
    lib.avh_video_preprocess.argtypes = [vp, i64, i32, i32, i32, ctypes.c_double, ctypes.c_double, vp, i32, vp]
    lib.avh_set_profiling.argtypes = [vp, i32]
    lib.avh_profile_json.argtypes = [vp, ctypes.c_char_p, i64]
    lib.avh_launch_count.restype = i64
    lib.avh_reset_launch_count.restype = None
    lib.avh_graph_launch_count.restype = i64
    for name in EXPORTS:
        fn = getattr(lib, name)
        if fn.restype is ctypes.c_int and name not in ("avh_abi_version",):
            fn.restype = i32
    if lib.avh_abi_version() != 1:
        raise RuntimeError("libavh_b200.so ABI version mismatch; rebuild with `python -m multimodalvc_b200.build --force`")
    _lib = lib
    return lib


def check(status):
    if status != 0:
        msg = load().avh_last_error()
        raise RuntimeError("libavh_b200: " + (msg.decode() if msg else "unknown error"))


def launch_count():
    return int(load().avh_launch_count())


def reset_launch_count():
    load().avh_reset_launch_count()
