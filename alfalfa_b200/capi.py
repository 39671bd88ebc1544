"""ctypes binding of libvp8gpu.so (the C ABI of include/vp8gpu.h).  Plumbing only: all compute is
in the shared library (CUDA kernels + C++ host code).  Importing this module never falls back to a
CPU implementation: if the library is missing the import fails loudly."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VP8GPU_LIB", os.path.join(_HERE, "libvp8gpu.so"))  # override only for tools/phase_profile.py

OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_LOGIC, ERR_CUDA, ERR_NOMEM = 0, -1, -2, -3, -4, -5


class Vp8Error(Exception):
    """base of the error classes mirroring util/exception.hh:76-98"""

    def __init__(self, code, msg=""):
        super().__init__("%s (vp8gpu status %d)" % (msg or self.__class__.__name__, code))
        self.code = code


class Invalid(Vp8Error):
    pass


class Unsupported(Vp8Error):
    pass


class LogicError(Vp8Error):
    pass


class CudaError(Vp8Error):
    pass


_ERR = {ERR_INVALID: Invalid, ERR_UNSUPPORTED: Unsupported, ERR_LOGIC: LogicError, ERR_CUDA: CudaError,
        ERR_NOMEM: CudaError}


class FrameDesc(C.Structure):
    _fields_ = [("width", C.c_uint16), ("height", C.c_uint16), ("mb_cols", C.c_uint16), ("mb_rows", C.c_uint16),
                ("key_frame", C.c_uint8), ("show_frame", C.c_uint8), ("loop_filter_level", C.c_uint8),
                ("sharpness", C.c_uint8), ("pad0", C.c_uint8 * 4), ("quant", C.c_uint16 * 24),
                ("n_tokens", C.c_uint32), ("n_split", C.c_uint32), ("refresh_last", C.c_uint8),
                ("refresh_golden", C.c_uint8), ("refresh_alternate", C.c_uint8), ("copy_to_golden", C.c_uint8),
                ("copy_to_alternate", C.c_uint8), ("pad1", C.c_uint8 * 3)]


class EncodeHeader(C.Structure):
    _fields_ = [("width", C.c_uint16), ("height", C.c_uint16), ("key_frame", C.c_uint8), ("show_frame", C.c_uint8),
                ("y_ac_qi", C.c_uint8), ("loop_filter_level", C.c_uint8), ("sharpness", C.c_uint8),
                ("optimize_token_probs", C.c_uint8), ("pad", C.c_uint8 * 2)]


class EncodeFeatures(C.Structure):
    _fields_ = [("log2_partitions", C.c_uint8), ("segmentation_enabled", C.c_uint8),
                ("update_mb_segmentation_map", C.c_uint8), ("update_segment_feature_data", C.c_uint8),
                ("segment_feature_absolute", C.c_uint8), ("segment_quant", C.c_int8 * 4), ("segment_lf", C.c_int8 * 4),
                ("segment_tree_probs", C.c_uint8 * 3), ("lf_delta_enabled", C.c_uint8), ("lf_delta_update", C.c_uint8),
                ("ref_lf_delta", C.c_int8 * 4), ("mode_lf_delta", C.c_int8 * 4), ("y_dc_delta", C.c_int8),
                ("y2_dc_delta", C.c_int8), ("y2_ac_delta", C.c_int8), ("uv_dc_delta", C.c_int8), ("uv_ac_delta", C.c_int8),
                ("refresh_golden", C.c_uint8), ("refresh_alternate", C.c_uint8), ("refresh_last", C.c_uint8),
                ("refresh_entropy_probs", C.c_uint8), ("copy_to_golden", C.c_uint8), ("copy_to_alternate", C.c_uint8),
                ("sign_bias_golden", C.c_uint8), ("sign_bias_alternate", C.c_uint8), ("pad", C.c_uint8 * 3),
                ("saved_coef_probs", C.c_void_p)]


class Job(C.Structure):
    _fields_ = [("desc", C.POINTER(FrameDesc)), ("mbs", C.c_void_p), ("tokens", C.c_void_p), ("split", C.c_void_p),
                ("refs", C.c_int32 * 3), ("out", C.c_int32)]


MB_DTYPE = np.dtype([("tok_off", "<u4"), ("tok_cnt", "<u2"), ("y_mode", "u1"), ("uv_mode", "u1"),
                     ("ref_frame", "u1"), ("segment_id", "u1"), ("lf_level", "u1"), ("flags", "u1"),
                     ("mv_x", "<i2"), ("mv_y", "<i2"), ("split_idx", "<u4"), ("reserved", "<u4"),
                     ("b_modes", "<u8")])

OPT_DEVICE_TOKENS = 1  # VP8GPU_OPT_DEVICE_TOKENS
QUALITY_BEST, QUALITY_REALTIME = 0, 1  # VP8GPU_QUALITY_* (EncoderQuality, encoder.hh:56-60)

# every symbol include/vp8gpu.h declares: name -> (restype, argtypes)
_vp = C.c_void_p
_pp = C.POINTER(C.c_void_p)
_u8p = C.c_void_p
SYMBOLS = {
    "vp8gpu_ctx_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, _pp]),
    "vp8gpu_ctx_destroy": (None, [_vp]),
    "vp8gpu_last_error": (C.c_char_p, [_vp]),
    "vp8gpu_frame_alloc": (C.c_int, [_vp, C.POINTER(C.c_int32)]),
    "vp8gpu_frame_retain": (C.c_int, [_vp, C.c_int32]),
    "vp8gpu_frame_release": (C.c_int, [_vp, C.c_int32]),
    "vp8gpu_frame_upload": (C.c_int, [_vp, C.c_int32, _u8p, C.c_size_t, _u8p, _u8p, C.c_size_t]),
    "vp8gpu_frame_download": (C.c_int, [_vp, C.c_int32, _u8p, C.c_size_t, _u8p, _u8p, C.c_size_t]),
    "vp8gpu_frame_download_display": (C.c_int, [_vp, C.c_int32, _u8p, C.c_size_t]),
    "vp8gpu_frame_download_display_async": (C.c_int, [_vp, C.c_int32, _u8p, C.c_size_t]),
    "vp8gpu_frame_hash": (C.c_int, [_vp, C.c_int32, C.POINTER(C.c_uint64)]),
    "vp8gpu_ctx_sync": (C.c_int, [_vp]),
    "vp8gpu_host_alloc": (C.c_int, [_pp, C.c_size_t]),
    "vp8gpu_host_free": (None, [_vp]),
    "vp8gpu_decode_parsed": (C.c_int, [_vp, C.c_int, C.POINTER(FrameDesc), _vp, _vp, _vp, C.POINTER(C.c_int32), C.c_int32]),
    "vp8gpu_decode_batch": (C.c_int, [_vp, C.c_int, C.POINTER(Job), C.c_int]),
    "vp8gpu_batch_upload": (C.c_int, [_vp, C.POINTER(Job), C.c_int, _pp]),
    "vp8gpu_batch_run": (C.c_int, [_vp, C.c_int, _vp, C.POINTER(C.c_float)]),
    "vp8gpu_batch_free": (None, [_vp, _vp]),
    "vp8gpu_batches_run": (C.c_int, [_vp, C.c_int, _pp, C.c_int, C.POINTER(C.c_float)]),
    "vp8gpu_batch_run_timed": (C.c_int, [_vp, C.c_int, _vp, C.POINTER(C.c_float)]),
    "vp8gpu_launch_count": (C.c_uint64, [_vp]),
    "vp8gpu_frames_in_use": (C.c_int, [_vp]),
    "vp8gpu_state_create": (C.c_int, [C.c_int, C.c_int, _pp]),
    "vp8gpu_state_clone": (C.c_int, [_vp, _pp]),
    "vp8gpu_state_destroy": (None, [_vp]),
    "vp8gpu_state_equal": (C.c_int, [_vp, _vp]),
    "vp8gpu_state_hash": (C.c_uint64, [_vp]),
    "vp8gpu_state_serialize": (C.c_size_t, [_vp, _u8p, C.c_size_t]),
    "vp8gpu_state_deserialize": (C.c_int, [C.c_char_p, C.c_size_t, _pp]),
    "vp8gpu_frame_bytes": (C.c_size_t, [_vp]),
    "vp8gpu_frame_export": (C.c_int, [_vp, C.c_int32, _vp, C.c_size_t]),
    "vp8gpu_frame_import": (C.c_int, [_vp, C.c_int32, _vp, C.c_size_t]),
    "vp8gpu_parsed_create": (C.c_int, [_pp]),
    "vp8gpu_parsed_destroy": (None, [_vp]),
    "vp8gpu_parsed_desc": (C.POINTER(FrameDesc), [_vp]),
    "vp8gpu_parsed_mbs": (_vp, [_vp]),
    "vp8gpu_parsed_tokens": (_vp, [_vp]),
    "vp8gpu_parsed_split": (_vp, [_vp]),
    "vp8gpu_parse_frame": (C.c_int, [_vp, C.c_char_p, C.c_size_t, _vp]),
    "vp8gpu_parsed_keep_labels": (C.c_int, [_vp, C.c_int]),
    "vp8gpu_parsed_serialize": (C.c_int, [_vp, _vp, C.c_size_t, C.POINTER(C.c_size_t)]),
    "vp8gpu_parse_frame_device": (C.c_int, [_vp, _vp, C.c_char_p, C.c_size_t, _vp]),
    "vp8gpu_ctx_set_option": (C.c_int, [_vp, C.c_int, C.c_int]),
    "vp8gpu_decoder_set_device_tokens": (C.c_int, [_vp, C.c_int]),
    "vp8gpu_decoder_create": (C.c_int, [_vp, _pp]),
    "vp8gpu_decoder_create_from": (C.c_int, [_vp, _vp, C.POINTER(C.c_int32), _pp]),
    "vp8gpu_decoder_clone": (C.c_int, [_vp, _pp]),
    "vp8gpu_decoder_destroy": (None, [_vp]),
    "vp8gpu_decoder_decode": (C.c_int, [_vp, C.c_char_p, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int32)]),
    "vp8gpu_decoder_decode_parsed": (C.c_int, [_vp, _vp, C.POINTER(C.c_int), C.POINTER(C.c_int32)]),
    "vp8gpu_decoder_state": (_vp, [_vp]),
    "vp8gpu_decoder_references": (C.c_int, [_vp, C.POINTER(C.c_int32)]),
    "vp8gpu_decoder_lane": (C.c_int, [_vp]),
    "vp8gpu_decoder_equal": (C.c_int, [_vp, _vp, C.POINTER(C.c_int)]),
    "vp8gpu_encoder_create": (C.c_int, [_vp, _pp]),
    "vp8gpu_encoder_destroy": (None, [_vp]),
    "vp8gpu_encoder_clone": (C.c_int, [_vp, _pp]),
    "vp8gpu_encoder_create_from_decoder": (C.c_int, [_vp, _vp, _pp]),
    "vp8gpu_encoder_export_decoder": (C.c_int, [_vp, _pp]),
    "vp8gpu_encoder_minihash": (C.c_int, [_vp, C.POINTER(C.c_uint32)]),
    "vp8gpu_encoder_set_two_pass": (C.c_int, [_vp, C.c_int]),
    "vp8gpu_encoder_set_quality": (C.c_int, [_vp, C.c_int]),
    "vp8gpu_encoder_update_residues": (C.c_int, [_vp, _u8p, C.c_size_t, _u8p, _u8p, C.c_size_t, _vp, C.c_int, C.c_int,
                                                 _u8p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "vp8gpu_encoder_reencode_as_interframe": (C.c_int, [_vp, _u8p, C.c_size_t, _u8p, _u8p, C.c_size_t, _vp, C.c_int,
                                                        _u8p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "vp8gpu_encoder_write_frame": (C.c_int, [_vp, _vp, _u8p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "vp8gpu_parsed_y_ac_qi": (C.c_int, [_vp]),
    "vp8gpu_encoder_set_writer": (C.c_int, [_vp, C.c_int]),
    "vp8gpu_encoder_encode_with_quantizer": (C.c_int, [_vp, _u8p, C.c_size_t, _u8p, _u8p, C.c_size_t, C.c_int, _u8p, C.c_size_t,
                                                       C.POINTER(C.c_size_t)]),
    "vp8gpu_encoder_encode_with_target_size": (C.c_int, [_vp, _u8p, C.c_size_t, _u8p, _u8p, C.c_size_t, C.c_size_t, _u8p,
                                                         C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_int)]),
    "vp8gpu_encoder_reconstruction": (C.c_int, [_vp, C.POINTER(C.c_int32)]),
    "vp8gpu_encoder_encode_with_minimum_ssim": (C.c_int, [_vp, _u8p, C.c_size_t, _u8p, _u8p, C.c_size_t, C.c_double, _u8p,
                                                          C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_int)]),
    "vp8gpu_encoder_estimate_frame_size": (C.c_int, [_vp, _u8p, C.c_size_t, _u8p, _u8p, C.c_size_t, C.c_int,
                                                     C.POINTER(C.c_size_t)]),
    "vp8gpu_decoder_serialize": (C.c_int, [_vp, _vp, C.c_size_t, C.POINTER(C.c_size_t)]),
    "vp8gpu_decoder_deserialize": (C.c_int, [_vp, C.c_char_p, C.c_size_t, _pp]),
    "vp8gpu_decoder_hash": (C.c_int, [_vp, C.POINTER(C.c_uint64)]),
    "vp8gpu_encoder_stats": (C.c_int, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vp8gpu_encoder_timeline": (C.c_int, [_vp, C.POINTER(C.c_double), C.c_int]),
    "vp8gpu_frame_ssim": (C.c_int, [_vp, C.c_int32, C.c_int32, C.POINTER(C.c_double)]),
    "vp8gpu_serialize_frame": (C.c_int, [C.POINTER(EncodeHeader), _vp, _vp, _vp, _vp, C.c_size_t, C.POINTER(C.c_size_t)]),
    "vp8gpu_serialize_frame_ex": (C.c_int, [C.POINTER(EncodeHeader), C.POINTER(EncodeFeatures), _vp, _vp, _vp, _vp, C.c_size_t,
                                            C.POINTER(C.c_size_t)]),
    "vp8gpu_comm_unique_id": (C.c_int, [_u8p]),
    "vp8gpu_comm_create": (C.c_int, [_vp, C.c_int, C.c_int, _u8p, _pp]),
    "vp8gpu_comm_destroy": (None, [_vp]),
    "vp8gpu_comm_broadcast_frames": (C.c_int, [_vp, C.c_int, C.c_int, C.POINTER(C.c_int32), C.c_int]),
    "vp8gpu_comm_broadcast_bytes": (C.c_int, [_vp, C.c_int, _vp, C.c_size_t]),
    "vp8gpu_comm_rank": (C.c_int, [_vp]),
    "vp8gpu_comm_size": (C.c_int, [_vp]),
    "vp8gpu_decode_ivf_stats": (None, [_vp, C.POINTER(C.c_double)]),
    "vp8gpu_decode_ivf": (C.c_int, [_vp, C.c_char_p, C.c_size_t, C.c_int, _u8p, C.c_size_t, C.POINTER(C.c_uint32),
                                    C.POINTER(C.c_uint32)]),
}

_lib = None


def lib():
    """load libvp8gpu.so (raises if it has not been built: there is no fallback path)"""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("libvp8gpu.so is not built: run __graft_entry__.build() "
                              "(alfalfa_b200/csrc/build.sh); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc, ctx=None, what=""):
    if rc == OK:
        return
    msg = what
    if ctx is not None:
        try:
            msg = "%s: %s" % (what, lib().vp8gpu_last_error(ctx).decode())
        except Exception:
            pass
    raise _ERR.get(rc, Vp8Error)(rc, msg)
