"""ctypes binding of include/kws_b200.h (the C-ABI is the product boundary)."""
from __future__ import annotations

import ctypes
from ctypes import (POINTER, Structure, c_char, c_char_p, c_double, c_float, c_int, c_int32, c_int64,
                    c_size_t, c_void_p)

from . import _build

KWS_OK = 0
KWS_ERR_INVALID_ARGUMENT = -1
KWS_ERR_CUDA = -2
KWS_ERR_ALLOC = -3
KWS_ERR_UNSUPPORTED = -4

PCM_F32 = 0
PCM_I16 = 1

PRECISION_FP32 = 0
PRECISION_TC_FP16 = 1

FRONTEND_FFT = 0
FRONTEND_TC = 1

DECODE_CTC = 0
DECODE_CTC2 = 1
DECODE_STRICT = 2


class InvalidArgumentError(ValueError):
    """What TensorFlow raised as ``errors::InvalidArgument`` in the reference ops."""


class KwsCudaError(RuntimeError):
    pass


class ModelConfig(Structure):
    _fields_ = [("n_mel", c_int32), ("hidden", c_int32), ("num_layers", c_int32),
                ("num_classes", c_int32), ("fft_size", c_int32), ("hop_size", c_int32)]


class ModelWeights(Structure):
    _fields_ = [("mel_basis", c_void_p),
                ("gates_kernel", c_void_p * 4), ("gates_bias", c_void_p * 4),
                ("cand_kernel", c_void_p * 4), ("cand_bias", c_void_p * 4),
                ("fc_w", c_void_p), ("fc_b", c_void_p)]


class OctbitWeights(Structure):
    _fields_ = [("gates_wq", c_void_p * 4), ("gates_scale", c_float * 4), ("gates_obias", c_void_p * 4),
                ("cand_wq", c_void_p * 4), ("cand_scale", c_float * 4), ("cand_obias", c_void_p * 4),
                ("fc_wq", c_void_p), ("fc_scale", c_float), ("fc_obias", c_void_p)]


class DecodeParams(Structure):
    _fields_ = [("mode", c_int32), ("lockout", c_int32), ("thres", c_double), ("loose_thres", c_double)]


class StreamConfig(Structure):
    _fields_ = [("n_streams", c_int64), ("max_chunk", c_int32), ("window_chunks", c_int32),
                ("vad_threshold", c_int32), ("decode_thres", c_double), ("keyword", c_char * 20)]


class ServerConfig(Structure):
    _fields_ = [("n_streams", c_int64), ("waves", c_int32), ("chunk_samples", c_int32), ("use_graphs", c_int32),
                ("stream", StreamConfig)]


class AttentionConfig(Structure):
    _fields_ = [(n, c_int32) for n in ("n_mel", "combine_frame", "hidden", "heads", "num_layers", "ffn",
                                       "num_classes", "use_relu")]


class AttentionWeights(Structure):
    _fields_ = [("w_in", c_void_p), ("b_in", c_void_p)] + \
               [(n, c_void_p * 8) for n in ("w_qkv", "b_qkv", "ln1_g", "ln1_b", "w_ff1", "b_ff1", "w_ff2", "b_ff2",
                                            "ln2_g", "ln2_b")] + \
               [("w_out", c_void_p), ("b_out", c_void_p)]


_SIGNATURES = {
    "kws_last_error": (c_char_p, []),
    "kws_abi_version": (c_int, []),
    "kws_device_count": (c_int, []),
    "kws_model_create": (c_int, [POINTER(ModelConfig), POINTER(ModelWeights), c_int, POINTER(c_void_p)]),
    "kws_model_destroy": (c_int, [c_void_p]),
    "kws_model_set_precision": (c_int, [c_void_p, c_int]),
    "kws_model_get_precision": (c_int, [c_void_p]),
    "kws_model_set_frontend": (c_int, [c_void_p, c_int]),
    "kws_model_get_frontend": (c_int, [c_void_p]),
    "kws_model_set_octbit": (c_int, [c_void_p, POINTER(OctbitWeights)]),
    "kws_model_is_octbit": (c_int, [c_void_p]),
    "kws_num_frames": (c_int, [c_void_p, c_int64]),
    "kws_model_reserve": (c_int, [c_void_p, c_int64, c_int32]),
    "kws_frontend_mel": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_int64, c_void_p, c_void_p]),
    "kws_frontend_mel_lens": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p]),
    "kws_gru_forward": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p,
                                c_void_p, c_void_p, c_void_p]),
    "kws_deploy_forward": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_int64, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_void_p]),
    "kws_deploy_forward_lens": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_int64, c_void_p, c_void_p,
                                        c_void_p, c_void_p, c_void_p, c_void_p]),
    "kws_ctc_decode": (c_int, [c_void_p, c_int64, c_int32, c_int32, c_void_p, POINTER(DecodeParams),
                               c_char_p, c_void_p, c_int32, c_void_p, c_void_p, c_void_p]),
    "kws_edit_distance": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_int32, c_void_p, c_void_p]),
    "kws_stream_create": (c_int, [c_void_p, POINTER(StreamConfig), POINTER(c_void_p)]),
    "kws_stream_destroy": (c_int, [c_void_p]),
    "kws_stream_reset": (c_int, [c_void_p, c_void_p]),
    "kws_stream_step": (c_int, [c_void_p, c_void_p, c_int32, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "kws_stream_step_host": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_void_p]),
    "kws_stream_max_frames": (c_int32, [c_void_p]),
    "kws_stream_state": (c_void_p, [c_void_p]),
    "kws_stream_copy_state": (c_int, [c_void_p, c_void_p, c_void_p]),
    "kws_stream_labels": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_void_p]),
    "kws_stream_record_bytes": (c_int64, [c_void_p]),
    "kws_stream_export": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "kws_stream_import": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "kws_server_create": (c_int, [c_void_p, POINTER(ServerConfig), POINTER(c_void_p)]),
    "kws_server_destroy": (c_int, [c_void_p]),
    "kws_server_info": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int32), POINTER(c_int32)]),
    "kws_server_reset": (c_int, [c_void_p]),
    "kws_server_ingest_slot": (c_void_p, [c_void_p, c_int32]),
    "kws_server_submit": (c_int, [c_void_p, c_int32]),
    "kws_server_wait": (c_int, [c_void_p, c_int32, POINTER(c_void_p), POINTER(c_double)]),
    "kws_server_serve": (c_int, [c_void_p, c_int32, c_int32]),
    "kws_server_stats": (c_int, [c_void_p, c_int, POINTER(c_double), POINTER(c_double), POINTER(c_double),
                                 POINTER(c_int64), POINTER(c_int64)]),
    "kws_server_set_copy_only": (c_int, [c_void_p, c_int]),
    "kws_server_wave_stream": (c_void_p, [c_void_p, c_int32]),
    "kws_server_export": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "kws_server_import": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "kws_octbit_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "kws_octbit_matmul": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_int, c_int, c_int64, c_int64,
                                  c_int64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "kws_octbit_matmul_exact": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_int64, c_int64, c_int64,
                                        c_void_p, c_void_p, c_size_t, c_void_p]),
    "kws_octize_weight": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, POINTER(c_double), c_void_p]),
    "kws_positional_encoding": (c_int, [c_int32, c_int32, c_void_p, c_void_p]),
    "kws_attention_create": (c_int, [POINTER(AttentionConfig), POINTER(AttentionWeights), c_int, POINTER(c_void_p)]),
    "kws_attention_destroy": (c_int, [c_void_p]),
    "kws_attention_frames": (c_int32, [c_void_p, c_int32]),
    "kws_attention_forward": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p]),
    "kws_attention_forward_lens": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "kws_debug_tc_gemm": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "kws_debug_att_linear": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int64, c_int32, c_int32, c_int,
                                     c_int, c_int, c_void_p, c_void_p]),
    "kws_debug_att_core": (c_int, [c_void_p, c_int64, c_int32, c_int32, c_int, c_void_p, c_void_p]),
    "kws_debug_att_core_lens": (c_int, [c_void_p, c_int64, c_int32, c_void_p, c_int32, c_int, c_void_p, c_void_p]),
    "kws_debug_att_add_layernorm": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int,
                                            c_void_p, c_void_p]),
    "kws_debug_att_add_layernorm_lens": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_int32,
                                                 c_int, c_void_p, c_void_p]),
    "kws_debug_tc_timeline": (c_int, [c_int, c_void_p, c_int]),
    "kws_debug_step_timing": (c_int, [c_int, c_void_p, c_void_p]),
    "kws_debug_mel_quads": (c_int, [c_void_p, c_int, c_void_p, c_int]),
}

EXPORTED_SYMBOLS = sorted(_SIGNATURES)

_lib = None


def load():
    """Build (if needed) and load libkws_b200.so; raises ImportError when impossible."""
    global _lib
    if _lib is None:
        path = _build.build()
        try:
            lib = ctypes.CDLL(path)
        except OSError as exc:           # pragma: no cover
            raise ImportError("cannot load %s: %s" % (path, exc))
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)      # AttributeError if the .so is missing a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error() -> str:
    msg = load().kws_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc: int):
    if rc == KWS_OK:
        return
    msg = last_error()
    if rc == KWS_ERR_INVALID_ARGUMENT:
        raise InvalidArgumentError(msg)
    if rc == KWS_ERR_ALLOC:
        raise MemoryError(msg)
    raise KwsCudaError("kws_b200 error %d: %s" % (rc, msg))
