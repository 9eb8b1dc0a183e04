"""ctypes binding of include/fo_b200.h.  Loading fails loudly if the library has not been built;
there is no Python/CPU fallback for any entry point."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FO_B200_LIB", os.path.join(HERE, "libfo_b200.so"))   # override: A/B runs of two builds

FO_F32, FO_BF16, FO_I16 = 0, 1, 2


class FoConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "feat_dim", "d_model", "n_heads", "ffn_dim", "n_layers", "chunk_size", "left_chunks",
        "input_layer_linear", "pos_max_len", "llm_dim", "adapter_kernel", "adapter_gelu",
        "has_encoder", "has_adapter", "sample_rate", "frame_len", "frame_shift", "frames_per_chunk",
        "context_frames", "max_sessions", "max_stream_frames", "ffn_conv_kernel", "adapter_batchnorm", "adapter_type",
        "post_norm", "concat_after", "ffn_multi_conv")]


class FoStats(C.Structure):
    _fields_ = [(n, C.c_int64) for n in (
        "stream_steps", "session_chunks", "offline_calls", "offline_frames", "kernel_launches",
        "sessions_in_use", "device_bytes", "graph_replays", "act_saturations")]


# every symbol include/fo_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_I32P = C.POINTER(C.c_int32)
_I64P = C.POINTER(C.c_int64)
SYMBOLS = {
    "fo_abi_version": (C.c_int, []),
    "fo_last_error": (C.c_char_p, []),
    "fo_create": (C.c_int, [C.POINTER(FoConfig), C.c_int, C.c_int, C.POINTER(_P)]),
    "fo_create_on_sms": (C.c_int, [C.POINTER(FoConfig), C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_P)]),
    "fo_destroy": (C.c_int, [_P]),
    "fo_load_tensor": (C.c_int, [_P, C.c_char_p, _P, _I64P, C.c_int]),
    "fo_finalize_weights": (C.c_int, [_P]),
    "fo_session_alloc": (C.c_int, [_P, C.c_int, _I32P]),
    "fo_session_reset": (C.c_int, [_P, C.c_int, _I32P]),
    "fo_session_free": (C.c_int, [_P, C.c_int, _I32P]),
    "fo_session_get_state": (C.c_int, [_P, C.c_int32, _I64P, _I64P]),
    "fo_session_set_pe_index": (C.c_int, [_P, C.c_int, _I32P, _I64P]),
    "fo_session_set_frames": (C.c_int, [_P, C.c_int32, C.c_int64]),
    "fo_session_export_kv": (C.c_int, [_P, C.c_int32, C.c_int, _P, _P, _I32P]),
    "fo_session_import_kv": (C.c_int, [_P, C.c_int32, C.c_int, _P, _P, C.c_int32]),
    "fo_session_export_adapter_cache": (C.c_int, [_P, C.c_int32, _P, _I32P]),
    "fo_session_import_adapter_cache": (C.c_int, [_P, C.c_int32, _P, C.c_int32]),
    "fo_session_export_adapter_cache_n": (C.c_int, [_P, C.c_int32, C.c_int, _P, _I32P]),
    "fo_session_import_adapter_cache_n": (C.c_int, [_P, C.c_int32, C.c_int, _P, C.c_int32]),
    "fo_session_export_ffn_cache": (C.c_int, [_P, C.c_int32, C.c_int, _P]),
    "fo_session_snapshot_bytes": (C.c_int, [_P, _I64P]),
    "fo_session_save": (C.c_int, [_P, _I32P, C.c_int, _P, _P]),
    "fo_session_restore": (C.c_int, [_P, _I32P, C.c_int, _P, _P]),
    "fo_fbank_stream": (C.c_int, [_P, _I32P, C.c_int, _P, C.c_int, C.c_float, _P, _P]),
    "fo_fbank_offline": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int64, C.c_float, _P, _P]),
    "fo_fbank_offline_packed": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_float, _P, _P]),
    "fo_encode_stream": (C.c_int, [_P, _I32P, C.c_int, _P, C.c_int, _P, _P, _P]),
    "fo_encode_stream_chunks": (C.c_int, [_P, _I32P, C.c_int, C.c_int, _P, C.c_int, _P, _P, _P]),
    "fo_encode_stream_chunks_v": (C.c_int, [_P, _I32P, _I32P, C.c_int, _P, C.c_int, _P, _P, _P]),
    "fo_stream_step": (C.c_int, [_P, _I32P, C.c_int, _P, C.c_int, C.c_float, _P, _P, _P]),
    "fo_stream_steps_v": (C.c_int, [_P, _I32P, _I32P, C.c_int, _P, C.c_int, C.c_float, _P, _P, _P]),
    "fo_fbank_stream_v": (C.c_int, [_P, _I32P, _I32P, C.c_int, _P, C.c_int, C.c_float, _P, _P]),
    "fo_encode_stream_steps_v": (C.c_int, [_P, _I32P, _I32P, C.c_int, _P, C.c_int, _P, _P, _P]),
    "fo_debug_trace_read": (C.c_int, [_P, _P, C.c_int64, _I64P]),
    "fo_debug_sm_ids": (C.c_int, [_P, C.c_int, C.c_int, _P, _P]),
    "fo_debug_plan": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "fo_debug_stack_plan": (C.c_int, [C.c_int] * 9 + [C.POINTER(C.c_int)] * 5),
    "fo_stream_step_async": (C.c_int, [_P, _I32P, C.c_int, _P, C.c_int, C.c_float, _P, _P, _P, C.POINTER(C.c_int64)]),
    "fo_stream_wait": (C.c_int, [_P, C.c_int64]),
    "fo_stream_step_embeds": (C.c_int, [_P, _I32P, C.c_int, _P, C.c_int, C.c_float, _P, _P, C.c_int64, C.c_int64, _P]),
    "fo_handoff_arm": (C.c_int, [_P, C.c_int, _P, C.c_int64, C.c_int64, _P, _P, _P, _P]),
    "fo_encode_offline": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P]),
    "fo_encode_offline_packed": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "fo_encode_offline_packed_pcm": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_float, C.c_int, C.c_int, _P, _P, _P, _P]),
    "fo_adapter_forward": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, _P, _P, _P, _P]),
    "fo_adapter_forward2": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P]),
    "fo_stats": (C.c_int, [_P, C.POINTER(FoStats)]),
    "fo_set_option": (C.c_int, [_P, C.c_char_p, C.c_int64]),
    "fo_get_option": (C.c_int, [_P, C.c_char_p, _I64P]),
    "fo_profile_dump": (C.c_int, [_P, C.c_char_p, C.c_int]),
    "fo_debug_gemm": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                C.POINTER(C.c_float), _P]),
    "fo_debug_attention": (C.c_int, [_P, C.c_int, C.c_int, _I32P, _I32P, _I32P] + [C.c_int] * 7 + [_P, _P, C.c_int, _P, _P, C.c_int,
                                                                                           _P, _P, _P, _P]),
}

FO_ATT_OFFLINE, FO_ATT_PACKED, FO_ATT_STREAM, FO_ATT_CHUNKS = 0, 1, 2, 3

_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """dlopen the in-tree library and bind every declared symbol (AttributeError if one is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "%s is missing: build it with `python -m freeze_omni_b200.build` (or __graft_entry__.build()). "
            "freeze_omni_b200 has no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.fo_abi_version() != 6:
        raise RuntimeError("libfo_b200.so ABI version mismatch")
    _lib = lib
    return lib


class FoError(RuntimeError):
    pass


def check(rc: int) -> None:
    if rc != 0:
        msg = load().fo_last_error()
        raise FoError("fo_b200 error %d: %s" % (rc, msg.decode() if msg else "?"))
