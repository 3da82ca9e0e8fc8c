"""ctypes binding of libqwen3tts_b200.so (C ABI declared in include/qwen3tts_b200.h).

The product path has NO CPU fallback: if the CUDA library is missing or fails to load, importing the engine
raises immediately.
"""
import ctypes as C
import os

from . import build as _build

MAXB = 32


class StackCfg(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("hidden_size", "num_layers", "num_heads", "num_kv_heads", "head_dim",
                                          "intermediate_size", "vocab_size")] + [("rms_eps", C.c_float)]


class EngineCfg(C.Structure):
    _fields_ = [("talker", StackCfg), ("cp", StackCfg), ("num_code_groups", C.c_int32),
                ("has_cp_projection", C.c_int32), ("codec_eos_token_id", C.c_int32), ("max_batch", C.c_int32),
                ("max_ctx", C.c_int32), ("device", C.c_int32)]


class Sampling(C.Structure):
    _fields_ = [("do_sample", C.c_int32), ("top_k", C.c_int32), ("top_p", C.c_float), ("temperature", C.c_float),
                ("repetition_penalty", C.c_float), ("subtalker_dosample", C.c_int32), ("subtalker_top_k", C.c_int32),
                ("subtalker_top_p", C.c_float), ("subtalker_temperature", C.c_float), ("min_new_tokens", C.c_int32),
                ("suppress_eos", C.c_int32), ("seed", C.c_uint64)]


class CodecCfg(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("codebook_size", "codebook_dim", "hidden_size", "latent_dim", "num_heads",
                                          "num_kv_heads", "head_dim", "sliding_window", "intermediate_size",
                                          "num_layers", "num_quantizers")] + \
               [("n_upsample_rates", C.c_int32), ("upsample_rates", C.c_int32 * 8),
                ("n_upsampling_ratios", C.c_int32), ("upsampling_ratios", C.c_int32 * 8),
                ("decoder_dim", C.c_int32), ("rms_eps", C.c_float), ("rope_theta", C.c_float),
                ("max_frames", C.c_int32), ("max_batch", C.c_int32), ("device", C.c_int32)]


class CodecEncCfg(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("num_filters", "kernel_size", "last_kernel_size", "residual_kernel_size",
                                          "compress", "n_ratios")] + \
               [("ratios", C.c_int32 * 8)] + \
               [(n, C.c_int32) for n in ("hidden_size", "num_layers", "num_heads", "head_dim", "intermediate_size",
                                          "sliding_window")] + \
               [("norm_eps", C.c_float)] + \
               [(n, C.c_int32) for n in ("codebook_size", "codebook_dim", "num_semantic_quantizers", "num_quantizers",
                                          "downsample_stride", "max_frames", "device")]


class SpkCfg(C.Structure):
    _fields_ = [("mel_dim", C.c_int32), ("enc_dim", C.c_int32), ("n_blocks", C.c_int32), ("channels", C.c_int32 * 8),
                ("kernel_sizes", C.c_int32 * 8), ("dilations", C.c_int32 * 8), ("attention_channels", C.c_int32),
                ("res2net_scale", C.c_int32), ("se_channels", C.c_int32), ("n_fft", C.c_int32), ("hop", C.c_int32),
                ("win", C.c_int32), ("device", C.c_int32)]


class TapGemmDesc(C.Structure):
    """q3_tap_gemm_desc: one tap-GEMM launch through the test hook q3_debug_tap_gemm."""
    _fields_ = [("a", C.c_void_p)] + [(n, C.c_int32) for n in ("B", "T", "K", "a_rows", "a_row0")] + \
               [("a_bs", C.c_int64), ("w", C.c_void_p)] + [(n, C.c_int32) for n in ("N", "Kp", "ntaps")] + \
               [("shifts", C.c_int32 * 8)] + [(n, C.c_int32) for n in ("bn", "act", "cmod")] + \
               [(n, C.c_void_p) for n in ("bias", "scale", "snake_ea", "snake_ib", "resid")] + \
               [("resid_bs", C.c_int64), ("out_raw", C.c_void_p), ("raw_bs", C.c_int64), ("out_act", C.c_void_p),
                ("act_bs", C.c_int64), ("max_ctas", C.c_int32)]


# every symbol include/qwen3tts_b200.h declares (tests/test_abi.py checks the header against this list)
AR_SYMBOLS = ["q3_abi_version", "q3_last_error", "q3_engine_create", "q3_engine_destroy", "q3_engine_load_tensor",
              "q3_engine_finalize", "q3_prefill", "q3_decode", "q3_get_progress", "q3_set_debug",
              "q3_algorithmic_bytes", "q3_set_profile", "q3_describe_frame_program", "q3_debug_time_phases", "q3_debug_set_skip",
              "q3_session_begin", "q3_admit", "q3_release_slots", "q3_append_trailing", "q3_set_hidden_capture"]
CODEC_SYMBOLS = ["q3_codec_create", "q3_codec_destroy", "q3_codec_load_tensor", "q3_codec_finalize",
                 "q3_codec_forward", "q3_codec_total_upsample", "q3_codec_last_launch_count", "q3_codec_debug_capture",
                 "q3_debug_tap_gemm",
                 "q3_codec_stream_open", "q3_codec_stream_step", "q3_codec_stream_reset", "q3_codec_stream_position", "q3_codec_stream_close",
                 "q3_codec_enc_create", "q3_codec_enc_destroy", "q3_codec_enc_load_tensor", "q3_codec_enc_finalize",
                 "q3_codec_enc_encode", "q3_codec_enc_frames", "q3_codec_enc_hop", "q3_codec_enc_last_launch_count",
                 "q3_codec_enc_debug_capture",
                 "q3_spk_create", "q3_spk_destroy", "q3_spk_load_tensor", "q3_spk_finalize", "q3_spk_frames", "q3_spk_mel",
                 "q3_spk_embed", "q3_spk_last_launch_count"]

_lib = None


def lib_path():
    return _build.LIB_PATH


def load():
    """Load (building first if the in-tree .so is stale/missing and nvcc is present)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    try:
        # no-op when lib/build.stamp matches the digest of csrc/ + include/ + flags; rebuilds a stale or missing .so
        path = _build.build(force=bool(os.environ.get("Q3_REBUILD")))
    except Exception as e:
        if not os.path.exists(path):
            raise
        import warnings
        warnings.warn(f"qwen3tts_b200: could not rebuild ({e!r}); loading the existing {path}", RuntimeWarning)
    try:
        import torch  # noqa: F401  (makes sure libcudart.so.12 is already mapped)
    except Exception:
        pass
    lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    lib.q3_abi_version.restype = C.c_int
    lib.q3_last_error.restype = C.c_char_p
    lib.q3_engine_create.argtypes = [C.POINTER(EngineCfg), C.POINTER(vp)]
    lib.q3_engine_destroy.argtypes = [vp]
    lib.q3_engine_destroy.restype = None
    lib.q3_engine_load_tensor.argtypes = [vp, C.c_char_p, vp, i64, i64]
    lib.q3_engine_finalize.argtypes = [vp]
    lib.q3_prefill.argtypes = [vp, i32, vp, C.POINTER(i32), vp, C.POINTER(i32), i32, vp, C.POINTER(Sampling), vp]
    lib.q3_decode.argtypes = [vp, i32, vp, i32, vp]
    lib.q3_session_begin.argtypes = [vp, i32, i32, vp, C.POINTER(Sampling), vp]
    lib.q3_release_slots.argtypes = [vp, i32, C.POINTER(i32), vp]
    lib.q3_append_trailing.argtypes = [vp, i32, vp, i32, vp]
    lib.q3_set_hidden_capture.argtypes = [vp, vp, i32]
    lib.q3_admit.argtypes = [vp, i32, C.POINTER(i32), C.POINTER(C.c_uint32), vp, C.POINTER(i32), vp, C.POINTER(i32), i32, vp]
    lib.q3_get_progress.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    lib.q3_set_debug.argtypes = [vp, vp, i32, vp, vp]
    lib.q3_set_profile.argtypes = [vp, vp]
    lib.q3_describe_frame_program.argtypes = [vp, C.POINTER(i32), i32]
    lib.q3_debug_set_skip.argtypes = [vp, i32]
    lib.q3_debug_time_phases.argtypes = [vp, i32, i32, i32, C.POINTER(C.c_float), vp]
    lib.q3_algorithmic_bytes.argtypes = [vp, i32, i32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    if hasattr(lib, "q3_codec_create"):
        lib.q3_codec_create.argtypes = [C.POINTER(CodecCfg), C.POINTER(vp)]
        lib.q3_codec_destroy.argtypes = [vp]
        lib.q3_codec_destroy.restype = None
        lib.q3_codec_load_tensor.argtypes = [vp, C.c_char_p, vp, C.POINTER(i64), i32]
        lib.q3_codec_finalize.argtypes = [vp]
        lib.q3_codec_forward.argtypes = [vp, vp, i32, i32, vp, vp]
        lib.q3_codec_stream_open.argtypes = [vp, i32, i32, C.POINTER(vp)]
        lib.q3_codec_stream_step.argtypes = [vp, vp, i32, vp, vp]
        lib.q3_codec_stream_reset.argtypes = [vp, vp]
        lib.q3_codec_stream_position.argtypes = [vp]
        lib.q3_codec_stream_close.argtypes = [vp]
        lib.q3_codec_stream_close.restype = None
        lib.q3_codec_total_upsample.argtypes = [vp]
        lib.q3_codec_last_launch_count.argtypes = [vp]
        lib.q3_codec_debug_capture.argtypes = [vp, i32, vp, i64]
        lib.q3_debug_tap_gemm.argtypes = [C.POINTER(TapGemmDesc), vp]
        lib.q3_codec_enc_create.argtypes = [C.POINTER(CodecEncCfg), C.POINTER(vp)]
        lib.q3_codec_enc_destroy.argtypes = [vp]
        lib.q3_codec_enc_destroy.restype = None
        lib.q3_codec_enc_load_tensor.argtypes = [vp, C.c_char_p, vp, C.POINTER(i64), i32]
        lib.q3_codec_enc_finalize.argtypes = [vp]
        lib.q3_codec_enc_encode.argtypes = [vp, vp, i32, i32, vp, vp]
        lib.q3_codec_enc_frames.argtypes = [vp, i32]
        lib.q3_codec_enc_hop.argtypes = [vp]
        lib.q3_codec_enc_last_launch_count.argtypes = [vp]
        lib.q3_codec_enc_debug_capture.argtypes = [vp, i32, vp, i64]
        lib.q3_spk_create.argtypes = [C.POINTER(SpkCfg), C.POINTER(vp)]
        lib.q3_spk_destroy.argtypes = [vp]
        lib.q3_spk_destroy.restype = None
        lib.q3_spk_load_tensor.argtypes = [vp, C.c_char_p, vp, C.POINTER(i64), i32]
        lib.q3_spk_finalize.argtypes = [vp]
        lib.q3_spk_frames.argtypes = [vp, i32]
        lib.q3_spk_mel.argtypes = [vp, vp, i32, i32, vp, vp]
        lib.q3_spk_embed.argtypes = [vp, vp, i32, i32, vp, i32, vp, vp]
        lib.q3_spk_last_launch_count.argtypes = [vp]
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise RuntimeError("qwen3tts_b200: " + load().q3_last_error().decode())
