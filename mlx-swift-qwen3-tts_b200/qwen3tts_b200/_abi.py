"""ctypes binding of include/qwen3tts_b200.h — the same symbols the Swift module map binds.

There is NO fallback: if libqwen3tts_b200.so is missing the import fails loudly, and every compute entry point
fails with Q3TTS_ERR_NO_DEVICE when no sm_100 GPU is visible.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("Q3TTS_LIB") or os.path.join(_HERE, "libqwen3tts_b200.so")  # Q3TTS_LIB: A/B measurements of two builds on one box

OK = 0
ERR_FILE_NOT_FOUND, ERR_DECODER_LOAD_FAILED, ERR_MODEL_NOT_LOADED, ERR_BAD_CONFIG, ERR_BAD_WEIGHTS = -1, -2, -3, -4, -5
ERR_CUDA, ERR_INVALID_ARG, ERR_CANCELLED, ERR_NO_DEVICE, ERR_CAPACITY = -6, -7, -8, -9, -10
F32, F16, BF16 = 0, 1, 2
DECODE_WHOLE, DECODE_FILE, DECODE_BATCHAPI, DECODE_STREAM = 0, 1, 2, 3
SAMPLE_RATE = 24000
SAMPLES_PER_FRAME = 1920

i32, i64, u64, f32 = C.c_int32, C.c_int64, C.c_uint64, C.c_float
p_i32, p_f32 = C.POINTER(C.c_int32), C.POINTER(C.c_float)


class Options(C.Structure):
    _fields_ = [("struct_size", i32), ("device", i32), ("cuda_stream", C.c_void_p), ("max_batch", i32), ("kv_capacity", i32),
                ("max_frames", i32), ("use_cuda_graph", i32), ("load_codec", i32), ("load_talker", i32),
                ("codec_max_frames", i32), ("codec_max_batch", i32), ("packed_gemm", i32), ("runtime_quantization", i32), ("lanes", i32), ("reserved", i32 * 5)]


class Info(C.Structure):
    _fields_ = [(n, i32) for n in ("hidden_size", "num_layers", "num_heads", "num_kv_heads", "head_dim", "intermediate_size",
                                   "vocab_size", "text_vocab_size", "text_hidden_size", "cp_hidden_size", "cp_num_layers",
                                   "cp_vocab_size", "num_code_groups", "quant_bits", "quant_group_size", "weight_dtype",
                                   "num_speakers", "has_codec", "codec_num_quantizers", "codec_total_upsample", "model_type",
                                   "codec_eos_id", "codec_pad_id", "max_batch", "kv_capacity", "max_frames")] + \
               [("device_bytes", i64), ("has_audio_encoder", i32), ("audio_encoder_hidden", i32), ("has_speaker_encoder", i32), ("speaker_embedding_dim", i32),
                ("checkpoint_quant_bits", i32), ("reserved", i32 * 3)]


class Request(C.Structure):
    _fields_ = [("struct_size", i32), ("text_ids", p_i32), ("n_text_ids", i32), ("instruct_ids", p_i32), ("n_instruct_ids", i32),
                ("speaker_id", i32), ("speaker_embedding", p_f32), ("speaker_embedding_dim", i32), ("ref_text_ids", p_i32),
                ("n_ref_text_ids", i32), ("ref_codes", p_i32), ("ref_frames", i32), ("temperature", f32), ("top_k", i32),
                ("top_p", f32), ("repetition_penalty", f32), ("max_tokens", i32), ("seed", u64), ("stream_variant", i32),
                ("forced_codes", p_i32), ("n_forced_frames", i32), ("code0_logits_out", p_f32), ("cp_logits_out", p_f32),
                ("logits_capacity_frames", i32), ("keep_invalid_frames", i32), ("reserved", i32 * 6)]


class Timing(C.Structure):
    _fields_ = [("device_ms", C.c_double), ("prefill_ms", C.c_double), ("decode_ms", C.c_double), ("kernel_launches", i64),
                ("graph_replays", i64), ("frames", i64), ("h2d_bytes", i64), ("d2h_bytes", i64), ("weight_bytes_per_frame", i64),
                ("talker_ms", C.c_double), ("codec_flops", i64), ("persistent_launches", i64), ("reserved", i64 * 3)]


# every symbol include/qwen3tts_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "q3tts_abi_version": (i32, []),
    "q3tts_default_options": (None, [C.POINTER(Options)]),
    "q3tts_default_request": (None, [C.POINTER(Request)]),
    "q3tts_create": (i32, [C.c_char_p, C.POINTER(Options), C.POINTER(C.c_void_p)]),
    "q3tts_destroy": (None, [C.c_void_p]),
    "q3tts_last_error": (C.c_char_p, [C.c_void_p]),
    "q3tts_get_info": (i32, [C.c_void_p, C.POINTER(Info)]),
    "q3tts_speaker_name": (i32, [C.c_void_p, i32, C.c_char_p, i32, p_i32]),
    "q3tts_speaker_id": (i32, [C.c_void_p, C.c_char_p]),
    "q3tts_clear_cache": (i32, [C.c_void_p]),
    "q3tts_get_timing": (i32, [C.c_void_p, C.POINTER(Timing)]),
    "q3tts_generate_codes": (i32, [C.c_void_p, C.POINTER(Request), p_i32, i32, p_i32]),
    "q3tts_generate_codes_batch": (i32, [C.c_void_p, C.POINTER(Request), i32, C.POINTER(p_i32), i32, p_i32]),
    "q3tts_stream_begin": (i32, [C.c_void_p, C.POINTER(Request), i32, C.POINTER(C.c_void_p)]),
    "q3tts_stream_next": (i32, [C.c_void_p, p_i32, p_i32, p_i32]),
    "q3tts_stream_next_audio": (i32, [C.c_void_p, p_f32, i32, p_i32, p_i32, p_i32, p_i32, p_i32]),
    "q3tts_stream_cancel": (i32, [C.c_void_p]),
    "q3tts_stream_free": (None, [C.c_void_p]),
    "q3tts_decode": (i32, [C.c_void_p, p_i32, i32, i32, p_f32]),
    "q3tts_decode_chunked": (i32, [C.c_void_p, p_i32, i32, i32, i32, i32, p_f32]),
    "q3tts_generate_pcm": (i32, [C.c_void_p, C.POINTER(Request), i32, p_f32, i64, C.POINTER(i64), p_i32]),
    "q3tts_generate_pcm_batch": (i32, [C.c_void_p, C.POINTER(Request), i32, i32, C.POINTER(p_f32), i64, C.POINTER(i64), p_i32]),
    "q3tts_mlx_quantize": (i32, [i32, C.c_void_p, i32, i32, i32, i32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "q3tts_dequantize": (i32, [i32, C.c_void_p, C.c_void_p, C.c_void_p, i32, i32, i32, i32, i32, i32, C.c_void_p]),
    "q3tts_quantized_matmul": (i32, [i32, p_f32, i32, C.c_void_p, C.c_void_p, C.c_void_p, i32, i32, i32, i32, i32, p_f32]),
    "q3tts_quantized_matmul_tc": (i32, [i32, p_f32, i32, C.c_void_p, C.c_void_p, C.c_void_p, i32, i32, i32, i32, i32, p_f32, i32, p_f32, p_f32]),
    "q3tts_conv_probe": (i32, [i32, p_f32, i32, i32, i32, p_f32, p_f32, i32, i32, i32, i32, i32, p_f32, p_f32, p_f32, p_f32, i32, i32, p_f32, p_f32]),
    "q3tts_attention_probe": (i32, [i32, i32, i32, i32, p_f32, i32, i32, i32, p_f32, p_f32, f32, p_f32, p_i32, p_i32, p_i32, i32, i32, p_f32, p_f32,
                                    p_f32]),
    "q3tts_codec_attention_probe": (i32, [i32, i32, p_f32, i32, i32, i32, i32, p_f32, p_f32]),
    "q3tts_codec_unit_probe": (i32, [i32, i32, i32, i32, i32, i32, p_f32, p_f32, p_f32, p_f32, p_f32, p_f32, p_f32, p_f32, p_f32, p_f32, i32, i32,
                                     i32, p_f32, p_f32]),
    "q3tts_codec_out_conv_probe": (i32, [i32, i32, p_f32, i32, i32, i32, p_f32, p_f32, i32, p_f32]),
    "q3tts_codec_rowop_probe": (i32, [i32, i32, p_f32, i32, i32, i32, i32, p_f32, p_f32, f32, p_f32]),
    "q3tts_profile_linear": (i32, [C.c_void_p, i32, i32, i32, C.POINTER(C.c_double), C.POINTER(i64), C.POINTER(i64)]),
    "q3tts_skinny_trace": (i32, [i32, i32, i32, i32, i32, i32, i32, C.POINTER(C.c_uint64), i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32),
                                 C.POINTER(C.c_double)]),
    "q3tts_skinny_trace_q": (i32, [i32, i32, i32, i32, i32, i32, i32, i32, C.POINTER(C.c_uint64), i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32),
                                   C.POINTER(C.c_double)]),
    "q3tts_sample_token": (i32, [C.c_void_p, p_f32, i32, f32, i32, f32, f32, p_i32, i32, u64, u64, p_i32]),
    "q3tts_sampler_probe": (i32, [i32, i32, p_f32, i32, i32, i32, i32, p_f32, p_i32, p_f32, p_f32, C.c_void_p, C.c_void_p, C.c_void_p, p_i32, p_f32]),
    "q3tts_sampler_slot_probe": (i32, [i32, i32, i32, i32, i32, i32, i32, i32, p_f32] + [p_i32] * 11 + [p_f32, p_i32, p_f32, p_f32, C.c_void_p, C.c_void_p, i32,
                                                                                            p_i32, i32, p_f32, i32, i32, p_i32]),
    "q3tts_rvq_embed": (i32, [C.c_void_p, p_i32, i32, i32, p_f32, p_f32, p_i32]),
    "q3tts_encode_reference_audio": (i32, [C.c_void_p, p_f32, i64, p_i32, i32, p_i32, p_i32, p_f32]),
    "q3tts_extract_speaker_embedding": (i32, [C.c_void_p, p_f32, i64, p_f32, i32, p_i32, p_f32]),
    "q3tts_clone": (i32, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "q3tts_safetensors_check": (i32, [C.c_char_p, p_i32, C.POINTER(i64)]),
}

_lib = None


def lib():
    """Load the CUDA library (once).  Raises RuntimeError if it has not been built — there is no CPU path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C mlx-swift-qwen3-tts_b200/csrc`). qwen3tts_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class Q3Error(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"q3tts status {status}: {message}")
        self.status = status
        self.message = message


def check(status: int, handle=None):
    if status != OK:
        msg = lib().q3tts_last_error(handle)
        raise Q3Error(status, msg.decode("utf-8", "replace") if msg else "")
