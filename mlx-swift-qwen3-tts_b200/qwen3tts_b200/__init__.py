"""qwen3tts_b200 — Python host of libqwen3tts_b200.so (B200 / sm_100a Qwen3-TTS engine).

`Qwen3TTSPipeline` mirrors the public API of hamptus/mlx-swift-qwen3-tts; `Engine` is the raw C-ABI seam.
There is no CPU path: importing works without a GPU (so symbols can be inspected), computing does not.
"""
from ._abi import (DECODE_BATCHAPI, DECODE_FILE, DECODE_STREAM, DECODE_WHOLE, LIB_PATH, SAMPLE_RATE, SAMPLES_PER_FRAME, Q3Error, lib)
from .engine import CodeStream, Engine, GenRequest, attention_probe, codec_attention_probe, codec_out_conv_probe, codec_rowop_probe, codec_unit_probe, conv_probe, dequantize, mlx_quantize, quantized_matmul, quantized_matmul_tc, safetensors_check, sampler_probe, sampler_slot_probe
from .pipeline import (AudioChunk, DecoderLoadFailed, FileNotFound, ModelNotLoaded, Qwen3TTSError, Qwen3TTSPipeline,
                       Qwen3TTSPipelineConfiguration, StreamingWAVWriter, SyntheticTokenizer, TextChunker)

__all__ = [n for n in dir() if not n.startswith("_")]
