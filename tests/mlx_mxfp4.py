"""Test support for MLX mxfp4 checkpoints: the reference dequantisation, the exact 8-bit affine container the engine holds the leaves in,
a quantiser for the checkpoint writer, and the writer.

An mxfp4 leaf (MLX `quantize(w, mode: "mxfp4")`, group 32) is `.weight` uint32 [out, in/8] -- E2M1 code j of a word at bits 4j, LSB first,
the word layout of 4-bit affine leaves -- and `.scales` uint8 [out, in/32], one E8M0 exponent byte e per group of 32; there is no `.biases`.
Element value = LUT[code] * 2^(e - 127).  Doubled, the LUT is the integers -12..12, so the same values are an 8-bit affine group of 32:
q = 2 * LUT[code] + 12, scale = 2^(e - 128), bias = -12 * 2^(e - 128), both held exactly in bf16 for e <= 251.  fp32(scale) * q and
+ fp32(bias) are then exact (powers of two times integers below 2^24), so the affine oracle (`oracle.mlx_quant.dequantize`) computes every
element exactly and rounds it once, as `mxfp4_dequantize` does; the only bit difference is code 8 (-0), which comes out as +0.

The oracle dequantises affine words only, so an mxfp4 checkpoint is written together with its CONTAINER TWIN: the same values as 8-bit
affine leaves of group 32 with bf16 scales and biases.  The oracle runs the twin; the engine runs both."""
from __future__ import annotations

import json
import os

import numpy as np
import torch

from oracle import checkpoint, mlx_quant

LUT = np.array([0.0, 0.5, 1.0, 1.5, 2.0, 3.0, 4.0, 6.0, -0.0, -0.5, -1.0, -1.5, -2.0, -3.0, -4.0, -6.0], np.float32)
Q8 = (2 * LUT + 12).astype(np.uint32)  # the container code of each E2M1 code
MAX_SCALE_BYTE = 251  # larger exponents overflow 24 * scale in fp32 or the bias in bf16; 255 is E8M0's NaN


def e8m0_to_f32(e) -> np.ndarray:
    """E8M0 bytes -> 2^(e - 127) as fp32; 255 -> NaN."""
    e = np.asarray(e, np.int32)
    return np.where(e == 255, np.nan, np.ldexp(1.0, e - 127)).astype(np.float32)


def mxfp4_dequantize(packed, scales_u8, out_dtype: str = "f32") -> np.ndarray:
    """MLX `dequantize(..., mode: "mxfp4")`: LUT[code] * 2^(e - 127), exact in fp32 for e <= 251, rounded once to `out_dtype`
    ('f32' | 'f16' | 'bf16'); returned as fp32 holding those values."""
    codes = mlx_quant.unpack(np.asarray(packed), 4)
    e = np.repeat(np.asarray(scales_u8, np.int64), 32, axis=1)
    assert e.shape == codes.shape and e.max(initial=0) <= MAX_SCALE_BYTE
    v = np.ldexp(LUT[codes].astype(np.float64), e - 127).astype(np.float32)
    return mlx_quant.round_to_dtype(v, out_dtype)


def mxfp4_quantize_codes(w: np.ndarray):
    """OCP MX quantisation of [out, in] fp32 weights (in % 32 == 0) -> (E2M1 codes uint32 [out, in], E8M0 bytes uint8 [out, in/32]).
    Shared exponent floor(log2(amax)) - 2 per group of 32, elements rounded to the nearest E2M1 value (ties to the even code) and
    saturated at +-6.  Only the checkpoint writer uses it: the engine is bound by the dequantisation semantics alone."""
    w = np.ascontiguousarray(w, dtype=np.float32)
    out, inn = w.shape
    assert inn % 32 == 0
    g = w.reshape(out, inn // 32, 32).astype(np.float64)
    amax = np.abs(g).max(axis=-1)
    _, ex = np.frexp(amax)  # amax = m * 2^ex with m in [0.5, 1): floor(log2(amax)) = ex - 1
    e = np.where(amax > 0, np.clip(ex - 1 - 2 + 127, 0, 254), 0).astype(np.int64)
    x = g / np.ldexp(1.0, e - 127)[..., None]
    order = np.array([0, 2, 4, 6, 1, 3, 5, 7])  # even codes first: argmin keeps the even code of a tie
    d = np.abs(np.abs(x)[..., None] - LUT[order].astype(np.float64))
    mag = order[np.argmin(d, axis=-1)]
    codes = (mag | np.where(x < 0, 8, 0)).astype(np.uint32)
    return codes.reshape(out, inn), e.astype(np.uint8)


def mxfp4_to_affine(packed, scales_u8):
    """The container twin of mxfp4 leaves: (8-bit words uint32 [out, in/4], scales, biases as fp32 holding their bf16 values [out, in/32]),
    for `oracle.mlx_quant.dequantize(..., group_size=32, bits=8)`."""
    codes = mlx_quant.unpack(np.asarray(packed), 4)
    e = np.asarray(scales_u8, np.int64)
    assert e.max(initial=0) <= MAX_SCALE_BYTE
    s = np.ldexp(1.0, e - 128).astype(np.float32)
    return mlx_quant.pack(Q8[codes], 8), s, (np.float32(-12) * s).astype(np.float32)


def _u32(a: np.ndarray) -> torch.Tensor:
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).view(torch.uint32)


def _bf16(a: np.ndarray) -> torch.Tensor:
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(torch.bfloat16)


def write_mxfp4_checkpoint(path: str, name: str = "tiny", seed: int = 0, init: str = "stress", quant_key: str = "quantization") -> tuple[str, str]:
    """An MLX mxfp4 checkpoint and its 8-bit g32 bf16 container twin, both made from `oracle.checkpoint`'s dense bf16 checkpoint of the same
    name / seed / init: every linear leaf is quantised with `mxfp4_quantize_codes`, embeddings stay dense.  quant_key = "quantization_config"
    gives the form `Qwen3Talker.load` dequantises offline to fp16.  Talker only (no speech tokenizer).  Returns (mxfp4 directory, twin
    directory); cached by a stamp file."""
    from safetensors.torch import load_file, save_file

    twin = f"{path}_as8"
    stamp = {"name": name, "seed": seed, "init": init, "quant_key": quant_key, "v": 1}
    stamps = [os.path.join(d, "mxfp4_stamp.json") for d in (path, twin)]
    if all(os.path.exists(s) and json.load(open(s)) == stamp for s in stamps):
        return path, twin
    dense = checkpoint.write_checkpoint(path + "_dense", name, bits=0, dtype="bf16", seed=seed, init=init, with_codec=False)
    t = load_file(os.path.join(dense, "model.safetensors"))
    packed, container = dict(t), dict(t)
    for k, v in t.items():
        if k.endswith(".weight") and v.dim() == 2 and "embedding" not in k:
            codes, e = mxfp4_quantize_codes(v.float().numpy())
            words = mlx_quant.pack(codes, 4)
            packed[k] = _u32(words)
            packed[k[:-7] + ".scales"] = torch.from_numpy(e)
            w8, s, b = mxfp4_to_affine(words, e)
            container.update({k: _u32(w8), k[:-7] + ".scales": _bf16(s), k[:-7] + ".biases": _bf16(b)})
    cfg = json.load(open(os.path.join(dense, "config.json")))
    for d, tensors, quant in ((path, packed, {"group_size": 32, "bits": 4, "mode": "mxfp4"}), (twin, container, {"group_size": 32, "bits": 8})):
        os.makedirs(d, exist_ok=True)
        save_file(tensors, os.path.join(d, "model.safetensors"))
        json.dump(dict(cfg, **{quant_key: quant}), open(os.path.join(d, "config.json"), "w"), indent=1)
        json.dump(stamp, open(os.path.join(d, "mxfp4_stamp.json"), "w"))
    return path, twin
