"""Test support for MLX affine checkpoints of 2, 3, 5 and 6 bits: the bit-stream packing and a checkpoint writer.

MLX packs the codes of a row as one little-endian, least-significant-bit-first bit stream: code j occupies bits [j*b, (j+1)*b) of the row's
bytes, stored as uint32 [out, in*b/32].  For b in {2, 4, 8} that is the word layout of `oracle.mlx_quant.pack` (element j of a word at bit
offset j*b, anchored on HF's Metal integration by tests/test_oracle_quant.py); for 3 and 6 bits MLX writes packs of 3 bytes (8 or 4 codes), for
5 bits packs of 5 bytes (8 codes) -- the same stream (SURVEY.md Appendix C).  The 3/5/6-bit packing is restated here from that description and
checked in tests/test_oracle_quant_widths.py against a stream built with numpy's packbits and against bytes written out by hand; it has not been
checked against MLX itself or another implementation, none being available where the tests run.

The oracle dequantises 4- and 8-bit words (`oracle.mlx_quant`).  A b-bit checkpoint is therefore written together with its CONTAINER TWIN: the
same codes, scales and biases packed as 4-bit (b = 2, 3) or 8-bit (b = 5, 6) words, which is what the engine widens the b-bit rows into at load.
The oracle runs the twin; the engine runs both."""
from __future__ import annotations

import json
import os

import numpy as np
import torch

from oracle import checkpoint, mlx_quant

BITS = (2, 3, 4, 5, 6, 8)  # the widths MLX's affine mode writes
CONTAINER = {2: 4, 3: 4, 4: 4, 5: 8, 6: 8, 8: 8}


def pack(q: np.ndarray, bits: int) -> np.ndarray:
    """[out, in] integer codes -> [out, in*bits/32] uint32 holding each row's LSB-first bit stream (in % 32 == 0)."""
    assert bits in BITS
    out, inn = q.shape
    assert inn % 32 == 0
    q = q.astype(np.uint64).reshape(out, inn // 32, 32)  # 32 codes fill `bits` whole words
    words = np.zeros((out, inn // 32, bits + 1), np.uint64)  # one spare word takes the (empty) spill of the last code
    for j in range(32):
        w, sh = divmod(j * bits, 32)
        v = q[:, :, j] << np.uint64(sh)
        words[:, :, w] |= v & np.uint64(0xFFFFFFFF)
        words[:, :, w + 1] |= v >> np.uint64(32)
    return words[:, :, :bits].astype(np.uint32).reshape(out, inn // 32 * bits)


def unpack(packed: np.ndarray, bits: int) -> np.ndarray:
    """Inverse of `pack`: [out, in*bits/32] uint32 -> [out, in] uint32 codes."""
    assert bits in BITS
    packed = np.ascontiguousarray(packed).view(np.uint32)
    out, words = packed.shape
    assert words % bits == 0
    p = packed.reshape(out, words // bits, bits).astype(np.uint64)
    p = np.concatenate([p, np.zeros_like(p[:, :, :1])], axis=-1)
    mask = np.uint64((1 << bits) - 1)
    q = np.empty((out, words // bits, 32), np.uint32)
    for j in range(32):
        w, sh = divmod(j * bits, 32)
        q[:, :, j] = (((p[:, :, w] | (p[:, :, w + 1] << np.uint64(32))) >> np.uint64(sh)) & mask).astype(np.uint32)
    return q.reshape(out, words // bits * 32)


def _u32(a: np.ndarray) -> torch.Tensor:
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).view(torch.uint32)


def write_width_checkpoint(path: str, name: str = "tiny", bits: int = 3, group: int = 64, seed: int = 0, init: str = "stress",
                           quant_key: str = "quantization") -> tuple[str, str]:
    """A b-bit MLX checkpoint and its container twin, both made from `oracle.checkpoint`'s dense bf16 checkpoint of the same name / seed /
    init: every linear leaf is quantised with `mlx_quant.quantize_codes` (group `group`, bf16 scales / biases), embeddings stay dense -- the
    leaves `oracle.checkpoint.write_checkpoint` quantises.  quant_key = "quantization_config" gives the form `Qwen3Talker.load` dequantises
    offline to fp16.  Talker only (no speech tokenizer).  Returns (b-bit directory, twin directory); cached by a stamp file."""
    from safetensors.torch import load_file, save_file

    cb = CONTAINER[bits]
    twin = f"{path}_as{cb}"
    stamp = {"name": name, "bits": bits, "group": group, "seed": seed, "init": init, "quant_key": quant_key, "v": 1}
    stamps = [os.path.join(d, "width_stamp.json") for d in (path, twin)]
    if all(os.path.exists(s) and json.load(open(s)) == stamp for s in stamps):
        return path, twin
    dense = checkpoint.write_checkpoint(path + "_dense", name, bits=0, dtype="bf16", seed=seed, init=init, with_codec=False)
    t = load_file(os.path.join(dense, "model.safetensors"))
    packed, container = dict(t), dict(t)
    for k, v in t.items():
        if k.endswith(".weight") and v.dim() == 2 and "embedding" not in k:
            q, s, b = mlx_quant.quantize_codes(v.float().numpy(), group, bits, "bf16")
            leaves = {k[:-7] + ".scales": torch.from_numpy(s).to(torch.bfloat16), k[:-7] + ".biases": torch.from_numpy(b).to(torch.bfloat16)}
            packed.update(leaves, **{k: _u32(pack(q, bits))})
            container.update(leaves, **{k: _u32(mlx_quant.pack(q, cb))})
    cfg = json.load(open(os.path.join(dense, "config.json")))
    for d, tensors, width in ((path, packed, bits), (twin, container, cb)):
        os.makedirs(d, exist_ok=True)
        save_file(tensors, os.path.join(d, "model.safetensors"))
        json.dump(dict(cfg, **{quant_key: {"group_size": group, "bits": width}}), open(os.path.join(d, "config.json"), "w"), indent=1)
        json.dump(stamp, open(os.path.join(d, "width_stamp.json"), "w"))
    return path, twin
