"""CPU: MLX affine checkpoints of 2, 3, 5 and 6 bits -- the bit-stream packing of tests/mlx_widths.py, the checkpoint writer at every width,
and the host-side refusals of the packed probes (no device needed).

MLX writes the codes of a row as one little-endian, LSB-first bit stream (code j at bits [j*b, (j+1)*b) of the row's bytes).  For 2, 4 and 8
bits that is the word layout of oracle/mlx_quant.py, which test_oracle_quant.py anchors on HF's Metal integration; the 3/5/6-bit packs are
checked here against a bit stream built independently with numpy's packbits, and by hand."""
import json
import os

import numpy as np
import pytest

import mlx_widths
from oracle import mlx_quant

WIDTHS = [2, 3, 4, 5, 6, 8]


def _bit_stream(q: np.ndarray, bits: int) -> np.ndarray:
    """Independent reference: every code's bits LSB first, concatenated per row, bytes little-endian -> uint32 words."""
    out, inn = q.shape
    shifts = np.arange(bits, dtype=np.uint32)
    stream = ((q.astype(np.uint32)[:, :, None] >> shifts) & 1).astype(np.uint8).reshape(out, inn * bits)
    return np.packbits(stream, axis=1, bitorder="little").view("<u4").astype(np.uint32)


@pytest.mark.parametrize("bits", WIDTHS)
def test_pack_is_the_lsb_first_bit_stream(bits):
    rng = np.random.default_rng(bits)
    q = rng.integers(0, 1 << bits, size=(7, 160)).astype(np.uint32)
    packed = mlx_widths.pack(q, bits)
    assert packed.shape == (7, 160 * bits // 32) and packed.dtype == np.uint32
    assert np.array_equal(packed, _bit_stream(q, bits))
    # code j at bit j*b of the row, read back one code at a time
    row = int.from_bytes(packed[3].astype("<u4").tobytes(), "little")
    assert [(row >> (j * bits)) & ((1 << bits) - 1) for j in range(160)] == q[3].tolist()


def test_pack_by_hand():
    # four 6-bit codes -> 3 bytes: 0b000001, 0b100000, 0b010101, 0b111111 LSB first
    q6 = np.array([[1, 32, 21, 63] * 8], np.uint32)
    b6 = mlx_widths.pack(q6, 6).astype("<u4").tobytes()
    assert b6[:3] == bytes([0b00000001, 0b01011000, 0b11111101])
    # eight 3-bit codes 0..7 -> 3 bytes: the stream 000 100 010 110 001 101 011 111 (each code LSB first)
    q3 = np.array([list(range(8)) * 4], np.uint32)
    b3 = mlx_widths.pack(q3, 3).astype("<u4").tobytes()
    assert b3[:3] == bytes([0b10001000, 0b11000110, 0b11111010])
    # eight 5-bit codes -> 5 bytes
    codes5 = [31, 0, 1, 16, 7, 24, 3, 30]
    q5 = np.array([codes5 * 4], np.uint32)
    b5 = mlx_widths.pack(q5, 5).astype("<u4").tobytes()
    want = sum(c << (5 * j) for j, c in enumerate(codes5)).to_bytes(5, "little")
    assert b5[:5] == want and want == bytes([0x1F, 0x04, 0x78, 0xF0, 0xF0])
    for q, bits in ((q6, 6), (q3, 3), (q5, 5)):
        assert np.array_equal(mlx_widths.unpack(mlx_widths.pack(q, bits), bits), q)


@pytest.mark.parametrize("bits", [2, 4, 8])
def test_stream_equals_word_packing(bits):
    """For widths that divide 32 the stream is the word definition: element j of a word at bit offset j*bits -- and, for 4 and 8 bits,
    exactly what oracle/mlx_quant.py packs."""
    rng = np.random.default_rng(40 + bits)
    q = rng.integers(0, 1 << bits, size=(5, 128)).astype(np.uint32)
    per = 32 // bits
    words = np.zeros((5, 128 // per), np.uint32)
    for j in range(per):
        words |= q[:, j::per] << np.uint32(j * bits)
    assert np.array_equal(mlx_widths.pack(q, bits), words)
    assert np.array_equal(_bit_stream(q, bits), words)
    if bits in (4, 8):
        assert np.array_equal(mlx_quant.pack(q, bits), words)


@pytest.mark.parametrize("group", [32, 64, 128])
def test_two_bit_dequantize_equals_hf_metal_affine(group):
    """test_dequantize_layout_equals_hf_metal_affine at 2 bits: HF's `_affine_dequantize_tensor` reads the 2-bit words to the weights the
    oracle computes from the same codes."""
    import torch

    mq_hf = pytest.importorskip("transformers.integrations.metal_quantization")
    rng = np.random.default_rng(200 + group)
    w = (rng.standard_normal((24, 256)) * 0.05).astype(np.float32)
    q, s, b = mlx_quant.quantize_codes(w, group, 2, "f32")
    mine = mlx_quant.dequantize(mlx_quant.pack(q, 4), s, b, group, 4, "f32")  # same codes in 4-bit words
    packed = mlx_widths.pack(q, 2)
    theirs = mq_hf._affine_dequantize_tensor(torch.from_numpy(packed.view(np.int32)), torch.from_numpy(s), torch.from_numpy(b), group, 2).numpy()
    assert np.array_equal(mine, theirs)


@pytest.mark.parametrize("bits", WIDTHS)
@pytest.mark.parametrize("group", [32, 64, 128])
def test_pack_unpack_roundtrip_every_width(bits, group):
    rng = np.random.default_rng(bits * 1000 + group)
    q = rng.integers(0, 1 << bits, size=(17, 2 * group)).astype(np.uint32)
    q[0] = (1 << bits) - 1  # all-maximal codes: a shifted mask would lose bits here
    assert np.array_equal(mlx_widths.unpack(mlx_widths.pack(q, bits), bits), q)


@pytest.mark.parametrize("bits", [2, 3, 5, 6])
@pytest.mark.parametrize("sdt", ["f32", "bf16", "f16"])
def test_quantize_dequantize_error_bound(bits, sdt):
    """Interior points land within half a step; MLX re-fits the scale so the dominant edge is exact, which can leave the far end of a
    group up to one step out (test_quantize_error_bound), so the bound for every element is one step."""
    rng = np.random.default_rng(bits + len(sdt))
    w = (rng.standard_normal((48, 256)) * 0.02).astype(np.float32)
    q, s, b = mlx_quant.quantize_codes(w, 64, bits, sdt)
    packed = mlx_widths.pack(q, bits)
    assert packed.shape == (48, 256 * bits // 32)
    assert np.array_equal(mlx_widths.unpack(packed, bits), q)
    cb = mlx_widths.CONTAINER[bits]
    deq = mlx_quant.dequantize(mlx_quant.pack(q, cb), s, b, 64, cb, "f32")
    step = np.repeat(np.abs(s), 64, axis=1)
    slack = {"f32": 1e-7, "bf16": 2 ** -8, "f16": 2 ** -11}[sdt] * np.abs(w).max() * 4
    assert np.all(np.abs(deq - w) <= step + slack + 1e-7)
    inner = (q > 0) & (q < (1 << bits) - 1)
    assert np.all(np.abs(deq - w)[inner] <= 0.5 * step[inner] * 1.001 + slack + 1e-7)


@pytest.mark.parametrize("bits,group", [(2, 64), (3, 32), (3, 64), (5, 64), (6, 64), (6, 128)])
def test_checkpoint_writer_every_width(bits, group, tmp_path):
    """mlx_widths.write_width_checkpoint: uint32 [out, in*b/32] leaves with [out, in/group] scales and biases, and a container twin that
    holds the same codes, scales and biases in 4/8-bit words."""
    import torch
    from safetensors.torch import load_file

    d, twin = mlx_widths.write_width_checkpoint(str(tmp_path / "ck"), "tiny", bits, group)
    cfg, tcfg = (json.load(open(os.path.join(p, "config.json"))) for p in (d, twin))
    cb = mlx_widths.CONTAINER[bits]
    assert cfg["quantization"] == {"group_size": group, "bits": bits} and tcfg["quantization"] == {"group_size": group, "bits": cb}
    t, tt = (load_file(os.path.join(p, "model.safetensors")) for p in (d, twin))
    assert set(t) == set(tt)
    n = 0
    for k, v in t.items():
        if not k.endswith(".weight") or k.replace(".weight", ".scales") not in t:
            assert np.array_equal(v.float().numpy(), tt[k].float().numpy()), k
            continue
        s = t[k.replace(".weight", ".scales")]
        out, inn = s.shape[0], s.shape[1] * group
        assert v.element_size() == 4 and not v.is_floating_point() and tuple(v.shape) == (out, inn * bits // 32), k
        assert t[k.replace(".weight", ".biases")].shape == s.shape
        codes = mlx_widths.unpack(v.view(torch.int32).numpy(), bits)
        assert np.array_equal(codes, mlx_quant.unpack(tt[k].view(torch.int32).numpy(), cb)), k
        n += 1
    assert n > 20


# ------------------------------------------------------------------------------------------------ CPU: refusals without a device
def _status(fn):
    import qwen3tts_b200 as q

    with pytest.raises(q.Q3Error) as e:
        fn()
    return e.value.status


def _raw_call(name, bits, group, in_f, out_f=8):
    """Call the C probe directly, so argument shapes the Python wrappers would derive cannot hide a refusal."""
    import ctypes as C

    from qwen3tts_b200 import _abi as A

    words = np.zeros(max(1, out_f * in_f * 8 // 32), np.uint32)  # large enough for any width
    s = np.zeros(max(1, out_f * in_f), np.float32)
    x = np.zeros(max(1, 2 * in_f), np.float32)
    y = np.zeros(max(1, 2 * out_f * in_f), np.float32)
    L = A.lib()
    if name == "dequantize":
        rc = L.q3tts_dequantize(0, words.ctypes.data, s.ctypes.data, s.ctypes.data, A.F32, out_f, in_f, group, bits, A.F32, y.ctypes.data)
    elif name == "quantized_matmul":
        rc = L.q3tts_quantized_matmul(0, x.ctypes.data_as(A.p_f32), 2, words.ctypes.data, s.ctypes.data, s.ctypes.data, A.F32, out_f, in_f, group, bits,
                                      y.ctypes.data_as(A.p_f32))
    else:
        rc = L.q3tts_quantized_matmul_tc(0, x.ctypes.data_as(A.p_f32), 2, words.ctypes.data, s.ctypes.data, s.ctypes.data, A.F32, out_f, in_f, group, bits,
                                         None, 0, None, y.ctypes.data_as(A.p_f32))
    return rc


@pytest.mark.parametrize("name", ["dequantize", "quantized_matmul", "quantized_matmul_tc"])
def test_packed_probes_refuse_bad_widths_without_a_device(name):
    """Bits 1 and 7, in_features not a multiple of 32 and group 16 at the new widths are refused by the host-side validation
    (Q3TTS_ERR_INVALID_ARG), before any device is looked for."""
    from qwen3tts_b200 import _abi as A

    cases = {"bits 1": (1, 64, 256), "bits 7": (7, 64, 256), "bits 9": (9, 64, 256),
             "3-bit in % 32": (3, 16, 272), "5-bit in % 32": (5, 8, 200), "6-bit group 16": (6, 16, 256), "3-bit group 16": (3, 16, 256),
             "2-bit group 256": (2, 256, 512), "in % group": (4, 64, 96)}
    for what, (bits, group, in_f) in cases.items():
        rc = _raw_call(name, bits, group, in_f)
        assert rc == A.ERR_INVALID_ARG, f"{name} {what}: status {rc}"


def test_python_wrapper_refusal_surfaces_as_q3error():
    import qwen3tts_b200 as q
    from qwen3tts_b200 import _abi as A

    q6 = np.zeros((4, 256), np.uint32)
    packed = mlx_widths.pack(q6, 6)
    s = np.ones((4, 16), np.float32)
    assert _status(lambda: q.dequantize(packed, s, s, 16, 6, "f32", "f32")) == A.ERR_INVALID_ARG
