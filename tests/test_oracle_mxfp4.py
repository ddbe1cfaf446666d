"""CPU: MLX mxfp4 -- the dequantisation of tests/mlx_mxfp4.py against HF's mxfp4 integration and torch's E8M0 type, the exactness of the
8-bit affine container twin, the checkpoint writer, and the host-side refusals of q3tts_mxfp4_to_affine (no device needed)."""
import json
import os

import numpy as np
import pytest
import torch

import mlx_mxfp4
from oracle import mlx_quant

ALL_E = np.arange(0, mlx_mxfp4.MAX_SCALE_BYTE + 1)


def _every_code_and_exponent():
    """Leaves holding every code (twice per group) in every group, one group per exponent 0..251, over an odd row count."""
    rows = 9
    groups = -(-len(ALL_E) // rows)
    e = np.resize(ALL_E, rows * groups).reshape(rows, groups).astype(np.uint8)
    codes = ((np.arange(groups * 32)[None, :] + 3 * np.arange(rows)[:, None]) % 16).astype(np.uint32)
    return mlx_quant.pack(codes, 4), e, codes


def _hf(packed, e, dtype):
    """HF `_convert_moe_packed_tensors` on the MLX words viewed as little-endian bytes [1, out, in/32, 16] -> [out, in]."""
    mx = pytest.importorskip("transformers.integrations.mxfp4")
    out, words = packed.shape
    blocks = torch.from_numpy(np.ascontiguousarray(packed).astype("<u4").view(np.uint8).reshape(1, out, words // 4, 16))
    scales = torch.from_numpy(np.ascontiguousarray(e)).reshape(1, out, words // 4)
    return mx._convert_moe_packed_tensors(blocks, scales, dtype=dtype)[0].transpose(0, 1).to(torch.float32).numpy()


@pytest.mark.parametrize("odt", ["f32", "bf16"])
def test_dequantize_equals_hf_mxfp4(odt):
    dtype = {"f32": torch.float32, "bf16": torch.bfloat16}[odt]
    packed, e, _ = _every_code_and_exponent()
    assert np.array_equal(mlx_mxfp4.mxfp4_dequantize(packed, e, odt).view(np.uint32), _hf(packed, e, dtype).view(np.uint32))
    rng = np.random.default_rng(7)
    packed = rng.integers(0, 2 ** 32, size=(13, 64), dtype=np.uint64).astype(np.uint32)  # random bytes
    e = rng.integers(0, mlx_mxfp4.MAX_SCALE_BYTE + 1, size=(13, 16)).astype(np.uint8)
    assert np.array_equal(mlx_mxfp4.mxfp4_dequantize(packed, e, odt).view(np.uint32), _hf(packed, e, dtype).view(np.uint32))


def test_e8m0_equals_torch_float8_e8m0fnu():
    b = np.arange(256, dtype=np.uint8)
    theirs = torch.from_numpy(b).view(torch.float8_e8m0fnu).to(torch.float32).numpy()
    mine = mlx_mxfp4.e8m0_to_f32(b)
    assert np.isnan(mine[255]) and np.isnan(theirs[255])
    assert np.array_equal(mine[:255].view(np.uint32), theirs[:255].view(np.uint32))


@pytest.mark.parametrize("odt", ["f32", "f16", "bf16"])
def test_container_twin_is_exact(odt):
    """Every code x every exponent 0..251: the twin through the affine oracle gives the mxfp4 values; bits differ only at code 8 (-0 -> +0)."""
    packed, e, codes = _every_code_and_exponent()
    w8, s, b = mlx_mxfp4.mxfp4_to_affine(packed, e)
    with np.errstate(over="ignore"):  # f16: large exponents round to inf on both sides
        want = mlx_mxfp4.mxfp4_dequantize(packed, e, odt)
        got = mlx_quant.dequantize(w8, s, b, 32, 8, odt)
    assert np.array_equal(got, want)
    same = got.view(np.uint32) == want.view(np.uint32)
    assert np.all(same[codes != 8]) and np.all(got[codes == 8].view(np.uint32) == 0)
    # the bf16 bit patterns of the container's scale and bias, from the exponent alone
    ee = e.astype(np.uint32)
    sb, bb = s.view(np.uint32) >> 16, b.view(np.uint32) >> 16
    assert np.all(round_trip_bf16(s) == s) and np.all(round_trip_bf16(b) == b)
    assert np.array_equal(sb, np.where(ee < 2, 0x20 << ee, (ee - 1) << 7))
    assert np.array_equal(bb, 0x8000 | ((ee + 2) << 7) | 0x40)
    assert np.array_equal(mlx_quant.unpack(w8, 8), mlx_mxfp4.Q8[codes])


def round_trip_bf16(a):
    return mlx_quant.round_to_dtype(a, "bf16")


def test_quantize_codes_follow_the_ocp_rule():
    # one group: amax 5.0 -> shared exponent floor(log2 5) - 2 = 0 -> e = 127; values land on the E2M1 grid, ties to even, saturate at 6
    w = np.zeros((1, 32), np.float32)
    w[0, :10] = [5.0, 0.25, 1.25, 2.5, 3.5, -0.75, -5.0, 0.1, -0.1, 1.75]
    codes, e = mlx_mxfp4.mxfp4_quantize_codes(w)
    assert e.tolist() == [[127]]
    assert codes[0, :10].tolist() == [6, 0, 2, 4, 6, 10, 14, 0, 8, 4]
    w[0, 0] = 7.9  # amax 7.9 -> exponent 0, saturated at 6
    codes, e = mlx_mxfp4.mxfp4_quantize_codes(w)
    assert e.tolist() == [[127]] and codes[0, 0] == 7
    rng = np.random.default_rng(3)
    w = (rng.standard_normal((16, 256)) * 0.03).astype(np.float32)
    codes, e = mlx_mxfp4.mxfp4_quantize_codes(w)
    deq = mlx_mxfp4.mxfp4_dequantize(mlx_quant.pack(codes, 4), e)
    unit = np.repeat(np.ldexp(1.0, e.astype(np.int64) - 127), 32, axis=1)
    assert np.all(np.abs(deq - w) <= 2 * unit)  # half the widest gap (4 -> 6) is one unit; saturation (amax < 8 units) costs at most two
    assert np.all(np.abs(deq).reshape(16, 8, 32).max(-1) > 0)


def test_checkpoint_writer(tmp_path):
    import torch as T
    from safetensors.torch import load_file

    for key in ("quantization", "quantization_config"):
        d, twin = mlx_mxfp4.write_mxfp4_checkpoint(str(tmp_path / key), "tiny", quant_key=key)
        cfg, tcfg = (json.load(open(os.path.join(p, "config.json"))) for p in (d, twin))
        assert cfg[key] == {"group_size": 32, "bits": 4, "mode": "mxfp4"} and tcfg[key] == {"group_size": 32, "bits": 8}
        t, tt = (load_file(os.path.join(p, "model.safetensors")) for p in (d, twin))
        n = 0
        for k, v in t.items():
            assert not k.endswith(".biases"), k
            if k.endswith(".scales"):
                continue
            if not k.endswith(".weight") or k.replace(".weight", ".scales") not in t:  # dense leaves are the same in both
                assert np.array_equal(v.float().numpy(), tt[k].float().numpy()), k
                continue
            s = t[k.replace(".weight", ".scales")]
            out, inn = s.shape[0], s.shape[1] * 32
            assert v.dtype == T.uint32 and tuple(v.shape) == (out, inn // 8), k
            assert s.dtype == T.uint8 and int(s.max()) <= mlx_mxfp4.MAX_SCALE_BYTE, k
            assert k.replace(".weight", ".biases") not in t
            tb = tt[k.replace(".weight", ".biases")]
            assert tt[k].dtype == T.uint32 and tuple(tt[k].shape) == (out, inn // 4), k
            assert tt[k.replace(".weight", ".scales")].dtype == T.bfloat16 and tb.dtype == T.bfloat16 and tuple(tb.shape) == (out, inn // 32)
            words, e = v.view(T.int32).numpy().view(np.uint32), s.numpy()
            want = mlx_mxfp4.mxfp4_dequantize(words, e)
            got = mlx_quant.dequantize(tt[k].view(T.int32).numpy().view(np.uint32), tt[k.replace(".weight", ".scales")],
                                       tb, 32, 8, "f32")
            assert np.array_equal(got, want), k
            n += 1
        assert n > 20


# ------------------------------------------------------------------------------------------------ CPU: refusals without a device
def test_probe_refuses_bad_arguments_without_a_device():
    """NULL pointers, in % 32 != 0 and scale bytes >= 252 are refused by the host-side validation (Q3TTS_ERR_INVALID_ARG) before any
    device is looked for."""
    from qwen3tts_b200 import _abi as A

    L = A.lib()
    out_f, in_f = 4, 64
    words = np.zeros(out_f * in_f // 8 + 64, np.uint32)
    codes = np.zeros(out_f * in_f, np.uint32)
    s16 = np.zeros(out_f * in_f, np.uint16)

    def call(scales, in_f=in_f, w=words.ctypes.data, c=codes.ctypes.data, so=s16.ctypes.data, bo=s16.ctypes.data):
        return L.q3tts_mxfp4_to_affine(0, w, None if scales is None else scales.ctypes.data, out_f, in_f, c, so, bo)

    good = np.full(out_f * in_f // 32 + 8, 127, np.uint8)
    cases = {"NULL packed": lambda: call(good, w=None), "NULL scales": lambda: call(None), "NULL codes": lambda: call(good, c=None),
             "NULL scales_out": lambda: call(good, so=None), "NULL biases_out": lambda: call(good, bo=None),
             "in % 32": lambda: call(good, in_f=48), "in 0": lambda: call(good, in_f=0)}
    for byte in (252, 254, 255):
        bad = good.copy()
        bad[out_f * in_f // 32 - 1] = byte  # the last group
        cases[f"scale byte {byte}"] = lambda bad=bad: call(bad)
    for what, fn in cases.items():
        assert fn() == A.ERR_INVALID_ARG, what


def test_python_wrapper_refusal_surfaces_as_q3error():
    import qwen3tts_b200 as q
    from qwen3tts_b200 import _abi as A

    e = np.full((4, 2), 252, np.uint8)
    with pytest.raises(q.Q3Error) as err:
        q.mxfp4_to_affine(np.zeros((4, 8), np.uint32), e)
    assert err.value.status == A.ERR_INVALID_ARG
