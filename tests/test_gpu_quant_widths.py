"""GPU: MLX affine checkpoints of 2, 3, 5 and 6 bits through the C ABI vs the CPU oracle.

The loader widens the b-bit rows into the 4-bit (2, 3 bits) or 8-bit (5, 6 bits) words the decode kernels read; codes, scales and biases are
copied unchanged.  So dequantisation is bit-exact, every decode path meets the bar of its existing 4/8-bit test, and a checkpoint and its
4/8-bit twin holding the same codes give identical bits.  The oracle dequantises 4- and 8-bit words only, so every reference is computed on
the container twin that tests/mlx_widths.py writes next to each b-bit checkpoint (same codes, scales and biases).  Bars: LOGIT_TOL as in test_gpu_talker.py, 1e-3 for the 2-slot persistent kernel
(test_two_utterance_persistent_kernel), the probe bars of test_quantized_matmul and tests/test_gpu_gemm_tc.py."""
import ctypes as C
import json
import os
import shutil

import numpy as np
import pytest

import mlx_widths
from conftest import CKPT_ROOT, TEXT_IDS, ckpt

pytestmark = pytest.mark.gpu

LOGIT_TOL = 1e-2
MMA_TOL = 1e-3
MARGIN_TOL = 2e-2
CONTAINER = {2: 4, 3: 4, 5: 8, 6: 8}
CKPTS = [(2, 64), (3, 64), (5, 64), (6, 64), (3, 32), (6, 128)]
F = 12


def _ck(bits, group, name="tiny", **kw):
    """(b-bit checkpoint, its container twin) -- cached under the test checkpoint root."""
    tag = f"width_{name}_b{bits}_g{group}" + "".join(f"_{k}{v}" for k, v in sorted(kw.items()))
    return mlx_widths.write_width_checkpoint(os.path.join(CKPT_ROOT, tag), name, bits, group, **kw)


def _forced():
    return np.random.default_rng(31).integers(0, 2048, size=(F, 16)).astype(np.int32)


def _greq(q, **kw):
    kw.setdefault("temperature", 0.0)
    return q.GenRequest(text_ids=TEXT_IDS, speaker_id=2861, keep_invalid_frames=True, **kw)


_REF = {}


def _reference(d, oracles):
    """The oracle's teacher-forced logits and free-running greedy ids (with margins) of checkpoint `d` (a container twin), computed once."""
    from oracle import talker as otalker

    if d not in _REF:
        rec, grec = {}, {}
        oracles(d).generate_codes(otalker.Request(text_ids=TEXT_IDS, speaker_id=2861, temperature=0.0, max_tokens=F), forced=_forced(), record=rec,
                                  filter_invalid=False)
        want = oracles(d).generate_codes(otalker.Request(text_ids=TEXT_IDS, speaker_id=2861, temperature=0.0, max_tokens=20), record=grec,
                                         filter_invalid=False)
        _REF[d] = (rec, want, grec["margins"])
    return _REF[d]


def _compare_greedy(got, want, margins):
    """test_gpu_talker._compare_greedy: ids match frame by frame; a first mismatch is only acceptable at an oracle near-tie."""
    for f in range(min(len(got), len(want))):
        for g in range(16):
            if got[f][g] != want[f][g]:
                assert margins[f][g] < MARGIN_TOL, f"ids diverge at frame {f} group {g} with oracle margin {margins[f][g]:.4f}"
                return
    assert len(got) == len(want)


def _logit_err(eng, q, rec):
    frames, lg = eng.generate_codes(_greq(q, max_tokens=F, forced_codes=_forced(), want_logits=F))
    assert frames.tolist() == _forced().tolist()
    return np.abs(lg["code0_logits"] - rec["code0_logits"]).max(), np.abs(lg["cp_logits"] - rec["cp_logits"]).max()


# ------------------------------------------------------------------------------------------------ dequantisation, bit-exact
@pytest.mark.parametrize("bits", [2, 3, 5, 6])
@pytest.mark.parametrize("sdt", ["bf16", "f16", "f32"])
@pytest.mark.parametrize("odt", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("group", [32, 64, 128])
def test_dequantize_bit_exact_widths(bits, sdt, odt, group):
    import qwen3tts_b200 as q
    from oracle import mlx_quant

    rng = np.random.default_rng(bits * 100 + group + len(sdt) * 7 + len(odt))
    w = (rng.standard_normal((97, 384)) * 0.05).astype(np.float32)  # odd row count: the last code of the last row is read
    w[3] = 0.0  # an all-zero row: scale clamps to 1e-7, q0 == 0 path
    w[4, :group] = 1.0  # constant group
    codes, s, b = mlx_quant.quantize_codes(w, group, bits, sdt)
    cb = CONTAINER[bits]
    want = mlx_quant.dequantize(mlx_quant.pack(codes, cb), s, b, group, cb, odt)
    got = q.dequantize(mlx_widths.pack(codes, bits), s, b, group, bits, sdt, odt)
    assert got.shape == want.shape
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), "dequantised weights are not bit-identical"
    # scale 1, bias 0: the output IS the codes; the last row holds only maximal codes (2^b - 1), which a shifted mask would cut
    codes = rng.integers(0, 1 << bits, size=(97, 384)).astype(np.uint32)
    codes[-1] = (1 << bits) - 1
    ones, zeros = np.ones((97, 384 // group), np.float32), np.zeros((97, 384 // group), np.float32)
    got = q.dequantize(mlx_widths.pack(codes, bits), ones, zeros, group, bits, sdt, odt)
    assert np.array_equal(got, codes.astype(np.float32))


# ------------------------------------------------------------------------------------------------ dequant-fused matmul probes
@pytest.mark.parametrize("bits", [3, 5, 6])
@pytest.mark.parametrize("sdt,group", [("bf16", 64), ("f16", 32), ("f32", 128)])
@pytest.mark.parametrize("shape", [(1, 1024, 1024), (2, 512, 2048), (5, 200, 1024), (19, 96, 256)])
def test_quantized_matmul_widths(bits, sdt, group, shape):
    """test_quantized_matmul's bar: the talker's GEMV on the widened words == x . dequant(W)^T at fp32-accumulation error."""
    import qwen3tts_b200 as q
    from oracle import mlx_quant

    m, out_f, in_f = shape
    rng = np.random.default_rng(m * 1000 + out_f + bits + group)
    w = (rng.standard_normal((out_f, in_f)) * 0.02).astype(np.float32)
    x = rng.standard_normal((m, in_f)).astype(np.float32)
    codes, s, b = mlx_quant.quantize_codes(w, group, bits, sdt)
    packed = mlx_widths.pack(codes, bits)
    wd = mlx_quant.dequantize(mlx_quant.pack(codes, CONTAINER[bits]), s, b, group, CONTAINER[bits], "f32")
    got = q.quantized_matmul(x, packed, s, b, group, bits, sdt)
    want = x.astype(np.float64) @ wd.astype(np.float64).T
    scale = np.abs(x).astype(np.float64) @ np.abs(wd).astype(np.float64).T
    assert np.all(np.abs(got - want) <= 4e-6 * scale + 1e-6), f"max err {np.abs(got - want).max():.3e}"


@pytest.mark.parametrize("bits", [3, 5, 6])
@pytest.mark.parametrize("sdt,group", [("bf16", 64), ("f16", 32), ("f32", 128)])
@pytest.mark.parametrize("shape", [(1, 1024, 1024), (24, 1024, 2048), (64, 3072, 1024), (128, 256, 512), (5, 160, 256)])
def test_dequant_fused_tensor_core_gemm_widths(bits, sdt, group, shape):
    """test_dequant_fused_tensor_core_gemm's bar: the tcgen05 GEMM on the widened words == fp16(x) . fp16(dequant(W))^T, fp32 accumulate."""
    import qwen3tts_b200 as q
    from oracle import mlx_quant

    m, out_f, in_f = shape
    rng = np.random.default_rng(m * 7 + out_f + bits + group)
    w = (rng.standard_normal((out_f, in_f)) * 0.02).astype(np.float32)
    w[5] = 0.0
    x = rng.standard_normal((m, in_f)).astype(np.float32)
    codes, s, b = mlx_quant.quantize_codes(w, group, bits, sdt)
    packed = mlx_widths.pack(codes, bits)
    wd = mlx_quant.dequantize(mlx_quant.pack(codes, CONTAINER[bits]), s, b, group, CONTAINER[bits], "f16").astype(np.float64)
    x16 = x.astype(np.float16).astype(np.float64)
    got = q.quantized_matmul_tc(x, packed, s, b, group, bits, sdt)
    want = x16 @ wd.T
    bound = 4e-6 * (np.abs(x16) @ np.abs(wd).T) + 1e-6
    assert np.all(np.abs(got - want) <= bound), f"max err {np.abs(got - want).max():.3e} (bound {bound.max():.3e})"


@pytest.mark.parametrize("bits", [3, 5, 6])
def test_dequant_fused_gemm_fold_swiglu_residual_widths(bits):
    """test_dequant_fused_gemm_fold_swiglu_residual at the new widths: folded RMSNorm weight, SwiGLU halves, residual."""
    import qwen3tts_b200 as q
    from oracle import mlx_quant

    rng = np.random.default_rng(bits)
    m, inter, in_f = 48, 1536, 1024
    w = (rng.standard_normal((2 * inter, in_f)) * 0.03).astype(np.float32)
    fold = rng.uniform(0.8, 1.2, in_f).astype(np.float32)
    x = rng.standard_normal((m, in_f)).astype(np.float32)
    codes, s, b = mlx_quant.quantize_codes(w, 64, bits, "bf16")
    packed = mlx_widths.pack(codes, bits)
    wd = (mlx_quant.dequantize(mlx_quant.pack(codes, CONTAINER[bits]), s, b, 64, CONTAINER[bits], "f32") * fold[None, :]).astype(np.float32).astype(np.float16).astype(np.float64)
    x16 = x.astype(np.float16).astype(np.float64)
    z = x16 @ wd.T
    gate, up = z[:, :inter], z[:, inter:]
    want = gate / (1 + np.exp(-gate)) * up
    got = q.quantized_matmul_tc(x, packed, s, b, 64, bits, "bf16", fold=fold, swiglu_halves=True)
    assert np.abs(got - want).max() <= 2e-5 * max(1.0, np.abs(want).max())
    res = rng.standard_normal((m, 2 * inter)).astype(np.float32)
    got2 = q.quantized_matmul_tc(x, packed, s, b, 64, bits, "bf16", fold=fold, residual=res)
    assert np.abs(got2 - (z + res)).max() <= 2e-5 * max(1.0, np.abs(z).max())


# ------------------------------------------------------------------------------------------------ every decode path
@pytest.mark.parametrize("bits,group", CKPTS)
def test_info_reports_checkpoint_and_container_widths(bits, group, engines):
    eng = engines(_ck(bits, group)[0], load_codec=False)
    assert eng.info.checkpoint_quant_bits == bits
    assert eng.info.quant_bits == CONTAINER[bits]
    assert eng.info.quant_group_size == group


@pytest.mark.parametrize("bits,group", CKPTS)
def test_persistent_frame_kernel(bits, group, engines, oracles):
    import qwen3tts_b200 as q

    d, twin = _ck(bits, group)
    rec, want, margins = _reference(twin, oracles)
    eng = engines(d, load_codec=False)
    e0, ec = _logit_err(eng, q, rec)
    assert eng.timing().persistent_launches >= 1
    print(f"[{bits}-bit g{group}] persistent kernel teacher-forced max-abs logit error: code0 {e0:.3e}, code predictor {ec:.3e}")
    assert e0 <= LOGIT_TOL and ec <= LOGIT_TOL
    got = eng.generate_codes(_greq(q, max_tokens=20))
    assert eng.timing().persistent_launches >= 1
    _compare_greedy(got.tolist(), want, margins)


@pytest.mark.parametrize("bits,group", CKPTS)
def test_cuda_graph_path(bits, group, oracles, monkeypatch):
    import qwen3tts_b200 as q

    d, twin = _ck(bits, group)
    rec, want, margins = _reference(twin, oracles)
    monkeypatch.setenv("Q3TTS_MEGAKERNEL", "0")
    eng = q.Engine(d, max_frames=256, load_codec=False)
    monkeypatch.delenv("Q3TTS_MEGAKERNEL")
    try:
        e0, ec = _logit_err(eng, q, rec)
        assert eng.timing().persistent_launches == 0 and eng.timing().graph_replays >= 1
        got = eng.generate_codes(_greq(q, max_tokens=20))
    finally:
        eng.close()
    print(f"[{bits}-bit g{group}] CUDA-graph path teacher-forced max-abs logit error: code0 {e0:.3e}, code predictor {ec:.3e}")
    assert e0 <= LOGIT_TOL and ec <= LOGIT_TOL
    _compare_greedy(got.tolist(), want, margins)


@pytest.mark.parametrize("bits,group", CKPTS)
def test_two_slot_persistent_mma_gemv(bits, group, engines, oracles):
    import qwen3tts_b200 as q

    d, twin = _ck(bits, group)
    rec, want, margins = _reference(twin, oracles)
    eng = engines(d, max_batch=2, load_codec=False)
    e0, ec = _logit_err(eng, q, rec)
    assert eng.timing().persistent_launches >= 1
    print(f"[{bits}-bit g{group}] two-slot persistent kernel max-abs logit error: code0 {e0:.3e}, code predictor {ec:.3e}")
    assert e0 <= MMA_TOL and ec <= MMA_TOL
    got = eng.generate_codes_batch([_greq(q, max_tokens=20), _greq(q, max_tokens=20)])
    assert eng.timing().persistent_launches >= 1
    for g in got:
        _compare_greedy(g.tolist(), want, margins)


@pytest.mark.parametrize("packed_gemm", [2, 1])
@pytest.mark.parametrize("bits,group", CKPTS)
def test_eight_slot_tensor_core_step(bits, group, packed_gemm, engines, oracles):
    """8 slots: the batched tensor-core step, on the fp16 copies (packed_gemm=2) and streaming the packed container (packed_gemm=1)."""
    import qwen3tts_b200 as q

    d, twin = _ck(bits, group)
    rec, want, margins = _reference(twin, oracles)
    eng = engines(d, max_batch=8, load_codec=False, packed_gemm=packed_gemm)
    e0, ec = _logit_err(eng, q, rec)
    assert eng.timing().persistent_launches == 0
    print(f"[{bits}-bit g{group}] 8-slot tensor-core step (packed_gemm={packed_gemm}) max-abs logit error: code0 {e0:.3e}, code predictor {ec:.3e}")
    assert e0 <= LOGIT_TOL and ec <= LOGIT_TOL
    got = eng.generate_codes_batch([_greq(q, max_tokens=20)] * 3)
    for g in got:
        _compare_greedy(g.tolist(), want, margins)


@pytest.mark.parametrize("bits,group", [(2, 64), (3, 32), (5, 64), (6, 128)])
def test_offline_dequant_load_branch_widths(bits, group, engines):
    """`quantization_config` without `quantization`: the leaves are widened, then dequantised offline to fp16 dense weights."""
    import qwen3tts_b200 as q
    from oracle import talker as otalker

    d, twin = _ck(bits, group, quant_key="quantization_config")
    eng = engines(d, load_codec=False)
    assert eng.info.quant_bits == 0 and eng.info.weight_dtype == 1 and eng.info.checkpoint_quant_bits == bits
    orc = otalker.TalkerOracle(twin)
    assert not orc.pre_quantized and orc.bits == CONTAINER[bits]
    rec, grec = {}, {}
    orc.generate_codes(otalker.Request(text_ids=TEXT_IDS, speaker_id=2861, temperature=0.0, max_tokens=F), forced=_forced(), record=rec, filter_invalid=False)
    e0, ec = _logit_err(eng, q, rec)
    print(f"[offline dequant {bits}-bit g{group}] max-abs logit error: code0 {e0:.3e}, code predictor {ec:.3e}")
    assert e0 <= LOGIT_TOL and ec <= LOGIT_TOL
    want = orc.generate_codes(otalker.Request(text_ids=TEXT_IDS, speaker_id=2861, temperature=0.0, max_tokens=20), record=grec, filter_invalid=False)
    _compare_greedy(eng.generate_codes(_greq(q, max_tokens=20)).tolist(), want, grec["margins"])


# ------------------------------------------------------------------------------------------------ the container is the only difference
@pytest.mark.parametrize("bits", [2, 3, 5, 6])
def test_container_is_the_only_difference(bits):
    import qwen3tts_b200 as q

    d, twin = _ck(bits, 64)
    for slots in (1, 8):
        out = []
        for path in (d, twin):
            eng = q.Engine(path, max_batch=slots, max_frames=64, load_codec=False)
            try:
                assert eng.info.quant_bits == CONTAINER[bits]
                _, lg = eng.generate_codes(_greq(q, max_tokens=F, forced_codes=_forced(), want_logits=F))
                ids = eng.generate_codes_batch([_greq(q, max_tokens=16, temperature=0.8, top_k=40, seed=s) for s in range(min(slots, 4))])
                out.append((lg["code0_logits"].copy(), lg["cp_logits"].copy(), [i.tolist() for i in ids]))
            finally:
                eng.close()
        assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1]), f"{bits}-bit vs its twin, {slots} slot(s): logits differ"
        assert out[0][2] == out[1][2], f"{bits}-bit vs its twin, {slots} slot(s): codes differ"


# ------------------------------------------------------------------------------------------------ refusals with a device
def _create_status(d):
    """q3tts_create on `d`: (status, handle pointer left behind)."""
    from qwen3tts_b200 import _abi as A

    L = A.lib()
    o = A.Options()
    L.q3tts_default_options(C.byref(o))
    o.max_frames, o.load_codec = 64, 0
    h = C.c_void_p()
    st = L.q3tts_create(str(d).encode(), C.byref(o), C.byref(h))
    if h.value:
        L.q3tts_destroy(h)
    return st, h.value


def _with_config(src, tag, **quant):
    dst = os.path.join(CKPT_ROOT, f"refuse_{tag}")
    shutil.rmtree(dst, ignore_errors=True)
    os.makedirs(dst)
    shutil.copy(os.path.join(src, "model.safetensors"), dst)
    cfg = json.load(open(os.path.join(src, "config.json")))
    cfg["quantization"].update(quant)
    json.dump(cfg, open(os.path.join(dst, "config.json"), "w"), indent=1)
    return dst


def test_create_refuses_unsupported_widths_and_mismatched_leaves():
    from qwen3tts_b200 import _abi as A

    cases = [("bits7", _ck(6, 64)[0], dict(bits=7), A.ERR_BAD_CONFIG),
             ("bits1", _ck(2, 64)[0], dict(bits=1), A.ERR_BAD_CONFIG),
             ("g16", _ck(3, 32)[0], dict(group_size=16), A.ERR_BAD_CONFIG),
             ("six_over_four", ckpt("tiny", 4), dict(bits=6), A.ERR_BAD_WEIGHTS),
             ("three_over_six", _ck(6, 64)[0], dict(bits=3), A.ERR_BAD_WEIGHTS)]
    for tag, src, quant, want in cases:
        d = _with_config(src, tag, **quant)
        st, h = _create_status(d)
        shutil.rmtree(d, ignore_errors=True)
        assert st == want and not h, f"{tag}: status {st}, handle {h}"


# ------------------------------------------------------------------------------------------------ full size
@pytest.mark.slow
@pytest.mark.parametrize("bits", [6, 3])
def test_full_size_widths_batch64_and_persistent(bits):
    """0.6B, g64, BASELINE init: the 64-row tensor-core step (strict 1e-2 teacher-forced logits on three rows, margin-checked greedy ids)
    and batch 1 on the persistent kernel (1e-2), as test_batch64_tensor_core_step_strict_logits_and_greedy and
    test_persistent_kernel_full_size_logits do for 4 and 8 bits."""
    import qwen3tts_b200 as q
    from oracle import talker as otalker

    d, twin = _ck(bits, 64, name="0.6b", init="baseline")
    orc = otalker.TalkerOracle(twin)  # the same codes, scales and biases in 8 / 4-bit words
    B, Ff = 64, 3
    rng = np.random.default_rng(11)
    ids = [rng.integers(0, 150000, size=int(rng.integers(8, 41)) + 9).tolist() for _ in range(B)]
    spk = [3066, 3065, 3010, 3061, 2861, 2873, 2864, 2875, 2878]
    forced = np.random.default_rng(4).integers(0, 2048, size=(B, Ff, 16)).astype(np.int32)

    def reqs(frames, with_forced):
        return [q.GenRequest(text_ids=ids[i], speaker_id=spk[i % len(spk)], temperature=0.0, max_tokens=frames, keep_invalid_frames=True,
                             forced_codes=forced[i] if with_forced else None) for i in range(B)]

    def oracle_logits(i):
        rec = {}
        orc.generate_codes(otalker.Request(text_ids=ids[i], speaker_id=spk[i % len(spk)], temperature=0.0, max_tokens=Ff), forced=forced[i], record=rec,
                           filter_invalid=False)
        return rec

    eng = q.Engine(d, max_batch=B, max_frames=64, load_codec=False)
    try:
        assert eng.info.checkpoint_quant_bits == bits and eng.info.quant_bits == CONTAINER[bits]
        for j in (0, 31, 63):
            r = reqs(Ff, True)
            r[j].want_logits = Ff
            _, lg = eng.generate_codes_batch(r)
            assert eng.timing().persistent_launches == 0
            rec = oracle_logits(j)
            e0, ec = np.abs(lg["code0_logits"] - rec["code0_logits"]).max(), np.abs(lg["cp_logits"] - rec["cp_logits"]).max()
            print(f"[0.6b {bits}-bit] row {j} of 64: code0 {e0:.3e}, code predictor {ec:.3e}")
            assert e0 <= LOGIT_TOL and ec <= LOGIT_TOL
        G = 4
        outs = eng.generate_codes_batch(reqs(G, False))
        for i in (0, 22, 50, 63):
            rec = {}
            want = orc.generate_codes(otalker.Request(text_ids=ids[i], speaker_id=spk[i % len(spk)], temperature=0.0, max_tokens=G), record=rec,
                                      filter_invalid=False)
            _compare_greedy(outs[i].tolist(), want, rec["margins"])
    finally:
        eng.close()
    eng = q.Engine(d, max_frames=64, load_codec=False)
    try:
        _, lg = eng.generate_codes(q.GenRequest(text_ids=ids[0], speaker_id=spk[0], temperature=0.0, max_tokens=Ff, forced_codes=forced[0],
                                                keep_invalid_frames=True, want_logits=Ff))
        assert eng.timing().persistent_launches >= 1
    finally:
        eng.close()
    rec = oracle_logits(0)
    e0, ec = np.abs(lg["code0_logits"] - rec["code0_logits"]).max(), np.abs(lg["cp_logits"] - rec["cp_logits"]).max()
    print(f"[0.6b {bits}-bit] batch 1, persistent kernel: code0 {e0:.3e}, code predictor {ec:.3e}")
    assert e0 <= LOGIT_TOL and ec <= LOGIT_TOL
