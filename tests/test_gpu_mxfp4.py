"""GPU: MLX mxfp4 checkpoints through the C ABI vs the CPU oracle.

The loader converts each mxfp4 leaf (E2M1 codes, one E8M0 byte per 32) into an exact 8-bit affine group of 32 with bf16 scale and bias, the
container every decode kernel already reads.  So the device container equals tests/mlx_mxfp4.py's `mxfp4_to_affine` bit for bit, its
dequantisation equals the mxfp4 values, every decode path meets the bar of its existing 4/8-bit test, and an mxfp4 checkpoint and its 8-bit
twin give identical bits.  The oracle dequantises affine words only, so every reference is computed on the twin.  Bars: LOGIT_TOL as in
test_gpu_talker.py, 1e-3 for the 2-slot persistent kernel, the probe bars of test_quantized_matmul_widths and
test_dequant_fused_tensor_core_gemm_widths."""
import ctypes as C
import json
import os
import shutil

import numpy as np
import pytest

import mlx_mxfp4
from conftest import CKPT_ROOT, TEXT_IDS, ckpt
from oracle import mlx_quant

pytestmark = pytest.mark.gpu

LOGIT_TOL = 1e-2
MMA_TOL = 1e-3
MARGIN_TOL = 2e-2
F = 12


def _ck(name="tiny", **kw):
    """(mxfp4 checkpoint, its 8-bit g32 twin) -- cached under the test checkpoint root."""
    tag = f"mxfp4_{name}" + "".join(f"_{k}{v}" for k, v in sorted(kw.items()))
    return mlx_mxfp4.write_mxfp4_checkpoint(os.path.join(CKPT_ROOT, tag), name, **kw)


def _forced():
    return np.random.default_rng(31).integers(0, 2048, size=(F, 16)).astype(np.int32)


def _greq(q, **kw):
    kw.setdefault("temperature", 0.0)
    return q.GenRequest(text_ids=TEXT_IDS, speaker_id=2861, keep_invalid_frames=True, **kw)


_REF = {}


def _reference(d, oracles):
    """The oracle's teacher-forced logits and free-running greedy ids (with margins) of checkpoint `d` (a twin), computed once."""
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


def _leaves(out_f, in_f, seed, scale=0.02):
    rng = np.random.default_rng(seed)
    w = (rng.standard_normal((out_f, in_f)) * scale).astype(np.float32)
    w[min(5, out_f - 1)] = 0.0
    codes, e = mlx_mxfp4.mxfp4_quantize_codes(w)
    return mlx_quant.pack(codes, 4), e


# ------------------------------------------------------------------------------------------------ the conversion probe
def test_probe_container_is_bit_exact():
    """Every code x every exponent 0..251 over an odd row count: codes, scales and biases == mxfp4_to_affine, bit for bit; dequantised
    through q3tts_dequantize (bits 8, group 32, bf16 scales) they equal the mxfp4 values in f32, f16 and bf16."""
    import qwen3tts_b200 as q

    rows = 9
    groups = -(-(mlx_mxfp4.MAX_SCALE_BYTE + 1) // rows)
    e = np.resize(np.arange(mlx_mxfp4.MAX_SCALE_BYTE + 1), rows * groups).reshape(rows, groups).astype(np.uint8)
    codes = ((np.arange(groups * 32)[None, :] + 5 * np.arange(rows)[:, None]) % 16).astype(np.uint32)
    packed = mlx_quant.pack(codes, 4)
    got_w, got_s, got_b = q.mxfp4_to_affine(packed, e)
    want_w, want_s, want_b = mlx_mxfp4.mxfp4_to_affine(packed, e)
    assert np.array_equal(got_w, want_w)
    assert np.array_equal(got_s.view(np.uint32), want_s.view(np.uint32)) and np.array_equal(got_b.view(np.uint32), want_b.view(np.uint32))
    for odt in ("f32", "f16", "bf16"):
        with np.errstate(over="ignore"):
            want = mlx_mxfp4.mxfp4_dequantize(packed, e, odt)
        got = q.dequantize(got_w, got_s, got_b, 32, 8, "bf16", odt)
        assert np.array_equal(got, want), odt
        assert np.array_equal(got.view(np.uint32)[codes != 8], want.view(np.uint32)[codes != 8]), odt


@pytest.mark.parametrize("shape", [(1, 1024, 1024), (2, 512, 2048), (5, 200, 1024), (19, 96, 256)])
def test_quantized_matmul_on_the_container(shape):
    """test_quantized_matmul_widths's bar: the talker's GEMV on the container == x . mxfp4(W)^T at fp32-accumulation error."""
    import qwen3tts_b200 as q

    m, out_f, in_f = shape
    packed, e = _leaves(out_f, in_f, m * 1000 + out_f)
    x = np.random.default_rng(m).standard_normal((m, in_f)).astype(np.float32)
    w8, s, b = q.mxfp4_to_affine(packed, e)
    wd = mlx_mxfp4.mxfp4_dequantize(packed, e).astype(np.float64)
    got = q.quantized_matmul(x, w8, s, b, 32, 8, "bf16")
    want = x.astype(np.float64) @ wd.T
    scale = np.abs(x).astype(np.float64) @ np.abs(wd).T
    assert np.all(np.abs(got - want) <= 4e-6 * scale + 1e-6), f"max err {np.abs(got - want).max():.3e}"


@pytest.mark.parametrize("shape", [(1, 1024, 1024), (24, 1024, 2048), (64, 3072, 1024), (128, 256, 512), (5, 160, 256)])
def test_dequant_fused_tensor_core_gemm_on_the_container(shape):
    """test_dequant_fused_tensor_core_gemm_widths's bar: the tcgen05 GEMM on the container == fp16(x) . fp16(mxfp4(W))^T, fp32 accumulate."""
    import qwen3tts_b200 as q

    m, out_f, in_f = shape
    packed, e = _leaves(out_f, in_f, m * 7 + out_f)
    x = np.random.default_rng(m + 1).standard_normal((m, in_f)).astype(np.float32)
    w8, s, b = q.mxfp4_to_affine(packed, e)
    wd = mlx_mxfp4.mxfp4_dequantize(packed, e, "f16").astype(np.float64)
    x16 = x.astype(np.float16).astype(np.float64)
    got = q.quantized_matmul_tc(x, w8, s, b, 32, 8, "bf16")
    want = x16 @ wd.T
    bound = 4e-6 * (np.abs(x16) @ np.abs(wd).T) + 1e-6
    assert np.all(np.abs(got - want) <= bound), f"max err {np.abs(got - want).max():.3e} (bound {bound.max():.3e})"


# ------------------------------------------------------------------------------------------------ every decode path
def test_info_reports_mode_and_widths(engines):
    eng = engines(_ck()[0], load_codec=False)
    i = eng.info
    assert (i.checkpoint_quant_mode, i.checkpoint_quant_bits, i.quant_bits, i.quant_group_size) == (1, 4, 8, 32)
    assert i.weight_dtype == 2  # Q3TTS_BF16: the container's scales
    twin = engines(_ck()[1], load_codec=False).info
    assert (twin.checkpoint_quant_mode, twin.checkpoint_quant_bits, twin.quant_bits, twin.quant_group_size) == (0, 8, 8, 32)
    affine = engines(ckpt("tiny", 4), load_codec=False).info
    assert affine.checkpoint_quant_mode == 0 and affine.checkpoint_quant_bits == 4


def test_persistent_frame_kernel(engines, oracles):
    import qwen3tts_b200 as q

    d, twin = _ck()
    rec, want, margins = _reference(twin, oracles)
    eng = engines(d, load_codec=False)
    e0, ec = _logit_err(eng, q, rec)
    assert eng.timing().persistent_launches >= 1
    print(f"[mxfp4] persistent kernel teacher-forced max-abs logit error: code0 {e0:.3e}, code predictor {ec:.3e}")
    assert e0 <= LOGIT_TOL and ec <= LOGIT_TOL
    got = eng.generate_codes(_greq(q, max_tokens=20))
    assert eng.timing().persistent_launches >= 1
    _compare_greedy(got.tolist(), want, margins)


def test_cuda_graph_path(oracles, monkeypatch):
    import qwen3tts_b200 as q

    d, twin = _ck()
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
    print(f"[mxfp4] CUDA-graph path teacher-forced max-abs logit error: code0 {e0:.3e}, code predictor {ec:.3e}")
    assert e0 <= LOGIT_TOL and ec <= LOGIT_TOL
    _compare_greedy(got.tolist(), want, margins)


def test_two_slot_persistent_mma_gemv(engines, oracles):
    import qwen3tts_b200 as q

    d, twin = _ck()
    rec, want, margins = _reference(twin, oracles)
    eng = engines(d, max_batch=2, load_codec=False)
    e0, ec = _logit_err(eng, q, rec)
    assert eng.timing().persistent_launches >= 1
    print(f"[mxfp4] two-slot persistent kernel max-abs logit error: code0 {e0:.3e}, code predictor {ec:.3e}")
    assert e0 <= MMA_TOL and ec <= MMA_TOL
    got = eng.generate_codes_batch([_greq(q, max_tokens=20), _greq(q, max_tokens=20)])
    assert eng.timing().persistent_launches >= 1
    for g in got:
        _compare_greedy(g.tolist(), want, margins)


@pytest.mark.parametrize("packed_gemm", [2, 1])
def test_eight_slot_tensor_core_step(packed_gemm, engines, oracles):
    """8 slots: the batched tensor-core step, on the fp16 copies (packed_gemm=2) and streaming the 8-bit container (packed_gemm=1)."""
    import qwen3tts_b200 as q

    d, twin = _ck()
    rec, want, margins = _reference(twin, oracles)
    eng = engines(d, max_batch=8, load_codec=False, packed_gemm=packed_gemm)
    e0, ec = _logit_err(eng, q, rec)
    assert eng.timing().persistent_launches == 0
    print(f"[mxfp4] 8-slot tensor-core step (packed_gemm={packed_gemm}) max-abs logit error: code0 {e0:.3e}, code predictor {ec:.3e}")
    assert e0 <= LOGIT_TOL and ec <= LOGIT_TOL
    got = eng.generate_codes_batch([_greq(q, max_tokens=20)] * 3)
    for g in got:
        _compare_greedy(g.tolist(), want, margins)


def test_offline_dequant_load_branch(engines):
    """`quantization_config` without `quantization`: the leaves are converted, then dequantised offline to fp16 dense weights."""
    import qwen3tts_b200 as q
    from oracle import talker as otalker

    d, twin = _ck(quant_key="quantization_config")
    eng = engines(d, load_codec=False)
    assert eng.info.quant_bits == 0 and eng.info.weight_dtype == 1 and eng.info.checkpoint_quant_bits == 4 and eng.info.checkpoint_quant_mode == 1
    orc = otalker.TalkerOracle(twin)
    assert not orc.pre_quantized and orc.bits == 8
    rec, grec = {}, {}
    orc.generate_codes(otalker.Request(text_ids=TEXT_IDS, speaker_id=2861, temperature=0.0, max_tokens=F), forced=_forced(), record=rec, filter_invalid=False)
    e0, ec = _logit_err(eng, q, rec)
    print(f"[offline dequant mxfp4] max-abs logit error: code0 {e0:.3e}, code predictor {ec:.3e}")
    assert e0 <= LOGIT_TOL and ec <= LOGIT_TOL
    want = orc.generate_codes(otalker.Request(text_ids=TEXT_IDS, speaker_id=2861, temperature=0.0, max_tokens=20), record=grec, filter_invalid=False)
    _compare_greedy(eng.generate_codes(_greq(q, max_tokens=20)).tolist(), want, grec["margins"])


# ------------------------------------------------------------------------------------------------ the container is the only difference
def test_container_is_the_only_difference():
    import qwen3tts_b200 as q

    d, twin = _ck()
    for slots in (1, 8):
        out = []
        for path in (d, twin):
            eng = q.Engine(path, max_batch=slots, max_frames=64, load_codec=False)
            try:
                assert eng.info.quant_bits == 8 and eng.info.quant_group_size == 32
                _, lg = eng.generate_codes(_greq(q, max_tokens=F, forced_codes=_forced(), want_logits=F))
                ids = eng.generate_codes_batch([_greq(q, max_tokens=16, temperature=0.8, top_k=40, seed=s) for s in range(min(slots, 4))])
                out.append((lg["code0_logits"].copy(), lg["cp_logits"].copy(), [i.tolist() for i in ids]))
            finally:
                eng.close()
        assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1]), f"mxfp4 vs its twin, {slots} slot(s): logits differ"
        assert out[0][2] == out[1][2], f"mxfp4 vs its twin, {slots} slot(s): codes differ"


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


def _variant(src, tag, quant=None, scale_byte=None):
    """A copy of checkpoint `src` with its `quantization` block replaced by `quant`, or with scale byte `scale_byte` in one mxfp4 leaf."""
    from safetensors.torch import load_file, save_file

    dst = os.path.join(CKPT_ROOT, f"refuse_mxfp4_{tag}")
    shutil.rmtree(dst, ignore_errors=True)
    os.makedirs(dst)
    cfg = json.load(open(os.path.join(src, "config.json")))
    if quant is not None:
        cfg["quantization"] = quant
    json.dump(cfg, open(os.path.join(dst, "config.json"), "w"), indent=1)
    if scale_byte is None:
        shutil.copy(os.path.join(src, "model.safetensors"), dst)
    else:
        t = load_file(os.path.join(src, "model.safetensors"))
        k = sorted(k for k in t if k.endswith(".scales"))[-1]
        t[k] = t[k].clone()
        t[k][-1, -1] = scale_byte
        save_file(t, os.path.join(dst, "model.safetensors"))
    return dst


def test_create_refuses_unsupported_modes_and_bad_leaves():
    from qwen3tts_b200 import _abi as A

    mx = _ck()[0]
    cases = [("nvfp4", mx, dict(quant={"group_size": 16, "bits": 4, "mode": "nvfp4"}), A.ERR_BAD_CONFIG),
             ("mxfp8", mx, dict(quant={"group_size": 32, "bits": 8, "mode": "mxfp8"}), A.ERR_BAD_CONFIG),
             ("unknown", mx, dict(quant={"group_size": 32, "bits": 4, "mode": "e2m1-please"}), A.ERR_BAD_CONFIG),
             ("bits8", mx, dict(quant={"group_size": 32, "bits": 8, "mode": "mxfp4"}), A.ERR_BAD_CONFIG),
             ("g64", mx, dict(quant={"group_size": 64, "bits": 4, "mode": "mxfp4"}), A.ERR_BAD_CONFIG),
             ("over_affine", ckpt("tiny", 4), dict(quant={"mode": "mxfp4"}), A.ERR_BAD_WEIGHTS),
             ("byte252", mx, dict(scale_byte=252), A.ERR_BAD_WEIGHTS),
             ("byte255", mx, dict(scale_byte=255), A.ERR_BAD_WEIGHTS)]
    for tag, src, kw, want in cases:
        d = _variant(src, tag, **kw)
        st, h = _create_status(d)
        shutil.rmtree(d, ignore_errors=True)
        assert st == want and not h, f"{tag}: status {st}, handle {h}"


# ------------------------------------------------------------------------------------------------ full size
@pytest.mark.slow
def test_full_size_mxfp4_batch64_and_persistent():
    """0.6B, BASELINE init: the 64-row tensor-core step (strict 1e-2 teacher-forced logits on three rows, margin-checked greedy ids) and
    batch 1 on the persistent kernel (1e-2), as test_full_size_widths_batch64_and_persistent does for 3 and 6 bits."""
    import qwen3tts_b200 as q
    from oracle import talker as otalker

    d, twin = _ck(name="0.6b", init="baseline")
    orc = otalker.TalkerOracle(twin)
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
        assert eng.info.checkpoint_quant_mode == 1 and eng.info.quant_bits == 8 and eng.info.quant_group_size == 32
        for j in (0, 31, 63):
            r = reqs(Ff, True)
            r[j].want_logits = Ff
            _, lg = eng.generate_codes_batch(r)
            assert eng.timing().persistent_launches == 0
            rec = oracle_logits(j)
            e0, ec = np.abs(lg["code0_logits"] - rec["code0_logits"]).max(), np.abs(lg["cp_logits"] - rec["cp_logits"]).max()
            print(f"[0.6b mxfp4] row {j} of 64: code0 {e0:.3e}, code predictor {ec:.3e}")
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
    print(f"[0.6b mxfp4] batch 1, persistent kernel: code0 {e0:.3e}, code predictor {ec:.3e}")
    assert e0 <= LOGIT_TOL and ec <= LOGIT_TOL
