"""GPU: registered voices (q3tts_voice).  A request with a voice installs the voice's prefilled K / V and prefills its firstText row
only; it must give the bits of the same request with the voice fields written inline -- greedy, sampled and teacher-forced, on every
decode path -- and q3tts_timing.prefill_rows shows which of the two ran."""
import threading

import numpy as np
import pytest

from conftest import TEXT_IDS

pytestmark = pytest.mark.gpu

EMB = (np.random.default_rng(7).standard_normal(256) * 0.5).astype(np.float32)  # tiny: hidden 256


def _codes(frames, mul=37):
    return (np.arange(16 * frames).reshape(16, frames) * mul % 2048).astype(np.int32)


KINDS = {
    "instruct": dict(instruct_ids=[41, 42, 43, 44, 45]),
    "instruct_speaker": dict(speaker_id=3066, instruct_ids=[41, 42, 43, 44, 45]),
    "icl": dict(ref_text_ids=[51, 52, 53, 54], ref_codes=_codes(7)),
    "icl_long": dict(ref_text_ids=list(range(51, 71)), ref_codes=_codes(48, 53)),
    "speaker_id": dict(speaker_id=2861),
    "speaker_embedding": dict(speaker_embedding=EMB),
    "role_only": dict(),
}
FORCED = np.random.default_rng(3).integers(0, 2048, size=(12, 16)).astype(np.int32)
MODES = {
    "greedy": dict(temperature=0.0, max_tokens=16),
    "sampled": dict(temperature=0.9, top_k=50, seed=1234, max_tokens=16),
    "forced": dict(temperature=0.0, forced_codes=FORCED, want_logits=len(FORCED)),
}
HANDLES = {  # (checkpoint fixture, Engine options): every decode path of the engine
    "persistent_1": ("tiny8", dict(max_batch=1)),
    "two_slot": ("tiny8", dict(max_batch=2)),
    "graph_1": ("tiny8", dict(max_batch=1, kv_capacity=600)),
    "tc_8": ("tiny8", dict(max_batch=8)),
    "tc_8_packed": ("tiny4", dict(max_batch=8, packed_gemm=1)),
    "bf16_runtime_q": ("tiny_bf16", dict(max_batch=1, runtime_quantization=True)),
}


def _prefix_positions(kind):
    n_front = len(kind.get("instruct_ids") or kind.get("ref_text_ids") or [])
    n_ref = kind["ref_codes"].shape[1] if "ref_codes" in kind and "instruct_ids" not in kind else 0
    has_spk = kind.get("speaker_id", -1) >= 0 or "speaker_embedding" in kind
    return n_front + n_ref + 3 + (5 if has_spk else 4)


def _run(eng, text_ids=TEXT_IDS, voice=None, kind=None, **mode):
    import qwen3tts_b200 as q

    req = q.GenRequest(text_ids=text_ids, voice=voice, keep_invalid_frames=True, **(kind if voice is None else {}), **mode)
    out = eng.generate_codes(req)
    frames, logits = out if req.want_logits else (out, None)
    return frames, logits, eng.timing()


def _same(a, b):
    fa, la, _ = a
    fb, lb, _ = b
    assert np.array_equal(fa, fb), "codes differ"
    if la is not None:
        for k in la:
            assert np.array_equal(la[k].view(np.uint32), lb[k].view(np.uint32)), f"{k} differ"


@pytest.mark.parametrize("handle", list(HANDLES))
def test_voice_equals_inline_bit_for_bit(handle, request, engines):
    import qwen3tts_b200 as q

    d, opts = HANDLES[handle]
    eng = engines(request.getfixturevalue(d), **opts)
    info = eng.info
    elem = 2 if opts["max_batch"] >= 3 else 4  # fp16 rings on tensor-core handles
    for name, kind in KINDS.items():
        with eng.create_voice(q.GenRequest(text_ids=TEXT_IDS, **kind)) as v:
            n = _prefix_positions(kind)
            assert v.prefix_positions == n, name
            assert v.device_bytes == n * 2 * info.num_layers * info.num_kv_heads * 128 * elem
            for mode, mkw in MODES.items():
                inline = _run(eng, kind=kind, **mkw)
                assert inline[2].prefill_rows == n + 1, (name, mode)
                voiced = _run(eng, voice=v, **mkw)
                assert voiced[2].prefill_rows == 1, (name, mode)
                if handle == "persistent_1":
                    assert voiced[2].persistent_launches > 0
                if handle == "graph_1":
                    assert voiced[2].persistent_launches == 0 and voiced[2].graph_replays > 0
                _same(voiced, inline)


@pytest.mark.parametrize("max_batch", [2, 4])
def test_mixed_admission(max_batch, tiny8, engines):
    """more requests than slots: voice A, inline A, voice B, no voice, voice A again -- continuous batching admits them in mixed rounds"""
    import qwen3tts_b200 as q

    eng = engines(tiny8, max_batch=max_batch)
    A, B = KINDS["icl"], KINDS["instruct_speaker"]
    with eng.create_voice(q.GenRequest(text_ids=TEXT_IDS, **A)) as va, eng.create_voice(q.GenRequest(text_ids=TEXT_IDS, **B)) as vb:
        texts = [TEXT_IDS[:3] + list(range(60 + 5 * i, 70 + 6 * i)) for i in range(5)]
        plan = [(va, A), (None, A), (vb, B), (None, {}), (va, A)]
        mk = lambda t, v, k: q.GenRequest(text_ids=t, voice=v, temperature=0.9, top_k=40, seed=11, max_tokens=14 + len(t) % 5,
                                          keep_invalid_frames=True, **(k if v is None else {}))
        got = eng.generate_codes_batch([mk(t, v, k) for t, (v, k) in zip(texts, plan)])
        want = [eng.generate_codes(mk(t, None, k)) for t, (_, k) in zip(texts, plan)]
        for g, w in zip(got, want):
            assert np.array_equal(g, w)


@pytest.mark.parametrize("max_batch", [1, 8])
def test_ring_wraps_and_window_trims_the_prefix(max_batch, tiny8, engines):
    """a 120-position ICL voice on a 208-position ring, 300 teacher-forced frames: the ring wraps and the window trims the prefix out"""
    import qwen3tts_b200 as q

    eng = engines(tiny8, max_batch=max_batch, kv_capacity=208, max_frames=320)
    kind = dict(ref_text_ids=list(range(51, 59)), ref_codes=_codes(105, 41))
    forced = np.random.default_rng(5).integers(0, 2048, size=(300, 16)).astype(np.int32)
    mode = dict(temperature=0.0, forced_codes=forced, want_logits=300)
    with eng.create_voice(q.GenRequest(text_ids=TEXT_IDS, **kind)) as v:
        assert v.prefix_positions == 120
        inline = _run(eng, kind=kind, **mode)
        voiced = _run(eng, voice=v, **mode)
    assert inline[2].prefill_rows == 121 and voiced[2].prefill_rows == 1
    assert np.array_equal(voiced[0], forced)
    _same(voiced, inline)


def test_stream_with_voice(tiny8, engines):
    import qwen3tts_b200 as q

    eng = engines(tiny8)
    kind = KINDS["icl_long"]
    mk = lambda v: q.GenRequest(text_ids=TEXT_IDS[:3] + list(range(100, 127)), voice=v, temperature=0.9, top_k=50, seed=3, max_tokens=40,
                                **(kind if v is None else {}))
    with eng.create_voice(q.GenRequest(text_ids=TEXT_IDS, **kind)) as v:
        for audio in (False, True):
            outs, rows = [], []
            for voice in (None, v):
                st = eng.stream(mk(voice), chunk_size=7)
                rows.append(eng.timing().prefill_rows)
                chunks = []
                try:
                    while True:
                        if audio:
                            pcm, rng, fin, done = st.next_audio()
                            chunks.append((pcm.view(np.uint32).tolist(), rng, fin))
                        else:
                            c, done = st.next_codes()
                            chunks.append(c.tolist())
                        if done:
                            break
                finally:
                    st.close()
                outs.append(chunks)
            assert rows == [_prefix_positions(kind) + 1, 1]
            assert len(outs[0]) > 1 and outs[0] == outs[1]


def test_voice_on_a_clone_from_another_thread(tiny8, engines):
    import qwen3tts_b200 as q

    parent = engines(tiny8, max_batch=2)
    kind = KINDS["speaker_embedding"]
    mode = dict(temperature=0.9, top_k=50, seed=77, max_tokens=20)
    clone = parent.clone()
    try:
        with parent.create_voice(q.GenRequest(text_ids=TEXT_IDS, **kind)) as v:
            want = _run(parent, kind=kind, **mode)
            res = {}
            t = threading.Thread(target=lambda: res.setdefault("got", _run(clone, voice=v, **mode)))
            t.start()
            t.join()
            assert res["got"][2].prefill_rows == 1
            _same(res["got"], want)
    finally:
        clone.close()


def test_lanes_with_voice_equal_single_lane_inline(tiny8, engines):
    import qwen3tts_b200 as q

    lanes = engines(tiny8, max_batch=2, lanes=2)
    single = engines(tiny8, max_batch=2)
    kind = KINDS["instruct"]
    texts = [TEXT_IDS[:3] + list(range(80 + 3 * i, 92 + 4 * i)) for i in range(5)]
    mk = lambda t, v: q.GenRequest(text_ids=t, voice=v, temperature=0.9, top_k=50, seed=5, max_tokens=12, **(kind if v is None else {}))
    with lanes.create_voice(q.GenRequest(text_ids=TEXT_IDS, **kind)) as v:
        got, gf = lanes.generate_pcm_batch([mk(t, v) for t in texts])
        assert lanes.timing().prefill_rows == len(texts)
    want, wf = single.generate_pcm_batch([mk(t, None) for t in texts])
    assert gf == wf
    for g, w in zip(got, want):
        assert np.array_equal(g.view(np.uint32), w.view(np.uint32))


def test_refusals_leave_the_handle_usable(tiny8, tiny4, engines):
    import qwen3tts_b200 as q

    eng = engines(tiny8)
    info = eng.info
    base = lambda: eng.generate_codes(q.GenRequest(text_ids=TEXT_IDS, speaker_id=2861, temperature=0.9, seed=9, max_tokens=10))
    before = base()

    def refused(status, fn):
        with pytest.raises(q.Q3Error) as e:
            fn()
        assert e.value.status == status, e.value.message
        assert np.array_equal(base(), before)
        return e.value.message

    with eng.create_voice(q.GenRequest(text_ids=TEXT_IDS, **KINDS["instruct"])) as v:
        refused(q._abi.ERR_INVALID_ARG, lambda: eng.generate_codes(q.GenRequest(text_ids=TEXT_IDS, voice=v, speaker_id=2861)))
        refused(q._abi.ERR_INVALID_ARG, lambda: eng.generate_codes(q.GenRequest(text_ids=TEXT_IDS, voice=v, instruct_ids=[41])))
        refused(q._abi.ERR_INVALID_ARG, lambda: eng.generate_codes(q.GenRequest(text_ids=[12] + TEXT_IDS[1:], voice=v)))
        # a too-short text still returns 0 frames
        assert len(eng.generate_codes(q.GenRequest(text_ids=TEXT_IDS[:8], voice=v, max_tokens=4))) == 0
        # handles that do not share this one's weights and options
        for other in (engines(tiny8, max_batch=2), engines(tiny4)):
            msg = refused(q._abi.ERR_INVALID_ARG, lambda: other.generate_codes(q.GenRequest(text_ids=TEXT_IDS, voice=v, max_tokens=4)))
            assert "clones" in msg
        # a batch refuses before running any of its requests
        refused(q._abi.ERR_INVALID_ARG, lambda: eng.generate_codes_batch([q.GenRequest(text_ids=TEXT_IDS, max_tokens=4),
                                                                          q.GenRequest(text_ids=TEXT_IDS, voice=v, speaker_id=1)]))
    small = engines(tiny8, kv_capacity=208)
    refused(q._abi.ERR_CAPACITY, lambda: small.create_voice(q.GenRequest(text_ids=TEXT_IDS, ref_text_ids=[51, 52, 53, 54], ref_codes=_codes(190))))
    st = eng.stream(q.GenRequest(text_ids=TEXT_IDS, speaker_id=2861, max_tokens=4))
    try:
        with pytest.raises(q.Q3Error) as e:
            eng.create_voice(q.GenRequest(text_ids=TEXT_IDS, speaker_id=2861))
        assert e.value.status == q._abi.ERR_INVALID_ARG
    finally:
        st.close()
    assert np.array_equal(base(), before)
    for bad in (dict(instruct_ids=[41, info.text_vocab_size]), dict(ref_text_ids=[51, 52], ref_codes=_codes(5) + info.vocab_size),
                dict(speaker_id=info.vocab_size), dict(text_ids=[info.text_vocab_size, 1, 2])):
        refused(q._abi.ERR_INVALID_ARG, lambda: eng.create_voice(q.GenRequest(**{"text_ids": TEXT_IDS, **bad})))


def test_free_order(tiny8):
    import qwen3tts_b200 as q

    kind = KINDS["speaker_id"]
    mode = dict(temperature=0.9, seed=21, max_tokens=10)
    eng = q.Engine(tiny8, max_frames=64, load_codec=False)
    want = _run(eng, kind=kind, **mode)
    v = eng.create_voice(q.GenRequest(text_ids=TEXT_IDS, **kind))
    _same(_run(eng, voice=v, **mode), want)
    v.close()  # voice first
    v = eng.create_voice(q.GenRequest(text_ids=TEXT_IDS, **kind))
    clone = eng.clone()
    eng.close()  # the creating handle first: the clone and the voice keep the weights
    _same(_run(clone, voice=v, **mode), want)
    clone.close()
    v.close()  # voice last, after every handle


LONG = ("The harbour was quiet before dawn, and the fishing boats rocked gently against their moorings while gulls circled overhead. "
        "Old Marta walked the length of the pier every morning, counting the boats and remembering the names of the sailors she had known. "
        "When the first light touched the water she would sit on the last bench and wait for the bakery to open across the square. "
        "Nobody in the village could say how long she had kept this habit, only that the morning did not feel complete without her.")


@pytest.mark.parametrize("what", ["to_file_icl", "to_file_instruct", "batch_instruct"])
def test_pipeline_calls_equal_inline(what, tiny8, tmp_path):
    """generate_to_file / generate_batch prefill the call's voice once; their bytes / samples equal what inline requests give"""
    import qwen3tts_b200 as q
    from oracle import pipeline as opipe

    p = q.Qwen3TTSPipeline(tiny8, q.Qwen3TTSPipelineConfiguration(max_batch=8))
    try:
        chunks = q.TextChunker.chunk(LONG, q.TextChunker.default_max_words)
        assert len(chunks) >= 3
        orig = p._request
        p._request = lambda *a, **kw: orig(*a, **{**kw, "max_tokens": 24, "temperature": 0.9})
        made = []
        create = p.engine.create_voice
        p.engine.create_voice = lambda r: made.append(create(r)) or made[-1]
        if what == "to_file_icl":
            fields = dict(reference_transcript="a quiet harbour", reference_audio_codes=_codes(48))
        else:
            fields = dict(speaker="aiden", instruct="a calm, low voice")
        if what == "batch_instruct":
            got = p.generate_batch(LONG, **fields)
            assert p.engine.timing().prefill_rows == len(chunks)  # one batched call, one row per chunk
            singles = [p.engine.generate_pcm(p._request(tc, **fields), q.DECODE_BATCHAPI)[0] for tc in chunks]
            want = opipe.crossfade_concat([s for s in singles if s.size], p.config.crossfade_samples)
            assert got.shape == want.shape and np.array_equal(got.view(np.uint32), want.view(np.uint32))
        else:
            n = p.generate_to_file(LONG, tmp_path / "v.wav", **fields)
            assert p.engine.timing().prefill_rows == len(chunks)
            w = q.StreamingWAVWriter(tmp_path / "inline.wav")
            for tc in chunks:
                pcm, _ = p.engine.generate_pcm(p._request(tc, **fields), q.DECODE_FILE)
                if pcm.size:
                    w.write(pcm)
            assert w.finalize() == n
            assert (tmp_path / "v.wav").read_bytes() == (tmp_path / "inline.wav").read_bytes()
        assert len(made) == 1 and made[0]._p is None, "the call's voice is created once and freed before the call returns"
    finally:
        p.close()
