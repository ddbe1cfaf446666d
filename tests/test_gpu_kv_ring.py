"""The talker's KV ring past its capacity, on every decode path (tiny checkpoints, through the C ABI).

An utterance's keys / values sit in a ring of kv_capacity positions: absolute position p at ring index p % kv_capacity, the live window
starting at win_start (trimmed to 192 keys every 15th frame step).  A single stream on default options wraps its ring after about 490
frames (~39 s of audio).  Capacity only changes WHERE a key is stored, never the order of any sum, so logits must be bit-identical across
capacities; a ring index that is off by one changes one key among ~200, which can hide inside a logit tolerance but not inside bit-identity.

Decode paths (chosen at handle creation; each test asserts the one it ran through q3tts_timing):
  P1  max_batch 1                        persistent frame kernel, fp32 rings
  P2  max_batch 1, Q3TTS_MEGAKERNEL=0    CUDA graph of small kernels (rope_attention_kernel), fp32 rings
  P3  max_batch 2                        two-row persistent frame kernel (tensor-core GEMV), fp32 rings
  P4  max_batch 4                        tensor-core step, fp16 rings
  P5  max_batch 4, Q3TTS_KV_F16=0        tensor-core step, fp32 rings
"""
import contextlib
import os

import numpy as np
import pytest

from conftest import TEXT_IDS, ckpt

pytestmark = pytest.mark.gpu

LOGIT_TOL = 1e-2   # the suite's teacher-forced bar (fp16 tensor-core operands)
FP32_TOL = 1e-3    # fp32-activation paths (test_two_utterance_persistent_kernel)
F = 480            # teacher-forced frames: P + F ~ 490 wraps a 208 ring twice and never a 512 ring
CAPS = [208, 211, 300]

PATHS = {
    "P1": dict(max_batch=1, env={}),
    "P2": dict(max_batch=1, env={"Q3TTS_MEGAKERNEL": "0"}),
    "P3": dict(max_batch=2, env={}),
    "P4": dict(max_batch=4, env={}),
    "P5": dict(max_batch=4, env={"Q3TTS_KV_F16": "0"}),
}
CKPTS = {"tiny8": lambda: ckpt("tiny", 8), "tiny4": lambda: ckpt("tiny", 4)}
CASES = [("P1", "tiny8"), ("P2", "tiny8"), ("P3", "tiny8"), ("P3", "tiny4"), ("P4", "tiny8"), ("P5", "tiny8")]


@contextlib.contextmanager
def _env(extra):
    old = {k: os.environ.get(k) for k in extra}
    os.environ.update(extra)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _engine(d, path, cap, max_frames=512):
    import qwen3tts_b200 as q

    with _env(PATHS[path]["env"]):  # read at handle creation
        return q.Engine(d, max_batch=PATHS[path]["max_batch"], kv_capacity=cap, max_frames=max_frames, load_codec=False)


def _assert_path(path, eng):
    t = eng.timing()
    if path in ("P1", "P3"):
        assert t.persistent_launches >= 1, (path, t.persistent_launches)
    elif path == "P2":
        assert t.persistent_launches == 0 and t.graph_replays >= 1, (path, t.persistent_launches, t.graph_replays)
    else:
        assert t.persistent_launches == 0, (path, t.persistent_launches)


def _forced(n, seed):
    return np.random.default_rng(seed).integers(0, 2048, size=(n, 16)).astype(np.int32)


def _logits(eng, req):
    frames, lg = eng.generate_codes(req)
    assert frames.tolist() == req.forced_codes.tolist()
    return lg["code0_logits"].copy(), lg["cp_logits"].copy()


FORCED = _forced(F, 31)


def _long_request():
    import qwen3tts_b200 as q

    return q.GenRequest(text_ids=TEXT_IDS, speaker_id=2861, temperature=0.0, max_tokens=F, forced_codes=FORCED, keep_invalid_frames=True,
                        want_logits=F)


@pytest.fixture(scope="module")
def ring_runs():
    """(path, checkpoint, capacity) -> (code0 logits, cp logits) of the long teacher-forced request, each run once."""
    cache = {}

    def get(path, ck, cap):
        key = (path, ck, cap)
        if key not in cache:
            eng = _engine(CKPTS[ck](), path, cap)
            try:
                cache[key] = _logits(eng, _long_request())
                _assert_path(path, eng)
            finally:
                eng.close()
        return cache[key]

    return get


@pytest.fixture(scope="module")
def oracle_long():
    """checkpoint -> oracle record of the long teacher-forced request (its result depends on neither path nor capacity)."""
    from oracle import talker as otalker

    cache = {}

    def get(ck):
        if ck not in cache:
            rec = {}
            o = otalker.TalkerOracle(CKPTS[ck]())
            o.generate_codes(otalker.Request(text_ids=TEXT_IDS, speaker_id=2861, temperature=0.0, max_tokens=F), forced=FORCED, record=rec,
                             filter_invalid=False)
            P = o.build_prompt(otalker.Request(text_ids=TEXT_IDS, speaker_id=2861))[0].shape[0]
            cache[ck] = (rec, P)
        return cache[ck]

    return get


# ------------------------------------------------------------------------------------------------ 1. capacity invariance
@pytest.mark.parametrize("path,ck", CASES)
def test_capacity_changes_no_bit(path, ck, ring_runs, oracle_long):
    """Wrapped rings (208: twice, 211 and 300: once) give the logits of a ring that never wraps (512), bit for bit."""
    _, P = oracle_long(ck)
    assert P + F > 2 * 208 and P + F < 512
    base = ring_runs(path, ck, 512)
    for cap in CAPS:
        got = ring_runs(path, ck, cap)
        for name, a, b in (("code0", got[0], base[0]), ("code predictor", got[1], base[1])):
            if not np.array_equal(a, b):
                f = int(np.argmax(np.any((a != b).reshape(len(a), -1), axis=1)))
                raise AssertionError(f"[{path} {ck}] {name} logits at kv_capacity {cap} differ from 512 from frame {f} (position {P + f}, "
                                     f"ring index {(P + f) % cap}); max diff {np.abs(a - b).max():.3e}")


def test_capacity_above_512_leaves_the_frame_kernel(tiny8, ring_runs):
    """The frame kernel splits a window into 4 key tiles of <= 128 keys, so a single-slot handle with kv_capacity > 512 takes the CUDA-graph
    path instead -- the same bits as that path at 512."""
    eng = _engine(tiny8, "P1", 640)
    try:
        got = _logits(eng, _long_request())
        t = eng.timing()
        assert t.persistent_launches == 0 and t.graph_replays >= 1, (t.persistent_launches, t.graph_replays)
        assert eng.info.kv_capacity == 640
    finally:
        eng.close()
    want = ring_runs("P2", "tiny8", 512)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


def test_capacity_below_208_is_raised_to_208(tiny8):
    """q3tts_create raises kv_capacity to 208 = window + 16 (a 192-key window plus 15 frames between trims and the current position)."""
    import qwen3tts_b200 as q

    eng = q.Engine(tiny8, kv_capacity=100, max_frames=16, load_codec=False)
    try:
        assert eng.info.kv_capacity == 208
    finally:
        eng.close()


# ------------------------------------------------------------------------------------------------ 2. oracle parity past the wrap
@pytest.mark.parametrize("path,ck", CASES)
def test_oracle_parity_past_the_wrap(path, ck, ring_runs, oracle_long):
    rec, P = oracle_long(ck)
    l0, lc = ring_runs(path, ck, 208)
    e0 = np.abs(l0 - rec["code0_logits"]).max()
    ec = np.abs(lc - rec["cp_logits"]).max()
    bar = LOGIT_TOL if path in ("P4", "P5") else FP32_TOL
    print(f"[{path} {ck}] kv_capacity 208, {F} frames after a {P}-position prompt (ring wrapped twice): max-abs logit error vs oracle "
          f"code0 {e0:.3e}, code predictor {ec:.3e} (bar {bar:.0e})")
    assert e0 <= bar and ec <= bar


# ------------------------------------------------------------------------------------------------ 3. long prefill at the capacity edge
REF_TEXT = [51, 52, 53, 54]


def _icl_request(R, n_frames, forced_seed=41):
    import qwen3tts_b200 as q

    ref = (np.arange(16 * R).reshape(16, R) * 37 % 2048).astype(np.int32)
    return q.GenRequest(text_ids=TEXT_IDS, ref_text_ids=REF_TEXT, ref_codes=ref, temperature=0.0, max_tokens=n_frames,
                        forced_codes=_forced(n_frames, forced_seed), keep_invalid_frames=True, want_logits=n_frames)


def test_prefill_of_capacity_minus_16(tiny8, ring_runs):
    """P = C - 16 (C = 512) through ICL reference frames: accepted; 40 frames cross the trims at steps 15 and 30 (the first drops
    P + 15 - 192 = 319 positions at once) and follow the oracle on P1, P2 and P4.  On P1 the window reaches S = P + 15 = 511 keys: all four
    128-key tiles of the frame kernel are full.  P2 gives the same bits at C = 512 and C = 1024.  P = C - 15 is refused with
    Q3TTS_ERR_CAPACITY and leaves the handle serving requests."""
    import qwen3tts_b200 as q
    from qwen3tts_b200 import _abi as A
    from oracle import talker as otalker

    C, n = 512, 40
    orc = otalker.TalkerOracle(tiny8)
    prompt_len = lambda R: orc.build_prompt(otalker.Request(text_ids=TEXT_IDS, ref_text_ids=REF_TEXT, ref_codes=np.zeros((16, R), np.int32)))[0].shape[0]
    R = 1 + (C - 16) - prompt_len(1)
    assert prompt_len(R) == C - 16 and prompt_len(R) + 15 == C - 1
    req = _icl_request(R, n)
    rec = {}
    orc.generate_codes(otalker.Request(text_ids=TEXT_IDS, ref_text_ids=REF_TEXT, ref_codes=req.ref_codes, temperature=0.0, max_tokens=n),
                       forced=req.forced_codes, record=rec, filter_invalid=False)
    got = {}
    for path in ("P1", "P2", "P4"):
        eng = _engine(tiny8, path, C, max_frames=64)
        try:
            got[path] = _logits(eng, req)
            _assert_path(path, eng)
            if path == "P1":  # one position more does not fit; the refusal leaves the handle usable
                with pytest.raises(q.Q3Error) as e:
                    eng.generate_codes(_icl_request(R + 1, n))
                assert e.value.status == A.ERR_CAPACITY
                short = _long_request()
                short.max_tokens, short.forced_codes, short.want_logits = 20, FORCED[:20], 20
                after = _logits(eng, short)
                base = ring_runs("P1", "tiny8", 512)
                assert np.array_equal(after[0], base[0][:20]) and np.array_equal(after[1], base[1][:20])
        finally:
            eng.close()
        e0 = np.abs(got[path][0] - rec["code0_logits"]).max()
        ec = np.abs(got[path][1] - rec["cp_logits"]).max()
        bar = LOGIT_TOL if path == "P4" else FP32_TOL
        print(f"[{path}] prefill of {C - 16} positions at kv_capacity {C}: max-abs logit error vs oracle code0 {e0:.3e}, code predictor {ec:.3e}")
        assert e0 <= bar and ec <= bar
    eng = _engine(tiny8, "P2", 1024, max_frames=64)
    try:
        wide = _logits(eng, req)
    finally:
        eng.close()
    assert np.array_equal(wide[0], got["P2"][0]) and np.array_equal(wide[1], got["P2"][1])


# ------------------------------------------------------------------------------------------------ 4. slot reuse, split admission, wrapped rings
def test_batch_on_wrapped_rings_equals_singles(tiny8):
    """A 4-slot handle at kv_capacity 208 serves 7 ICL requests (prompts of 20..192 positions).  Their admission estimates (ref text + ref
    frames + 10 rows each, csrc/api.cu run_batch) exceed max_prefill_rows() = max(2 * 4, 208, 96 * 4) = 384 for the first four, so admission
    takes several prefill passes; requests 0, 2, 4 and 5 wrap their ring (request 0 twice), the others do not; slots are reused after
    wrapped utterances.  The text keeps EOS suppressed, so every utterance runs its max_tokens.  Codes equal what the same handle gives each
    request alone, bit for bit, greedy and sampled."""
    import qwen3tts_b200 as q

    spec = [(180, 230), (12, 40), (100, 150), (60, 20), (150, 60), (30, 250), (8, 10)]  # (reference frames, frames)
    ests = [len(REF_TEXT) + R + 10 for R, _ in spec]
    assert sum(ests[:4]) > 384
    eng = q.Engine(tiny8, max_batch=4, kv_capacity=208, max_frames=512, load_codec=False)
    try:
        assert eng.info.kv_capacity == 208
        for sampled in (False, True):
            reqs = []
            for i, (R, n) in enumerate(spec):
                ref = (np.arange(16 * R).reshape(16, R) * (31 + i) % 2048).astype(np.int32)
                text = [11, 21, 22] + list(range(100 + 3 * i, 100 + 3 * i + n + 7))  # n + 10 ids: n + 1 trailing rows
                reqs.append(q.GenRequest(text_ids=text, ref_text_ids=REF_TEXT, ref_codes=ref, temperature=0.9 if sampled else 0.0,
                                         top_k=50 if sampled else 0, seed=500 + i, max_tokens=n, keep_invalid_frames=True))
            batch = [b.tolist() for b in eng.generate_codes_batch(reqs)]
            assert eng.timing().persistent_launches == 0
            wrapped = [R + 12 + len(b) > 208 for (R, _), b in zip(spec, batch)]
            assert [len(b) for b in batch] == [n for _, n in spec]
            assert wrapped == [True, False, True, False, True, True, False], wrapped
            singles = [eng.generate_codes(r).tolist() for r in reqs]
            for i in range(len(reqs)):
                assert batch[i] == singles[i], f"request {i} ({'sampled' if sampled else 'greedy'}) differs between the batch and alone"
    finally:
        eng.close()
