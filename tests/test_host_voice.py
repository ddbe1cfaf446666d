"""CPU: the registered-voice ABI (q3tts_voice_*, q3tts_request.voice, q3tts_timing.prefill_rows).  The new fields take space from
`reserved`, so every existing field keeps its offset and both structs keep their size; refusals that need no device return at once."""
import ctypes
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# sizeof / offsetof on x86-64 Linux before the voice fields existed
REQUEST_SIZE = 184
REQUEST_OFFSETS = {"struct_size": 0, "text_ids": 8, "n_text_ids": 16, "instruct_ids": 24, "n_instruct_ids": 32, "speaker_id": 36,
                   "speaker_embedding": 40, "speaker_embedding_dim": 48, "ref_text_ids": 56, "n_ref_text_ids": 64, "ref_codes": 72,
                   "ref_frames": 80, "temperature": 84, "top_k": 88, "top_p": 92, "repetition_penalty": 96, "max_tokens": 100, "seed": 104,
                   "stream_variant": 112, "forced_codes": 120, "n_forced_frames": 128, "code0_logits_out": 136, "cp_logits_out": 144,
                   "logits_capacity_frames": 152, "keep_invalid_frames": 156}
TIMING_SIZE = 120
TIMING_OFFSETS = {"device_ms": 0, "prefill_ms": 8, "decode_ms": 16, "kernel_launches": 24, "graph_replays": 32, "frames": 40, "h2d_bytes": 48,
                  "d2h_bytes": 56, "weight_bytes_per_frame": 64, "talker_ms": 72, "codec_flops": 80, "persistent_launches": 88}
NEW_REQUEST = {"voice": 160, "reserved": 168}
NEW_TIMING = {"prefill_rows": 96, "reserved": 104}


def _offsets(S):
    return {n: getattr(S, n).offset for n, _ in S._fields_}


def test_ctypes_layout_keeps_every_existing_field():
    from qwen3tts_b200 import _abi

    assert ctypes.sizeof(_abi.Request) == REQUEST_SIZE and ctypes.sizeof(_abi.Timing) == TIMING_SIZE
    assert _offsets(_abi.Request) == {**REQUEST_OFFSETS, **NEW_REQUEST}
    assert _offsets(_abi.Timing) == {**TIMING_OFFSETS, **NEW_TIMING}
    assert NEW_REQUEST["voice"] % 8 == 0


def test_c_compiler_agrees_with_the_mirror(tmp_path):
    cc = shutil.which("cc") or shutil.which("gcc") or shutil.which("clang")
    if cc is None:
        pytest.skip("no C compiler")
    from qwen3tts_b200 import _abi

    fields = [("q3tts_request", f) for f, _ in _abi.Request._fields_] + [("q3tts_timing", f) for f, _ in _abi.Timing._fields_]
    src = ["#include <stddef.h>", "#include <stdio.h>", '#include "qwen3tts_b200.h"', "int main(void) {",
           '  printf("q3tts_request sizeof %zu\\n", sizeof(q3tts_request));', '  printf("q3tts_timing sizeof %zu\\n", sizeof(q3tts_timing));']
    src += [f'  printf("{s} {f} %zu\\n", offsetof({s}, {f}));' for s, f in fields]
    src += ["  return 0;", "}"]
    (tmp_path / "layout.c").write_text("\n".join(src) + "\n")
    exe = tmp_path / "layout"
    subprocess.run([cc, "-std=c99", "-I", os.path.join(ROOT, "include"), str(tmp_path / "layout.c"), "-o", str(exe)], check=True)
    got = {}
    for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines():
        s, f, v = line.split()
        got[(s, f)] = int(v)
    assert got[("q3tts_request", "sizeof")] == ctypes.sizeof(_abi.Request) == REQUEST_SIZE
    assert got[("q3tts_timing", "sizeof")] == ctypes.sizeof(_abi.Timing) == TIMING_SIZE
    for s, S in (("q3tts_request", _abi.Request), ("q3tts_timing", _abi.Timing)):
        for f, off in _offsets(S).items():
            assert got[(s, f)] == off, (s, f, got[(s, f)], off)


def test_default_request_has_no_voice():
    import qwen3tts_b200 as q
    from qwen3tts_b200 import _abi

    r = _abi.Request()
    ctypes.memset(ctypes.byref(r), 0xAB, ctypes.sizeof(r))
    q.lib().q3tts_default_request(ctypes.byref(r))
    assert r.voice is None and r.struct_size == REQUEST_SIZE


def test_voice_calls_refuse_null_before_any_device():
    import qwen3tts_b200 as q
    from qwen3tts_b200 import _abi

    L = q.lib()
    r = _abi.Request()
    L.q3tts_default_request(ctypes.byref(r))
    out = ctypes.c_void_p(0x1234)
    assert L.q3tts_voice_create(None, ctypes.byref(r), ctypes.byref(out)) == _abi.ERR_INVALID_ARG
    assert out.value is None  # cleared even when refused
    assert L.q3tts_voice_create(None, ctypes.byref(r), None) == _abi.ERR_INVALID_ARG
    assert L.q3tts_voice_create(None, None, None) == _abi.ERR_INVALID_ARG
    n, b = _abi.i32(7), _abi.i64(7)
    assert L.q3tts_voice_info(None, ctypes.byref(n), ctypes.byref(b)) == _abi.ERR_INVALID_ARG
    L.q3tts_voice_free(None)  # no-op


def test_genrequest_carries_the_voice_pointer():
    import qwen3tts_b200 as q

    class FakeVoice:  # what to_c reads of a Voice
        ptr = 0x1000

    r = q.GenRequest(text_ids=list(range(12)), voice=FakeVoice()).to_c()
    assert r.voice == 0x1000 and r.speaker_id == -1 and not r.instruct_ids and not r.ref_codes
    assert q.GenRequest(text_ids=list(range(12))).to_c().voice is None
