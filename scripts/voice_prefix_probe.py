"""What a registered voice (q3tts_voice) saves, measured in one run on one GPU, with the card's name and power limit.

  1. batch-1 time to first audio (q3tts_stream_begin -> first q3tts_stream_next_audio, wall clock) with the voice inline and with
     a voice, alternating, for an ICL clone of a 6 s reference (75 frames, 20-id transcript) and a VoiceDesign instruct of 40 ids, on
     0.6B MLX 4-bit and on 1.7B bf16 runtime-quantised at load (BASELINE init); with prefill_ms / prefill_rows of each arm;
  2. a config-5-shaped generate_to_file (24 text chunks x 600 frames, 32-slot handle, 1.7B runtime-quantised) as CustomVoice and as
     an ICL clone: wall time and audio-s/s of the pipeline as it runs now (one voice per call) against inline requests;
  3. q3tts_voice_create wall time and device bytes per voice.
Every output of the voice arm is compared bit for bit with the inline arm's.  Prints one JSON document; --out writes it too.

    python scripts/voice_prefix_probe.py --reps 7 --out voice_prefix.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "mlx-swift-qwen3-tts_b200"))

import numpy as np  # noqa: E402

INIT = "baseline"
CKPT_ROOT = os.environ.get("Q3TTS_TEST_CKPT", "/tmp/q3tts_test_ckpt")


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return out.strip().splitlines()[0] if out.strip() else "unknown"


def stats(xs):
    xs = np.asarray(xs, dtype=np.float64)
    return {"median": float(np.median(xs)), "min": float(xs.min()), "max": float(xs.max()), "n": int(xs.size)}


def checkpoints():
    from oracle import checkpoint

    d06 = checkpoint.write_checkpoint(os.path.join(CKPT_ROOT, f"0.6b_b4_bf16_s0_init{INIT}"), "0.6b", bits=4, dtype="bf16", seed=0, init=INIT)
    d17 = checkpoint.write_checkpoint(os.path.join(CKPT_ROOT, f"1.7b-cv_b0_bf16_s0_init{INIT}_enc"), "1.7b-cv", bits=0, dtype="bf16", seed=0,
                                      init=INIT, encoder="full", speaker_encoder="full")
    return d06, d17


def voice_cases():
    rng = np.random.default_rng(1)
    role = [151644, 77091, 198]  # <|im_start|> assistant \n
    return {
        "icl_clone_6s": dict(ref_text_ids=[int(i) for i in rng.integers(1000, 50000, 20)], ref_codes=rng.integers(0, 2048, (16, 75)).astype(np.int32)),
        "voice_design_40": dict(instruct_ids=[int(i) for i in rng.integers(1000, 50000, 40)]),
    }, role


def ttfa(q, d, rtq, reps, warmup):
    eng = q.Engine(d, max_batch=1, runtime_quantization=rtq)
    cases, role = voice_cases()
    text = role + [int(i) for i in np.random.default_rng(2).integers(1000, 50000, 24)]
    res = {}
    try:
        for name, fields in cases.items():
            t0 = time.perf_counter()
            v = eng.create_voice(q.GenRequest(text_ids=text, **fields))
            create_ms = (time.perf_counter() - t0) * 1e3
            arms = {"inline": dict(fields), "voice": dict(voice=v)}
            rec = {a: {"ttfa_ms": [], "prefill_ms": [], "prefill_rows": set()} for a in arms}
            first = {}
            identical = True
            for i in range(warmup + reps):
                for arm, kw in arms.items():
                    req = q.GenRequest(text_ids=text, temperature=0.85, seed=100 + i, max_tokens=60, **kw)
                    t0 = time.perf_counter()
                    st = eng.stream(req, 12)
                    tm = eng.timing()
                    pcm, _, _, _ = st.next_audio()
                    dt = (time.perf_counter() - t0) * 1e3
                    st.close()
                    first[arm] = pcm.view(np.uint32).copy()
                    if i >= warmup:
                        rec[arm]["ttfa_ms"].append(dt)
                        rec[arm]["prefill_ms"].append(tm.prefill_ms)
                        rec[arm]["prefill_rows"].add(int(tm.prefill_rows))
                identical &= bool(np.array_equal(first["inline"], first["voice"])) and first["inline"].size > 0
            res[name] = {"prefix_positions": v.prefix_positions, "voice_device_bytes": v.device_bytes, "voice_create_ms": create_ms,
                         "first_audio_identical": identical,
                         **{arm: {"ttfa_ms": stats(r["ttfa_ms"]), "prefill_ms": stats(r["prefill_ms"]), "prefill_rows": sorted(r["prefill_rows"])}
                            for arm, r in rec.items()}}
            v.close()
    finally:
        eng.close()
    return res


def config5(q, d17, reps):
    p = q.Qwen3TTSPipeline(d17, q.Qwen3TTSPipelineConfiguration(max_batch=32))
    sentence = "The quick brown fox jumps over the lazy dog near the quiet river bank while the evening light fades slowly. "
    text = sentence * 24
    chunks = q.TextChunker.chunk(text, q.TextChunker.default_max_words)
    tt = np.arange(24000 * 6) / 24000.0
    clip = (0.2 * np.sin(2 * np.pi * 220 * tt) * np.sin(2 * np.pi * 3 * tt) + 0.05 * np.random.default_rng(5).standard_normal(tt.size)).astype(np.float32)
    codes = p.encode_reference_audio(clip)
    voice_call = p._call_voice
    inline_call = lambda n, voice, **f: (voice, None)  # noqa: E731  what the pipeline did before voices: every chunk inline
    res = {"text_chunks": len(chunks)}
    try:
        with tempfile.TemporaryDirectory() as td:
            for tag, kw in (("custom_voice", dict(speaker="aiden", instruct="Speak slowly, in a warm and calm voice.")),
                            ("icl_clone", dict(reference_transcript="This is the reference recording.", reference_audio_codes=codes))):
                p.generate_to_file(sentence * 2, os.path.join(td, "warm.wav"), **kw)  # warm-up: graphs, workspaces
                wall = {"inline": [], "voice": []}
                files = {}
                identical = True
                for i in range(reps):
                    for arm, fn in (("inline", inline_call), ("voice", voice_call)):
                        p._call_voice = fn
                        path = os.path.join(td, f"{tag}_{arm}.wav")
                        t0 = time.perf_counter()
                        n = p.generate_to_file(text, path, **kw)
                        wall[arm].append(time.perf_counter() - t0)
                        files[arm] = open(path, "rb").read()
                        rows = p.engine.timing().prefill_rows
                    identical &= files["inline"] == files["voice"]
                res[tag] = {"audio_s": n / 24000.0, "files_identical": identical, "last_call_prefill_rows_voice": int(rows),
                            **{arm: {"wall_s": stats(w), "audio_s_per_s_median": n / 24000.0 / float(np.median(w))} for arm, w in wall.items()}}
    finally:
        p._call_voice = voice_call
        p.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--config5-reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import qwen3tts_b200 as q

    out = {"card": card()}

    def emit():  # after every section: a run cut short keeps what it measured
        s = json.dumps(out, indent=1)
        print(s, flush=True)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                f.write(s)

    d06, d17 = checkpoints()
    out["ttfa_batch1"] = {"0.6b_mlx4": ttfa(q, d06, False, a.reps, a.warmup)}
    emit()
    out["ttfa_batch1"]["1.7b_bf16_runtime_q"] = ttfa(q, d17, True, a.reps, a.warmup)
    emit()
    out["config5_generate_to_file"] = config5(q, d17, a.config5_reps)
    out["card_after"] = card()
    emit()


if __name__ == "__main__":
    main()
