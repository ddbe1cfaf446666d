#!/usr/bin/env python
"""bench.py — BASELINE.json metric on the B200 engine (and, with --impl reference, on the CPU restatement).

Workload of the headline line (BASELINE.json configs[1]): Qwen3-TTS-12Hz-0.6B, MLX 4-bit g64, `generateStream` semantics (stream
sampler variant, temperature 0.85, chunk 12, codec windows 18 / 8+18), `--batch` independent utterances per GPU (default 64) with
8-40 text ids from seed 1 and different speakers, `--frames` frames each (default 36 = two decode windows).  Synthetic seeded weights
drawn with BASELINE.md's init (every matrix N(0, 0.02^2), norms 1; no network).  One *step* = one such batch: prompt assembly +
prefill + 36 frame steps + windowed codec decode to PCM.

  value    = audio seconds produced by all GPUs / device time of the step (CUDA events on the engine's stream: talker span + codec
             passes; ids are tiny so "inputs resident" only excludes the PCM read-back);
  e2e      = the same through the public C-ABI call (`q3tts_generate_pcm_batch`) with host buffers, wall clock, including the H2D
             of ids/codes and the D2H of every PCM sample;
  roofline = the dominant kernel of the step (the <= 128-row tcgen05 GEMM that streams the packed weights), measured live with CUDA
             events over the 113 linear launches of one talker decode step (q3tts_profile_linear): ALGORITHMIC bytes (packed codes +
             scales + biases, SURVEY.md §8d) / average launch time, against MEASURED_PEAKS.json hbm_gbs; `traffic` = ncu dram bytes
             per launch of the same kernel, keyed by (model, bits) in profiles/traffic.json;
  latency  = batch-1 view (the reference's only mode): ms per frame of the persistent frame kernel and the MEASURED wall-clock
             time to the first audio chunk through q3tts_stream_begin -> q3tts_stream_next_audio;
  config3  = BASELINE.json configs[2]: 1.7B bf16, 512 utterances x 125 frames sharded over the ranks, whole-sequence decode, with the
             NCCL gather of lengths + PCM to rank 0 AFTER the timed region (its time reported separately);
  config4  = BASELINE.json configs[3]: codec decode only, 128 clips x 750 frames sharded over the ranks, chunkedDecode(100, 10) and
             whole-sequence T = 750;
  config5  = BASELINE.json configs[4] (one GPU): 1.7B CustomVoice generateToFile of a long text (chunk-parallel) as CustomVoice and as an
             ICL clone, with the reference-audio and speaker encoders timed on a 6 s clip.

Multi-GPU: request-parallel replicas (SURVEY.md §8e) — one process per GPU (torchrun), each with its own shard of utterances (weak
scaling on the headline line); NCCL carries only the barrier, the max-over-ranks time, the sums, and the result gather.

`--dump-outputs DIR` writes what the last timed step returned to its caller as DIR/*.npy (see dump_outputs).  Every step's requests
are drawn from its index, so the same arguments give the same inputs on every run and two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "mlx-swift-qwen3-tts_b200"))

import numpy as np  # noqa: E402

METRIC = "audio-sec generated per sec (RTFx)"
UNIT = "audio-sec/s"
SPEAKERS = [3066, 3065, 3010, 3061, 2861, 2873, 2864, 2875, 2878]
INIT = "baseline"  # oracle.checkpoint init: BASELINE.md §3


def make_requests(q, n, frames, seed, rank=0, lo=8, hi=41, temperature=0.85, stream=True):
    rng = np.random.default_rng(seed * 1000 + rank)
    reqs = []
    for i in range(n):
        n_ids = int(rng.integers(lo, hi)) + 9  # text ids + the 9 template ids
        ids = rng.integers(0, 150000, size=n_ids).tolist()
        reqs.append(q.GenRequest(text_ids=ids, speaker_id=SPEAKERS[i % len(SPEAKERS)], temperature=temperature, max_tokens=frames,
                                 seed=seed * 100000 + rank * 1000 + i, stream_variant=stream))
    return reqs


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.p, self.first = index, [], None, 0

    def mark(self):
        """samples before this point (warm-up) are not reported"""
        self.first = len(self.rows)

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def snapshot(self, last=None):
        rows = self.rows[self.first:last] or self.rows[-1:]
        sm = [float(r[0]) for r in rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}

    def stop(self):
        if self.p:
            self.p.terminate()


def ckpt_path(model, bits):
    """Same cache layout as tests/conftest.py::ckpt, so a box that already ran the GPU tests does not write the 1-6 GB files twice."""
    root = os.environ.get("Q3TTS_TEST_CKPT", "/tmp/q3tts_test_ckpt")
    return os.path.join(root, f"{model}_b{bits}_bf16_s0_init{INIT}")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return j.get("hbm_gbs", 6650.0), j.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, "fallback"


def dump_outputs(out_dir, pcm, frames, n_samples, suffix="", budget=63 << 20):
    """--dump-outputs: what the last timed q3tts_generate_pcm_batch call returned -- every utterance's PCM (float32, zero-padded to
    `n_samples`), its length in samples and its frame count -- as .npy files, so two builds can be compared output for output on
    identical inputs.  Above `budget` bytes of PCM (64 MB in all with the small per-utterance arrays) a fixed seeded sample of
    utterances is written; `utterance.npy` names the rows."""
    rows = np.arange(len(pcm))
    keep = max(1, budget // (4 * max(1, n_samples)))
    if keep < len(pcm):
        rows = np.sort(np.random.default_rng(0).choice(len(pcm), keep, replace=False))
    block = np.zeros((len(rows), n_samples), dtype=np.float32)
    for j, i in enumerate(rows):
        block[j, :pcm[i].size] = pcm[i]
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in (("pcm", block[:, :budget // 4]), ("pcm_samples", [pcm[i].size for i in rows]), ("frames", [frames[i] for i in rows]),
                      ("utterance", rows)):
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), np.asarray(arr, dtype=np.float32 if name == "pcm" else np.float64))


def workload_config(a, world):
    wfmt = f"{a.bits}-bit g64" if a.bits else "bf16"
    return {"workload": f"Qwen3-TTS-12Hz-{a.model} {wfmt} generateStream: {a.batch} utterances/GPU x {a.frames} frames, 8-40 text ids, stream windows 18/8+18 "
                        f"(BASELINE.json configs[1]; weights N(0, 0.02^2), norms 1)",
            "model": a.model, "bits": a.bits, "batch_per_gpu": a.batch, "frames": a.frames, "parallelism": f"request-parallel x{world}",
            "cache": "a frame-step walks 103 layer passes of weights (0.6B 4-bit: 0.93 GB packed = the algorithmic bytes; 3.3 GB as the fp16 operand copies the "
                     "default GEMM mode streams) + the KV rings of 64 utterances, >> L2 126 MB for the talker stack; the code predictor's five layers "
                     "are re-read 15x per frame and stay L2-resident by design; no explicit flush between steps (each step = 36 frame-steps)"}


# --------------------------------------------------------------------------------------------------- CPU restatement arm
def cpu_sample(ckpt_dir, frames, reps, warmup):
    """Times the CPU restatement of the reference graph (oracle/, torch-CPU fp32, all host threads) on a bounded sample of the SAME
    workload: ONE of the step's utterances at a time (batch 1 is the reference's only mode, Qwen3TTSPipeline.swift:484-624) — the
    stream-variant loop for `frames` frames, then the stream's codec windows (18, then 8 + 18).  Audio is counted like the GPU arm
    counts it: decoded PCM samples / 24000 (frames whose code0 is outside [0, 2048) produce none)."""
    import torch

    from oracle import codec as ocodec, pipeline as opipe, talker as otalker

    torch.set_num_threads(os.cpu_count() or 1)
    orc = otalker.TalkerOracle(ckpt_dir)
    cdc = ocodec.load_codec(ckpt_dir)
    rng = np.random.default_rng(1)
    times = []
    for it in range(warmup + reps):
        ids = rng.integers(0, 150000, size=int(rng.integers(8, 41)) + 9).tolist()
        n = frames if it >= warmup else 3  # warm-up runs only page the weights in
        t0 = time.perf_counter()
        fr = orc.generate_codes(otalker.Request(text_ids=ids, speaker_id=SPEAKERS[it % len(SPEAKERS)], temperature=0.85, max_tokens=n, seed=it,
                                                stream_variant=True), filter_invalid=False)
        chunks = opipe.stream_chunks(cdc, [fr[i:i + 12] for i in range(0, len(fr), 12)])
        samples = sum(int(c["samples"].size) for c in chunks)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append((samples / 24000.0, dt))
    audio = sum(a for a, _ in times)
    secs = sum(t for _, t in times)
    return audio / max(secs, 1e-9), secs / max(1, len(times))


def cpu_sample_text(frames):
    return (f"1 of the step's utterances per timed run (batch 1 = the reference's only mode): {frames} frames of the stream-variant loop + the stream's "
            f"codec windows (18, 8+18), audio counted as decoded PCM samples / 24000; CPU restatement of the reference graph (torch fp32, all host "
            f"threads), not MLX")


# --------------------------------------------------------------------------------------------------- extra blocks (all ranks)
def ckpt_17b_dir():
    return os.path.join(os.environ.get("Q3TTS_TEST_CKPT", "/tmp/q3tts_test_ckpt"), f"1.7b-cv_b0_bf16_s0_init{INIT}_enc")


def write_ckpt_17b(checkpoint):
    """ONE synthetic 1.7B checkpoint for configs 3 and 5: bf16, BASELINE init, `tts_model_type` custom_voice, with the ICL reference-audio encoder
    and the ECAPA speaker encoder (config 3 ignores the last three)."""
    return checkpoint.write_checkpoint(ckpt_17b_dir(), "1.7b-cv", bits=0, dtype="bf16", seed=0, init=INIT, encoder="full", speaker_encoder="full")


def run_config3(q, checkpoint, dist, a, rank, local_rank, world):
    """BASELINE.json configs[2]: 1.7B bf16, 512 synthetic utterances (ids 20-60 long, seed 2), 125 frames each, request-parallel."""
    import torch

    from qwen3tts_b200 import parallel

    d = ckpt_17b_dir()
    if rank == 0:
        write_ckpt_17b(checkpoint)
    if world > 1:
        dist.barrier()
    total, frames, B = a.config3_utterances, 125, 64
    idx = parallel.shard_indices(total, rank, world)
    # `--config3-handles` lanes per GPU: a batched frame step is a chain of ~570 dependent launches that leaves the SMs > 85 % idle, so
    # independent chains overlap (measured at 1.7B bf16, 512 utterances: 997 / 1408 / 1575 / 1712 audio-s/s with 1 / 2 / 3 / 4 handles fed from
    # host threads; one 128-row chain gains 1.24x over one 64-row chain).  Requests are independent (SURVEY.md §8e): which lane serves one
    # does not change its result.
    H = max(1, a.config3_handles)
    eng = q.Engine(d, device=local_rank, max_batch=B, max_frames=128, kv_capacity=512, lanes=H)  # q3tts_options.lanes: H chains inside ONE call
    up = eng.info.codec_total_upsample
    allreq = make_requests(q, total, frames, 2, 0, lo=20, hi=61, temperature=0.85, stream=False)
    mine = [allreq[i] for i in idx]
    eng.generate_pcm_batch(mine[:min(len(mine), B * H)], q.DECODE_WHOLE)  # warm-up: clones, graphs, workspaces
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    # one public call with the rank's whole share: the library splits it over its lanes (this handle + clones sharing its weights), every
    # lane batches continuously over its 64 slots
    pcm, _ = eng.generate_pcm_batch(mine, q.DECODE_WHOLE)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    tm = eng.timing()
    pcm = list(pcm)
    # device time of the call: the lanes overlap; q3tts_timing.device_ms is the slowest lane's CUDA-event span (talker + codec of its share)
    dev_s = (tm.device_ms if H > 1 else tm.talker_ms + tm.decode_ms) * 1e-3
    launches = int(tm.kernel_launches)
    samples = sum(int(p.size) for p in pcm)
    dev = torch.device("cuda", local_rank)
    t_wall, sums = parallel.aggregate(dist if world > 1 else None, dev, wall, samples, (launches,))
    t_dev, _ = parallel.aggregate(dist if world > 1 else None, dev, dev_s, 0)
    # result gather (north star: "NCCL only to gather results"): lengths + PCM of all 512 utterances to rank 0, outside the timed region
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    g0 = time.perf_counter()
    allpcm, lengths, moved = parallel.gather_pcm(dist if world > 1 else None, dev, pcm, total, rank, world)
    torch.cuda.synchronize()
    gather_s = time.perf_counter() - g0
    eng.close()
    if rank != 0:
        return None
    assert allpcm is not None and len(allpcm) == total and all(int(p.size) == l for p, l in zip(allpcm, lengths))
    return {"workload": f"BASELINE.json configs[2]: Qwen3-TTS-12Hz-1.7B (assumed dims H 2048 / MLP 6144, 2048->1024 code-predictor projection) bf16, "
                        f"{total} utterances x 125 frames sharded over {world} GPU(s), batches of {B}, {H} lane(s) per GPU (q3tts_options.lanes: one q3tts_generate_pcm_batch call per rank), whole-sequence decode",
            "lanes_per_gpu": H,
            "value": sums[0] / 24000.0 / t_dev, "e2e": sums[0] / 24000.0 / t_wall, "unit": UNIT, "n_gpus": world, "utterances": total,
            "device_s": t_dev, "wall_s": t_wall, "gpu_launches": int(sums[1]), "dtype": "bf16 weights -> f16 operands x f32 accumulate",
            "result_gather": {"collective": "all_reduce(lengths) + gather(PCM) to rank 0 over NCCL" if world > 1 else "single rank: no collective",
                              "seconds": gather_s, "bytes_into_rank0": moved, "utterances_on_rank0": len(allpcm)}}


def run_config5(q, checkpoint, a, local_rank):
    """BASELINE.json configs[4]: 1.7B CustomVoice long-text generateToFile with chunking + ICL reference-audio encode / clone (rank 0,
    one GPU).  Through the mirrored Swift API (qwen3tts_b200.Qwen3TTSPipeline): `encode_reference_audio` and `extract_speaker_embedding`
    of a 6 s clip, then two files of the same 24-sentence text -- (a) CustomVoice: speaker + instruct, (b) clone: reference transcript +
    the ICL codes -- with the reference's defaults (temperature 0.85, maxTokens 600 per text chunk, runtime 4/6-bit quantisation of the
    bf16 checkpoint ON).  Random weights never emit EOS, so every text chunk runs its 600 frames (48 s of audio)."""
    import tempfile

    d = write_ckpt_17b(checkpoint)
    t0 = time.perf_counter()
    p = q.Qwen3TTSPipeline(d, q.Qwen3TTSPipelineConfiguration(device=local_rank, max_batch=32))
    load_s = time.perf_counter() - t0
    try:
        assert p.supports_custom_voice and p.supports_icl and p.supports_voice_cloning
        tt = np.arange(24000 * 6) / 24000.0
        clip = (0.2 * np.sin(2 * np.pi * 220 * tt) * np.sin(2 * np.pi * 3 * tt) + 0.05 * np.random.default_rng(5).standard_normal(tt.size)).astype(np.float32)
        p.encode_reference_audio(clip)  # warm-up at the measured length (workspaces grow on first use)
        p.extract_speaker_embedding(clip)
        t0 = time.perf_counter()
        codes = p.encode_reference_audio(clip)
        enc_ms = (time.perf_counter() - t0) * 1e3
        enc_dev_ms = p.engine.timing().device_ms
        t0 = time.perf_counter()
        emb = p.extract_speaker_embedding(clip)
        spk_ms = (time.perf_counter() - t0) * 1e3
        spk_dev_ms = p.engine.timing().device_ms
        sentence = "The quick brown fox jumps over the lazy dog near the quiet river bank while the evening light fades slowly. "
        text = sentence * 24
        chunks = q.TextChunker.chunk(text, q.TextChunker.default_max_words)
        res = {}
        with tempfile.TemporaryDirectory() as td:
            for tag, kw in (("custom_voice", dict(speaker="aiden", instruct="Speak slowly, in a warm and calm voice.")),
                            ("icl_clone", dict(reference_transcript="This is the reference recording.", reference_audio_codes=codes))):
                path = os.path.join(td, tag + ".wav")
                if tag == "custom_voice":
                    p.generate_to_file(sentence * 2, path, **kw)  # warm-up: graphs, workspaces
                t0 = time.perf_counter()
                n = p.generate_to_file(text, path, **kw)
                wall = time.perf_counter() - t0
                res[tag] = {"samples": int(n), "audio_s": n / 24000.0, "wall_s": wall, "value": n / 24000.0 / wall, "unit": UNIT, "file_bytes": os.path.getsize(path)}
        return {"workload": "BASELINE.json configs[4]: Qwen3-TTS-12Hz-1.7B CustomVoice (assumed dims, bf16 checkpoint, runtime 4/6-bit quantisation at load = the "
                            f"reference's default), generateToFile of a {len(text.split())}-word text = {len(chunks)} text chunks x 600 frames run as ONE batch on a "
                            "32-slot handle, 16+8 codec windows, 16-bit WAV on disk; wall clock through the mirrored Swift API incl. tokenisation, H2D / D2H and the file write",
                "text_chunks": len(chunks), "load_s": load_s, **res,
                "encode_reference_audio": {"clip_s": 6.0, "frames": int(codes.shape[1]), "quantizers": int(codes.shape[0]), "wall_ms": enc_ms, "device_ms": enc_dev_ms},
                "extract_speaker_embedding": {"clip_s": 6.0, "dim": int(emb.size), "wall_ms": spk_ms, "device_ms": spk_dev_ms}}
    finally:
        p.close()


def run_config4(q, ckpt_dir, dist, a, rank, local_rank, world, tf):
    """BASELINE.json configs[3]: codec decode only, codes int32 [128, 750, 16] uniform in [0, 2048), seed 3; batch axis split over ranks."""
    import torch

    from qwen3tts_b200 import parallel

    clips_total, T = a.config4_clips, 750
    idx = parallel.shard_indices(clips_total, rank, world)
    codes = np.random.default_rng(3).integers(0, 2048, size=(clips_total, T, 16)).astype(np.int32)[idx]
    eng = q.Engine(ckpt_dir, device=local_rank, load_talker=False, codec_max_frames=3000)
    up = eng.info.codec_total_upsample
    res = {}
    dev = torch.device("cuda", local_rank)
    for mode in ("chunked", "whole"):
        fn = (lambda c: eng.decode_chunked(c, 100, 10)) if mode == "chunked" else eng.decode
        fn(codes[: min(4, len(codes))])  # warm-up at the measured window shape
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dev_ms, flops = 0.0, 0
        part = 32  # clips per call: bounds the host PCM buffer (32 x 1.44 M floats = 184 MB)
        for b0 in range(0, len(codes), part):
            fn(codes[b0:b0 + part])
            tm = eng.timing()
            dev_ms += tm.decode_ms
            flops += int(tm.codec_flops)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        samples = len(codes) * T * up
        t_dev, sums = parallel.aggregate(dist if world > 1 else None, dev, dev_ms * 1e-3, samples, (flops,))
        t_wall, _ = parallel.aggregate(dist if world > 1 else None, dev, wall, 0)
        res[mode] = {"samples_per_s": sums[0] / t_dev, "e2e_samples_per_s": sums[0] / t_wall, "device_s": t_dev, "wall_s": t_wall,
                     "tflops": sums[1] / t_dev / 1e12, "tensor_frac_of_peak": sums[1] / t_dev / 1e12 / (tf * world)}
    eng.close()
    if rank != 0:
        return None
    return {"workload": f"BASELINE.json configs[3]: speech_tokenizer decode only, {clips_total} clips x 750 frames (60 s) sharded over {world} GPU(s); "
                        "chunked = chunkedDecode(100, 10) -> windows of 110 stacked on the batch axis; whole = one T = 750 pass per clip",
            "unit": "samples/s", "peak_tflops_per_gpu": tf, "n_gpus": world, **res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--frames", type=int, default=36)
    ap.add_argument("--bits", type=int, default=4)
    ap.add_argument("--model", default="0.6b")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline line only (no latency / config3 / config4 blocks)")
    ap.add_argument("--config3", default="on", choices=["on", "off"])
    ap.add_argument("--config4", default="on", choices=["on", "off"])
    ap.add_argument("--config5", default="on", choices=["on", "off"])
    ap.add_argument("--config3-utterances", type=int, default=512)
    ap.add_argument("--config3-handles", type=int, default=4, help="q3tts_options.lanes of config3's handle: launch chains served concurrently per GPU (1 = one chain)")
    ap.add_argument("--config4-clips", type=int, default=128)
    ap.add_argument("--packed-gemm", type=int, default=0, choices=[0, 1, 2],
                    help="q3tts_options.packed_gemm of the measured handle: 1 = packed weights dequantised inside the tcgen05 GEMM, 2 / 0 = fp16 operand copies")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (PCM, samples and frames per utterance) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA engine (--impl b200)")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert world == max(1, a.gpus) or world == 1, f"WORLD_SIZE {world} != --gpus {a.gpus}"
    config = workload_config(a, max(1, a.gpus))
    fused_mode = a.bits in (4, 8) and (a.packed_gemm == 1 or (a.packed_gemm == 0 and os.environ.get("Q3TTS_SKINNY_Q", "0") not in ("", "0")))

    from oracle import checkpoint

    ckpt_dir = ckpt_path(a.model, a.bits)

    if a.impl == "reference":
        # The reference's own implementation of the path cannot run here (Swift + MLX, SURVEY.md §8c): this arm times the CPU
        # restatement (oracle/) on the host cores, rank 0 only, on a bounded sample of the SAME workload (see cpu_sample).
        if rank != 0:
            return
        checkpoint.write_checkpoint(ckpt_dir, a.model, bits=a.bits, dtype="bf16", seed=0, init=INIT)
        steps = max(1, a.steps)  # ~4 s of CPU work per step
        v, sec = cpu_sample(ckpt_dir, a.frames, steps, min(a.warmup, 1))
        cores = os.cpu_count() or 1
        # what THIS arm runs, in its own words (ADVICE r1): one utterance of the GPU arm's workload per step, batch 1
        config = dict(config)
        config["sampled_from"] = config["workload"]
        config["workload"] = (f"bounded sample of the GPU arm's workload: 1 utterance x {a.frames} frames per step (batch 1 = the reference's only mode), "
                              f"same stream windows 18/8+18, audio counted as decoded PCM samples; CPU restatement of the reference graph (oracle/), all host cores")
        config["batch_per_gpu"] = 1
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": steps, "warmup": min(a.warmup, 1),
                "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": cpu_sample_text(a.frames)},
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return

    # stdout carries exactly ONE JSON line.  Native libraries write there too (NCCL prints "NCCL version ..." from C on its first
    # communicator in this image, whatever NCCL_DEBUG says): file descriptor 1 points at stderr for the whole run and the JSON line
    # goes to the saved descriptor at the end.
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist

    import qwen3tts_b200 as q

    if world > 1:
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if rank == 0:
        checkpoint.write_checkpoint(ckpt_dir, a.model, bits=a.bits, dtype="bf16", seed=0, init=INIT)
    if world > 1:
        dist.barrier()

    # torch's own CUDA state (lazy init on first use) is brought up BEFORE the warm-up steps: initialising it at the
    # synchronize() that opens the timed region stalled kernel submission inside the first timed step on some boxes.
    torch.cuda.set_device(local_rank)
    torch.zeros(8, device="cuda").sum().item()
    torch.cuda.synchronize()
    eng = q.Engine(ckpt_dir, device=local_rank, max_batch=a.batch, max_frames=max(64, a.frames), kv_capacity=512, packed_gemm=a.packed_gemm)
    up = eng.info.codec_total_upsample
    out_bufs = [np.zeros(a.frames * up, dtype=np.float32) for _ in range(a.batch)]

    def step(i):
        reqs = make_requests(q, a.batch, a.frames, i, rank)
        t0 = time.perf_counter()
        pcm, frames = eng.generate_pcm_batch(reqs, q.DECODE_STREAM, out_buffers=out_bufs)
        wall = time.perf_counter() - t0
        tm = eng.timing()
        samples = int(sum(p.size for p in pcm))
        return {"wall": wall, "dev": (tm.talker_ms + tm.decode_ms) * 1e-3, "talker": tm.talker_ms * 1e-3, "decode": tm.decode_ms * 1e-3,
                "samples": samples, "frames": int(tm.frames), "launches": int(tm.kernel_launches), "h2d": int(tm.h2d_bytes), "d2h": int(tm.d2h_bytes),
                "codec_flops": int(tm.codec_flops), "bytes_frame": int(tm.weight_bytes_per_frame), "prefill": tm.prefill_ms * 1e-3,
                "out": (pcm, frames)}

    # nvidia-smi is started BEFORE the warm-up steps: its start-up (NVML init takes driver locks for tens to hundreds of ms on a
    # box without persistence mode) would otherwise stall kernel submission inside the first timed step; it keeps sampling
    # through the timed region, and only the samples taken after the warm-up are reported.
    sampler = ClockSampler(local_rank)
    sampler.start()
    for i in range(a.warmup):
        step(1000 + i)
    sampler.mark()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_begin = time.perf_counter()
    res = [step(i) for i in range(a.steps)]
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_total = time.perf_counter() - t_begin
    clocks = sampler.snapshot()
    n_clock_rows = len(sampler.rows)
    if a.dump_outputs:  # before the extra blocks below reuse out_bufs
        dump_outputs(a.dump_outputs, *res[-1]["out"], a.frames * up, f"_rank{rank}" if world > 1 else "")

    dev = sum(r["dev"] for r in res)
    wall = sum(r["wall"] for r in res)
    samples = sum(r["samples"] for r in res)
    stats = torch.tensor([dev, wall, t_total], dtype=torch.float64, device="cuda")
    sums = torch.tensor([samples, sum(r["launches"] for r in res), sum(r["h2d"] for r in res), sum(r["d2h"] for r in res)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)  # time = max over ranks
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)   # work = sum over ranks
    dev_max, wall_max, total_max = [float(x) for x in stats.tolist()]
    samples_all, launches_all, h2d_all, d2h_all = [float(x) for x in sums.tolist()]
    audio_s = samples_all / 24000.0

    hbm, tf, src = peaks()
    roof = lat = cpu_base = inflight = None
    extras = not a.no_extras
    if rank == 0 and extras:
        # ---- roofline of the dominant kernel, live (SURVEY.md §8d: algorithmic bytes = the weights as stored)
        iters = 20
        ms, n, nbytes = eng.profile_linear(0, a.batch, iters)
        packed = eng.info.quant_bits in (4, 8)
        fused = fused_mode
        streamed = nbytes  # bytes one launch set streams from HBM: the packed weights, or their fp16 copies (2 B / parameter)
        if packed and not fused and 3 <= a.batch <= 128:
            streamed = int(nbytes * 2.0 / (a.bits / 8.0 + 4.0 / 64.0))  # packed = bits/8 + (2+2)/64 B per parameter
        if 3 <= a.batch <= 128:
            kname = ("tc_skinny_q_kernel (tcgen05 / TMEM split-K cluster GEMM, MLX-packed weights streamed and dequantised in-kernel)" if fused
                     else "tc_skinny_kernel (tcgen05 / TMEM split-K cluster GEMM over fp16 operand copies of the weights)")
        elif a.batch > 128:
            kname = "tc_gemm_kernel (128-row-tile tcgen05 GEMM)"
        else:
            kname = "linear_kernel (dequant-fused GEMV)"
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")  # dram__bytes_read+write per launch from the committed ncu --set full captures
        key = f"{a.model}:{a.bits}:m{a.batch}"
        if os.path.exists(tp):
            traffic = (json.load(open(tp)).get(key) or {}).get("dram_bytes_per_launch")
        alg = nbytes / (n / iters)
        ach = nbytes * iters / (ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": kname + f"; the {n // iters} linear launches of one talker decode step at m = {a.batch} rows, replayed as a CUDA graph",
                "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm, "traffic": traffic, "traffic_key": key,
                "traffic_over_algorithmic": (traffic / alg) if traffic else None, "peak_source": src, "launches_timed": n,
                "algorithmic_bytes_per_launch": alg, "streamed_bytes_per_launch": streamed / (n / iters), "avg_launch_us": ms * 1e3 / n,
                "note": "latency-bound: ~600 dependent launches per frame-step, each far below the bytes one launch could move (DESIGN.md §3.2)"}
        # ---- batch-1 latency view (the reference's only mode), max_batch = 1 handle: persistent frame kernel + codec
        e1 = q.Engine(ckpt_dir, device=local_rank, max_batch=1, max_frames=64)
        r1 = q.GenRequest(text_ids=list(range(1000, 1024)), speaker_id=2861, temperature=0.85, max_tokens=36, stream_variant=True, keep_invalid_frames=True)
        e1.generate_codes(r1)
        e1.generate_codes(r1)
        t1 = e1.timing()
        msf = (t1.talker_ms - t1.prefill_ms) / max(1, t1.frames)
        ttfc = []
        for rep in range(4):  # wall clock: q3tts_stream_begin -> first q3tts_stream_next_audio returns (prefill + 18 frames + first window + D2H)
            w0 = time.perf_counter()
            st = e1.stream(r1, 12)
            s0, _, _, _ = st.next_audio()
            w1 = time.perf_counter()
            st.close()
            if rep:
                ttfc.append(((w1 - w0) * 1e3, int(s0.size)))
        ms1, n1, nb1 = eng.profile_linear(0, 1, iters)
        msc, nc, nbc = eng.profile_linear(1, 1, iters)
        lat = {"batch1_path": "persistent frame kernel (1 cooperative launch per run of frames)" if t1.persistent_launches else "CUDA graph of per-op kernels",
               "batch1_ms_per_frame": msf, "batch1_rtfx": 80.0 / msf, "batch1_prefill_ms": t1.prefill_ms,
               "batch1_frame_roofline_frac": (t1.weight_bytes_per_frame / (msf * 1e-3) / 1e9) / hbm,
               "batch1_frame_algorithmic_bytes": int(t1.weight_bytes_per_frame),
               "batch1_linear_gbs_talker_step": nb1 * iters / (ms1 * 1e-3) / 1e9, "batch1_linear_gbs_cp_pass_L2": nbc * iters / (msc * 1e-3) / 1e9,
               "time_to_first_chunk_ms": float(np.median([t for t, _ in ttfc])), "time_to_first_chunk_samples": ttfc[0][1],
               "time_to_first_chunk_how": "measured wall clock, q3tts_stream_begin -> first q3tts_stream_next_audio (18-frame window), median of 3",
               "like_for_like_single_stream_rtfx": 80.0 / msf}
        e1.close()
        # ---- the same step with several batches IN FLIGHT (not the headline: BASELINE.json configs[1] is one batch of 64): H handles on H host
        # threads, each generating `steps` of the headline's batches through the same public call with its own host buffers
        H = 4
        more = [eng.clone() for _ in range(H - 1)]  # q3tts_clone: shares eng's weights
        handles = [eng] + more
        bufs = [out_bufs] + [[np.zeros(a.frames * up, dtype=np.float32) for _ in range(a.batch)] for _ in more]
        got = [0] * H

        def serve(h, n_steps, seed0):
            for i in range(n_steps):
                pcm, _ = handles[h].generate_pcm_batch(make_requests(q, a.batch, a.frames, seed0 + 10 * h + i, rank), q.DECODE_STREAM, out_buffers=bufs[h])
                got[h] += int(sum(p.size for p in pcm))

        def run_all(n_steps, seed0):
            th = [threading.Thread(target=serve, args=(h, n_steps, seed0)) for h in range(H)]
            t0 = time.perf_counter()
            for t in th:
                t.start()
            for t in th:
                t.join()
            return time.perf_counter() - t0

        run_all(1, 2000)
        got = [0] * H
        torch.cuda.synchronize()
        w_inflight = run_all(a.steps, 3000)
        inflight = {"what": f"{H} handles on {H} host threads, {a.steps} batches of the headline workload each ({a.batch} utterances x {a.frames} frames, stream windows), "
                            "q3tts_generate_pcm_batch with host buffers, wall clock; NOT the headline configuration (one batch of 64 at a time) -- it shows what the "
                            "latency-bound launch chain leaves on the table when more than one batch is pending (DESIGN.md §7)",
                    "handles": H, "e2e_value": sum(got) / 24000.0 / w_inflight, "unit": UNIT, "wall_s": w_inflight, "utterances_in_flight": H * a.batch}
        for e in more:
            e.close()
        if world == 1 and not a.no_cpu_baseline:
            v, sec = cpu_sample(ckpt_dir, a.frames, 2, 1)
            cpu_base = {"value": v, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
                        "sample": cpu_sample_text(a.frames) + f"; 2 timed runs of {sec:.1f} s after a 3-frame warm-up",
                        "single_stream_gpu_over_cpu": (80.0 / msf) / max(v, 1e-9)}
    eng_bytes = int(res[0]["bytes_frame"])
    talker_ms_frame = (sum(r["talker"] - r["prefill"] for r in res)) / a.steps / a.frames * 1e3
    eng.close()
    ab = None
    if rank == 0 and extras and a.bits in (4, 8) and 3 <= a.batch <= 128:
        # the other weight-operand mode of the 3..128-row GEMMs on the same workload (2 steps after 1 warm-up): SURVEY.md §8 row a9
        other = 2 if a.packed_gemm == 1 else 1
        eng = q.Engine(ckpt_dir, device=local_rank, max_batch=a.batch, max_frames=max(64, a.frames), kv_capacity=512, packed_gemm=other)
        step(2000)
        r2 = [step(2001 + i) for i in range(2)]
        ab = {"packed_gemm": other, "what": "packed 4/8-bit weights dequantised inside the tcgen05 GEMM" if other == 1 else "fp16 operand copies",
              "value": sum(r["samples"] for r in r2) / 24000.0 / sum(r["dev"] for r in r2), "unit": UNIT,
              "ms_per_frame_step_batch": sum(r["talker"] - r["prefill"] for r in r2) / 2 / a.frames * 1e3}
        eng.close()

    cfg3 = cfg4 = cfg5 = None
    if extras and a.config4 == "on":
        cfg4 = run_config4(q, ckpt_dir, dist, a, rank, local_rank, world, tf)
    if extras and a.config3 == "on":
        cfg3 = run_config3(q, checkpoint, dist, a, rank, local_rank, world)
    if extras and a.config5 == "on" and world == 1:
        cfg5 = run_config5(q, checkpoint, a, local_rank)
    clocks_all = sampler.snapshot()
    sampler.stop()

    if rank == 0:
        codec_sps = samples / max(1e-9, sum(r["decode"] for r in res))
        packed = a.bits in (4, 8)
        line = {"metric": METRIC, "value": audio_s / dev_max, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": dev_max / a.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": ((f"u{a.bits} g64 weights dequantised inside the GEMM to f16 operands x f32 accumulate, f32 residual stream" if fused_mode else
                           f"u{a.bits} g64 weights dequantised at load to f16 operands x f32 accumulate, f32 residual stream") if packed
                          else "bf16 weights -> f16 operands x f32 accumulate, f32 residual stream") if a.batch >= 3 else "f32 activations, packed weights",
                "data": "synthetic", "config": config,
                "e2e": {"value": audio_s / wall_max, "unit": UNIT, "h2d_bytes_per_step": h2d_all / world / a.steps, "d2h_bytes_per_step": d2h_all / world / a.steps,
                        "ms_per_step": wall_max / a.steps * 1e3},
                "gpu_launches": int(launches_all), "clocks": clocks, "clocks_whole_run": clocks_all, "roofline": roof, "cpu_baseline": cpu_base, "latency": lat,
                "codec": {"samples_per_s_rank0": codec_sps, "tflops_rank0": sum(r["codec_flops"] for r in res) / max(1e-9, sum(r["decode"] for r in res)) / 1e12,
                          "peak_tflops": tf, "share_of_step": sum(r["decode"] for r in res) / max(1e-9, dev)},
                "talker": {"ms_per_frame_step_batch": talker_ms_frame, "prefill_ms_per_step": sum(r["prefill"] for r in res) / a.steps * 1e3,
                           "share_of_step": sum(r["talker"] for r in res) / max(1e-9, dev), "algorithmic_weight_bytes_per_frame_step": eng_bytes,
                           "frame_step_hbm_frac": (eng_bytes / max(1e-9, talker_ms_frame * 1e-3) / 1e9) / hbm},
                "other_weight_operand_mode": ab, "batches_in_flight": inflight, "config3": cfg3, "config4": cfg4, "config5": cfg5,
                "wall_s_timed_region": total_max}
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    os.close(json_fd)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
