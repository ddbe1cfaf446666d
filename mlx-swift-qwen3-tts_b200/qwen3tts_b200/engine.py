"""Thin, typed wrapper over the C ABI: one `Engine` = one q3tts_handle (one GPU, one stream).

This is the seam the reference crosses with `Qwen3Talker.generateCodes / generateStream` and
`AudioDecoder.mlxDecode / chunkedDecode` (SURVEY.md §8b); everything above it (chat template, tokeniser, text
chunking, WAV files) lives in `pipeline.py`, as it lives in Swift on the reference side.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _abi as A


@dataclass
class GenRequest:
    """Python-side `q3tts_request` (ids already templated + tokenised)."""
    text_ids: list
    speaker_id: int = -1
    speaker_embedding: np.ndarray | None = None
    instruct_ids: list | None = None
    ref_text_ids: list | None = None
    ref_codes: np.ndarray | None = None  # [16][T_ref]
    temperature: float = 0.9
    top_k: int = 0
    top_p: float = 1.0
    repetition_penalty: float = 1.05
    max_tokens: int = 1200
    seed: int = 0
    stream_variant: bool = False
    forced_codes: np.ndarray | None = None  # [F][16]
    keep_invalid_frames: bool = False
    want_logits: int = 0  # frames of logits to capture (one request per call)
    voice: "Voice | None" = None  # a registered voice (Engine.create_voice): leave the voice fields above at their defaults

    def to_c(self) -> A.Request:
        """-> q3tts_request whose pointers reference numpy buffers kept alive by the returned struct itself (`r._keep`): the
        caller holds the struct for as long as the C side may read it (a call, or the lifetime of a stream).  Nothing is
        stored on the dataclass, so the same GenRequest may appear several times in one batch."""
        r = A.Request()
        A.lib().q3tts_default_request(C.byref(r))
        keep = []
        r._keep = keep

        def ints(a):
            arr = np.ascontiguousarray(np.asarray(a, dtype=np.int32))
            keep.append(arr)
            return arr.ctypes.data_as(A.p_i32), int(arr.size)

        r.text_ids, r.n_text_ids = ints(self.text_ids)
        if self.instruct_ids is not None and len(self.instruct_ids):
            r.instruct_ids, r.n_instruct_ids = ints(self.instruct_ids)
        r.speaker_id = int(self.speaker_id)
        if self.speaker_embedding is not None:
            e = np.ascontiguousarray(np.asarray(self.speaker_embedding, dtype=np.float32).reshape(-1))
            keep.append(e)
            r.speaker_embedding = e.ctypes.data_as(A.p_f32)
            r.speaker_embedding_dim = int(e.size)
        if self.ref_text_ids is not None and len(self.ref_text_ids):
            r.ref_text_ids, r.n_ref_text_ids = ints(self.ref_text_ids)
        if self.ref_codes is not None:
            rc = np.ascontiguousarray(np.asarray(self.ref_codes, dtype=np.int32))
            keep.append(rc)
            r.ref_codes = rc.ctypes.data_as(A.p_i32)
            r.ref_frames = int(rc.shape[1]) if rc.ndim == 2 else 0
        r.temperature = float(self.temperature)
        r.top_k = int(self.top_k)
        r.top_p = float(self.top_p)
        r.repetition_penalty = float(self.repetition_penalty)
        r.max_tokens = int(self.max_tokens)
        r.seed = int(self.seed)
        r.stream_variant = 1 if self.stream_variant else 0
        if self.forced_codes is not None:
            fc = np.ascontiguousarray(np.asarray(self.forced_codes, dtype=np.int32).reshape(-1, 16))
            keep.append(fc)
            r.forced_codes = fc.ctypes.data_as(A.p_i32)
            r.n_forced_frames = int(fc.shape[0])
        r.keep_invalid_frames = 1 if self.keep_invalid_frames else 0
        if self.voice is not None:
            r.voice = self.voice.ptr
            keep.append(self.voice)  # a voice is not freed while a struct that names it lives
        return r


def _attach_logits(r: "A.Request", frames: int, info) -> dict:
    l0 = np.zeros((frames, info.vocab_size), dtype=np.float32)
    lc = np.zeros((frames, 15, info.cp_vocab_size), dtype=np.float32)
    r.code0_logits_out = l0.ctypes.data_as(A.p_f32)
    r.cp_logits_out = lc.ctypes.data_as(A.p_f32)
    r.logits_capacity_frames = frames
    r._keep.extend([l0, lc])
    return {"code0_logits": l0, "cp_logits": lc}


class Voice:
    """`q3tts_voice`: the prefilled prompt prefix of one voice (Engine.create_voice).  Requests that set `voice=` give the bits of the
    same requests with the voice fields written inline; the handle that made it and its clones accept it."""

    def __init__(self, ptr):
        self._p = ptr
        n, b = A.i32(0), A.i64(0)
        A.check(A.lib().q3tts_voice_info(self._p, C.byref(n), C.byref(b)), None)
        self.prefix_positions, self.device_bytes = n.value, b.value

    @property
    def ptr(self):
        if not self._p:
            raise ValueError("the voice is closed")
        return self._p

    def close(self):
        if getattr(self, "_p", None):
            A.lib().q3tts_voice_free(self._p)
            self._p = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class CodeStream:
    """`q3tts_stream`: code chunks (`next_codes`) or decoded AudioChunks (`next_audio`)."""

    def __init__(self, engine: "Engine", ptr, chunk_size: int, req_keepalive):
        self._e, self._p, self.chunk_size, self._keep = engine, ptr, chunk_size, req_keepalive
        self.done = False

    def next_codes(self):
        out = np.zeros((self.chunk_size, 16), dtype=np.int32)
        n, done = A.i32(0), A.i32(0)
        A.check(A.lib().q3tts_stream_next(self._p, out.ctypes.data_as(A.p_i32), C.byref(n), C.byref(done)), self._e._h)
        self.done = bool(done.value)
        return out[: n.value].copy(), self.done

    def next_audio(self):
        cap = 18 * A.SAMPLES_PER_FRAME
        out = np.zeros(cap, dtype=np.float32)
        n, t0, t1, fin, done = A.i32(0), A.i32(0), A.i32(0), A.i32(0), A.i32(0)
        A.check(A.lib().q3tts_stream_next_audio(self._p, out.ctypes.data_as(A.p_f32), cap, C.byref(n), C.byref(t0), C.byref(t1),
                                                C.byref(fin), C.byref(done)), self._e._h)
        self.done = bool(done.value)
        return out[: n.value].copy(), (t0.value, t1.value), bool(fin.value), self.done

    def cancel(self):
        A.lib().q3tts_stream_cancel(self._p)

    def close(self):
        if self._p:
            A.lib().q3tts_stream_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Engine:
    def __init__(self, model_dir: str, device: int = 0, max_batch: int = 1, kv_capacity: int = 512, max_frames: int = 2400,
                 use_cuda_graph: bool = True, load_codec: bool = True, load_talker: bool = True, codec_max_frames: int = 2400,
                 cuda_stream: int | None = None, packed_gemm: int = 0, runtime_quantization: bool = False, lanes: int = 1):
        L = A.lib()
        o = A.Options()
        L.q3tts_default_options(C.byref(o))
        o.device, o.max_batch, o.kv_capacity, o.max_frames = device, max_batch, kv_capacity, max_frames
        o.use_cuda_graph = 1 if use_cuda_graph else 0
        o.load_codec, o.load_talker, o.codec_max_frames = int(load_codec), int(load_talker), codec_max_frames
        o.packed_gemm = int(packed_gemm)
        o.runtime_quantization = 1 if runtime_quantization else 0
        o.lanes = int(lanes)
        if cuda_stream:
            o.cuda_stream = C.c_void_p(cuda_stream)
        h = C.c_void_p()
        st = L.q3tts_create(str(model_dir).encode(), C.byref(o), C.byref(h))
        A.check(st, None)
        self._h = h
        self.info = A.Info()
        A.check(L.q3tts_get_info(self._h, C.byref(self.info)), self._h)

    def clone(self) -> "Engine":
        """A second handle on the same device sharing this one's talker weights (q3tts_clone): own stream, KV rings, buffers and codec.
        Serve more than `max_batch` pending requests through 2-4 handles from as many threads."""
        h = C.c_void_p()
        A.check(A.lib().q3tts_clone(self._h, C.byref(h)), None)
        e = Engine.__new__(Engine)
        e._h = h
        e.info = A.Info()
        A.check(A.lib().q3tts_get_info(e._h, C.byref(e.info)), e._h)
        return e

    def close(self):
        if getattr(self, "_h", None):
            A.lib().q3tts_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- info
    def speakers(self) -> dict:
        out = {}
        buf = C.create_string_buffer(256)
        for i in range(self.info.num_speakers):
            sid = A.i32(0)
            A.check(A.lib().q3tts_speaker_name(self._h, i, buf, 256, C.byref(sid)), self._h)
            out[buf.value.decode()] = sid.value
        return out

    def speaker_id(self, name: str) -> int:
        return A.lib().q3tts_speaker_id(self._h, name.lower().encode())

    def timing(self) -> A.Timing:
        t = A.Timing()
        A.check(A.lib().q3tts_get_timing(self._h, C.byref(t)), self._h)
        return t

    def clear_cache(self):
        A.check(A.lib().q3tts_clear_cache(self._h), self._h)

    # ---- talker
    def create_voice(self, req: GenRequest) -> Voice:
        """q3tts_voice_create: prefill the voice part of `req` (instruct / speaker / ICL fields and the role ids text_ids[:3]) once."""
        r = req.to_c()
        p = C.c_void_p()
        A.check(A.lib().q3tts_voice_create(self._h, C.byref(r), C.byref(p)), self._h)
        v = Voice(p)
        v.role_ids = [int(i) for i in req.text_ids[:3]]
        return v

    def generate_codes(self, req: GenRequest, capacity: int | None = None):
        """-> frames int32 [F,16]  (+ dict of logits when req.want_logits)."""
        cap = capacity or max(req.max_tokens, 0 if req.forced_codes is None else len(req.forced_codes), 1)
        r = req.to_c()
        out = np.zeros((cap, 16), dtype=np.int32)
        n = A.i32(0)
        logits = _attach_logits(r, req.want_logits, self.info) if req.want_logits else None
        A.check(A.lib().q3tts_generate_codes(self._h, C.byref(r), out.ctypes.data_as(A.p_i32), cap, C.byref(n)), self._h)
        frames = out[: n.value].copy()
        return (frames, logits) if req.want_logits else frames

    def generate_codes_batch(self, reqs: list, capacity: int | None = None):
        """-> list of frames [F_i,16]; when ONE request has want_logits set: (list, logits dict of that request)."""
        n = len(reqs)
        cap = capacity or max([max(r.max_tokens, 0 if r.forced_codes is None else len(r.forced_codes), 1) for r in reqs] + [1])
        structs = [r.to_c() for r in reqs]  # held until the call returns (they own the buffers the C side reads)
        logits = None
        for r, st in zip(reqs, structs):
            if r.want_logits:
                logits = _attach_logits(st, r.want_logits, self.info)
        arr = (A.Request * n)(*structs)
        outs = [np.zeros((cap, 16), dtype=np.int32) for _ in range(n)]
        ptrs = (A.p_i32 * n)(*[o.ctypes.data_as(A.p_i32) for o in outs])
        counts = (A.i32 * n)()
        A.check(A.lib().q3tts_generate_codes_batch(self._h, arr, n, ptrs, cap, counts), self._h)
        del structs
        res = [outs[i][: counts[i]].copy() for i in range(n)]
        return (res, logits) if logits is not None else res

    def stream(self, req: GenRequest, chunk_size: int = 12) -> CodeStream:
        r = req.to_c()
        p = C.c_void_p()
        A.check(A.lib().q3tts_stream_begin(self._h, C.byref(r), chunk_size, C.byref(p)), self._h)
        return CodeStream(self, p, chunk_size, r)  # the stream keeps the struct (and with it the id buffers) alive

    # ---- codec
    def decode(self, codes: np.ndarray) -> np.ndarray:
        """codes int32 [B,F,16] -> pcm float32 [B, F*1920]  (`AudioDecoder.mlxDecode`)."""
        codes = np.ascontiguousarray(np.asarray(codes, dtype=np.int32))
        if codes.ndim == 2:
            codes = codes[None]
        B, F, _ = codes.shape
        out = np.zeros((B, F * self.info.codec_total_upsample), dtype=np.float32)
        A.check(A.lib().q3tts_decode(self._h, codes.ctypes.data_as(A.p_i32), B, F, out.ctypes.data_as(A.p_f32)), self._h)
        return out

    def decode_chunked(self, codes: np.ndarray, chunk_size: int = 100, left_context: int = 10) -> np.ndarray:
        codes = np.ascontiguousarray(np.asarray(codes, dtype=np.int32))
        if codes.ndim == 2:
            codes = codes[None]
        B, F, _ = codes.shape
        out = np.zeros((B, F * self.info.codec_total_upsample), dtype=np.float32)
        A.check(A.lib().q3tts_decode_chunked(self._h, codes.ctypes.data_as(A.p_i32), B, F, chunk_size, left_context,
                                             out.ctypes.data_as(A.p_f32)), self._h)
        return out

    def rvq_embed(self, codes: np.ndarray):
        codes = np.ascontiguousarray(np.asarray(codes, dtype=np.int32))
        if codes.ndim == 2:
            codes = codes[None]
        B, F, _ = codes.shape
        D = 4096
        first = np.zeros((B * F, D), dtype=np.float32)
        rest = np.zeros((B * F, D), dtype=np.float32)
        dim = A.i32(0)
        # first query the dim with an empty call
        A.check(A.lib().q3tts_rvq_embed(self._h, codes.ctypes.data_as(A.p_i32), 0, 0, first.ctypes.data_as(A.p_f32),
                                        rest.ctypes.data_as(A.p_f32), C.byref(dim)), self._h)
        first = np.zeros((B * F, dim.value), dtype=np.float32)
        rest = np.zeros((B * F, dim.value), dtype=np.float32)
        A.check(A.lib().q3tts_rvq_embed(self._h, codes.ctypes.data_as(A.p_i32), B, F, first.ctypes.data_as(A.p_f32),
                                        rest.ctypes.data_as(A.p_f32), C.byref(dim)), self._h)
        return first.reshape(B, F, -1), rest.reshape(B, F, -1)

    # ---- ICL reference-audio encoder
    def encode_reference_audio(self, samples, want_latent: bool = False):
        """24 kHz mono float32 samples -> codes int32 [16, T] (the `ref_codes` layout), or None without encoder weights
        (`Qwen3TTSPipeline.encodeReferenceAudio`).  want_latent: also return the quantiser input [T, hidden]."""
        if not self.info.has_audio_encoder:
            return (None, None) if want_latent else None
        a = np.ascontiguousarray(np.asarray(samples, dtype=np.float32).reshape(-1))
        cap = (a.size + 1919) // 1920 + 2
        codes = np.zeros((64, cap), dtype=np.int32)
        lat = np.zeros((cap, self.info.audio_encoder_hidden), dtype=np.float32) if want_latent else None
        n, nq = A.i32(0), A.i32(0)
        A.check(A.lib().q3tts_encode_reference_audio(self._h, a.ctypes.data_as(A.p_f32), a.size, codes.ctypes.data_as(A.p_i32), cap, C.byref(n), C.byref(nq),
                                                     lat.ctypes.data_as(A.p_f32) if want_latent else None), self._h)
        out = codes.reshape(-1)[: nq.value * n.value].reshape(nq.value, n.value).copy()
        return (out, lat[: n.value].copy()) if want_latent else out

    # ---- ECAPA-TDNN speaker encoder
    def extract_speaker_embedding(self, samples, want_mels: bool = False):
        """24 kHz mono float32 samples -> speaker embedding float32 [speaker_embedding_dim] (the `speaker_embedding` request field), or
        None without `speaker_encoder.*` weights (`Qwen3TTSPipeline.extractSpeakerEmbedding`).  want_mels: also return the log-mel
        input [frames, 128]."""
        if not self.info.has_speaker_encoder:
            return (None, None) if want_mels else None
        a = np.ascontiguousarray(np.asarray(samples, dtype=np.float32).reshape(-1))
        dim = self.info.speaker_embedding_dim
        emb = np.zeros(dim, dtype=np.float32)
        mels = np.zeros((a.size // 256 + 1, 128), dtype=np.float32) if want_mels else None
        n = A.i32(0)
        A.check(A.lib().q3tts_extract_speaker_embedding(self._h, a.ctypes.data_as(A.p_f32), a.size, emb.ctypes.data_as(A.p_f32), dim, C.byref(n),
                                                        mels.ctypes.data_as(A.p_f32) if want_mels else None), self._h)
        emb = emb[: n.value].copy()
        return (emb, mels) if want_mels else emb

    # ---- fused
    def generate_pcm(self, req: GenRequest, mode: int = A.DECODE_WHOLE):
        cap = max(req.max_tokens, 1) * self.info.codec_total_upsample
        out = np.zeros(cap, dtype=np.float32)
        n, frames = A.i64(0), A.i32(0)
        r = req.to_c()
        A.check(A.lib().q3tts_generate_pcm(self._h, C.byref(r), mode, out.ctypes.data_as(A.p_f32), cap, C.byref(n), C.byref(frames)), self._h)
        return out[: n.value].copy(), frames.value

    def generate_pcm_batch(self, reqs: list, mode: int = A.DECODE_WHOLE, out_buffers: list | None = None):
        n = len(reqs)
        cap = max([max(r.max_tokens, 1) for r in reqs] + [1]) * self.info.codec_total_upsample
        outs = out_buffers or [np.zeros(cap, dtype=np.float32) for _ in range(n)]
        structs = [r.to_c() for r in reqs]
        arr = (A.Request * n)(*structs)
        ptrs = (A.p_f32 * n)(*[o.ctypes.data_as(A.p_f32) for o in outs])
        ns = (A.i64 * n)()
        fr = (A.i32 * n)()
        A.check(A.lib().q3tts_generate_pcm_batch(self._h, arr, n, mode, ptrs, cap, ns, fr), self._h)
        return [outs[i][: ns[i]] for i in range(n)], [fr[i] for i in range(n)]

    def profile_linear(self, which: int = 0, m: int = 1, iters: int = 20):
        """-> (ms_total, launches, bytes_per_iter) of the talker-step (which=0) / code-predictor-pass (which=1) linear launches."""
        ms, n, b = C.c_double(0), A.i64(0), A.i64(0)
        A.check(A.lib().q3tts_profile_linear(self._h, which, m, iters, C.byref(ms), C.byref(n), C.byref(b)), self._h)
        return ms.value, n.value, b.value

    def sample_token(self, logits, temperature=0.9, top_k=0, top_p=1.0, repetition_penalty=1.05, token_set=None, seed=0, counter=0) -> int:
        lg = np.ascontiguousarray(np.asarray(logits, dtype=np.float32))
        ts = np.ascontiguousarray(np.asarray(sorted(token_set) if token_set else [], dtype=np.int32))
        out = A.i32(-1)
        A.check(A.lib().q3tts_sample_token(self._h, lg.ctypes.data_as(A.p_f32), lg.size, temperature, top_k, top_p, repetition_penalty,
                                           ts.ctypes.data_as(A.p_i32) if ts.size else None, int(ts.size), seed, counter, C.byref(out)), self._h)
        return out.value


_DT = {"f32": A.F32, "f16": A.F16, "bf16": A.BF16}


def safetensors_check(path: str):
    """`q3tts_safetensors_check`: (n_tensors, data_bytes) of a well-formed file, raises Q3Error otherwise.  Needs no GPU."""
    n, b = A.i32(0), A.i64(0)
    A.check(A.lib().q3tts_safetensors_check(str(path).encode(), C.byref(n), C.byref(b)), None)
    return n.value, b.value


def _raw16(a, dtype: str) -> np.ndarray:
    """fp32 numpy values that are exactly representable in `dtype` -> raw uint16 / float32 storage."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    if dtype == "f32":
        return a
    if dtype == "f16":
        return a.astype(np.float16).view(np.uint16)
    return (a.view(np.uint32) >> 16).astype(np.uint16)


def dequantize(packed, scales, biases, group_size=64, bits=4, scale_dtype="bf16", out_dtype="f32", device=0) -> np.ndarray:
    """`q3tts_dequantize` probe.  scales/biases: fp32 numpy holding `scale_dtype`-representable values.
    Returns fp32 numpy holding the `out_dtype` values."""
    packed = np.ascontiguousarray(packed, dtype=np.uint32)
    out_f, words = packed.shape
    in_f = words * 32 // bits
    s, b = _raw16(scales, scale_dtype), _raw16(biases, scale_dtype)
    if out_dtype == "f32":
        out = np.zeros((out_f, in_f), dtype=np.float32)
    else:
        out = np.zeros((out_f, in_f), dtype=np.uint16)
    A.check(A.lib().q3tts_dequantize(device, packed.ctypes.data, s.ctypes.data, b.ctypes.data, _DT[scale_dtype], out_f, in_f,
                                     group_size, bits, _DT[out_dtype], out.ctypes.data), None)
    if out_dtype == "f16":
        return out.view(np.float16).astype(np.float32)
    if out_dtype == "bf16":
        return (out.astype(np.uint32) << 16).view(np.float32)
    return out


def mlx_quantize(w, bits=4, dtype="bf16", device=0):
    """`q3tts_mlx_quantize` probe: w fp32 numpy holding `dtype`-representable values -> (codes uint8 [out, in], scales, biases as fp32 numpy
    holding the `dtype` values)."""
    w = np.ascontiguousarray(w, dtype=np.float32)
    out_f, in_f = w.shape
    raw = _raw16(w, dtype) if dtype != "f32" else w
    codes = np.zeros((out_f, in_f), dtype=np.uint8)
    g = (out_f, in_f // 64)
    s = np.zeros(g, dtype=np.float32 if dtype == "f32" else np.uint16)
    b = np.zeros_like(s)
    A.check(A.lib().q3tts_mlx_quantize(device, raw.ctypes.data, _DT[dtype], out_f, in_f, bits, codes.ctypes.data, s.ctypes.data, b.ctypes.data), None)
    if dtype == "f16":
        return codes, s.view(np.float16).astype(np.float32), b.view(np.float16).astype(np.float32)
    if dtype == "bf16":
        return codes, (s.astype(np.uint32) << 16).view(np.float32), (b.astype(np.uint32) << 16).view(np.float32)
    return codes, s, b


def mxfp4_to_affine(packed, scales, device=0):
    """`q3tts_mxfp4_to_affine` probe: MLX mxfp4 leaves (packed uint32 [out, in/8], E8M0 scale bytes uint8 [out, in/32]) -> the exact 8-bit
    affine container the loader keeps: (codes uint32 [out, in/4] in 8-bit words, scales, biases as fp32 numpy holding the bf16 values).
    `dequantize` / `quantized_matmul` / `quantized_matmul_tc` take them with group_size=32, bits=8, scale_dtype="bf16"."""
    packed = np.ascontiguousarray(packed, dtype=np.uint32)
    scales = np.ascontiguousarray(scales, dtype=np.uint8)
    out_f, words = packed.shape
    in_f = words * 8
    codes = np.zeros((out_f, in_f // 4), dtype=np.uint32)
    s = np.zeros((out_f, in_f // 32), dtype=np.uint16)
    b = np.zeros_like(s)
    A.check(A.lib().q3tts_mxfp4_to_affine(device, packed.ctypes.data, scales.ctypes.data, out_f, in_f, codes.ctypes.data, s.ctypes.data,
                                          b.ctypes.data), None)
    return codes, (s.astype(np.uint32) << 16).view(np.float32), (b.astype(np.uint32) << 16).view(np.float32)


def quantized_matmul(x, packed, scales, biases, group_size=64, bits=4, scale_dtype="bf16", device=0) -> np.ndarray:
    """`q3tts_quantized_matmul` probe: y = x @ dequant(W)^T with the talker's GEMV kernels.  bits=0: `packed` is a dense
    fp32-valued weight matrix stored as `scale_dtype`."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    m, in_f = x.shape
    if bits:
        w = np.ascontiguousarray(packed, dtype=np.uint32)
        out_f = w.shape[0]
        s, b = _raw16(scales, scale_dtype), _raw16(biases, scale_dtype)
        sp, bp = s.ctypes.data, b.ctypes.data
    else:
        w = _raw16(packed, scale_dtype)
        out_f = w.shape[0]
        sp = bp = None
    y = np.zeros((m, out_f), dtype=np.float32)
    A.check(A.lib().q3tts_quantized_matmul(device, x.ctypes.data_as(A.p_f32), m, w.ctypes.data, sp, bp, _DT[scale_dtype], out_f, in_f,
                                           group_size, bits, y.ctypes.data_as(A.p_f32)), None)
    return y


def quantized_matmul_tc(x, packed, scales, biases, group_size=64, bits=4, scale_dtype="bf16", fold=None, swiglu_halves=False, residual=None, device=0):
    """`q3tts_quantized_matmul_tc` probe: the dequant-fused tcgen05 GEMM of batched decode (m <= 128 rows)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    m, in_f = x.shape
    w = np.ascontiguousarray(packed, dtype=np.uint32)
    out_f = w.shape[0]
    s, b = _raw16(scales, scale_dtype), _raw16(biases, scale_dtype)
    n_out = out_f // 2 if swiglu_halves else out_f
    y = np.zeros((m, n_out), dtype=np.float32)
    f = None if fold is None else np.ascontiguousarray(fold, dtype=np.float32)
    r = None if residual is None else np.ascontiguousarray(residual, dtype=np.float32)
    pf = lambda a: None if a is None else a.ctypes.data_as(A.p_f32)
    A.check(A.lib().q3tts_quantized_matmul_tc(device, x.ctypes.data_as(A.p_f32), m, w.ctypes.data, s.ctypes.data, b.ctypes.data, _DT[scale_dtype], out_f, in_f,
                                              group_size, bits, pf(f), 1 if swiglu_halves else 0, pf(r), y.ctypes.data_as(A.p_f32)), None)
    return y


def conv_probe(x, w, bias=None, ntap=1, dil=1, act=0, swiglu=False, res=None, scale=None, snake=None, use_tensor_cores=True, device=0):
    """`q3tts_conv_probe`: x [B,T,cin], w [ntap,N,cin] -> (y32, y16) each [B,T,N or N/2] (fp32 numpy)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    w = np.ascontiguousarray(w, dtype=np.float32)
    B, T, cin = x.shape
    nt, N, _ = w.shape
    assert nt == ntap
    n_out = N // 2 if swiglu else N
    f = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float32).ctypes.data_as(A.p_f32)
    keep = [np.ascontiguousarray(a, dtype=np.float32) if a is not None else None for a in (bias, res, scale)]
    ea = ieb = None
    sch = 0
    if snake is not None:
        ea, ieb = [np.ascontiguousarray(a, dtype=np.float32) for a in snake]
        sch = int(ea.size)
    y32 = np.zeros((B, T, n_out), dtype=np.float32)
    y16 = np.zeros((B, T, n_out), dtype=np.float32)
    p = lambda a: None if a is None else a.ctypes.data_as(A.p_f32)
    A.check(A.lib().q3tts_conv_probe(device, p(x), B, T, cin, p(w), p(keep[0]), N, ntap, dil, act, 1 if swiglu else 0, p(keep[1]), p(keep[2]),
                                     p(ea), p(ieb), sch, 1 if use_tensor_cores else 0, p(y32), p(y16)), None)
    return y32, y16


def attention_probe(kernel, qkv, heads, kv_heads, q_norm, k_norm, eps, inv_freq, row_slot, row_pos, win_start, k_ring, v_ring,
                    kv_f16=False, out_f16=False, device=0):
    """`q3tts_attention_probe`: one talker attention launch.  qkv [m, (heads + 2*kv_heads)*128]; k_ring / v_ring
    [n_slots, kv_heads, capacity, 128] (not modified); win_start [n_slots] or None.  -> (out [m, heads*128], k_ring, v_ring after
    the launch), fp32 numpy (fp16 values widened)."""
    f = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    i = lambda a: np.ascontiguousarray(a, dtype=np.int32)
    qkv, q_norm, k_norm, inv_freq = f(qkv), f(q_norm), f(k_norm), f(inv_freq)
    row_slot, row_pos = i(row_slot), i(row_pos)
    win = None if win_start is None else i(win_start)
    k_out, v_out = f(k_ring).copy(), f(v_ring).copy()
    n_slots, _, capacity, _ = k_out.shape
    m = qkv.shape[0]
    out = np.zeros((m, heads * 128), dtype=np.float32)
    pf, pi = (lambda a: a.ctypes.data_as(A.p_f32)), (lambda a: None if a is None else a.ctypes.data_as(A.p_i32))
    A.check(A.lib().q3tts_attention_probe(device, kernel, int(bool(kv_f16)), int(bool(out_f16)), pf(qkv), m, heads, kv_heads, pf(q_norm), pf(k_norm),
                                          eps, pf(inv_freq), pi(row_slot), pi(row_pos), pi(win), n_slots, capacity, pf(k_out), pf(v_out), pf(out)), None)
    return out, k_out, v_out


def _f32(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float32)


def _pf(a):
    return None if a is None else a.ctypes.data_as(A.p_f32)


def codec_attention_probe(kernel, qkv, nh, nkv, inv_freq=None, device=0):
    """`q3tts_codec_attention_probe`: qkv [B, T, (nh + 2*nkv)*64]; inv_freq [32] or None (no RoPE).
    -> (out [B, T, nh*64], qkv after the in-place RoPE), fp32 numpy (fp16 outputs widened)."""
    q = _f32(qkv).copy()
    B, T, _ = q.shape
    f = _f32(inv_freq)
    out = np.zeros((B, T, nh * 64), dtype=np.float32)
    A.check(A.lib().q3tts_codec_attention_probe(device, kernel, _pf(q), B, T, nh, nkv, _pf(f), _pf(out)), None)
    return out, q


def codec_unit_probe(form, a, w7, b7, ea2, ieb2, w1, b1, res, ea3, ieb3, dil, in_place=False, emit_residual=True, weight_reps=1, device=0):
    """`q3tts_codec_unit_probe`: one vocoder residual unit.  a, res [B, T, C]; w7 [7, C, C]; w1 [C, C]; b7 / b1 [C] or None.
    -> (x' [B, T, C] or None when not emitted, snake3(x') [B, T, C]), fp16 values widened to fp32."""
    a, res = _f32(a), _f32(res)
    B, T, C = a.shape
    keep = [_f32(v) for v in (w7, b7, ea2, ieb2, w1, b1, ea3, ieb3)]
    x_out = np.zeros((B, T, C), dtype=np.float32) if emit_residual else None
    out = np.zeros((B, T, C), dtype=np.float32)
    A.check(A.lib().q3tts_codec_unit_probe(device, form, B, T, C, dil, _pf(a), *[_pf(v) for v in keep[:6]], _pf(res), _pf(keep[6]), _pf(keep[7]),
                                           int(bool(in_place)), int(bool(emit_residual)), weight_reps, _pf(x_out), _pf(out)), None)
    return x_out, out


def codec_out_conv_probe(kernel, x, w, bias, strip=0, device=0):
    """`q3tts_codec_out_conv_probe`: x [B, T, C], w [7, C], bias [1] -> pcm [B, T] (clipped, NaN -> 0)."""
    x, w, b = _f32(x), _f32(w), _f32(np.reshape(bias, (1,)))
    B, T, C = x.shape
    y = np.zeros((B, T), dtype=np.float32)
    A.check(A.lib().q3tts_codec_out_conv_probe(device, kernel, _pf(x), B, T, C, _pf(w), _pf(b), strip, _pf(y)), None)
    return y


CODEC_ROWOPS = {"dwconv7": 0, "layernorm": 1, "layernorm_f16": 2, "rmsnorm_f16": 3, "snake": 4, "silu_mul": 5}


def codec_rowop_probe(op, x, C, w=None, b=None, eps=1e-6, T=0, device=0):
    """`q3tts_codec_rowop_probe`: x [rows, ldx] -> y [rows, C] (fp16 outputs widened).  op is a key of CODEC_ROWOPS."""
    x = _f32(x)
    rows, ldx = x.shape
    w, b = _f32(w), _f32(b)
    y = np.zeros((rows, C), dtype=np.float32)
    A.check(A.lib().q3tts_codec_rowop_probe(device, CODEC_ROWOPS[op], _pf(x), rows, ldx, C, T, _pf(w), _pf(b), eps, _pf(y)), None)
    return y


def sampler_probe(form, logits, temperature, top_k, top_p, repetition_penalty, seed, counter, token_sets=None, codec_vocab=0,
                  want_processed=False, n_rows=None, device=0):
    """`q3tts_sampler_probe`: the device sampler on each row of logits [n, V] (or one row [V] shared by n_rows rows).  The sampling
    arguments are scalars or arrays of n; token_sets is [n, 128] uint32 bitmaps or None.  form 0 = sample_kernel's form, 1 = the
    frame kernel's.  -> (ids int32 [n], processed [n, V] fp32 or None)."""
    lg = _f32(logits)
    V = lg.shape[-1]
    n = lg.shape[0] if lg.ndim == 2 else int(n_rows or 1)
    ld = V if lg.ndim == 2 else 0
    row = lambda a, dt: np.ascontiguousarray(np.broadcast_to(np.asarray(a, dtype=dt), (n,)))
    t, k, p, r = row(temperature, np.float32), row(top_k, np.int32), row(top_p, np.float32), row(repetition_penalty, np.float32)
    sd, ct = row(seed, np.uint64), row(counter, np.uint64)
    sets = None if token_sets is None else np.ascontiguousarray(np.broadcast_to(np.asarray(token_sets, dtype=np.uint32), (n, 128)))
    ids = np.zeros(n, np.int32)
    proc = np.zeros((n, V), np.float32) if want_processed else None
    pi = lambda a: a.ctypes.data_as(A.p_i32)
    A.check(A.lib().q3tts_sampler_probe(device, form, _pf(lg), n, V, ld, codec_vocab, _pf(t), pi(k), _pf(p), _pf(r),
                                        None if sets is None else sets.ctypes.data, sd.ctypes.data, ct.ctypes.data, pi(ids), _pf(proc)), None)
    return ids, proc


SLOT_FIELDS = ("active", "finished", "step", "max_tokens", "trailing_idx", "total_text", "consecutive_pad", "n_forced", "stream_variant",
               "frame_alive", "logits_cap")


def sampler_slot_probe(form, group, logits, state, sampling, token_sets, cur_codes, eos_id, pad_id, codec_vocab, forced=None,
                       dump_slot=0, dump_frames=None, device=0):
    """`q3tts_sampler_slot_probe`: one sampling point of `group` for every slot of logits [n, V].  state: {SLOT_FIELDS name: int [n]};
    sampling: {temperature, top_k, top_p, repetition_penalty, seed: [n]}; token_sets uint32 [n, 16, set_words]; cur_codes int [n, 16];
    forced int [n, max_frames, 16] or None; dump_frames: rows of the logits dump of slot dump_slot, or None (no dump).
    -> (state after the launch, token_sets, cur_codes, dump [dump_frames, V] or None); the inputs are not modified."""
    lg = _f32(logits)
    n, V = lg.shape
    st = {f: np.array(np.broadcast_to(np.asarray(state[f], dtype=np.int32), (n,))) for f in SLOT_FIELDS}
    row = lambda name, dt: np.ascontiguousarray(np.broadcast_to(np.asarray(sampling[name], dtype=dt), (n,)))
    t, k, p, r = row("temperature", np.float32), row("top_k", np.int32), row("top_p", np.float32), row("repetition_penalty", np.float32)
    sd = row("seed", np.uint64)
    sets = np.array(token_sets, dtype=np.uint32)
    assert sets.ndim == 3 and sets.shape[:2] == (n, 16)
    codes = np.array(cur_codes, dtype=np.int32).reshape(n, 16)
    fz = None if forced is None else np.ascontiguousarray(forced, dtype=np.int32)
    max_frames = 0 if fz is None else fz.shape[1]
    dump = None if dump_frames is None else np.zeros((dump_frames, V), np.float32)
    pi = lambda a: None if a is None else a.ctypes.data_as(A.p_i32)
    A.check(A.lib().q3tts_sampler_slot_probe(device, form, group, n, V, codec_vocab, eos_id, pad_id, _pf(lg), *[pi(st[f]) for f in SLOT_FIELDS],
                                             _pf(t), pi(k), _pf(p), _pf(r), sd.ctypes.data, sets.ctypes.data, sets.shape[2], pi(fz), max_frames,
                                             _pf(dump), dump_slot, 0 if dump_frames is None else dump_frames, pi(codes)), None)
    return st, sets, codes, dump
