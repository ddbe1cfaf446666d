"""Host-side mirror of the reference's public Swift API (`Qwen3TTSPipeline.swift`), same names, argument meaning and
error behaviour, over the C ABI.  The Swift package in ../swift/ is the drop-in for Swift hosts; this module is the
same surface for Python hosts and for the parity tests (no Swift toolchain in this image).

Mapping (reference file:line -> here)
    Qwen3TTSPipeline.init(modelPath:configuration:)            :118  -> Qwen3TTSPipeline(model_path, configuration)
    generate(text:speaker:temperature:maxTokens:)              :244  -> generate(text, speaker=...)
    generate(text:speakerEmbedding:temperature:maxTokens:)     :279  -> generate(text, speaker_embedding=...)
    generateStream(...) -> AsyncThrowingStream<AudioChunk>     :323  -> generate_stream(...) -> iterator of AudioChunk
    generateVoiceDesign / generateCustomVoice (+Stream)        :355-480
    generateToFile(...) async throws -> Int                    :644  -> generate_to_file(...)
    generateBatch(...) async -> [Float]                        :774  -> generate_batch(...)
    (no counterpart: a registered voice, q3tts_voice)                -> prepare_voice(...) -> Voice; voice= on every generate*
    clearCache()                                               :951
    availableSpeakers / supports* / modelType / sampleRate     :65-104
    AudioChunk :6-19, Qwen3TTSPipelineConfiguration :22-54, Qwen3TTSError :985-1000
Host-only helpers restated from the reference because the API needs them: TextChunker (Utilities/TextChunker.swift),
StreamingWAVWriter (Utilities/AudioSampleWriter.swift:44-106).
"""
from __future__ import annotations

import os
import struct
from dataclasses import dataclass

import numpy as np

from . import _abi as A
from .engine import Engine, GenRequest, Voice


@dataclass
class AudioChunk:  # Qwen3TTSPipeline.swift:6-19
    samples: np.ndarray
    token_range: range
    is_final: bool


@dataclass
class Qwen3TTSPipelineConfiguration:  # Qwen3TTSPipeline.swift:22-54
    apply_runtime_quantization: bool = True  # :25, :184: a checkpoint without a `quantization` block is quantised 4/6-bit at load
    default_temperature: float = 0.85
    default_max_tokens: int = 2400
    default_streaming_chunk_size: int = 12
    crossfade_samples: int = 480
    # engine-side options (no reference counterpart)
    device: int = 0
    max_batch: int = 1
    lanes: int = 1  # q3tts_options.lanes: launch chains served side by side when a call carries more than max_batch requests
    kv_capacity: int = 512
    use_cuda_graph: bool = True
    seed: int = 0


class Qwen3TTSError(Exception):  # Qwen3TTSPipeline.swift:985-1000
    pass


class FileNotFound(Qwen3TTSError):
    def __init__(self, file):
        super().__init__(f"Required file not found: {file}")


class DecoderLoadFailed(Qwen3TTSError):
    def __init__(self):
        super().__init__("Failed to load MLX audio decoder")


class ModelNotLoaded(Qwen3TTSError):
    def __init__(self):
        super().__init__("Model is not loaded")


class TextChunker:
    """Utilities/TextChunker.swift:5-155 (host string logic, unchanged by the engine)."""
    default_max_words = 35
    min_words = 8
    _conjunctions = [" and then ", " and ", " but ", " or ", " so ", " because ", " when ", " while ", " although ", " however ",
                     " therefore ", " meanwhile ", " afterwards ", " finally ", " then "]
    _starters = [" in the ", " on the ", " at the ", " for the ", " with the ", " to the ", " from the ", " into the ", " onto the "]

    @staticmethod
    def _words(s):
        return [w for w in s.split(" ") if w]

    @classmethod
    def chunk(cls, text: str, max_words: int = 35):
        trimmed = text.strip()
        if not trimmed:
            return []
        if len(cls._words(trimmed)) <= max_words:
            return [trimmed]
        chunks, remaining = [], trimmed
        while remaining:
            c = cls._natural_break(remaining, max_words)
            if c.strip():
                chunks.append(c.strip())
            remaining = remaining[len(c):].strip()
        return chunks

    @classmethod
    def _natural_break(cls, text, max_words):
        words = cls._words(text)
        if len(words) <= max_words:
            return text
        window = " ".join(words[:max_words])
        ok = lambda c: len(cls._words(c)) >= cls.min_words
        end = cls._sentence_end(window)
        if end is not None and ok(window[:end]):
            return window[:end]
        for ch in (";", ":", ","):
            i = window.rfind(ch)
            if i >= 0 and ok(window[: i + 1]):
                return window[: i + 1]
        low = window.lower()
        for group in (cls._conjunctions, cls._starters):
            for k in group:
                i = low.rfind(k)
                if i >= 0 and ok(window[:i]):
                    return window[:i]
        return window

    @classmethod
    def _sentence_end(cls, text):
        last = None
        for i, ch in enumerate(text):
            if ch in ".!?" and (i + 1 == len(text) or text[i + 1].isspace()) and i >= cls.min_words * 4:
                last = i + 1
        return last

    @staticmethod
    def estimate_tokens(text):
        return max(50, len([w for w in text.split(" ") if w]) * 5)


class StreamingWAVWriter:
    """Utilities/AudioSampleWriter.swift:44-106: 44-byte placeholder header, 16-bit PCM `Int16(clamped * 32767)`
    (truncation toward zero), header patched on finalize."""

    def __init__(self, path, sample_rate=24000):
        self.path, self.sample_rate, self.sample_count = path, sample_rate, 0
        self._f = open(path, "wb")
        self._f.write(b"\0" * 44)

    def write(self, samples):
        s = np.clip(np.asarray(samples, dtype=np.float32), -1.0, 1.0)
        self._f.write(np.trunc(s * np.float32(32767.0)).astype("<i2").tobytes())
        self.sample_count += int(s.size)

    def finalize(self):
        data = self.sample_count * 2
        hdr = b"RIFF" + struct.pack("<I", 36 + data) + b"WAVEfmt " + struct.pack("<IHHIIHH", 16, 1, 1, self.sample_rate,
                                                                                  self.sample_rate * 2, 2, 16) + b"data" + struct.pack("<I", data)
        self._f.seek(0)
        self._f.write(hdr)
        self._f.close()
        return self.sample_count


class SyntheticTokenizer:
    """Deterministic stand-in used ONLY with synthetic checkpoints (no tokenizer.json on disk): special tokens map
    to fixed ids, every other whitespace-separated word / punctuation run hashes into the text vocabulary.  The
    reference's BPE (Tokenizer/Qwen3Tokenizer.swift) is host string code outside the engine boundary."""

    def __init__(self, text_vocab_size: int, reserved_top: int = 64):
        self.n = max(16, text_vocab_size - reserved_top)
        self.special = {"<|im_start|>": self.n + 1, "<|im_end|>": self.n + 2, "\n": self.n + 3, "assistant": self.n + 4, "user": self.n + 5}

    def encode(self, text: str):
        import re

        ids = []
        for tok in re.findall(r"<\|im_start\|>|<\|im_end\|>|\n|[A-Za-z0-9']+|[^\sA-Za-z0-9']", text):
            if tok in self.special:
                ids.append(self.special[tok])
            else:
                h = 2166136261
                for b in tok.encode("utf-8"):
                    h = ((h ^ b) * 16777619) & 0xFFFFFFFF
                ids.append(h % self.n)
        return ids


def _load_tokenizer(model_path, text_vocab):
    tj = os.path.join(model_path, "tokenizer.json")
    if os.path.exists(tj):
        try:
            from tokenizers import Tokenizer

            t = Tokenizer.from_file(tj)

            class _HF:
                def encode(self, text):
                    # quote normalisation of Qwen3Tokenizer.encode (Tokenizer/Qwen3Tokenizer.swift:165-190)
                    for a, b in (("‘", "'"), ("’", "'"), ("“", '"'), ("”", '"')):
                        text = text.replace(a, b)
                    return t.encode(text, add_special_tokens=False).ids

            return _HF()
        except Exception:
            pass
    return SyntheticTokenizer(text_vocab)


class Qwen3TTSPipeline:
    sample_rate = 24000  # Qwen3TTSPipeline.swift:65

    def __init__(self, model_path, configuration: Qwen3TTSPipelineConfiguration | None = None, tokenizer=None):
        self.config = configuration or Qwen3TTSPipelineConfiguration()
        model_path = str(model_path)
        try:
            self.engine = Engine(model_path, device=self.config.device, max_batch=self.config.max_batch,
                                 kv_capacity=self.config.kv_capacity, max_frames=max(self.config.default_max_tokens, 600),
                                 use_cuda_graph=self.config.use_cuda_graph, runtime_quantization=self.config.apply_runtime_quantization,
                                 lanes=self.config.lanes)
        except A.Q3Error as e:
            if e.status == A.ERR_FILE_NOT_FOUND:
                raise FileNotFound(e.message.split(": ", 1)[-1]) from e
            if e.status == A.ERR_DECODER_LOAD_FAILED:
                raise DecoderLoadFailed() from e
            raise
        self.info = self.engine.info
        self._speakers = self.engine.speakers()
        self.tokenizer = tokenizer or _load_tokenizer(model_path, self.info.text_vocab_size)

    # ---- properties (Qwen3TTSPipeline.swift:76-104)
    @property
    def available_speakers(self):
        return sorted(self._speakers.keys())

    @property
    def supports_voice_cloning(self):
        return bool(self.info.has_speaker_encoder)  # speakerEncoder?.isWeightsLoaded (Qwen3TTSPipeline.swift:82-84)

    @property
    def supports_icl(self):
        return bool(self.info.has_audio_encoder)  # audioEncoder != nil (Qwen3TTSPipeline.swift:87-89)

    @property
    def model_type(self):
        return {0: None, 1: "voice_design", 2: "custom_voice"}[self.info.model_type]

    @property
    def supports_voice_design(self):
        return self.info.model_type == 1

    @property
    def supports_custom_voice(self):
        return self.info.model_type == 2

    # ---- request assembly (host string side of Model/Qwen3Talker.swift:338-414)
    def _request(self, text, speaker="", instruct=None, speaker_embedding=None, reference_transcript=None, reference_audio_codes=None,
                 temperature=None, max_tokens=None, stream_variant=False, voice=None) -> GenRequest:
        enc = self.tokenizer.encode
        chat = f"<|im_start|>assistant\n{text}<|im_end|>\n<|im_start|>assistant\n"  # :344
        if voice is not None:  # the voice's prefilled prefix stands for every voice field
            if speaker or instruct or speaker_embedding is not None or reference_transcript or reference_audio_codes is not None:
                raise ValueError("voice= replaces speaker, instruct, speaker_embedding and the reference fields: pass one or the other")
            return GenRequest(text_ids=enc(chat), voice=voice,
                              temperature=self.config.default_temperature if temperature is None else temperature,
                              max_tokens=self.config.default_max_tokens if max_tokens is None else max_tokens,
                              seed=self.config.seed, stream_variant=stream_variant)
        spk_id = self._speakers.get(speaker.lower(), -1) if speaker else -1  # :339-340
        instruct_ids = None
        ref_ids = None
        use_icl = reference_audio_codes is not None and reference_transcript is not None and len(reference_transcript) > 0  # :338
        if instruct:
            instruct_ids = enc(f"<|im_start|>user\n{instruct}<|im_end|>\n")  # :391
        elif use_icl:
            ref_ids = enc(f"<|im_start|>user\n{reference_transcript}<|im_end|>\n")  # :396
        elif speaker and spk_id < 0 and speaker_embedding is None:
            instruct_ids = enc(f"<|im_start|>user\n{speaker}<|im_end|>\n")  # backward compat: prompt as instruct (:408-413)
        return GenRequest(
            text_ids=enc(chat), speaker_id=spk_id,
            speaker_embedding=None if (spk_id >= 0 or speaker_embedding is None) else np.asarray(speaker_embedding, dtype=np.float32),
            instruct_ids=instruct_ids, ref_text_ids=ref_ids,
            ref_codes=None if not use_icl or instruct else np.asarray(reference_audio_codes, dtype=np.int32),
            temperature=self.config.default_temperature if temperature is None else temperature,
            max_tokens=self.config.default_max_tokens if max_tokens is None else max_tokens,
            seed=self.config.seed, stream_variant=stream_variant)

    # ---- registered voices (no reference counterpart)
    def prepare_voice(self, speaker="", instruct=None, speaker_embedding=None, reference_transcript=None, reference_audio_codes=None) -> Voice:
        """Prefill the voice part of the prompt once (q3tts_voice_create), from the same fields and rules as a request.  Pass the result
        as `voice=` to any generate* call of this pipeline: the output is bit for bit what the fields written inline give, without
        prefilling them again.  Free it with close() (or a `with` block); it may outlive the pipeline."""
        return self.engine.create_voice(self._request("", speaker=speaker, instruct=instruct, speaker_embedding=speaker_embedding,
                                                      reference_transcript=reference_transcript, reference_audio_codes=reference_audio_codes))

    def _call_voice(self, n_chunks, voice, **fields):
        """(voice to use, voice to free at the end) of a call that runs n_chunks generations with the same voice fields."""
        if voice is not None or n_chunks <= 1:
            return voice, None
        own = self.prepare_voice(**fields)
        return own, own

    def _chunk_request(self, text, voice, own, fields, **kw) -> GenRequest:
        """The request of one chunk: with the call's voice, unless the chunk's role ids differ from a voice the call made itself
        (a tokenizer may merge the role's last id into the text), which then runs with its fields inline."""
        if voice is not None:
            req = self._request(text, voice=voice, **kw)
            if voice is not own or list(req.text_ids[:3]) == voice.role_ids:
                return req
        return self._request(text, **fields, **kw)

    # ---- simple generation (:244-306, 355-381, 424-451)
    def generate(self, text, speaker="", speaker_embedding=None, temperature=None, max_tokens=None, instruct=None, voice=None):
        req = self._request(text, speaker=speaker, instruct=instruct, speaker_embedding=speaker_embedding, temperature=temperature,
                            max_tokens=max_tokens, voice=voice)
        pcm, _ = self.engine.generate_pcm(req, A.DECODE_WHOLE)
        return pcm

    def generate_voice_design(self, text, voice_description=None, temperature=None, max_tokens=None, voice=None):
        return self.generate(text, speaker="", instruct=voice_description, temperature=temperature, max_tokens=max_tokens, voice=voice)

    def generate_custom_voice(self, text, speaker="", instruct=None, temperature=None, max_tokens=None, voice=None):
        return self.generate(text, speaker=speaker, instruct=instruct, temperature=temperature, max_tokens=max_tokens, voice=voice)

    # ---- streaming (:323-340, 392-408, 463-480, 484-624)
    def generate_stream(self, text, speaker="", speaker_embedding=None, temperature=None, max_tokens=None, chunk_size=None, instruct=None,
                        voice=None):
        req = self._request(text, speaker=speaker, instruct=instruct, speaker_embedding=speaker_embedding, temperature=temperature,
                            max_tokens=max_tokens, stream_variant=True, voice=voice)
        st = self.engine.stream(req, chunk_size or self.config.default_streaming_chunk_size)
        try:
            while True:
                samples, (t0, t1), is_final, done = st.next_audio()
                yield AudioChunk(samples, range(t0, t1), is_final)
                if done:
                    break
        finally:
            st.close()

    def generate_stream_voice_design(self, text, voice_description=None, **kw):
        return self.generate_stream(text, speaker="", instruct=voice_description, **kw)

    def generate_stream_custom_voice(self, text, speaker="", instruct=None, **kw):
        return self.generate_stream(text, speaker=speaker, instruct=instruct, **kw)

    # ---- file output (:644-757)
    def generate_to_file(self, text, output_url, speaker="", instruct=None, speaker_embedding=None, reference_transcript=None,
                         reference_audio_codes=None, temperature=None, on_progress=None, voice=None) -> int:
        chunks = TextChunker.chunk(text, TextChunker.default_max_words)
        if not chunks:
            return 0
        fields = dict(speaker=speaker, instruct=instruct, speaker_embedding=speaker_embedding, reference_transcript=reference_transcript,
                      reference_audio_codes=reference_audio_codes)
        # every chunk repeats the same voice: a call of several chunks prefills it once (a voice of its own, freed before returning)
        voice, own = self._call_voice(len(chunks), voice, **fields)
        try:
            return self._generate_to_file(chunks, output_url, voice, own, fields, temperature, on_progress)
        finally:
            if own is not None:
                own.close()

    def _generate_to_file(self, chunks, output_url, voice, own, fields, temperature, on_progress) -> int:
        writer = StreamingWAVWriter(output_url)
        # Every text chunk is an independent generation with a fresh KV cache (Qwen3TTSPipeline.swift:668-691), so a handle with
        # several slots runs `max_batch` chunks at a time through the batched path; a handle's numeric path is fixed at creation,
        # so the samples of a chunk do not depend on how many chunks shared its steps.  The file is written in chunk order.
        group = max(1, int(self.info.max_batch)) * max(1, int(self.config.lanes))
        for g0 in range(0, len(chunks), group):
            part = chunks[g0: g0 + group]
            if on_progress:
                on_progress(g0 / len(chunks))
            reqs = [self._chunk_request(tc, voice, own, fields, temperature=temperature, max_tokens=600) for tc in part]  # :690
            if len(reqs) == 1:
                outs = [self.engine.generate_pcm(reqs[0], A.DECODE_FILE)]
            else:
                pcms, frames = self.engine.generate_pcm_batch(reqs, A.DECODE_FILE)
                outs = list(zip(pcms, frames))
            for pcm, frames in outs:
                if frames == 0 or pcm.size == 0:
                    continue
                writer.write(pcm)
        if on_progress:
            on_progress(1.0)
        return writer.finalize()

    # ---- batch (:774-898)
    def generate_batch(self, text, speaker="", instruct=None, speaker_embedding=None, reference_transcript=None, temperature=None,
                       on_progress=None, voice=None):
        chunks = TextChunker.chunk(text, TextChunker.default_max_words)
        if not chunks:
            return np.zeros(0, np.float32)
        if len(chunks) == 1:  # single-chunk shortcut drops speakerEmbedding / instruct, as the reference does (:791-796)
            if on_progress:
                on_progress(0.0)
            out = self.generate(chunks[0], speaker=speaker if voice is None else "", temperature=temperature, voice=voice)
            if on_progress:
                on_progress(1.0)
            return out
        # generateBatch forwards the transcript but not the codes, so ICL stays off (:813-822)
        fields = dict(speaker=speaker, instruct=instruct, speaker_embedding=speaker_embedding)
        voice, own = self._call_voice(len(chunks), voice, **fields)
        try:
            return self._generate_batch(chunks, voice, own, fields, temperature, on_progress)
        finally:
            if own is not None:
                own.close()

    def _generate_batch(self, chunks, voice, own, fields, temperature, on_progress):
        cf = self.config.crossfade_samples
        all_s, tail = [], np.zeros(0, np.float32)
        # chunks are independent generations (:813-864): a handle with several slots runs `max_batch` of them per batched call, the
        # crossfade below consumes them in chunk order
        group = max(1, int(self.info.max_batch)) * max(1, int(self.config.lanes))
        done: dict = {}
        for i, tc in enumerate(chunks):
            if on_progress:
                on_progress(i / len(chunks))
            if i not in done:
                reqs = [self._chunk_request(c, voice, own, fields, temperature=temperature, max_tokens=600) for c in chunks[i: i + group]]
                if len(reqs) == 1:
                    done[i] = self.engine.generate_pcm(reqs[0], A.DECODE_BATCHAPI)
                else:
                    pcms, fr = self.engine.generate_pcm_batch(reqs, A.DECODE_BATCHAPI)
                    for j in range(len(reqs)):
                        done[i + j] = (pcms[j], fr[j])
            ch, frames = done.pop(i)
            if frames == 0 or ch.size == 0:
                continue
            last = i == len(chunks) - 1
            if tail.size and cf > 0:  # crossfade (:869-879)
                n = min(cf, tail.size, ch.size)
                k = np.arange(n, dtype=np.float32)
                all_s.append(tail[:n] * ((np.float32(n) - k) / np.float32(n)) + ch[:n] * (k / np.float32(n)))
                ch = ch[n:]
            if last:
                all_s.append(ch)
            elif ch.size > cf:
                all_s.append(ch[: ch.size - cf])
                tail = ch[ch.size - cf:]
            else:
                tail = ch
        if on_progress:
            on_progress(1.0)
        return np.concatenate(all_s) if all_s else np.zeros(0, np.float32)

    # ---- voice cloning inputs (:906-945).  Both encoders run on the device when the checkpoint carries their weights; without them the
    # calls return nil like the reference
    def extract_speaker_embedding(self, audio_samples):
        """[Float] speaker embedding of reference audio, or None without a speaker encoder (Qwen3TTSPipeline.swift:906-919)."""
        emb = self.engine.extract_speaker_embedding(audio_samples)
        return None if emb is None or emb.size == 0 else emb

    def encode_reference_audio(self, audio_samples):
        """[[Int32]] [num_quantizers][time] of 24 kHz reference audio, or None without an encoder (Qwen3TTSPipeline.swift:924-945)."""
        codes = self.engine.encode_reference_audio(audio_samples)
        return None if codes is None or codes.size == 0 else codes

    def clear_cache(self):  # :951-956
        self.engine.clear_cache()

    def close(self):
        self.engine.close()

    @staticmethod
    def wav_to_float_samples(data: bytes):  # :1006-1020
        if len(data) <= 44:
            return np.zeros(0, np.float32)
        return np.frombuffer(data[44: 44 + (len(data) - 44) // 2 * 2], dtype="<i2").astype(np.float32) / np.float32(32767.0)
