/*
 * qwen3tts_b200.h — C ABI of libqwen3tts_b200.so (CUDA, sm_100a only; no CPU fallback).
 *
 * The reference (hamptus/mlx-swift-qwen3-tts, Swift on MLX) has no FFI layer: its seam is the set of calls
 * `Qwen3TTSPipeline` makes into its MLX-backed classes.  Each entry point below replaces one of those calls;
 * the citation names the reference interface it stands in for (paths relative to
 * /root/reference/Sources/Qwen3TTS/).  The Swift module map that binds this header is in
 * mlx-swift-qwen3-tts_b200/swift/Sources/CQwen3TTSB200/, the Python ctypes binding used by the tests in
 * mlx-swift-qwen3-tts_b200/qwen3tts_b200/_abi.py; INTEGRATION.md shows the reference-side patch.
 *
 * Conventions
 *   - plain pointers and sizes only; the caller owns every buffer; inputs are copied before the call returns;
 *   - every function returns a q3tts_status (0 = ok, negative = error); q3tts_last_error() gives the text;
 *   - generation calls do NOT fail on "too short" / "no codes": they return Q3TTS_OK with 0 frames, like the
 *     reference returns [] (Model/Qwen3Talker.swift:348-352, 602-604);
 *   - one handle = one CUDA device + one stream; calls on a handle are serialised by an internal mutex
 *     (the reference is `@unchecked Sendable` with no locking, Qwen3TTSPipeline.swift:63);
 *   - token ids in, codes / PCM out: chat templating and BPE stay in the host language
 *     (Tokenizer/Qwen3Tokenizer.swift, Utilities/TextChunker.swift are outside this boundary).
 */
#ifndef QWEN3TTS_B200_H
#define QWEN3TTS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define Q3TTS_ABI_VERSION 1
#define Q3TTS_SAMPLE_RATE 24000      /* Qwen3TTSPipeline.swift:65 */
#define Q3TTS_SAMPLES_PER_FRAME 1920 /* Qwen3TTSPipeline.swift:522; Vocoder/SpeechTokenizer.swift:82 */

typedef struct q3tts_handle q3tts_handle;
typedef struct q3tts_stream q3tts_stream;
typedef struct q3tts_voice q3tts_voice; /* a registered voice: see q3tts_voice_create */

typedef enum q3tts_status {
  Q3TTS_OK = 0,
  Q3TTS_ERR_FILE_NOT_FOUND = -1,      /* Qwen3TTSError.fileNotFound      (Qwen3TTSPipeline.swift:986) */
  Q3TTS_ERR_DECODER_LOAD_FAILED = -2, /* Qwen3TTSError.decoderLoadFailed (Qwen3TTSPipeline.swift:987) */
  Q3TTS_ERR_MODEL_NOT_LOADED = -3,    /* Qwen3TTSError.modelNotLoaded    (Qwen3TTSPipeline.swift:988) */
  Q3TTS_ERR_BAD_CONFIG = -4,
  Q3TTS_ERR_BAD_WEIGHTS = -5,
  Q3TTS_ERR_CUDA = -6,
  Q3TTS_ERR_INVALID_ARG = -7,
  Q3TTS_ERR_CANCELLED = -8,
  Q3TTS_ERR_NO_DEVICE = -9, /* no sm_100 GPU: the library never computes on the CPU */
  Q3TTS_ERR_CAPACITY = -10
} q3tts_status;

/* dtypes of raw buffers crossing the ABI */
typedef enum q3tts_dtype { Q3TTS_F32 = 0, Q3TTS_F16 = 1, Q3TTS_BF16 = 2 } q3tts_dtype;

/* ---- options: replaces Qwen3TTSPipelineConfiguration's device/loader side + DeviceSelector
 *      (Qwen3TTSPipeline.swift:22-54, Utilities/DeviceSelector.swift:9-32) ------------------------------- */
typedef struct q3tts_options {
  int32_t struct_size;      /* sizeof(q3tts_options), for forward compatibility */
  int32_t device;           /* CUDA ordinal */
  void* cuda_stream;        /* cudaStream_t to run on, or NULL: the library creates its own */
  int32_t max_batch;        /* concurrent utterances the handle can hold (1 = the reference's behaviour) */
  int32_t kv_capacity;      /* KV ring capacity per utterance in positions (>= prefill + 16); 0 = 512; values below 208 (a
                               192-key window + 16) are raised to 208; above 512 a 1-2 slot handle runs the CUDA-graph step */
  int32_t max_frames;       /* per-utterance frame buffer (>= max_tokens); 0 = 2400 (Qwen3TTSPipeline.swift:42) */
  int32_t use_cuda_graph;   /* 1: frame step replayed as a CUDA graph (the reference's analogue is MLX compile{}) */
  int32_t load_codec;       /* 0: talker only */
  int32_t load_talker;      /* 0: codec only (BASELINE config 4) */
  int32_t codec_max_frames; /* largest T of one codec decode window; 0 = 2400 */
  int32_t codec_max_batch;  /* largest B of one codec decode call; 0 = 8 */
  int32_t packed_gemm;      /* 3..128-row decode GEMMs of a quantised checkpoint: 1 = stream the PACKED 4/8-bit weights and dequantise
                               inside the tcgen05 kernel (QuantizedLayerFactory.swift:56's quantizedMatmul; 0.5625 B/param from HBM),
                               2 = fp16 operand copies made at load (2 B/param), 0 = the faster of the two as measured (DESIGN.md 3.2;
                               today 2; env Q3TTS_SKINNY_Q=1 flips it).  Same bits either way (the copies ARE the dequantised values). */
  int32_t runtime_quantization; /* Qwen3TTSPipelineConfiguration.applyRuntimeQuantization (Qwen3TTSPipeline.swift:25, 184, 961-980): a checkpoint
                               without a `quantization` block is MLX-quantised at load, group 64, 6 bits for embeddings / q,k,v projections /
                               heads, 4 bits for the rest (codes held in an 8-bit container).  0 = run the checkpoint as stored.
                               Checkpoints with a `quantization` block are never re-quantised; MLX affine checkpoints of 2, 3, 4, 5, 6
                               and 8 bits with group_size 32, 64 or 128 load as stored (q3tts_info.checkpoint_quant_bits), and MLX mxfp4
                               checkpoints (mode "mxfp4", bits 4, group_size 32) load as exact 8-bit affine groups of 32 */
  int32_t lanes;            /* > 1: q3tts_generate_pcm_batch / q3tts_generate_codes_batch calls with more than max_batch requests are split over
                               `lanes` handles (this one + lazily created q3tts_clone()s sharing its weights), each served by a worker thread
                               of the call: several latency-bound launch chains overlap on the device (see q3tts_clone).  The threads live
                               only inside the call and never call back into the host.  0 / 1 = one chain (continuous batching over max_batch slots) */
  int32_t reserved[5];
} q3tts_options;

typedef struct q3tts_info {
  int32_t hidden_size, num_layers, num_heads, num_kv_heads, head_dim, intermediate_size;
  int32_t vocab_size, text_vocab_size, text_hidden_size;
  int32_t cp_hidden_size, cp_num_layers, cp_vocab_size, num_code_groups;
  int32_t quant_bits, quant_group_size; /* 0 bits = dense weights */
  int32_t weight_dtype;                 /* q3tts_dtype of dense / scale tensors */
  int32_t num_speakers;                 /* availableSpeakers (Qwen3TTSPipeline.swift:77-79) */
  int32_t has_codec, codec_num_quantizers, codec_total_upsample;
  int32_t model_type; /* 0 base, 1 voice_design, 2 custom_voice (Qwen3TTSPipeline.swift:92-104) */
  int32_t codec_eos_id, codec_pad_id;
  int32_t max_batch, kv_capacity, max_frames;
  int64_t device_bytes; /* HBM held by the handle */
  int32_t has_audio_encoder;    /* supportsICL (Qwen3TTSPipeline.swift:87-89): speech_tokenizer/model.safetensors carries `encoder.*` */
  int32_t audio_encoder_hidden; /* width of the quantiser input (q3tts_encode_reference_audio latent_out) */
  int32_t has_speaker_encoder;   /* model.safetensors carries `speaker_encoder.*` (Qwen3TTSPipeline.swift:82-84, 155-169) */
  int32_t speaker_embedding_dim; /* enc_dim of the ECAPA-TDNN (1024 in the reference) */
  int32_t checkpoint_quant_bits; /* width of the MLX-packed leaves on disk (2, 3, 4, 5, 6 or 8); 0 = dense checkpoint, runtime-quantised
                                    or not.  quant_bits is the width the kernels stream: 2 / 3-bit codes are held in 4-bit words and 5 / 6-bit
                                    codes in 8-bit words, unchanged (DESIGN.md §1) */
  int32_t checkpoint_quant_mode; /* 0 = MLX affine leaves or a dense checkpoint, 1 = MLX mxfp4 leaves (E2M1 codes, one E8M0 scale byte per
                                    32): held as exact 8-bit affine groups of 32 with bf16 scales and biases, so checkpoint_quant_bits is 4,
                                    quant_bits 8 and quant_group_size 32 (DESIGN.md §1; q3tts_mxfp4_to_affine) */
  int32_t reserved[2];
} q3tts_info;

/* ---- one utterance; replaces the argument list of Qwen3Talker.generateCodes / generateStream
 *      (Model/Qwen3Talker.swift:327-337, 633-644).  All ids are already templated + tokenised by the host. */
typedef struct q3tts_request {
  int32_t struct_size;
  const int32_t* text_ids; /* "<|im_start|>assistant\n{text}<|im_end|>\n<|im_start|>assistant\n" (:344) */
  int32_t n_text_ids;
  const int32_t* instruct_ids; /* "<|im_start|>user\n{instruct}<|im_end|>\n" or NULL (:389-394, 408-413) */
  int32_t n_instruct_ids;
  int32_t speaker_id;             /* codec_embedding row = config.spk_id[name.lowercased()], -1 = none (:370-373) */
  const float* speaker_embedding; /* [speaker_embedding_dim] == hidden_size, or NULL (:374-376) */
  int32_t speaker_embedding_dim;
  const int32_t* ref_text_ids; /* ICL "<|im_start|>user\n{transcript}<|im_end|>\n" or NULL (:396-398) */
  int32_t n_ref_text_ids;
  const int32_t* ref_codes; /* ICL codes [16][ref_frames] row-major, only row 0 is consumed (:402-403) */
  int32_t ref_frames;
  float temperature;        /* 0 = greedy (argmax BEFORE the valid-id mask, :301-305) */
  int32_t top_k;            /* 0 = off (reference default, :277) */
  float top_p;              /* 1 = off.  Extension: the reference has no top-p */
  float repetition_penalty; /* 1.05 in the reference (:279); set-based, division for every sign (:288-299) */
  int32_t max_tokens;
  uint64_t seed;          /* counter-based sampler stream (documented in DESIGN.md; MLX's is not reproducible) */
  int32_t stream_variant; /* 1 = generateStream's loop: no repetition penalty on code-predictor groups (:821) */
  /* --- diagnostics / parity hooks (all optional) --- */
  const int32_t* forced_codes; /* teacher forcing [n_forced_frames][16]: ids fed back instead of the sampled ones */
  int32_t n_forced_frames;
  float* code0_logits_out;    /* [frames][vocab_size]     raw codec_head logits of every sampled frame */
  float* cp_logits_out;       /* [frames][15][cp_vocab]   raw lm_head logits of every code-predictor pass */
  int32_t logits_capacity_frames;
  int32_t keep_invalid_frames; /* 1: skip the final code0 in [0,2048) filter (:571-576) */
  const q3tts_voice* voice;     /* a voice of q3tts_voice_create whose prefilled prompt prefix replaces the voice fields, or NULL
                                   (every field written inline, prefilled with the request).  Rules at q3tts_voice_create */
  int32_t reserved[4];
} q3tts_request;

/* decode scheduling of the fused text->PCM calls (Qwen3TTSPipeline.swift) */
typedef enum q3tts_decode_mode {
  Q3TTS_DECODE_WHOLE = 0,    /* generate():      one whole-sequence decode (Model/Qwen3Talker.swift:606-613) */
  Q3TTS_DECODE_FILE = 1,     /* generateToFile(): windows of 16 frames + 8 left context (:700-740) */
  Q3TTS_DECODE_BATCHAPI = 2, /* generateBatch():  windows of 24 + 8 (:827-829) */
  Q3TTS_DECODE_STREAM = 3    /* generateStream(): first window 18, then 8 + 18 (:520-561) */
} q3tts_decode_mode;

typedef struct q3tts_timing {
  double device_ms;        /* CUDA-event time of the last call's device work on the handle's stream */
  double prefill_ms;       /* part of device_ms spent in prefill */
  double decode_ms;        /* part spent in the codec decoder */
  int64_t kernel_launches; /* kernels this library launched in the last call (graph nodes counted per replay) */
  int64_t graph_replays;
  int64_t frames;          /* talker frames produced (before the validity filter) */
  int64_t h2d_bytes, d2h_bytes;
  int64_t weight_bytes_per_frame; /* algorithmic bytes streamed per 12.5 Hz frame (SURVEY.md §8d): weights counted in the 4 / 8-bit
                                     words the kernels read, so a 3-bit checkpoint counts as 4-bit and a 5 / 6-bit one as 8-bit */
  double talker_ms;               /* CUDA-event time of prompt assembly + prefill + all frame steps of the last call */
  int64_t codec_flops;            /* algorithmic flops of the codec passes of the last call (SURVEY.md §8d) */
  int64_t persistent_launches;    /* launches of the persistent frame kernel in the last call (0 = CUDA-graph / eager path) */
  int64_t prefill_rows;           /* talker rows the last call's prefill computed (q3tts_stream_begin included): the whole prompt of an
                                     inline request, 1 of a request with a voice */
  int64_t reserved[2];
} q3tts_timing;

/* ------------------------------------------------------------------------------------------------------
 * lifecycle — replaces Qwen3TTSPipeline.init(modelPath:configuration:) (Qwen3TTSPipeline.swift:118-232):
 * config.json, model.safetensors, speech_tokenizer/{config.json|configuration.json|speech_tokenizer_config.json}
 * + speech_tokenizer/model.safetensors; key remap of Qwen3Talker.load (Model/Qwen3Talker.swift:114-270) and
 * AudioDecoder.sanitize (Vocoder/AudioDecoder.swift:196-305).
 * ---------------------------------------------------------------------------------------------------- */
int32_t q3tts_abi_version(void);
void q3tts_default_options(q3tts_options* opts);
void q3tts_default_request(q3tts_request* req);
q3tts_status q3tts_create(const char* model_dir, const q3tts_options* opts, q3tts_handle** out);
/* A second handle on the same device that SHARES the parent's talker weights (packed / dense tensors and their fp16 tensor-core copies;
 * reference counted: parent and clones may be destroyed in any order) and owns everything mutable: stream, KV rings, slot state,
 * activation buffers, CUDA graphs, codec instance.  Same options as the parent.  Purpose: a batched decode step is a latency-bound chain
 * of ~570 dependent launches that leaves the SMs mostly idle; a host with more than max_batch pending requests serves them through 2-4
 * handles from as many threads (1.7B bf16, 512 utterances: 997 / 1 408 / 1 575 / 1 712 audio-s/s with 1 / 2 / 3 / 4 handles) without
 * paying for the weights again.  Results per request are bit-identical to the parent's.  The reference-audio and speaker encoders stay
 * with the parent.  No reference counterpart (the reference serves one utterance at a time). */
q3tts_status q3tts_clone(q3tts_handle* parent, q3tts_handle** out);
void q3tts_destroy(q3tts_handle* h);
/* error text of the last failing call on `h`; h == NULL: of the last failing q3tts_create on this thread */
const char* q3tts_last_error(const q3tts_handle* h);
q3tts_status q3tts_get_info(const q3tts_handle* h, q3tts_info* out);
/* availableSpeakers / config.spk_id (Qwen3TTSPipeline.swift:77-79; Model/Qwen3Talker.swift:339-340) */
q3tts_status q3tts_speaker_name(const q3tts_handle* h, int32_t index, char* name_out, int32_t capacity, int32_t* id_out);
int32_t q3tts_speaker_id(const q3tts_handle* h, const char* lowercased_name); /* -1 if unknown */
/* Qwen3Talker.clearGenerationCache + AudioDecoder.clearCompiledCache + Memory.clearCache
 * (Qwen3TTSPipeline.swift:951-956): drops CUDA graphs and scratch; weights stay resident */
q3tts_status q3tts_clear_cache(q3tts_handle* h);
q3tts_status q3tts_get_timing(const q3tts_handle* h, q3tts_timing* out);

/* ------------------------------------------------------------------------------------------------------
 * talker — replaces Qwen3Talker.generateCodes (Model/Qwen3Talker.swift:327-577).
 * codes_out: [capacity_frames][16] int32; *frames_out <= min(max_tokens, capacity_frames).
 * ---------------------------------------------------------------------------------------------------- */
q3tts_status q3tts_generate_codes(q3tts_handle* h, const q3tts_request* req, int32_t* codes_out,
                                  int32_t capacity_frames, int32_t* frames_out);
/* request-parallel batch of independent utterances on one GPU (continuous batching over max_batch slots);
 * codes_out[i] -> [capacity_frames][16]; same per-utterance results as n calls of q3tts_generate_codes */
q3tts_status q3tts_generate_codes_batch(q3tts_handle* h, const q3tts_request* reqs, int32_t n_requests,
                                        int32_t* const* codes_out, int32_t capacity_frames, int32_t* frames_out);

/* replaces Qwen3Talker.generateStream (Model/Qwen3Talker.swift:633-885): code chunks of `chunk_size` frames
 * (:831-835), final partial chunk (:871-873).  q3tts_stream_next is the cancellation point (:771).
 * A stream owns talker slot 0 of its handle from q3tts_stream_begin until q3tts_stream_free: meanwhile a second
 * q3tts_stream_begin and every q3tts_generate_* call on that handle fail with Q3TTS_ERR_INVALID_ARG (the codec calls
 * q3tts_decode* stay available).  q3tts_stream_cancel may be called from any thread. */
q3tts_status q3tts_stream_begin(q3tts_handle* h, const q3tts_request* req, int32_t chunk_size, q3tts_stream** out);
q3tts_status q3tts_stream_next(q3tts_stream* s, int32_t* codes_out /*[chunk_size][16]*/, int32_t* frames_out,
                               int32_t* done_out);
/* replaces the consumer half of _generateStreamImpl (Qwen3TTSPipeline.swift:572-607): yields AudioChunk
 * {samples, tokenRange, isFinal}; windows 18 / 8+18; the trailing empty isFinal chunk is delivered too (:607).
 * pcm_out capacity must be >= (decode_chunk) * 1920 floats where decode_chunk = 18. */
q3tts_status q3tts_stream_next_audio(q3tts_stream* s, float* pcm_out, int32_t capacity_samples, int32_t* samples_out,
                                     int32_t* token_start_out, int32_t* token_end_out, int32_t* is_final_out,
                                     int32_t* done_out);
q3tts_status q3tts_stream_cancel(q3tts_stream* s);
void q3tts_stream_free(q3tts_stream* s);

/* ------------------------------------------------------------------------------------------------------
 * registered voices (no reference counterpart: the reference prefills every prompt whole).  Every prompt row before the
 * first text id depends only on the voice: [instruct | ICL transcript + ICL codes] + role ids + the codec rows with the speaker
 * (Model/Qwen3Talker.swift:344-433).  q3tts_voice_create prefills those P - 1 rows once and keeps their talker K / V (every layer
 * and kv head, in the handle's ring element type: fp16 on handles of >= 3 slots, fp32 otherwise); a request with `voice` set
 * installs them into its slot's KV ring and prefills its one remaining row.
 *
 *   - Input: `voice` is read for instruct_ids, speaker_id / speaker_embedding, ref_text_ids + ref_codes / ref_frames (the same
 *     precedence rules as a request) and text_ids[0..2] (the role ids; n_text_ids >= 3).  Sampling and diagnostic fields are ignored.
 *     Ids and codes are validated with the same checks and errors as a request.  P - 1 prefix positions: P + 16 <= kv_capacity, or
 *     Q3TTS_ERR_CAPACITY.  Not while a stream is open on the handle (Q3TTS_ERR_INVALID_ARG, as q3tts_generate_*).
 *   - Output contract: a request with voice = v gives the same codes, code0_logits_out / cp_logits_out and PCM, bit for bit, as the
 *     same request with v's fields written inline and voice = NULL -- on every decode path, greedy, sampled and teacher-forced.
 *   - Exclusive fields: a request with a voice leaves instruct_ids, ref_text_ids, ref_codes and speaker_embedding NULL and
 *     speaker_id at -1, and its text_ids[0..2] equal the voice's role ids; otherwise the call returns Q3TTS_ERR_INVALID_ARG before
 *     any device work.  A request with fewer than 9 text ids still returns 0 frames with Q3TTS_OK (its text is not read).
 *   - Handles: a voice is accepted by the handle that created it and by that handle's clones (the same weights and options, so the
 *     same numeric path and KV element type); any other handle returns Q3TTS_ERR_INVALID_ARG.  Streams (q3tts_stream_begin), batches
 *     and q3tts_options.lanes accept voices; requests with and without voices, and with different voices, mix in one call.
 *   - Lifetime and threads: a voice is immutable once created and may be used from several threads at once by the handles that
 *     accept it.  It holds a reference on the shared weights: a voice, its handle and the handle's clones may be freed in any order.
 *     Freeing a voice while a call that uses it is running is a caller error.
 * ---------------------------------------------------------------------------------------------------- */
q3tts_status q3tts_voice_create(q3tts_handle* h, const q3tts_request* voice, q3tts_voice** out);
/* prefix positions (P - 1) and the device bytes the voice holds (P - 1 positions x 2 x layers x kv_heads x 128 elements) */
q3tts_status q3tts_voice_info(const q3tts_voice* v, int32_t* prefix_positions_out, int64_t* device_bytes_out);
void q3tts_voice_free(q3tts_voice* v);

/* ------------------------------------------------------------------------------------------------------
 * codec — replaces AudioDecoder.mlxDecode / decode / chunkedDecode (Vocoder/AudioDecoder.swift:157-182) and
 * Qwen3TTSSpeechTokenizerDecoder.callAsFunction / chunkedDecode (Vocoder/SpeechTokenizer.swift:904-987).
 * codes: [B][F][16] int32 (the layout mlxDecode takes, before its own transpose); pcm_out: [B][F*1920] fp32.
 * ---------------------------------------------------------------------------------------------------- */
q3tts_status q3tts_decode(q3tts_handle* h, const int32_t* codes, int32_t batch, int32_t frames, float* pcm_out);
q3tts_status q3tts_decode_chunked(q3tts_handle* h, const int32_t* codes, int32_t batch, int32_t frames,
                                  int32_t chunk_size, int32_t left_context, float* pcm_out);

/* ------------------------------------------------------------------------------------------------------
 * ICL reference-audio encoder -- replaces Qwen3TTSPipeline.encodeReferenceAudio (Qwen3TTSPipeline.swift:924-945), i.e.
 * Qwen3TTSAudioEncoder.encode (Vocoder/Qwen3TTSAudioEncoder.swift:526-572): 24 kHz mono PCM -> SEANet CNN -> bidirectional
 * transformer -> stride-2 downsample -> split residual vector quantiser (nearest codeword per layer) -> the first 16 code rows.
 * codes_out: [quantizers][frames] int32 row-major -- exactly the `ref_codes` layout q3tts_request takes; *frames_out =
 * ceil(ceil(n / 960) / 2) (one frame per 1920 samples, the last one completed by zero padding).  Without encoder weights in the
 * checkpoint the call returns Q3TTS_OK with *frames_out = 0 (the reference returns nil).  latent_out (optional,
 * [frames][audio_encoder_hidden] fp32) receives the quantiser's input, for parity probes.
 * ---------------------------------------------------------------------------------------------------- */
q3tts_status q3tts_encode_reference_audio(q3tts_handle* h, const float* samples, int64_t n_samples, int32_t* codes_out,
                                          int32_t capacity_frames, int32_t* frames_out, int32_t* quantizers_out, float* latent_out);

/* ECAPA-TDNN speaker encoder -- replaces Qwen3TTSPipeline.extractSpeakerEmbedding (Qwen3TTSPipeline.swift:906-919), i.e.
 * SpeakerEncoder.extractEmbedding (SpeakerEncoder/SpeakerEncoder.swift:526-542): 24 kHz mono PCM -> log-mel (reflect-padded STFT 1024 / hop
 * 256, symmetric Hann, 128 Slaney mel bins, log(clip(., 1e-5))) -> TimeDelayNet / SE-Res2Net blocks -> attentive statistics pooling -> 1x1
 * conv.  embedding_out: [speaker_embedding_dim] fp32 -- exactly what q3tts_request.speaker_embedding takes.  Without the weights the call
 * returns Q3TTS_OK with *dim_out = 0 (the reference returns nil).  mels_out (optional, [n_samples / 256 + 1][128] fp32) receives the
 * log-mel input, for parity probes.  Needs at least 1024 samples (5 frames: the reflect padding of the dilation-4 block indexes frame 4). */
q3tts_status q3tts_extract_speaker_embedding(q3tts_handle* h, const float* samples, int64_t n_samples, float* embedding_out, int32_t capacity,
                                             int32_t* dim_out, float* mels_out);

/* ------------------------------------------------------------------------------------------------------
 * fused text -> PCM — the bodies of Qwen3TTSPipeline.generate (:244-306), generateToFile's per-text-chunk work
 * (:681-744) and generateBatch's (:813-864): generateCodes, then decode as `mode` schedules it, NaN/Inf scrub
 * and clamp (:565-570, 726-732).  *samples_out <= capacity_samples; needs frames*1920 floats.
 * ---------------------------------------------------------------------------------------------------- */
q3tts_status q3tts_generate_pcm(q3tts_handle* h, const q3tts_request* req, int32_t mode, float* pcm_out,
                                int64_t capacity_samples, int64_t* samples_out, int32_t* frames_out);
q3tts_status q3tts_generate_pcm_batch(q3tts_handle* h, const q3tts_request* reqs, int32_t n_requests, int32_t mode,
                                      float* const* pcm_out, int64_t capacity_samples, int64_t* samples_out,
                                      int32_t* frames_out);

/* ------------------------------------------------------------------------------------------------------
 * parity probes (single ops the reference reaches through MLX; host buffers in and out)
 * ---------------------------------------------------------------------------------------------------- */
/* MLX `dequantized(w, scales:, biases:, groupSize:, bits:, dtype:)` as called at Model/Qwen3Talker.swift:156.
 * packed [out][in*bits/32] uint32, scales/biases [out][in/group] of `scale_dtype`; out [out][in] of `out_dtype`.
 * Contract: deq32 = fp32(scale)*q (rounded) + fp32(bias) (rounded); result = round_to_nearest_even(deq32).
 * bits 2, 3, 4, 5, 6 or 8: a row is one little-endian LSB-first bit stream, code j at bits [j*bits, (j+1)*bits) (for 2 / 4 / 8 bits:
 * element j of a word at bit offset j*bits).  Bits 2 / 3 / 5 / 6 need group_size 32, 64 or 128 and in % 32 == 0; they are widened on
 * the device into the 4 / 8-bit words the loader keeps, then run the same kernel.  The same widths and rules hold for
 * q3tts_quantized_matmul and q3tts_quantized_matmul_tc; arguments are checked before any device is touched. */
/* MLX `quantize(w, group_size: 64, bits)` (affine) on the device -- the quantiser behind q3tts_options.runtime_quantization
 * (Qwen3TTSPipeline.applyMixedQuantization, Qwen3TTSPipeline.swift:961-980; bits 4, 6 or 8).  w: [out_f][in_f] of w_dtype (host);
 * codes8_out: [out_f][in_f] bytes, one code per byte (the 8-bit container, = MLX-packed 8-bit words); scales_out / biases_out:
 * [out_f][in_f / 64] of w_dtype.  Bit-exact against oracle/mlx_quant.py:quantize_codes. */
q3tts_status q3tts_mlx_quantize(int32_t device, const void* w, int32_t w_dtype, int32_t out_f, int32_t in_f, int32_t bits, uint32_t* codes8_out,
                                void* scales_out, void* biases_out);
q3tts_status q3tts_dequantize(int32_t device, const uint32_t* packed, const void* scales, const void* biases,
                              int32_t scale_dtype, int32_t out_features, int32_t in_features, int32_t group_size,
                              int32_t bits, int32_t out_dtype, void* out);
/* The load-time conversion of an MLX mxfp4 leaf (config `mode` "mxfp4") on host buffers.  packed [out][in/8] uint32, E2M1 code j of a
 * word at bits 4j (LSB first); scales [out][in/32] E8M0 bytes, element = lut[code] * 2^(byte - 127) with
 * lut = {0, .5, 1, 1.5, 2, 3, 4, 6, -0, -.5, -1, -1.5, -2, -3, -4, -6}.  Output: the same values as an 8-bit affine group of 32:
 * codes8_out [out][in/4] uint32 (q = 2 * lut[code] + 12, the 8-bit word layout of q3tts_dequantize), scales_out / biases_out
 * [out][in/32] bf16 (2^(byte - 128) and -12 * 2^(byte - 128)).  q3tts_dequantize, q3tts_quantized_matmul and
 * q3tts_quantized_matmul_tc take them with bits 8, group_size 32 and Q3TTS_BF16 scales and give the E2M1 values exactly (-0 as +0).
 * NULL pointers, in % 32 != 0 and scale bytes >= 252 (values the container cannot hold; 255 is E8M0's NaN) are refused with
 * Q3TTS_ERR_INVALID_ARG before any device is touched. */
q3tts_status q3tts_mxfp4_to_affine(int32_t device, const uint32_t* packed, const uint8_t* scales, int32_t out_features, int32_t in_features,
                                   uint32_t* codes8_out, void* scales_out, void* biases_out);
/* MLXNN.QuantizedLinear / quantized_matmul (Model/QuantizedLayerFactory.swift:56): y[m][out] = x[m][in] . W^T,
 * fp32 activations, the same kernels the talker uses for m rows. */
q3tts_status q3tts_quantized_matmul(int32_t device, const float* x, int32_t m, const uint32_t* packed,
                                    const void* scales, const void* biases, int32_t scale_dtype,
                                    int32_t out_features, int32_t in_features, int32_t group_size, int32_t bits,
                                    float* y);
/* The same contraction on the tensor-core path batched decode takes (csrc/gemm_skinny_q.cu): the packed matrix is the streamed
 * operand of a tcgen05 GEMM for m <= 128 rows, dequantised inside the kernel; activations rounded to fp16, fp32 accumulate.
 * fold (fp32 [in_features] or NULL): multiplied into the dequantised columns before their fp16 rounding (a folded RMSNorm weight).
 * swiglu_halves = 1: the packed rows are [gate ; up] (out_features / 2 each) and y[m][i] = silu(gate_i . x) * up_i . x for
 * i < out_features / 2 (Model/Qwen3Layers.swift:236); 0: y[m][out_features].  residual (fp32 [m][out] or NULL) is added. */
q3tts_status q3tts_quantized_matmul_tc(int32_t device, const float* x, int32_t m, const uint32_t* packed, const void* scales,
                                       const void* biases, int32_t scale_dtype, int32_t out_features, int32_t in_features,
                                       int32_t group_size, int32_t bits, const float* fold, int32_t swiglu_halves,
                                       const float* residual, float* y);
/* Qwen3Talker.sampleToken (Model/Qwen3Talker.swift:274-322) on one logits row; `counter` selects the position in
 * the request's sampler stream; token_set = ids already generated for this group (may be NULL). */
q3tts_status q3tts_sample_token(q3tts_handle* h, const float* logits, int32_t vocab, float temperature, int32_t top_k,
                                float top_p, float repetition_penalty, const int32_t* token_set, int32_t n_token_set,
                                uint64_t seed, uint64_t counter, int32_t* id_out);
/* The engine's device sampler (sampleToken, Model/Qwen3Talker.swift:274-322) on n_rows rows, one CTA per row, on host buffers.
 * form: 0 = the 512-thread form the CUDA-graph path and q3tts_sample_token run, 1 = the form of the persistent frame kernel (named
 * barrier 1 over warps 0-14 of a 512-thread CTA).  logits [n_rows][ld] fp32, V entries per row (ld = 0: every row reads row 0).
 * Per row r: temperature, top_k, top_p, repetition_penalty, seed and counter (the position in the sampler stream); token_sets
 * [n_rows][128] uint32 bitmaps (bit i % 32 of word i / 32 = id i is in the set) or NULL.  The valid-id mask applies when V == codec_vocab.
 * ids_out [n_rows]; processed_out [n_rows][V] or NULL: the row just before the Gumbel step (for greedy rows, right after the penalty),
 * -inf where removed.  1 <= V <= 4096, 1 <= n_rows <= 65535, ld = 0 or >= V, temperature / top_p / repetition_penalty finite and
 * top_p > 0; anything else returns Q3TTS_ERR_INVALID_ARG without touching the device. */
q3tts_status q3tts_sampler_probe(int32_t device, int32_t form, const float* logits, int32_t n_rows, int32_t V, int32_t ld, int32_t codec_vocab,
                                 const float* temperature, const int32_t* top_k, const float* top_p, const float* repetition_penalty,
                                 const uint32_t* token_sets, const uint64_t* seed, const uint64_t* counter, int32_t* ids_out,
                                 float* processed_out);
/* One sampling point of one group for n_slots slots, with the generation loop's per-slot rules, as the engine runs it: form 0 = the
 * sampler launch of the CUDA-graph path, 1 = the form of the persistent frame kernel.  group 0 = code0 (EOS / pad suppressed while
 * trailing_idx < total_text, the EOS and 7-pad stops unless the slot is forced, max_tokens, sets frame_alive); group g >= 1 = code-predictor
 * group g - 1 (nothing unless frame_alive; the id is added to the slot's set of group g; stream_variant drops the penalty).
 * logits [n_slots][V].  Slot state, one int32 array of n_slots per field, in/out: active, finished, step, max_tokens, trailing_idx,
 * total_text, consecutive_pad, n_forced, stream_variant, frame_alive, logits_cap.  Sampling fields per slot: temperature, top_k,
 * top_p, repetition_penalty, seed (the counter is step * 16 + group).  token_sets [n_slots][16][set_words] in/out (set_words * 32 >= V);
 * forced [n_slots][max_frames][16] or NULL (read when n_forced > 0); cur_codes [n_slots][16] in/out (a sampled slot writes [s][group]).
 * dump [dump_frames][V] or NULL: slot dump_slot's raw logits land in row `step` while step < logits_cap.  Arguments are validated on
 * the host (see q3tts_sampler_probe; also step >= 0, step < max_frames for forced slots, logits_cap[dump_slot] <= dump_frames). */
q3tts_status q3tts_sampler_slot_probe(int32_t device, int32_t form, int32_t group, int32_t n_slots, int32_t V, int32_t codec_vocab, int32_t eos_id,
                                      int32_t pad_id, const float* logits, int32_t* active, int32_t* finished, int32_t* step, int32_t* max_tokens,
                                      int32_t* trailing_idx, int32_t* total_text, int32_t* consecutive_pad, int32_t* n_forced,
                                      int32_t* stream_variant, int32_t* frame_alive, int32_t* logits_cap, const float* temperature,
                                      const int32_t* top_k, const float* top_p, const float* repetition_penalty, const uint64_t* seed,
                                      uint32_t* token_sets, int32_t set_words, const int32_t* forced, int32_t max_frames, float* dump,
                                      int32_t dump_slot, int32_t dump_frames, int32_t* cur_codes);
/* SplitResidualVectorQuantizer code -> embedding lookup (Vocoder/SpeechTokenizer.swift:504-506, 566-582, 684-691),
 * bit-exact contract: fp32 gather-sum in codebook order.  codes [B][F][16]; first_out/rest_out [B][F][dim] fp32
 * (rvq_first and rvq_rest sums before their 1x1 output projections). */
q3tts_status q3tts_rvq_embed(q3tts_handle* h, const int32_t* codes, int32_t batch, int32_t frames, float* first_out,
                             float* rest_out, int32_t* dim_out);

/* `MLX.loadArrays(url:)` front end (Qwen3TTSPipeline.swift:142; Vocoder/AudioDecoder.swift:141) without a device: parses and
 * bounds-checks the header of a .safetensors file exactly as q3tts_create does (every offset inside the file, byte count ==
 * product(shape) * sizeof(dtype)), so a corrupt checkpoint is rejected before anything is sized from it.
 * Returns Q3TTS_OK and the tensor count, Q3TTS_ERR_FILE_NOT_FOUND or Q3TTS_ERR_BAD_WEIGHTS (text via q3tts_last_error(NULL)). */
q3tts_status q3tts_safetensors_check(const char* path, int32_t* n_tensors_out, int64_t* data_bytes_out);

/* MLX `Conv1d` / `ConvTransposed1d` (polyphase) / `Linear` as the codec calls them (Vocoder/SpeechTokenizer.swift:142, 179,
 * 230, 726, 791), through the engine's implicit-GEMM kernels:  y[b,t,n] = epi(bias[n] + sum_tap x[b, t-(ntap-1-tap)*dil, :] . w[tap][n][:])
 * x [B][T][cin] fp32, w [ntap][N][cin] fp32.  use_tensor_cores = 1: tcgen05/TMEM path (operands rounded to fp16, fp32
 * accumulate); 0: fp32 SIMT path.  act: 0 none, 1 exact-erf GELU, 2 SiLU.  swiglu = 1: columns (2i, 2i+1) = (gate, up) ->
 * N/2 outputs.  res/scale: y = res + scale[n]*y (either may be NULL).  snake_ea/snake_ieb [snake_ch]: SnakeBeta applied to
 * the fp16 copy only.  y32 / y16 (fp16 values widened to fp32) are [B][T][N or N/2]; either may be NULL. */
q3tts_status q3tts_conv_probe(int32_t device, const float* x, int32_t B, int32_t T, int32_t cin, const float* w, const float* bias,
                              int32_t N, int32_t ntap, int32_t dil, int32_t act, int32_t swiglu, const float* res,
                              const float* scale, const float* snake_ea, const float* snake_ieb, int32_t snake_ch,
                              int32_t use_tensor_cores, float* y32, float* y16);

/* One talker attention launch as the engine issues it (head_dim 128, scale 1/sqrt(128)), on host buffers:
 * kernel: 0 = rope_attention (decode: one row per slot, appends that row's k/v), 1 = qk_norm_rope_append + attention (prefill),
 *         2 = cp_pass0_attention (rows 2s, 2s+1 at positions 0, 1; fp16 out, fp32 cache).
 * qkv [m][(heads + 2*kv_heads)*128]; row_slot / row_pos [m]; win_start [n_slots] or NULL (= 0);
 * k_ring / v_ring [n_slots][kv_heads][capacity][128] fp32, in/out (rounded to fp16 on upload when kv_f16, widened back);
 * out [m][heads*128] fp32 (fp16 values widened when out_f16).
 * Everything is validated before the launch: heads / kv_heads in {1, 2, 4}, slots in range, 0 <= win_start <= pos,
 * pos - win_start + 1 <= capacity, one row per slot for kernel 0, rows (2s, 2s+1) of slot s at positions (0, 1) with an fp32
 * cache and fp16 output for kernel 2.  Anything else returns Q3TTS_ERR_INVALID_ARG without touching the device. */
q3tts_status q3tts_attention_probe(int32_t device, int32_t kernel, int32_t kv_f16, int32_t out_f16, const float* qkv, int32_t m,
                                   int32_t heads, int32_t kv_heads, const float* q_norm, const float* k_norm, float eps,
                                   const float* inv_freq, const int32_t* row_slot, const int32_t* row_pos, const int32_t* win_start,
                                   int32_t n_slots, int32_t capacity, float* k_ring, float* v_ring, float* out);

/* Codec-decoder kernels one launch at a time, through the engine's own launchers, on host buffers.  Every argument is validated on
 * the host first: anything out of range returns Q3TTS_ERR_INVALID_ARG without touching the device.  Outputs no launch writes read
 * as 3.4e38 (fp32) or NaN (fp16).
 *
 * Codec-transformer attention (head_dim 64, scale 1/sqrt(64)).  kernel: 0 = the tcgen05 pipeline's fp16-output launch on the
 * mma.sync kernel, 1 = the SIMT pipeline's fp32 kernel (causal), 2 = its bidirectional form (ICL
 * encoder), 3 = the fp16-output SIMT kernel (the fallback of kernel 0's launcher).  qkv [B][T][(nh + 2*nkv)*64] fp32, in/out: when
 * inv_freq [32] is given the codec RoPE runs on it first, in place (positions t = row % T), and the roped rows come back.
 * out [B][T][nh*64] fp32 (fp16 values widened for kernels 0 and 3).  1 <= B <= 64, 1 <= T <= 2400, nh <= 64, nh % nkv == 0. */
q3tts_status q3tts_codec_attention_probe(int32_t device, int32_t kernel, float* qkv, int32_t B, int32_t T, int32_t nh, int32_t nkv,
                                         const float* inv_freq, float* out);

/* One DecoderResidualUnit of the vocoder (Vocoder/SpeechTokenizer.swift:696-718) on fp16 operands:
 *   x' = res + conv1x1(snake2(conv7_dil(a) + b7)) + b1,   out = snake3(x')
 * form: 1 = the fused kernel (codec_unit), 0 = the two tensor-core GEMM launches the decoder uses when the fused kernel does not take
 * the shape.  a = snake1(x) and res = x [B][T][C] fp32 (rounded to fp16 on upload); w7 [7][C][C] (tap 6 reads row t, tap 0 row
 * t - 6*dil), w1 [C][C] ([out][in]); b7 / b1 [C] or NULL; SnakeBeta parameters ea / ieb [C] (v + ieb * sin^2(v * ea)).
 * weight_reps (1..32): copies of each fp16 weight laid out as the decoder stores them.  emit_residual: x' is stored (fp16) and
 * returned in x_out (NULL otherwise); in_place: x' overwrites the residual buffer.  snake_out = out (fp16 widened).
 * C % 32 == 0, 32 <= C <= 1536; form 1 also needs C <= 192, 128 + 6*dil <= 192 and B * ceil(T / 128) >= 32. */
q3tts_status q3tts_codec_unit_probe(int32_t device, int32_t form, int32_t B, int32_t T, int32_t C, int32_t dil, const float* a,
                                    const float* w7, const float* b7, const float* ea2, const float* ieb2, const float* w1, const float* b1,
                                    const float* res, const float* ea3, const float* ieb3, int32_t in_place, int32_t emit_residual,
                                    int32_t weight_reps, float* x_out, float* snake_out);

/* DecoderOutputConv (causal 7 taps, C -> 1, then clip(-1, 1), NaN -> 0): y[b][t] from x [B][T][C], w [7][C] (tap 6 reads row t),
 * bias [1].  kernel: 0 = the streaming fp16 kernel (C in {32, 64, 96, 128}; strip = outputs per warp, a multiple of 32, 0 = the
 * default), 1 = the SIMT kernel on fp32 input, 2 = the SIMT kernel on fp16 input (C <= 256 for both), 3 = the tcgen05 GEMM's pcm
 * epilogue (C % 8 == 0).  fp16 kernels round x on upload. */
q3tts_status q3tts_codec_out_conv_probe(int32_t device, int32_t kernel, const float* x, int32_t B, int32_t T, int32_t C, const float* w,
                                        const float* bias, int32_t strip, float* y);

/* Row-wise codec ops on x [rows][ldx] -> y [rows][C]:  op 0 = causal depthwise conv k7 (w [7][C], b [C]; rows = B * T, tap 6 reads
 * row t), 1 = LayerNorm (w, b [C], eps; fp32 out), 2 = LayerNorm with fp16 out, 3 = RMSNorm with fp16 out (w [C] or NULL, ldx >= C),
 * 4 = SnakeBeta (w = ea, b = ieb), 5 = silu(x[:, :C]) * x[:, C:] (ldx = 2C).  Other ops take ldx = C. */
q3tts_status q3tts_codec_rowop_probe(int32_t device, int32_t op, const float* x, int32_t rows, int32_t ldx, int32_t C, int32_t T,
                                     const float* w, const float* b, float eps, float* y);

/* ------------------------------------------------------------------------------------------------------
 * measurement hook (bench.py roofline): runs the dequant-fused linear launches of ONE talker decode step
 * (which = 0: 28 x {qkv, o, gate|up, down} + codec_head) or ONE code-predictor pass (which = 1) for `m` activation
 * rows, `iters` times back to back on the handle's stream, bracketed by CUDA events.  Same kernels, weights and
 * shapes as the frame step; no reference counterpart (the reference has no benchmark, SURVEY.md §6).
 * ---------------------------------------------------------------------------------------------------- */
q3tts_status q3tts_profile_linear(q3tts_handle* h, int32_t which, int32_t m, int32_t iters, double* ms_out,
                                  int64_t* launches_out, int64_t* bytes_per_iter_out);

/* measurement hook (scripts/skinny_trace.py): `iters` back-to-back launches (one CUDA graph, programmatic dependent launch,
 * a different weight matrix each) of the <= 128-row split-K cluster GEMM (csrc/gemm_skinny.cu) for an [M x K] . [N x K]^T
 * linear; returns the average time per launch and, for the LAST launch, 16 stamps per CTA: [0]/[9] %globaltimer at entry /
 * exit, [1..8] clock64 at entry, after setup, first operand stage landed, accumulator complete, partial sums shipped,
 * peers' partial sums landed, epilogue done, exit.  No reference counterpart. */
q3tts_status q3tts_skinny_trace(int32_t device, int32_t M, int32_t N, int32_t K, int32_t swiglu, int32_t residual, int32_t iters,
                                uint64_t* stamps_out, int32_t capacity_ctas, int32_t* tiles_out, int32_t* split_out,
                                int32_t* stages_out, double* avg_us_out);

/* the same measurement for the dequant-fused kernel (csrc/gemm_skinny_q.cu): bits = 4 / 8 streams MLX-packed weights (group 64, fp16
 * scales), bits = 0 is q3tts_skinny_trace.  Extra stamps: [14] all k-blocks dequantised (warp 3), [15] dependency on the predecessor
 * launch resolved (warp 3). */
q3tts_status q3tts_skinny_trace_q(int32_t device, int32_t M, int32_t N, int32_t K, int32_t bits, int32_t swiglu, int32_t residual, int32_t iters,
                                  uint64_t* stamps_out, int32_t capacity_ctas, int32_t* tiles_out, int32_t* split_out,
                                  int32_t* stages_out, double* avg_us_out);

#ifdef __cplusplus
}
#endif
#endif /* QWEN3TTS_B200_H */
