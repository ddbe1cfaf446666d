// Qwen3TTSPipeline over the C ABI — same public surface as the reference's Sources/Qwen3TTS/Qwen3TTSPipeline.swift
// (AudioChunk :6-19, Qwen3TTSPipelineConfiguration :22-54, init :118, generate :244/:279, generateStream :323,
// VoiceDesign/CustomVoice :355-480, generateToFile :644, generateBatch :774, clearCache :951, Qwen3TTSError :985).
// The tokenizer (Tokenizer/Qwen3Tokenizer.swift), TextChunker and WAV writers of the reference are pure Swift and are
// reused unchanged; only the MLX-backed members (Qwen3Talker, AudioDecoder) are replaced by the handle.
// COMPILE-UNTESTED (no Swift toolchain in the build image).
import CQwen3TTSB200
import Foundation

public struct AudioChunk: Sendable {
    public let samples: [Float]
    public let tokenRange: Range<Int>
    public let isFinal: Bool
    public init(samples: [Float], tokenRange: Range<Int>, isFinal: Bool) {
        self.samples = samples; self.tokenRange = tokenRange; self.isFinal = isFinal
    }
}

public struct Qwen3TTSPipelineConfiguration: Sendable {
    public var applyRuntimeQuantization: Bool   // q3tts_options.runtime_quantization: mixed 4/6-bit MLX quantisation at load
    public var defaultTemperature: Float
    public var defaultMaxTokens: Int
    public var defaultStreamingChunkSize: Int
    public var crossfadeSamples: Int
    public var device: Int32 = 0                // CUDA ordinal (replaces MLX_DEVICE / DeviceSelector)
    public var seed: UInt64 = 0
    public var maxBatch: Int32 = 1              // q3tts_options.max_batch: utterance slots of the handle (text chunks of generateToFile run batched)
    public var lanes: Int32 = 1                 // q3tts_options.lanes: launch chains served side by side for calls with more than maxBatch requests
    public init(applyRuntimeQuantization: Bool = true, defaultTemperature: Float = 0.85, defaultMaxTokens: Int = 2400,
                defaultStreamingChunkSize: Int = 12, crossfadeSamples: Int = 480) {
        self.applyRuntimeQuantization = applyRuntimeQuantization
        self.defaultTemperature = defaultTemperature
        self.defaultMaxTokens = defaultMaxTokens
        self.defaultStreamingChunkSize = defaultStreamingChunkSize
        self.crossfadeSamples = crossfadeSamples
    }
    public static let `default` = Qwen3TTSPipelineConfiguration()
}

public enum Qwen3TTSError: LocalizedError {
    case fileNotFound(String)
    case decoderLoadFailed
    case modelNotLoaded
    case engine(Int32, String)
    public var errorDescription: String? {
        switch self {
        case .fileNotFound(let f): return "Required file not found: \(f)"
        case .decoderLoadFailed: return "Failed to load MLX audio decoder"
        case .modelNotLoaded: return "Model is not loaded"
        case .engine(let s, let m): return "qwen3tts_b200 status \(s): \(m)"
        }
    }
}

/// A registered voice (q3tts_voice): the prompt prefix of one speaker / instruct / ICL reference, prefilled once by
/// `Qwen3TTSPipeline.prepareVoice`.  Requests made with it give the bits of the same requests with the fields written inline.
/// Immutable; usable from several threads; may outlive the pipeline.  Freed when the last reference goes.
public final class Qwen3TTSVoice: @unchecked Sendable {
    let pointer: OpaquePointer
    let roleIds: [Int32]
    public let prefixPositions: Int
    public let deviceBytes: Int64
    init(pointer: OpaquePointer, roleIds: [Int32]) {
        self.pointer = pointer
        self.roleIds = roleIds
        var n: Int32 = 0
        var b: Int64 = 0
        _ = q3tts_voice_info(pointer, &n, &b)
        prefixPositions = Int(n)
        deviceBytes = b
    }
    deinit { q3tts_voice_free(pointer) }
}

public final class Qwen3TTSPipeline: @unchecked Sendable {
    public static let sampleRate: Int = 24000

    private var handle: OpaquePointer?
    private let tokenizer: Qwen3Tokenizer          // reference's pure-Swift BPE, unchanged
    private let pipelineConfig: Qwen3TTSPipelineConfiguration
    private var info = q3tts_info()
    private var speakerIds: [String: Int32] = [:]

    public var availableSpeakers: [String] { speakerIds.keys.sorted() }
    public var supportsVoiceCloning: Bool { info.has_speaker_encoder != 0 }   // speakerEncoder?.isWeightsLoaded (:82-84)
    public var supportsICL: Bool { info.has_audio_encoder != 0 }              // audioEncoder != nil (:87-89)
    public var modelType: String? { info.model_type == 1 ? "voice_design" : (info.model_type == 2 ? "custom_voice" : nil) }
    public var supportsVoiceDesign: Bool { info.model_type == 1 }
    public var supportsCustomVoice: Bool { info.model_type == 2 }

    public init(modelPath: URL, configuration: Qwen3TTSPipelineConfiguration = .default) throws {
        pipelineConfig = configuration
        tokenizer = Qwen3Tokenizer(modelPath: modelPath)
        var opts = q3tts_options()
        q3tts_default_options(&opts)
        opts.device = configuration.device
        opts.runtime_quantization = configuration.applyRuntimeQuantization ? 1 : 0
        opts.max_batch = max(1, configuration.maxBatch)
        opts.lanes = max(1, configuration.lanes)
        opts.max_frames = Int32(max(configuration.defaultMaxTokens, 600))
        var h: OpaquePointer?
        let st = q3tts_create(modelPath.path, &opts, &h)
        guard st == Q3TTS_OK, let hh = h else {
            let msg = String(cString: q3tts_last_error(nil))
            switch st {
            case Q3TTS_ERR_FILE_NOT_FOUND: throw Qwen3TTSError.fileNotFound(msg.components(separatedBy: ": ").last ?? msg)
            case Q3TTS_ERR_DECODER_LOAD_FAILED: throw Qwen3TTSError.decoderLoadFailed
            default: throw Qwen3TTSError.engine(st.rawValue, msg)
            }
        }
        handle = hh
        q3tts_get_info(hh, &info)
        var buf = [CChar](repeating: 0, count: 256)
        for i in 0..<info.num_speakers {
            var sid: Int32 = 0
            if q3tts_speaker_name(hh, i, &buf, 256, &sid) == Q3TTS_OK { speakerIds[String(cString: buf)] = sid }
        }
    }

    deinit { if let h = handle { q3tts_destroy(h) } }

    // MARK: request assembly — the string side of Qwen3Talker.generateCodes (Model/Qwen3Talker.swift:338-414)
    private struct Ids {
        var text: [Int32]; var instruct: [Int32] = []; var refText: [Int32] = []; var refCodes: [Int32] = []; var refFrames: Int32 = 0
        var speakerId: Int32 = -1; var embedding: [Float] = []
        var voice: Qwen3TTSVoice? = nil   // replaces every voice field above
    }
    /// the ids of `text` in a voice; nil when a voice made by the call itself does not match the chunk's role ids
    private func voiceIds(text: String, voice: Qwen3TTSVoice, strict: Bool) -> Ids? {
        var ids = Ids(text: tokenizer.encode(text: "<|im_start|>assistant\n\(text)<|im_end|>\n<|im_start|>assistant\n"))
        if !strict && Array(ids.text.prefix(3)) != voice.roleIds { return nil }
        ids.voice = voice
        return ids
    }
    private func makeIds(text: String, speaker: String, instruct: String?, speakerEmbedding: [Float]?, referenceTranscript: String?,
                         referenceAudioCodes: [[Int32]]?) -> Ids {
        var ids = Ids(text: tokenizer.encode(text: "<|im_start|>assistant\n\(text)<|im_end|>\n<|im_start|>assistant\n"))
        ids.speakerId = speakerIds[speaker.lowercased()] ?? -1
        let useICL = referenceAudioCodes != nil && referenceTranscript != nil && !referenceTranscript!.isEmpty
        if let ins = instruct, !ins.isEmpty {
            ids.instruct = tokenizer.encode(text: "<|im_start|>user\n\(ins)<|im_end|>\n")
        } else if useICL, let codes = referenceAudioCodes, let tr = referenceTranscript {
            ids.refText = tokenizer.encode(text: "<|im_start|>user\n\(tr)<|im_end|>\n")
            ids.refFrames = Int32(codes.first?.count ?? 0)
            ids.refCodes = codes.flatMap { $0 }
        } else if !speaker.isEmpty && ids.speakerId < 0 && speakerEmbedding == nil {
            ids.instruct = tokenizer.encode(text: "<|im_start|>user\n\(speaker)<|im_end|>\n")
        }
        if ids.speakerId < 0, let e = speakerEmbedding { ids.embedding = e }
        return ids
    }
    private func withRequest<R>(_ ids: Ids, temperature: Float, maxTokens: Int, streamVariant: Bool, _ body: (inout q3tts_request) -> R) -> R {
        var req = q3tts_request()
        q3tts_default_request(&req)
        return ids.text.withUnsafeBufferPointer { tp in
            ids.instruct.withUnsafeBufferPointer { ip in
                ids.refText.withUnsafeBufferPointer { rp in
                    ids.refCodes.withUnsafeBufferPointer { cp in
                        ids.embedding.withUnsafeBufferPointer { ep in
                            req.text_ids = tp.baseAddress; req.n_text_ids = Int32(tp.count)
                            if !ids.instruct.isEmpty { req.instruct_ids = ip.baseAddress; req.n_instruct_ids = Int32(ip.count) }
                            if !ids.refText.isEmpty { req.ref_text_ids = rp.baseAddress; req.n_ref_text_ids = Int32(rp.count)
                                                      req.ref_codes = cp.baseAddress; req.ref_frames = ids.refFrames }
                            req.speaker_id = ids.speakerId
                            if !ids.embedding.isEmpty { req.speaker_embedding = ep.baseAddress; req.speaker_embedding_dim = Int32(ep.count) }
                            req.temperature = temperature
                            req.max_tokens = Int32(maxTokens)
                            req.seed = pipelineConfig.seed
                            req.stream_variant = streamVariant ? 1 : 0
                            req.voice = ids.voice?.pointer
                            return body(&req)
                        }
                    }
                }
            }
        }
    }
    private func pcm(_ ids: Ids, mode: q3tts_decode_mode, temperature: Float, maxTokens: Int) -> [Float] {
        guard let h = handle else { return [] }
        var out = [Float](repeating: 0, count: max(maxTokens, 1) * Int(Q3TTS_SAMPLES_PER_FRAME))
        var n: Int64 = 0
        var frames: Int32 = 0
        let cap = Int64(out.count)
        let st = withRequest(ids, temperature: temperature, maxTokens: maxTokens, streamVariant: false) { req in
            out.withUnsafeMutableBufferPointer { q3tts_generate_pcm(h, &req, Int32(mode.rawValue), $0.baseAddress, cap, &n, &frames) }
        }
        guard st == Q3TTS_OK else { return [] }   // generation APIs do not throw in the reference either
        return Array(out.prefix(Int(n)))
    }

    // MARK: registered voices (no reference counterpart)
    /// Prefill the voice part of the prompt once (q3tts_voice_create), from the same fields and rules as a request.
    public func prepareVoice(speaker: String = "", instruct: String? = nil, speakerEmbedding: [Float]? = nil, referenceTranscript: String? = nil,
                             referenceAudioCodes: [[Int32]]? = nil) throws -> Qwen3TTSVoice {
        guard let h = handle else { throw Qwen3TTSError.modelNotLoaded }
        let ids = makeIds(text: "", speaker: speaker, instruct: instruct, speakerEmbedding: speakerEmbedding, referenceTranscript: referenceTranscript,
                          referenceAudioCodes: referenceAudioCodes)
        var v: OpaquePointer?
        let st = withRequest(ids, temperature: 0, maxTokens: 0, streamVariant: false) { req in q3tts_voice_create(h, &req, &v) }
        guard st == Q3TTS_OK, let vv = v else { throw Qwen3TTSError.engine(st.rawValue, String(cString: q3tts_last_error(h))) }
        return Qwen3TTSVoice(pointer: vv, roleIds: Array(ids.text.prefix(3)))
    }
    /// a voice for a call of several chunks that repeat the same fields (nil: run them inline)
    private func callVoice(chunks: Int, voice: Qwen3TTSVoice?, speaker: String, instruct: String?, speakerEmbedding: [Float]?,
                           referenceTranscript: String?, referenceAudioCodes: [[Int32]]?) -> (Qwen3TTSVoice?, Bool) {
        if let v = voice { return (v, true) }
        guard chunks > 1 else { return (nil, false) }
        return ((try? prepareVoice(speaker: speaker, instruct: instruct, speakerEmbedding: speakerEmbedding, referenceTranscript: referenceTranscript,
                                   referenceAudioCodes: referenceAudioCodes)), false)
    }

    // MARK: simple generation (:244-306)
    public func generate(text: String, voice: Qwen3TTSVoice, temperature: Float? = nil, maxTokens: Int? = nil) -> [Float] {
        guard let ids = voiceIds(text: text, voice: voice, strict: true) else { return [] }
        return pcm(ids, mode: Q3TTS_DECODE_WHOLE, temperature: temperature ?? pipelineConfig.defaultTemperature, maxTokens: maxTokens ?? pipelineConfig.defaultMaxTokens)
    }
    public func generate(text: String, speaker: String, temperature: Float? = nil, maxTokens: Int? = nil) -> [Float] {
        pcm(makeIds(text: text, speaker: speaker, instruct: nil, speakerEmbedding: nil, referenceTranscript: nil, referenceAudioCodes: nil),
            mode: Q3TTS_DECODE_WHOLE, temperature: temperature ?? pipelineConfig.defaultTemperature, maxTokens: maxTokens ?? pipelineConfig.defaultMaxTokens)
    }
    public func generate(text: String, speakerEmbedding: [Float], temperature: Float? = nil, maxTokens: Int? = nil) -> [Float] {
        pcm(makeIds(text: text, speaker: "", instruct: nil, speakerEmbedding: speakerEmbedding, referenceTranscript: nil, referenceAudioCodes: nil),
            mode: Q3TTS_DECODE_WHOLE, temperature: temperature ?? pipelineConfig.defaultTemperature, maxTokens: maxTokens ?? pipelineConfig.defaultMaxTokens)
    }
    public func generateVoiceDesign(text: String, voiceDescription: String, temperature: Float? = nil, maxTokens: Int? = nil) -> [Float] {
        pcm(makeIds(text: text, speaker: "", instruct: voiceDescription, speakerEmbedding: nil, referenceTranscript: nil, referenceAudioCodes: nil),
            mode: Q3TTS_DECODE_WHOLE, temperature: temperature ?? pipelineConfig.defaultTemperature, maxTokens: maxTokens ?? pipelineConfig.defaultMaxTokens)
    }
    public func generateCustomVoice(text: String, speaker: String, instruct: String, temperature: Float? = nil, maxTokens: Int? = nil) -> [Float] {
        pcm(makeIds(text: text, speaker: speaker, instruct: instruct, speakerEmbedding: nil, referenceTranscript: nil, referenceAudioCodes: nil),
            mode: Q3TTS_DECODE_WHOLE, temperature: temperature ?? pipelineConfig.defaultTemperature, maxTokens: maxTokens ?? pipelineConfig.defaultMaxTokens)
    }

    // MARK: streaming (:323-340, 484-624): q3tts_stream_next_audio IS the consumer loop (windows 18 / 8+18, final empty chunk)
    public func generateStream(text: String, speaker: String = "", speakerEmbedding: [Float]? = nil, temperature: Float? = nil,
                               maxTokens: Int? = nil, chunkSize: Int? = nil) -> AsyncThrowingStream<AudioChunk, Error> {
        streamImpl(text: text, speaker: speaker, instruct: nil, speakerEmbedding: speakerEmbedding, temperature: temperature, maxTokens: maxTokens, chunkSize: chunkSize)
    }
    public func generateStreamVoiceDesign(text: String, voiceDescription: String, temperature: Float? = nil, maxTokens: Int? = nil,
                                          chunkSize: Int? = nil) -> AsyncThrowingStream<AudioChunk, Error> {
        streamImpl(text: text, speaker: "", instruct: voiceDescription, speakerEmbedding: nil, temperature: temperature, maxTokens: maxTokens, chunkSize: chunkSize)
    }
    public func generateStreamCustomVoice(text: String, speaker: String, instruct: String, temperature: Float? = nil, maxTokens: Int? = nil,
                                          chunkSize: Int? = nil) -> AsyncThrowingStream<AudioChunk, Error> {
        streamImpl(text: text, speaker: speaker, instruct: instruct, speakerEmbedding: nil, temperature: temperature, maxTokens: maxTokens, chunkSize: chunkSize)
    }
    public func generateStream(text: String, voice: Qwen3TTSVoice, temperature: Float? = nil, maxTokens: Int? = nil,
                               chunkSize: Int? = nil) -> AsyncThrowingStream<AudioChunk, Error> {
        streamImpl(text: text, speaker: "", instruct: nil, speakerEmbedding: nil, temperature: temperature, maxTokens: maxTokens, chunkSize: chunkSize,
                   voice: voice)
    }
    private func streamImpl(text: String, speaker: String, instruct: String?, speakerEmbedding: [Float]?, temperature: Float?, maxTokens: Int?,
                            chunkSize: Int?, voice: Qwen3TTSVoice? = nil) -> AsyncThrowingStream<AudioChunk, Error> {
        let ids = voice.flatMap { voiceIds(text: text, voice: $0, strict: true) }
            ?? makeIds(text: text, speaker: speaker, instruct: instruct, speakerEmbedding: speakerEmbedding, referenceTranscript: nil, referenceAudioCodes: nil)
        let temp = temperature ?? pipelineConfig.defaultTemperature
        let tokens = maxTokens ?? pipelineConfig.defaultMaxTokens
        let chunk = Int32(chunkSize ?? pipelineConfig.defaultStreamingChunkSize)
        return AsyncThrowingStream { continuation in
            Task { [self] in
                guard let h = handle else { continuation.finish(throwing: Qwen3TTSError.modelNotLoaded); return }
                var stream: OpaquePointer?
                let st = withRequest(ids, temperature: temp, maxTokens: tokens, streamVariant: true) { req in q3tts_stream_begin(h, &req, chunk, &stream) }
                guard st == Q3TTS_OK, let s = stream else {
                    continuation.finish(throwing: Qwen3TTSError.engine(st.rawValue, String(cString: q3tts_last_error(h)))); return
                }
                defer { q3tts_stream_free(s) }
                var buf = [Float](repeating: 0, count: 18 * Int(Q3TTS_SAMPLES_PER_FRAME))
                while true {
                    if Task.isCancelled { q3tts_stream_cancel(s) }
                    var n: Int32 = 0, t0: Int32 = 0, t1: Int32 = 0, fin: Int32 = 0, done: Int32 = 0
                    let cap = Int32(buf.count)
                    let rc = buf.withUnsafeMutableBufferPointer { q3tts_stream_next_audio(s, $0.baseAddress, cap, &n, &t0, &t1, &fin, &done) }
                    if rc != Q3TTS_OK { continuation.finish(throwing: Qwen3TTSError.engine(rc.rawValue, String(cString: q3tts_last_error(h)))); return }
                    continuation.yield(AudioChunk(samples: Array(buf.prefix(Int(n))), tokenRange: Int(t0)..<Int(t1), isFinal: fin != 0))
                    if done != 0 { break }
                }
                continuation.finish()
            }
        }
    }

    // MARK: file output (:644-757): TextChunker + StreamingWAVWriter are the reference's own Swift sources
    public func generateToFile(text: String, speaker: String = "", instruct: String? = nil, speakerEmbedding: [Float]? = nil,
                               referenceTranscript: String? = nil, referenceAudioCodes: [[Int32]]? = nil, outputURL: URL,
                               temperature: Float? = nil, onProgress: ((Float) -> Void)? = nil, voice: Qwen3TTSVoice? = nil) async throws -> Int {
        let temp = temperature ?? pipelineConfig.defaultTemperature
        let chunks = TextChunker.chunk(text, maxWords: TextChunker.defaultMaxWords)
        guard !chunks.isEmpty else { return 0 }
        // every chunk repeats the same voice: several chunks prefill it once (a voice of the call's own, freed when the call returns)
        let (v, strict) = callVoice(chunks: chunks.count, voice: voice, speaker: speaker, instruct: instruct, speakerEmbedding: speakerEmbedding,
                                    referenceTranscript: referenceTranscript, referenceAudioCodes: referenceAudioCodes)
        let writer = try StreamingWAVWriter(to: outputURL)
        for (i, c) in chunks.enumerated() {
            if Task.isCancelled { break }
            onProgress?(Float(i) / Float(chunks.count))
            let ids = v.flatMap { voiceIds(text: c, voice: $0, strict: strict) }
                ?? makeIds(text: c, speaker: speaker, instruct: instruct, speakerEmbedding: speakerEmbedding,
                           referenceTranscript: referenceTranscript, referenceAudioCodes: referenceAudioCodes)
            let samples = pcm(ids, mode: Q3TTS_DECODE_FILE, temperature: temp, maxTokens: 600)
            if !samples.isEmpty { try writer.write(samples: samples) }
        }
        onProgress?(1.0)
        return writer.finalize().sampleCount
    }

    // MARK: batch (:774-898)
    public func generateBatch(text: String, speaker: String = "", instruct: String? = nil, speakerEmbedding: [Float]? = nil,
                              referenceTranscript: String? = nil, temperature: Float? = nil, onProgress: ((Float) -> Void)? = nil,
                              voice: Qwen3TTSVoice? = nil) async -> [Float] {
        let temp = temperature ?? pipelineConfig.defaultTemperature
        let crossfade = pipelineConfig.crossfadeSamples
        let chunks = TextChunker.chunk(text, maxWords: TextChunker.defaultMaxWords)
        guard !chunks.isEmpty else { return [] }
        if chunks.count == 1 {
            onProgress?(0)
            let s = voice.map { generate(text: chunks[0], voice: $0, temperature: temp) } ?? generate(text: chunks[0], speaker: speaker, temperature: temp)
            onProgress?(1)
            return s
        }
        let (v, strict) = callVoice(chunks: chunks.count, voice: voice, speaker: speaker, instruct: instruct, speakerEmbedding: speakerEmbedding,
                                    referenceTranscript: nil, referenceAudioCodes: nil)
        var all: [Float] = [], tail: [Float] = []
        for (i, c) in chunks.enumerated() {
            if Task.isCancelled { return all }
            onProgress?(Float(i) / Float(chunks.count))
            let ids = v.flatMap { voiceIds(text: c, voice: $0, strict: strict) }
                ?? makeIds(text: c, speaker: speaker, instruct: instruct, speakerEmbedding: speakerEmbedding, referenceTranscript: nil, referenceAudioCodes: nil)
            var s = pcm(ids, mode: Q3TTS_DECODE_BATCHAPI, temperature: temp, maxTokens: 600)
            if s.isEmpty { continue }
            if !tail.isEmpty && crossfade > 0 {
                let n = min(crossfade, tail.count, s.count)
                for k in 0..<n { all.append(tail[k] * Float(n - k) / Float(n) + s[k] * Float(k) / Float(n)) }
                s = Array(s.dropFirst(n))
            }
            if i == chunks.count - 1 { all.append(contentsOf: s) }
            else if s.count > crossfade { all.append(contentsOf: s.dropLast(crossfade)); tail = Array(s.suffix(crossfade)) }
            else { tail = s }
        }
        onProgress?(1.0)
        return all
    }

    /// :906 — ECAPA-TDNN on the device; nil without `speaker_encoder.*` weights
    public func extractSpeakerEmbedding(audioSamples: [Float]) -> [Float]? {
        guard let h = handle, info.has_speaker_encoder != 0, audioSamples.count >= 1024 else { return nil }
        var emb = [Float](repeating: 0, count: Int(info.speaker_embedding_dim))
        var dim: Int32 = 0
        let st = q3tts_extract_speaker_embedding(h, audioSamples, Int64(audioSamples.count), &emb, Int32(emb.count), &dim, nil)
        guard st == Q3TTS_OK, dim > 0 else { return nil }
        return Array(emb.prefix(Int(dim)))
    }

    /// :924 — SEANet + transformer + split RVQ on the device; [num_quantizers][time], nil without `encoder.*` weights
    public func encodeReferenceAudio(audioSamples: [Float]) -> [[Int32]]? {
        guard let h = handle, info.has_audio_encoder != 0, !audioSamples.isEmpty else { return nil }
        let cap = (audioSamples.count + 1919) / 1920 + 2
        var codes = [Int32](repeating: 0, count: 64 * cap)
        var frames: Int32 = 0, quantizers: Int32 = 0
        let st = q3tts_encode_reference_audio(h, audioSamples, Int64(audioSamples.count), &codes, Int32(cap), &frames, &quantizers, nil)
        guard st == Q3TTS_OK, frames > 0 else { return nil }
        let T = Int(frames)
        return (0..<Int(quantizers)).map { q in Array(codes[(q * T)..<((q + 1) * T)]) }
    }
    public func clearCache() { if let h = handle { _ = q3tts_clear_cache(h) } }      // :951
}
