/* thewhisper_b200 -- C-ABI of the B200-native Whisper hot path (log-mel -> encoder -> decoder -> tokens).
 *
 * This is the drop-in boundary below `thestage_speechkit.nvidia.ASRPipeline.__call__`
 * (reference: /root/reference/thestage_speechkit/nvidia/asr_pipeline.py:30-92).  The reference has no native
 * code and no FFI: everything numeric is reached through `transformers` (un-vendored), so each entry point cites
 * the Python call it replaces (TF = transformers 5.5.0 as installed; the reference pins 4.52.3):
 *
 *   bw_logmel            TF/models/whisper/feature_extraction_whisper.py:135-164  (_torch_extract_fbank_features)
 *   bw_encode            TF/models/whisper/modeling_whisper.py:593-647 (WhisperEncoder.forward) + :331-336 (cross K/V)
 *   bw_decode_begin/run  TF/generation/utils.py:2743-2809 (_sample loop) over modeling_whisper.py:691-796,1081 and
 *                        the processors TF/generation/logits_process.py:1812-2043
 *   bw_word_timestamps   TF/models/whisper/generation_whisper.py:241-381 (_extract_token_timestamps, DTW :64-115)
 *
 * Conventions: plain C, no torch types.  Every function returns 0 on success and a negative code on error; the
 * message is available from bw_last_error() (thread-local).  Nothing throws across the boundary.  Device pointers
 * are caller-owned (the Python host passes torch storage); `stream` is a cudaStream_t cast to void* and all work
 * is enqueued asynchronously on it.  One engine per GPU / process; an engine is not re-entrant.
 * There is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef THEWHISPER_B200_H_
#define THEWHISPER_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BW_ABI_VERSION 2

typedef struct bw_engine bw_engine;

#ifndef THEWHISPER_B200_TYPES_
#define THEWHISPER_B200_TYPES_
typedef struct bw_config {
  int32_t d_model;      /* 1280 */
  int32_t n_heads;      /* 20  (head_dim must be 64) */
  int32_t ffn;          /* 5120 */
  int32_t enc_layers;   /* 32 */
  int32_t dec_layers;   /* 32 (4 for turbo) */
  int32_t n_mels;       /* 128 */
  int32_t vocab;        /* 51866 */
  int32_t max_source_positions; /* S: 1500 (30 s), 1000, 750, 500 -- set by chunk_length_s */
  int32_t max_target_positions; /* 448 */
  int32_t max_audios;   /* A: audios per encode/decode call */
  int32_t max_beams;    /* G <= 8 sequences sharing one audio's cross K/V */
  int32_t n_align_heads;/* alignment heads for word timestamps (0 = off) */
  int32_t max_align_steps; /* rows of alignment scores kept per audio (<= max_target_positions) */
  int32_t dtype;        /* 16-bit element type of weights / activations / KV caches: 0 = bfloat16, 1 = float16 (what the reference's
                           streaming and benchmark paths run: REF streaming_pipeline.py:369-370); accumulation is fp32 in both */
} bw_config;

typedef struct bw_decode_opts {
  int32_t begin_index;        /* prompt length: positions < begin_index are teacher-forced */
  int32_t eos_token, pad_token;
  int32_t timestamp_rules;    /* 1 = WhisperTimeStampLogitsProcessor on */
  int32_t timestamp_begin, no_timestamps_token, max_initial_timestamp_index; /* -1 = none */
  const int32_t* suppress_tokens; int32_t n_suppress;             /* host arrays */
  const int32_t* begin_suppress_tokens; int32_t n_begin_suppress;
  int32_t record_alignment;   /* 1 = keep cross-attention scores of the alignment heads */
} bw_decode_opts;
#endif /* THEWHISPER_B200_TYPES_ */

const char* bw_last_error(void);
int bw_abi_version(void);
int bw_device_count(void);
/* bit 0: the persistent decoder-step kernel is launched cooperatively; bit 1: the batched step uses programmatic dependent
 * launch.  Both are on by default and are cleared (once, process-wide) if the driver cannot capture such a launch in a graph;
 * valid after the first bw_decode_begin. */
int bw_runtime_flags(void);

/* ---- lifetime ---------------------------------------------------------------------------------------------- */
int bw_engine_create(const bw_config* cfg, bw_engine** out);
void bw_engine_destroy(bw_engine* e);
/* Bind one weight tensor by name (device pointer, must outlive the engine).  Matrices are 16-bit (bw_config::dtype) row-major
 * [out, in] (torch Linear layout), vectors fp32.  Names: see DESIGN.md "weights". */
int bw_engine_set_tensor(bw_engine* e, const char* name, const void* device_ptr);
/* slaney mel filter bank [201, n_mels] fp32 on the HOST (TF/audio_utils.py:453-544), copied to the device. */
int bw_engine_set_mel_filters(bw_engine* e, const float* bank_host);
/* alignment heads as (layer, head) pairs on the host */
int bw_engine_set_alignment_heads(bw_engine* e, const int32_t* layer_head_pairs, int32_t n);
/* checks that every tensor is bound and allocates the workspace + KV caches */
int bw_engine_finalize(bw_engine* e);
/* device pointer + size of an internal buffer ("mel_tm", "x_enc", "enc_out", "logits", "tokens", "align", ...) */
int bw_engine_buffer(bw_engine* e, const char* name, void** device_ptr, size_t* bytes);

/* ---- hot path ------------------------------------------------------------------------------------------------ */
/* pcm: device fp32 [B, n_samples], n_samples == 320 * max_source_positions (chunk already zero-padded/truncated).
 * Writes the engine's mel buffer; if mel_f32_out != NULL also the reference layout [B, n_mels, frames] fp32. */
int bw_logmel(bw_engine* e, const float* pcm, int32_t B, int32_t n_samples, float* mel_f32_out, void* stream);
/* load externally computed features instead (device fp32 [B, n_mels, frames]) */
int bw_set_mel(bw_engine* e, const float* mel_f32, int32_t B, void* stream);
/* conv stem + encoder layers + final LayerNorm + cross-attention K/V projection of every decoder layer */
int bw_encode(bw_engine* e, int32_t B, void* stream);
/* start a decode over A audios x G sequences; prompt_host: [A*G, prompt_len] int32 */
int bw_decode_begin(bw_engine* e, int32_t A, int32_t G, const int32_t* prompt_host, int32_t prompt_len,
                    const bw_decode_opts* opts, void* stream);
/* run n decoder steps (one CUDA-graph launch each, no host synchronisation) */
int bw_decode_run(bw_engine* e, int32_t n_steps, void* stream);
/* kernels launched by bw_decode_run since the engine was created (kernel nodes of the step graph x graph launches);
 * bench.py reports it as part of "gpu_launches" */
long long bw_decode_kernel_launches(bw_engine* e);
/* synchronises the stream; tokens_host [A*G, max_target_positions], finished_host [A*G] (either may be NULL) */
int bw_decode_read(bw_engine* e, int32_t* tokens_host, int32_t* finished_host, int32_t* pos_host, void* stream);
/* beam search support: reorder sequences (new sequence i continues old sequence parent[i]) by permuting the
 * per-token block table; overwrite the token just selected.  Host arrays of A*G entries. */
int bw_decode_reorder(bw_engine* e, const int32_t* parent_host, const int32_t* next_token_host, void* stream);
/* beam search step: upload the running scores [A*G], run one decoder step, download each sequence's 2*G best
 * continuations (score = running score + processed log-prob, token id; -inf / -1 when fewer exist).
 * Replaces the log_softmax + processors + topk part of TF/generation/utils.py:3254-3275; the beam bookkeeping
 * (:2945-3072) stays on the host (thewhisper_b200/beam.py). */
int bw_decode_beam_step(bw_engine* e, const float* run_scores_host, float* cand_scores_host, int32_t* cand_tokens_host,
                        void* stream);
/* word timestamps for sequence slot `audio` (= the audio index when decoding one sequence per audio): n_tokens generated tokens
 * starting at alignment row 0, num_frames valid encoder frames (<= S); out_host [n_tokens + 1] seconds */
int bw_word_timestamps(bw_engine* e, int32_t audio, int32_t n_tokens, int32_t num_frames, double time_precision,
                       float* out_host, void* stream);
/* the same for n audios in one pass (4 kernel launches + one D2H whatever n is): audio[i], n_tokens[i], num_frames[i];
 * out_host [n][out_pitch] floats, out_pitch >= max n_tokens + 1 */
int bw_word_timestamps_batch(bw_engine* e, int32_t n, const int32_t* audio, const int32_t* n_tokens, const int32_t* num_frames,
                             double time_precision, float* out_host, int32_t out_pitch, void* stream);
/* beam search: alignment scores are kept per SEQUENCE slot (audio * G + beam); row t of item i is read from slot
 * slot_map[i * map_pitch + t] -- the slot that was the returned sequence's ancestor at step t, i.e. what
 * `_extract_token_timestamps` selects with `beam_indices` (TF/models/whisper/generation_whisper.py:265-301). */
int bw_word_timestamps_gather(bw_engine* e, int32_t n, const int32_t* slot_map, int32_t map_pitch, const int32_t* n_tokens,
                              const int32_t* num_frames, double time_precision, float* out_host, int32_t out_pitch, void* stream);

/* ---- host-side post-processing (no CUDA) ---------------------------------------------------------------------- */
/* Seam merge of overlapping chunks: the reference's patched `_find_longest_common_sequence`
 * (REF thestage_speechkit/__init__.py:5-134, installed at :137-139).  tokens: the n_seq sequences concatenated, lens[n_seq];
 * ts: NULL, or one (start, end) pair of doubles per token (NaN = Python None); out_tokens / out_ts sized for the sum of
 * lens.  Returns 0, or -3 where Python would raise TypeError (a float end compared with None). */
int bw_host_merge_overlapping(const int32_t* tokens, const int32_t* lens, int32_t n_seq, const double* ts,
                              int32_t* out_tokens, double* out_ts, int32_t* out_len);

/* Token ids -> text / segment chunks / word chunks: what the reference's pipeline does after every generate()
 * (AutomaticSpeechRecognitionPipeline.postprocess, TF/pipelines/automatic_speech_recognition.py:603-611 ->
 * WhisperTokenizer._decode_asr + _collate_word_timestamps / _combine_tokens_into_words, TF/models/whisper/tokenization_whisper.py,
 * with the seam merge above).  A bw_host_vocab is built once per tokenizer:
 *   bytes / offsets[n_vocab + 1]: the bytes id i contributes to decoded text (byte-level pieces already mapped back to bytes);
 *   kind[i]: 0 text or timestamp id, 1 special id that is not a language, 2 + k language k of language_names (n_languages NUL-terminated
 *   UTF-8 names back to back); timestamp_begin = id of <|notimestamps|> + 1; render_begin = last special id + 1 (ids from there on are
 *   written as "<|seconds|>" when words are split); eos / sot / startofprev ids; cleanup_spaces = the tokenizer's
 *   clean_up_tokenization_spaces. */
typedef struct bw_host_vocab bw_host_vocab;
int bw_host_vocab_create(const uint8_t* bytes, const int64_t* offsets, int32_t n_vocab, const int32_t* kind, const char* language_names,
                         int32_t n_languages, int32_t timestamp_begin, int32_t render_begin, int32_t eos_id, int32_t sot_id,
                         int32_t startofprev_id, int32_t cleanup_spaces, bw_host_vocab** out);
void bw_host_vocab_destroy(bw_host_vocab* v);
/* One `_decode_asr` call over n_out windows: tokens = their ids back to back (lens[n_out]); token_ts / ts_lens = the per-token end times
 * of word mode, back to back (NULL otherwise); strides[n_out][3] = (chunk_len, stride_left, stride_right) seconds where has_stride[i].
 * mode: 0 text only, 1 segment timestamps (return_timestamps=True), 2 word timestamps (return_timestamps="word").  default_language:
 * index into language_names used for word splitting while no language token has been seen, or -1.
 * The result is a JSON document {"text": ..., "warn": bool, "chunks": [...]} ("chunks" as the original's `optional["chunks"]`, absent when the
 * original returns {}; "warn" = the original logs its missing-end-timestamp warning) in a buffer owned by `v`, valid until the next call.
 * Returns 0, or -4 where the original raises IndexError (message in bw_last_error). */
int bw_host_decode_asr(bw_host_vocab* v, const int32_t* tokens, const int32_t* lens, int32_t n_out, const double* token_ts, const int32_t* ts_lens,
                       const double* strides, const uint8_t* has_stride, int32_t mode, int32_t return_language, double time_precision,
                       int32_t default_language, const char** json_out, int64_t* json_len);

/* ---- single-op entry points (used by the parity tests; same kernels as the engine) --------------------------- */
/* C[M,N] = epi(A[M,K] W[N,K]^T): impl 0 = tcgen05, 1 = CUDA-core comparator, 2 = tcgen05 CTA pairs (cta_group::2, persistent).  out_is_f32 selects the output type. */
int bw_op_gemm(const void* A, const void* W, int32_t M, int32_t N, int32_t K, const float* bias, float alpha, int32_t act,
               const float* residual, void* out, int32_t out_is_f32, int32_t impl, int32_t force_bn, void* stream);
/* The two building blocks of the batched (tensor-core) decoder step.  Split-K GEMM: split z of `ksplit` writes the raw fp32 partial
 * sums of its k range at out_partials + z * M * N ([ksplit_used][M][N]; *ksplit_used <= ksplit); W has n_valid (<= N) rows in
 * memory, rows beyond read as zero (tied LM head).  force_bn: 0 auto, 32 (decoder tile), 64, 128, 256. */
int bw_op_gemm_splitk(const void* A, const void* W, int32_t M, int32_t N, int32_t K, int32_t n_valid, int32_t ksplit, int32_t force_bn,
                      float* out_partials, int32_t* ksplit_used, void* stream);
/* The decoder-step projection (gemm_dec.cu): weights as the 128-row MMA operand, Q activation rows as the N operand, K split over
 * CTAs.  Writes the raw fp32 partial sums [*ksplit_used][Q][N] (want_split = 0: one split); W has n_valid (<= N) rows in memory. */
int bw_op_gemm_dec(const void* X, const void* W, int32_t Q, int32_t N, int32_t K, int32_t n_valid, int32_t want_split, float* out_partials,
                   int32_t* ksplit_used, void* stream);
/* h[q, n] = bf16(GELU(sum_s partials[s][q][n] + bias[n])) */
int bw_op_gelu_bias(const float* partials, int32_t nsplit, const float* bias, void* h_bf16, int32_t Q, int32_t N, void* stream);
/* x[q] += bias + sum_s partials[s][q] (s ascending: deterministic), y[q] = LayerNorm(x[q]) as bf16 (y may be NULL). */
int bw_op_resid_ln(float* x, const float* partials, int32_t nsplit, const float* bias, const float* ln_g, const float* ln_b, void* y_bf16,
                   int32_t Q, int32_t D, void* stream);
/* qkv [B*S, 3D] bf16 -> out [B*S, D] bf16; vt_scratch [B, H, 64, Spad] bf16 (Spad = S rounded up to 8).
   impl 0 = tcgen05 (one query tile per CTA), 1 = CUDA-core comparator, 2 = tcgen05 ping-pong (two query tiles per CTA, O in TMEM),
   3 = ping-pong reading V tiles from the qkv rows as an MN-major operand (vt_scratch unused). */
int bw_op_attn_enc(const void* qkv, void* vt_scratch, void* out, int32_t B, int32_t S, int32_t H, int32_t impl, void* stream);
int bw_op_layernorm(const float* x, const float* g, const float* b, void* out, int32_t out_is_f32, int32_t rows, int32_t D,
                    void* stream);
/* out[M,N] fp32 = epi(LN?(x[M,K]) W[N,K]^T), M <= 8 */
int bw_op_gemv(const float* x, const float* ln_g, const float* ln_b, const void* W, int32_t M, int32_t N, int32_t K,
               const float* bias, float alpha, int32_t act, const float* residual, float* out, void* stream);
/* causal self-attention of one decoder step over positions 0..*pos. qkv [Q,3D] fp32 (q pre-scaled), or nsplit raw partial sums
   [nsplit][Q][3D] + qkv_bias, q scaled by q_alpha (batched path). append = 1: the k/v of this step are rounded to 16 bit and written
   to kc/vc at *pos (batched path). anc [Q,Tmax] or NULL. elem_dtype 0 = bf16, 1 = fp16 (dispatch to the _bf16 / _f16 build). */
int bw_op_self_attn(const float* qkv, int32_t nsplit, const float* qkv_bias, float q_alpha, void* kc, void* vc, const int32_t* anc,
                    int32_t append, void* out, int32_t out_is_f32, const int32_t* pos_dev, int32_t Q, int32_t H, int32_t Tmax,
                    int32_t elem_dtype, void* stream);
/* cross-attention of A*G query rows over kc/vc [A,H,S,64]. impl 0 = the engine's policy, 1 = split kernel, 2 = streaming kernel.
   part_o / part_ml / counters: caller-owned scratch of the sizes in decode.cuh; counters must be zero on entry and are zero on
   return. align / head_slots / Ha / Tcap / step_base: the word-timestamp capture (align may be NULL). */
int bw_op_cross_attn(const float* q, int32_t nsplit, const float* q_bias, float q_alpha, const void* kc, const void* vc,
                     void* out, int32_t out_is_f32, float* part_o, float* part_ml, uint32_t* counters, int32_t A, int32_t G,
                     int32_t H, int32_t S, float* align, const int32_t* head_slots, int32_t Ha, int32_t Tcap, int32_t step_base,
                     const int32_t* pos_dev, int32_t impl, int32_t elem_dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* THEWHISPER_B200_H_ */
