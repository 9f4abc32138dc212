// The public C-ABI (include/thewhisper_b200.h).  The engine exists twice in this library -- api.cu and every kernel source compiled
// with 16-bit elements = bfloat16 (symbols *_bf16) and = float16 (symbols *_f16) -- and this file is the only place that knows it:
// bw_engine_create picks the build from bw_config::dtype, every other entry point forwards to the build its engine belongs to.
// The single-op entry points (bw_op_*) are the bf16 build's.
#include "../../include/thewhisper_b200.h"

#define BW_RENAME_SUFFIX _bf16
#include "abi_rename.h"
#undef THEWHISPER_B200_H_
#include "../../include/thewhisper_b200.h"
#include "abi_unrename.h"
#undef BW_CAT
#undef BW_CAT2
#define BW_RENAME_SUFFIX _f16
#include "abi_rename.h"
#undef THEWHISPER_B200_H_
#include "../../include/thewhisper_b200.h"
#include "abi_unrename.h"

struct bw_engine {
  int f16;
  void* impl;
};

namespace {
thread_local int g_last_f16 = 0;  // which build reported the most recent status on this thread (bw_last_error)
}
#define BW_B(e) reinterpret_cast<bw_engine_bf16*>((e)->impl)
#define BW_H(e) reinterpret_cast<bw_engine_f16*>((e)->impl)
// forward an engine call; a null engine goes to the bf16 build, whose argument check reports it
#define BW_FWD(name, e, ...)                                                                      \
  do {                                                                                            \
    if (!(e)) { g_last_f16 = 0; return name##_bf16(nullptr, ##__VA_ARGS__); }                      \
    g_last_f16 = (e)->f16;                                                                        \
    return (e)->f16 ? name##_f16(BW_H(e), ##__VA_ARGS__) : name##_bf16(BW_B(e), ##__VA_ARGS__);    \
  } while (0)

extern "C" {

const char* bw_last_error(void) { return g_last_f16 ? bw_last_error_f16() : bw_last_error_bf16(); }
int bw_abi_version(void) { return BW_ABI_VERSION; }
int bw_device_count(void) { return bw_device_count_bf16(); }
int bw_runtime_flags(void) { return bw_runtime_flags_bf16() | bw_runtime_flags_f16(); }

int bw_engine_create(const bw_config* cfg, bw_engine** out) {
  if (!cfg || !out || (cfg->dtype != 0 && cfg->dtype != 1)) {
    g_last_f16 = 0;
    return bw_engine_create_bf16(nullptr, nullptr);  // reports "null argument"; an unknown dtype is treated the same way
  }
  bw_engine* e = new bw_engine{cfg->dtype, nullptr};
  g_last_f16 = e->f16;
  int rc;
  if (e->f16) {
    bw_engine_f16* h = nullptr;
    rc = bw_engine_create_f16(cfg, &h);
    e->impl = h;
  } else {
    bw_engine_bf16* h = nullptr;
    rc = bw_engine_create_bf16(cfg, &h);
    e->impl = h;
  }
  if (rc != 0) {
    delete e;
    return rc;
  }
  *out = e;
  return 0;
}
void bw_engine_destroy(bw_engine* e) {
  if (!e) return;
  if (e->f16) bw_engine_destroy_f16(BW_H(e));
  else bw_engine_destroy_bf16(BW_B(e));
  delete e;
}
int bw_engine_set_tensor(bw_engine* e, const char* name, const void* p) { BW_FWD(bw_engine_set_tensor, e, name, p); }
int bw_engine_set_mel_filters(bw_engine* e, const float* bank) { BW_FWD(bw_engine_set_mel_filters, e, bank); }
int bw_engine_set_alignment_heads(bw_engine* e, const int32_t* pairs, int32_t n) { BW_FWD(bw_engine_set_alignment_heads, e, pairs, n); }
int bw_engine_finalize(bw_engine* e) { BW_FWD(bw_engine_finalize, e); }
int bw_engine_buffer(bw_engine* e, const char* name, void** p, size_t* bytes) { BW_FWD(bw_engine_buffer, e, name, p, bytes); }
int bw_logmel(bw_engine* e, const float* pcm, int32_t B, int32_t n_samples, float* mel_f32_out, void* stream) {
  BW_FWD(bw_logmel, e, pcm, B, n_samples, mel_f32_out, stream);
}
int bw_set_mel(bw_engine* e, const float* mel, int32_t B, void* stream) { BW_FWD(bw_set_mel, e, mel, B, stream); }
int bw_encode(bw_engine* e, int32_t B, void* stream) { BW_FWD(bw_encode, e, B, stream); }
int bw_decode_begin(bw_engine* e, int32_t A, int32_t G, const int32_t* prompt, int32_t plen, const bw_decode_opts* opts, void* stream) {
  BW_FWD(bw_decode_begin, e, A, G, prompt, plen, opts, stream);
}
int bw_decode_run(bw_engine* e, int32_t n_steps, void* stream) { BW_FWD(bw_decode_run, e, n_steps, stream); }
long long bw_decode_kernel_launches(bw_engine* e) {
  if (!e) return -1;
  return e->f16 ? bw_decode_kernel_launches_f16(BW_H(e)) : bw_decode_kernel_launches_bf16(BW_B(e));
}
int bw_decode_read(bw_engine* e, int32_t* tokens, int32_t* finished, int32_t* pos, void* stream) { BW_FWD(bw_decode_read, e, tokens, finished, pos, stream); }
int bw_decode_reorder(bw_engine* e, const int32_t* parent, const int32_t* next_token, void* stream) {
  BW_FWD(bw_decode_reorder, e, parent, next_token, stream);
}
int bw_decode_beam_step(bw_engine* e, const float* run_scores, float* cand_scores, int32_t* cand_tokens, void* stream) {
  BW_FWD(bw_decode_beam_step, e, run_scores, cand_scores, cand_tokens, stream);
}
int bw_word_timestamps(bw_engine* e, int32_t audio, int32_t n_tokens, int32_t num_frames, double time_precision, float* out_host, void* stream) {
  BW_FWD(bw_word_timestamps, e, audio, n_tokens, num_frames, time_precision, out_host, stream);
}
int bw_word_timestamps_batch(bw_engine* e, int32_t n, const int32_t* audio, const int32_t* n_tokens, const int32_t* num_frames,
                             double time_precision, float* out_host, int32_t out_pitch, void* stream) {
  BW_FWD(bw_word_timestamps_batch, e, n, audio, n_tokens, num_frames, time_precision, out_host, out_pitch, stream);
}
int bw_word_timestamps_gather(bw_engine* e, int32_t n, const int32_t* slot_map, int32_t map_pitch, const int32_t* n_tokens,
                              const int32_t* num_frames, double time_precision, float* out_host, int32_t out_pitch, void* stream) {
  BW_FWD(bw_word_timestamps_gather, e, n, slot_map, map_pitch, n_tokens, num_frames, time_precision, out_host, out_pitch, stream);
}

// ---- single ops: the bf16 build ------------------------------------------------------------------------------------------------
int bw_op_gemm(const void* A, const void* W, int32_t M, int32_t N, int32_t K, const float* bias, float alpha, int32_t act,
               const float* residual, void* out, int32_t out_is_f32, int32_t impl, int32_t force_bn, void* stream) {
  g_last_f16 = 0;
  return bw_op_gemm_bf16(A, W, M, N, K, bias, alpha, act, residual, out, out_is_f32, impl, force_bn, stream);
}
int bw_op_gemm_splitk(const void* A, const void* W, int32_t M, int32_t N, int32_t K, int32_t n_valid, int32_t ksplit, int32_t force_bn,
                      float* out_partials, int32_t* ksplit_used, void* stream) {
  g_last_f16 = 0;
  return bw_op_gemm_splitk_bf16(A, W, M, N, K, n_valid, ksplit, force_bn, out_partials, ksplit_used, stream);
}
int bw_op_gemm_dec(const void* X, const void* W, int32_t Q, int32_t N, int32_t K, int32_t n_valid, int32_t want_split, float* out_partials,
                   int32_t* ksplit_used, void* stream) {
  g_last_f16 = 0;
  return bw_op_gemm_dec_bf16(X, W, Q, N, K, n_valid, want_split, out_partials, ksplit_used, stream);
}
int bw_op_gelu_bias(const float* partials, int32_t nsplit, const float* bias, void* h_bf16, int32_t Q, int32_t N, void* stream) {
  g_last_f16 = 0;
  return bw_op_gelu_bias_bf16(partials, nsplit, bias, h_bf16, Q, N, stream);
}
int bw_op_resid_ln(float* x, const float* partials, int32_t nsplit, const float* bias, const float* ln_g, const float* ln_b, void* y_bf16,
                   int32_t Q, int32_t D, void* stream) {
  g_last_f16 = 0;
  return bw_op_resid_ln_bf16(x, partials, nsplit, bias, ln_g, ln_b, y_bf16, Q, D, stream);
}
int bw_op_attn_enc(const void* qkv, void* vt_scratch, void* out, int32_t B, int32_t S, int32_t H, int32_t impl, void* stream) {
  g_last_f16 = 0;
  return bw_op_attn_enc_bf16(qkv, vt_scratch, out, B, S, H, impl, stream);
}
int bw_op_layernorm(const float* x, const float* g, const float* b, void* out, int32_t out_is_f32, int32_t rows, int32_t D, void* stream) {
  g_last_f16 = 0;
  return bw_op_layernorm_bf16(x, g, b, out, out_is_f32, rows, D, stream);
}
int bw_op_gemv(const float* x, const float* ln_g, const float* ln_b, const void* W, int32_t M, int32_t N, int32_t K, const float* bias,
               float alpha, int32_t act, const float* residual, float* out, void* stream) {
  g_last_f16 = 0;
  return bw_op_gemv_bf16(x, ln_g, ln_b, W, M, N, K, bias, alpha, act, residual, out, stream);
}

// ---- single ops with a 16-bit cache operand: the build elem_dtype names ---------------------------------------------------------
int bw_op_self_attn(const float* qkv, int32_t nsplit, const float* qkv_bias, float q_alpha, void* kc, void* vc, const int32_t* anc,
                    int32_t append, void* out, int32_t out_is_f32, const int32_t* pos_dev, int32_t Q, int32_t H, int32_t Tmax,
                    int32_t elem_dtype, void* stream) {
  g_last_f16 = elem_dtype == 1;
  if (elem_dtype == 1)
    return bw_op_self_attn_f16(qkv, nsplit, qkv_bias, q_alpha, kc, vc, anc, append, out, out_is_f32, pos_dev, Q, H, Tmax, elem_dtype, stream);
  // an unknown elem_dtype: the bf16 build reports it
  return bw_op_self_attn_bf16(qkv, nsplit, qkv_bias, q_alpha, kc, vc, anc, append, out, out_is_f32, pos_dev, Q, H, Tmax,
                              elem_dtype, stream);
}
int bw_op_cross_attn(const float* q, int32_t nsplit, const float* q_bias, float q_alpha, const void* kc, const void* vc,
                     void* out, int32_t out_is_f32, float* part_o, float* part_ml, uint32_t* counters, int32_t A, int32_t G,
                     int32_t H, int32_t S, float* align, const int32_t* head_slots, int32_t Ha, int32_t Tcap, int32_t step_base,
                     const int32_t* pos_dev, int32_t impl, int32_t elem_dtype, void* stream) {
  g_last_f16 = elem_dtype == 1;
  if (elem_dtype == 1)
    return bw_op_cross_attn_f16(q, nsplit, q_bias, q_alpha, kc, vc, out, out_is_f32, part_o, part_ml, counters, A, G, H, S, align,
                                head_slots, Ha, Tcap, step_base, pos_dev, impl, elem_dtype, stream);
  return bw_op_cross_attn_bf16(q, nsplit, q_bias, q_alpha, kc, vc, out, out_is_f32, part_o, part_ml, counters, A, G, H, S, align,
                               head_slots, Ha, Tcap, step_base, pos_dev, impl, elem_dtype, stream);
}

}  // extern "C"
