// Decoder-step kernels (q_len = 1, HBM-bound weight / KV streaming) and their argument blocks.
#pragma once
#include "common.cuh"

namespace BW_NS {

// out[m, n] = epi( LN?(x[m, :]) . W[n, :] )   for m < M <= 8 rows per launch
struct GemvArgs {
  const float* x = nullptr;  // [M, K] fp32 rows (pitch ldx)
  int ldx = 0;
  const float* ln_g = nullptr;  // optional LayerNorm (eps 1e-5) applied to x rows first
  const float* ln_b = nullptr;
  const bf16* W = nullptr;  // [N, K]
  int N = 0, K = 0, M = 0;
  const float* bias = nullptr;
  float alpha = 1.0f;
  int alpha_cols = 0;  // alpha applies to columns [0, alpha_cols)
  int act = 0;         // 1 = exact GELU
  const float* residual = nullptr;  // [M, ldo] (may alias out)
  float* out = nullptr;
  int ldo = 0;
  // optional self-KV scatter (fused QKV projection): columns [D,2D) -> kc, [2D,3D) -> vc at row (seq0+m, *pos)
  bf16* kc = nullptr;
  bf16* vc = nullptr;
  int D = 0, Tmax = 0, seq0 = 0;
  const int* pos = nullptr;
};

struct SelfAttnArgs {
  const float* qkv = nullptr;  // [Q, 3D] fp32 (q already scaled)
  const bf16* kc = nullptr;    // [Q, Tmax, D]
  const bf16* vc = nullptr;
  const int* anc = nullptr;    // [Q, Tmax] sequence slot holding position s for sequence q (null = own slot)
  float* out = nullptr;        // [Q, D] fp32 (per-op GEMV path) ...
  bf16* out_bf16 = nullptr;    // ... or bf16 (operand of the batched path's tcgen05 out-projection); exactly one of the two
  const int* pos = nullptr;
  int H = 0, D = 0, Tmax = 0;
  // batched path: the fused QKV GEMM leaves k / v of the current token in qkv (fp32, + bias); the (sequence, head) CTA rounds them to
  // bf16, appends them to the cache at position *pos and attends over them (the GEMV path appends in its own epilogue)
  bf16* kc_w = nullptr;
  bf16* vc_w = nullptr;
  // batched path, split-K projection: qkv holds nsplit raw partial sums ([split][Q][3D], split_stride apart); the kernel adds them in
  // order, then the bias (qkv_bias [3D]) and scales q by q_alpha.  nsplit = 0: qkv is final (per-op / ksplit = 1 paths).
  int nsplit = 0;
  long long split_stride = 0;
  const float* qkv_bias = nullptr;
  float q_alpha = 1.0f;
};

constexpr int XSPLIT = 12;   // key splits per (audio, head) in cross attention (<= 128 keys each: S <= 1536)
constexpr int MAXG = 8;      // max sequences (beams) sharing one audio's cross K/V

struct CrossAttnArgs {
  const float* q = nullptr;  // [Q, D] fp32 (scaled), Q = A*G
  const bf16* kc = nullptr;  // [A, H, S, 64]
  const bf16* vc = nullptr;  // [A, H, S, 64]
  float* out = nullptr;      // [Q, D] fp32, or
  bf16* out_bf16 = nullptr;  // [Q, D] bf16 (batched path)
  float* part_o = nullptr;   // [A, H, XSPLIT, G, 64]
  float* part_ml = nullptr;  // [A, H, XSPLIT, G, 2]
  unsigned* counters = nullptr;  // [A*H], zero between launches
  int S = 0, H = 0, D = 0, G = 1;
  // word timestamps: raw scores of alignment heads (beam 0 of each audio) -> align[(a*Ha + slot)*Tcap + step][S]
  float* align = nullptr;
  int align_slot = -1;  // slot of THIS layer's head `align_head`, resolved per launch via head_slots
  const int* head_slots = nullptr;  // [H] slot per head for this layer or -1
  int Ha = 0, Tcap = 0, step_base = 0;
  const int* pos = nullptr;
  // batched path, split-K cross-q projection: q holds nsplit raw partial sums ([split][Q][D]); summed in order, + q_bias, * q_alpha
  int nsplit = 0;
  long long split_stride = 0;
  const float* q_bias = nullptr;
  float q_alpha = 1.0f;
};

struct SelectArgs {
  const float* logits = nullptr;  // [Q, ldl], ldl >= V
  int V = 0, Q = 0, Tmax = 0, ldl = 0;
  int* tokens = nullptr;       // [Q, Tmax]
  int* finished = nullptr;     // [Q]
  int* pos = nullptr;          // device scalar, advanced by the last block
  unsigned* done_ctr = nullptr;
  const unsigned* suppress_bits = nullptr;        // bitmap [ceil(V/32)]
  const unsigned* begin_suppress_bits = nullptr;  // bitmap, applied when pos+1 == begin_index
  int begin_index = 0;  // prompt length
  int eos = 0, pad = 0;
  int ts_rules = 0, ts_begin = 0, no_ts = 0, max_initial_ts = -1;
  float* out_lse = nullptr;  // optional [Q]: log-sum-exp of the raw logits (parity / beam search)
  // beam search: per sequence the n_cand (<= 16) best continuations, running score included
  int n_cand = 0;
  const float* run_scores = nullptr;  // [Q]
  float* cand_scores = nullptr;       // [Q, n_cand]
  int* cand_tokens = nullptr;         // [Q, n_cand]
};

// ---- persistent one-kernel-per-step decoder (decode_mega.cu) ----
struct MegaLayer {
  const float *ln1g, *ln1b, *bqkv, *bo, *ln2g, *ln2b, *xbq, *xbo, *ln3g, *ln3b, *b1, *b2;
  const bf16 *wqkv, *wo, *xwq, *xwo, *w1, *w2;
  bf16 *self_k, *self_v;
  const bf16 *cross_k, *cross_v;
  const int* head_slots;  // [H] or null
};

constexpr int MEGA_MAXL = 32;
constexpr int MEGA_DEFAULT_FLAGS = 64;  // MegaArgs::flags when BW_MEGA_FLAGS is unset (bit 6 measured -1.2 %, bit-exact: r1_v8)
constexpr int MEGA_TRACE_N = 264;  // barriers per step that the optional trace records

struct MegaArgs {
  // the per-layer pointer table travels in the kernel parameter block (constant bank, ~8 KB: CUDA >= 12.1 allows 32 KB),
  // so no phase spends registers or a dependent global load on it
  MegaLayer layers[MEGA_MAXL];
  int L, D, H, ffn, V, S, Tmax, Q;
  int ldl;  // row pitch of logits (V rounded up to 32: rows stay 16-byte aligned for the batched path's tcgen05 LM head)
  const bf16* embed;
  const float* dec_pos;
  const float *lnf_g, *lnf_b;
  const int* tokens;
  const int* pos;
  float *dx, *dqkv, *dattn, *dq, *dh, *logits;
  float *part_o, *part_ml;  // cross-attention partials [Q][H][nsplit][64], [..][2]
  unsigned* xcounters;      // [Q*H]
  unsigned* bar;
  int nsplit;
  // alignment (word timestamps)
  float* align;
  int Ha, Tcap, step_base;
  long long* trace;  // optional barrier timeline (debug)
  int flags;         // bit0: no L2 prefetch two phases ahead; bit1: force single-buffered weight slabs (experiments);
                     // bit6 (64): the staging warps do not wait for the DMA warp
  // greedy token selection fused behind the LM head (no timestamp rules, one beam): masked arg-max by 64-bit atomicMax,
  // the last CTA to finish writes the token, handles EOS / pad and advances the position -- no select kernel
  int fuse_select;
  const unsigned* suppress_bits;
  const unsigned* begin_suppress_bits;
  int begin_index, eos, pad;
  int* finished;
  int* tokens_rw;
  int* pos_rw;
  unsigned long long* sel_best;  // [Q], zero between steps
  unsigned* sel_ctr;             // zero between steps
  int p0_off;        // set by the launcher: byte offset of the second slab region (0: single-buffered slabs)
};

// Returns -3 when the configuration is outside what the persistent kernel supports (caller uses the per-op path).
int launch_decode_mega(cudaStream_t st, const MegaArgs& a, int num_sms);
extern int g_mega_coop;  // 1: the persistent step kernels are launched cooperatively (co-residency guaranteed by the driver)
int launch_gemv(cudaStream_t st, const GemvArgs& a);
int launch_embed(cudaStream_t st, const bf16* E, const float* P, const int* tokens, const int* pos, float* x, int Q, int D, int Tmax);
int launch_self_attn(cudaStream_t st, const SelfAttnArgs& a, int Q);
// impl: 0 = the engine's policy (streaming kernel from BW_XATTN_STREAM_MIN CTAs, default 296), 1 = split kernel, 2 = streaming kernel
int launch_cross_attn(cudaStream_t st, const CrossAttnArgs& a, int A, int impl = 0);
int launch_select(cudaStream_t st, const SelectArgs& a);
// x[q] += bias + sum_{s < nsplit} part[s][q]  (fixed order: deterministic), then y[q] = LayerNorm(x[q]) as bf16.
// nsplit = 0: LayerNorm only.  part: [nsplit][Q][D] fp32 partial sums of a split-K GEMM (gemm_tc_split).
int launch_resid_ln(cudaStream_t st, float* x, const float* part, int nsplit, long long split_stride, const float* bias, const float* g,
                    const float* b, bf16* y, int Q, int D);

}  // namespace bw
