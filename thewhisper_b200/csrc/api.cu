// C-ABI (include/thewhisper_b200.h) and the engine that sequences the kernels: encoder pass, cross-K/V projection,
// CUDA-graph decode steps.  Host C++ only orchestrates; all arithmetic is in the .cu kernels of this directory.
#include <limits.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <tuple>
#include <vector>

// This file is compiled once per element type (bf16: namespace bw, symbols *_bf16; -DBW_F16: namespace bw_f16, symbols *_f16);
// abi.cu defines the public names of include/thewhisper_b200.h and dispatches on bw_config::dtype.
#ifdef BW_F16
#define BW_RENAME_SUFFIX _f16
#define BW_API_NS bw_api_f16
#else
#define BW_RENAME_SUFFIX _bf16
#define BW_API_NS bw_api
#endif
#include "abi_rename.h"
#include "../../include/thewhisper_b200.h"
#include "decode.cuh"
#include "kernels.h"

namespace BW_NS {

static thread_local char g_err[1024] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* get_error() { return g_err; }
int g_pdl = 0;
static int g_pdl_enabled = -1;  // BW_PDL (default on); cleared if a step with programmatic launches cannot be captured

size_t word_timestamps_work_floats(int Ha, int Tcap, int S);  // timestamps.cu
int word_timestamps_batch_device(cudaStream_t st, const float* align, int Ha, int Tcap, int S, const int* items_dev, const int* slot_map_dev,
                                 int map_pitch, int n, int maxT, int maxNF, double time_precision, float* work, float* out_dev);

namespace {

struct EncLayer {
  const float *ln1g, *ln1b, *bqkv, *bo, *ln2g, *ln2b, *b1, *b2;
  const bf16 *wqkv, *wo, *w1, *w2;
};
struct DecLayer {
  const float *ln1g, *ln1b, *bqkv, *bo, *ln2g, *ln2b, *xbq, *xbv, *xbo, *ln3g, *ln3b, *b1, *b2;
  const bf16 *wqkv, *wo, *xwq, *xwk, *xwv, *xwo, *w1, *w2;
};

// Everything a captured step graph bakes in as kernel parameters: a decode that differs in any of these gets its own graph
// (round-1 advisor: eos / pad / timestamp ids were missing, a second decode with other ids replayed the old ones).
struct GraphKey {
  int A, G, begin_index, ts_rules, align, variant, eos, pad, ts_begin, no_ts;
  bool operator<(const GraphKey& o) const {
    return std::tie(A, G, begin_index, ts_rules, align, variant, eos, pad, ts_begin, no_ts) <
           std::tie(o.A, o.G, o.begin_index, o.ts_rules, o.align, o.variant, o.eos, o.pad, o.ts_begin, o.no_ts);
  }
};

}  // namespace
}  // namespace bw

using namespace BW_NS;

struct bw_engine {
  bw_config cfg;
  std::map<std::string, const void*> tensors;
  bool finalized = false;
  int D, H, S, F, V, Vp, Tmax, Spad;
  // resolved weights
  const bf16 *conv1_w = nullptr, *conv2_w = nullptr, *embed = nullptr;
  const float *conv1_b = nullptr, *conv2_b = nullptr, *enc_pos = nullptr, *enc_lnf_g = nullptr, *enc_lnf_b = nullptr;
  const float *dec_pos = nullptr, *dec_lnf_g = nullptr, *dec_lnf_b = nullptr;
  std::vector<EncLayer> enc;
  std::vector<DecLayer> dec;
  LogmelPlan* mel_plan = nullptr;
  std::vector<int> align_pairs;
  // encoder workspace
  bf16 *mel_tm = nullptr, *h1 = nullptr, *xn = nullptr, *qkv = nullptr, *vt = nullptr, *ao = nullptr, *hbuf = nullptr, *enc_out = nullptr;
  float *x_enc = nullptr, *mel_scratch = nullptr;
  unsigned* mel_max = nullptr;
  // caches
  bf16 *cross_k = nullptr, *cross_v = nullptr;  // [L][A][H][S][64]
  bf16 *self_k = nullptr, *self_v = nullptr;    // [L][Q][Tmax][D]
  // decoder state
  int *tokens = nullptr, *finished = nullptr, *pos = nullptr, *anc = nullptr, *anc_tmp = nullptr, *head_slots = nullptr;
  unsigned *done_ctr = nullptr, *xcounters = nullptr, *sup_bits = nullptr, *bsup_bits = nullptr, *sel_ctr = nullptr;
  unsigned long long* sel_best = nullptr;
  float *dx = nullptr, *dqkv = nullptr, *dattn = nullptr, *dq = nullptr, *dh = nullptr, *logits = nullptr, *part_o = nullptr,
        *part_ml = nullptr, *align = nullptr, *lse = nullptr, *ts_work = nullptr, *ts_out = nullptr;
  int *reorder_tmp = nullptr, *cand_tokens = nullptr, *ts_items = nullptr, *ts_map = nullptr;
  float *run_scores = nullptr, *cand_scores = nullptr;
  size_t align_bytes = 0;
  // current decode session
  int A = 0, G = 1, Q = 0;
  bw_decode_opts opts{};
  bool use_anc = false;
  std::map<GraphKey, cudaGraphExec_t> graphs;
  cudaGraphExec_t cur_graph = nullptr;
  std::map<cudaGraphExec_t, int> graph_kernels;  // kernel nodes of each captured step graph
  long long step_kernel_launches = 0;            // kernels launched by bw_decode_run so far (graph path)
  bool no_graph = false, simt = false, no_mega = false, no_fused_select = false;  // env switches, read ONCE at engine creation
  int mega_flags = MEGA_DEFAULT_FLAGS;  // BW_MEGA_FLAGS (experiment switches of the persistent step kernel), read once at engine creation
  // batched (tensor-core) decoder step: bf16 GEMM operands [Qpad][D] / [Qpad][ffn], split-K partial sums [BSPLIT][Qm][D]
  bf16 *dbn = nullptr, *dba = nullptr, *dbh = nullptr;
  float* dpart = nullptr;
  int batch_min = 3;  // sequences from which a step runs on the tcgen05 path (BW_BATCH_MIN)
  bool gemm2 = true;  // encoder GEMMs on the CTA-pair kernel (BW_GEMM2=0: first-generation kernel only)
  bool attn2 = true;  // encoder attention on the ping-pong kernel (BW_ATTN2=0: first-generation kernel)
  bool attn_vdirect = true;   // ... reading V tiles from the qkv rows (MN-major operand) instead of a transposed copy (BW_ATTN_VDIRECT=0: transposed copy)
  long long gemm2_min_rows = 1024;
  bool enc_graph = true;   // the encoder pass of a batch size runs as one CUDA graph from its second call on (BW_ENC_GRAPH=0: stream launches)
  bool enc_pdl = false;    // BW_ENC_PDL=1: ... with its kernels chained by programmatic dependent launch (measured in r2o: no gain, 5.000 vs 5.005 ms at B = 1)
  std::map<int, cudaGraphExec_t> enc_graphs;
  std::map<int, int> enc_calls;
  int num_sms = 148;
  unsigned* mega_bar = nullptr;
  long long* mega_trace = nullptr;
  std::map<std::string, std::pair<void*, size_t>> buffers;
};

namespace BW_API_NS {

template <typename T>
int dalloc(bw_engine* e, const char* name, T** p, size_t count, bool zero = true) {
  const size_t bytes = count * sizeof(T);
  BW_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(p), bytes ? bytes : 16));
  if (zero) BW_CUDA_OK(cudaMemset(*p, 0, bytes ? bytes : 16));
  e->buffers[name] = std::make_pair(static_cast<void*>(*p), bytes);
  return 0;
}

template <typename T>
int need(bw_engine* e, const std::string& name, const T** out) {
  auto it = e->tensors.find(name);
  BW_CHECK(it != e->tensors.end() && it->second != nullptr, "weight '%s' is not bound", name.c_str());
  *out = static_cast<const T*>(it->second);
  return 0;
}

int gemm(bw_engine* e, cudaStream_t st, const GemmA& a, const bf16* W, int B, int rows, int N, int K, const GemmEpi& epi) {
  if (e->simt) return gemm_simt(st, a, W, B, rows, N, K, epi);
  // plain row-major activations of all B items are one [B * rows, K] matrix: the CTA-pair kernel tiles it without per-item tails
  if (e->gemm2 && a.kwrap >= K && a.pitch == K && a.batch_stride == (long long)rows * K && !epi.pos && gemm_tc2_supported(B * rows, N, K) &&
      (long long)B * rows >= e->gemm2_min_rows)
    return gemm_tc2(st, a.base, W, B * rows, N, K, rows, epi, 0);
  return gemm_tc(st, a, W, B, rows, N, K, epi, 0);
}

GemmA plainA(const bf16* base, int rows, int K) {
  GemmA a;
  a.base = base;
  a.batch_stride = (long long)rows * K;
  a.pitch = K;
  a.rows_base = rows;
  a.kwrap = INT_MAX;
  return a;
}

GemmEpi plainEpi(int rows, int ld) {
  GemmEpi ep;
  ep.batch_stride = (long long)rows * ld;
  ep.row_stride = ld;
  ep.head_stride = 64;
  return ep;
}

int encode_impl(bw_engine* e, int B, cudaStream_t st) {
  const int D = e->D, S = e->S, F = e->F, H = e->H, ffn = e->cfg.ffn, nm = e->cfg.n_mels;
  // ---- conv stem as two wrapping-coordinate GEMMs (modeling_whisper.py:619-625)
  {
    GemmA a;
    a.base = e->mel_tm; a.batch_stride = (long long)(F + 2) * nm; a.pitch = nm; a.rows_base = F + 2; a.kwrap = nm;
    GemmEpi ep;
    ep.bias = e->conv1_b; ep.act = 1;
    ep.out_bf16 = e->h1 + D;  // row t -> padded row t+1
    ep.batch_stride = (long long)(F + 2) * D; ep.row_stride = D;
    if (int rc = gemm(e, st, a, e->conv1_w, B, F, D, 3 * nm, ep)) return rc;
  }
  {
    GemmA a;
    a.base = e->h1; a.batch_stride = (long long)(F + 2) * D; a.pitch = 2 * D; a.rows_base = (F + 2) / 2; a.kwrap = 2 * D;
    GemmEpi ep;
    ep.bias = e->conv2_b; ep.act = 1; ep.pos = e->enc_pos;
    ep.out_f32 = e->x_enc;
    ep.batch_stride = (long long)S * D; ep.row_stride = D;
    if (int rc = gemm(e, st, a, e->conv2_w, B, S, D, 3 * D, ep)) return rc;
  }
  const float scale = 0.125f;  // head_dim^-1/2, head_dim = 64 (applied inside the attention kernels)
  (void)scale;
  for (size_t l = 0; l < e->enc.size(); ++l) {
    const EncLayer& L = e->enc[l];
    if (int rc = layernorm_bf16(st, e->x_enc, L.ln1g, L.ln1b, e->xn, B * S, D)) return rc;
    {
      GemmEpi ep = plainEpi(S, 3 * D);
      ep.bias = L.bqkv; ep.out_bf16 = e->qkv;
      if (int rc = gemm(e, st, plainA(e->xn, S, D), L.wqkv, B, S, 3 * D, D, ep)) return rc;
    }
    if (e->simt) {
      if (int rc = attn_enc_simt(st, e->qkv, e->ao, B, S, H)) return rc;
    } else {
      if (e->attn2 && e->attn_vdirect) {  // V tiles straight from the qkv rows (MN-major tcgen05 operand): no transposed copy
        if (int rc = attn_enc_tc2(st, e->qkv, nullptr, e->ao, B, S, e->Spad, H)) return rc;
      } else {
        if (int rc = transpose_v(st, e->qkv, e->vt, B, S, e->Spad, H)) return rc;
        if (int rc = (e->attn2 ? attn_enc_tc2 : attn_enc_tc)(st, e->qkv, e->vt, e->ao, B, S, e->Spad, H)) return rc;
      }
    }
    {
      GemmEpi ep = plainEpi(S, D);
      ep.bias = L.bo; ep.residual = e->x_enc; ep.out_f32 = e->x_enc;
      if (int rc = gemm(e, st, plainA(e->ao, S, D), L.wo, B, S, D, D, ep)) return rc;
    }
    if (int rc = layernorm_bf16(st, e->x_enc, L.ln2g, L.ln2b, e->xn, B * S, D)) return rc;
    {
      GemmEpi ep = plainEpi(S, ffn);
      ep.bias = L.b1; ep.act = 1; ep.out_bf16 = e->hbuf;
      if (int rc = gemm(e, st, plainA(e->xn, S, D), L.w1, B, S, ffn, D, ep)) return rc;
    }
    {
      GemmEpi ep = plainEpi(S, D);
      ep.bias = L.b2; ep.residual = e->x_enc; ep.out_f32 = e->x_enc;
      if (int rc = gemm(e, st, plainA(e->hbuf, S, ffn), L.w2, B, S, D, ffn, ep)) return rc;
    }
  }
  if (int rc = layernorm_bf16(st, e->x_enc, e->enc_lnf_g, e->enc_lnf_b, e->enc_out, B * S, D)) return rc;
  // ---- cross-attention K/V of every decoder layer, written head-major: [L][A][H][S][64]
  const long long per_layer = (long long)e->cfg.max_audios * H * S * 64;
  for (size_t l = 0; l < e->dec.size(); ++l) {
    const DecLayer& L = e->dec[l];
    GemmEpi ep;
    ep.batch_stride = (long long)H * S * 64; ep.row_stride = 64; ep.head_stride = (long long)S * 64;
    ep.out_bf16 = e->cross_k + l * per_layer;
    if (int rc = gemm(e, st, plainA(e->enc_out, S, D), L.xwk, B, S, D, D, ep)) return rc;
    ep.bias = L.xbv;
    ep.out_bf16 = e->cross_v + l * per_layer;
    if (int rc = gemm(e, st, plainA(e->enc_out, S, D), L.xwv, B, S, D, D, ep)) return rc;
  }
  return 0;
}

constexpr int DPART_PER_ROW = 20480;  // floats of split-K partial sums per sequence: ksplit * N <= (SMs / n_tiles) * (n_tiles * 128) < 20480

// One decoder step for Q >= 3 sequences on the tensor cores.  Every projection is a weight-streaming tcgen05 GEMM (gemm_dec.cu:
// weights = 128-row MMA operand, activations = N operand, K split so that a launch is one DRAM round trip) that leaves raw split-K
// partial sums; the kernel that consumes them adds them in a fixed order together with bias / scale / activation:
//   resid_ln (residual update + LayerNorm), the attention kernels (q / k / v), gelu_bias (fc1 -> fc2 operand).
// 12 launches per layer in one CUDA graph, chained by programmatic dependent launch; weights are read once per step whatever Q is
// (the GEMV path runs 2*Q*params flops on the fp32 pipes: 46 ms per step at Q = 64, profiles/r2a_summary.md).
int step_batched_impl(bw_engine* e, cudaStream_t st);
int step_batched(bw_engine* e, cudaStream_t st) {
  // programmatic dependent launch for every kernel of the step (BW_PDL=0: plain stream order)
  if (g_pdl_enabled < 0) {
    const char* ev = getenv("BW_PDL");
    g_pdl_enabled = (ev && ev[0] == '0') ? 0 : 1;
  }
  g_pdl = g_pdl_enabled;
  const int rc = step_batched_impl(e, st);
  g_pdl = 0;
  return rc;
}
int step_batched_impl(bw_engine* e, cudaStream_t st) {
  const int D = e->D, H = e->H, S = e->S, ffn = e->cfg.ffn, Tmax = e->Tmax, Q = e->Q, A = e->A, G = e->G;
  const long long self_layer = (long long)e->cfg.max_audios * e->cfg.max_beams * Tmax * D;
  const long long cross_layer = (long long)e->cfg.max_audios * H * S * 64;
  // raw partial sums of out[Q, N] = in[Q, K] W[N, K]^T into dpart ([split][Q][N]); returns the split count
  auto proj = [&](const bf16* in, int K, const bf16* W, int N, int* ns) {
    const DecGemmPlan pl = gemm_dec_plan(Q, N, K, e->num_sms, true);
    BW_CHECK((long long)pl.ksplit * N <= DPART_PER_ROW, "batched step: %d splits x N=%d exceed the partial-sum buffer", pl.ksplit, N);
    GemmEpi ep;
    ep.out_f32 = e->dpart; ep.row_stride = N;
    *ns = pl.ksplit;
    return gemm_dec(st, in, W, Q, N, K, 0, ep, pl, (long long)Q * N);
  };
  if (int rc = launch_embed(st, e->embed, e->dec_pos, e->tokens, e->pos, e->dx, Q, D, Tmax)) return rc;
  int ns = 0;                  // partial sums of the previous residual GEMM still to be folded into dx
  const float* pbias = nullptr;
  for (size_t l = 0; l < e->dec.size(); ++l) {
    const DecLayer& L = e->dec[l];
    bf16* kc = e->self_k + l * self_layer;
    bf16* vc = e->self_v + l * self_layer;
    // dx += fc2 partials of layer l-1 (+ b2); LN1 -> dbn
    if (int rc = launch_resid_ln(st, e->dx, e->dpart, ns, (long long)Q * D, pbias, L.ln1g, L.ln1b, e->dbn, Q, D)) return rc;
    if (int rc = proj(e->dbn, D, L.wqkv, 3 * D, &ns)) return rc;
    {
      SelfAttnArgs s;
      s.qkv = e->dpart; s.nsplit = ns; s.split_stride = (long long)Q * 3 * D; s.qkv_bias = L.bqkv; s.q_alpha = 0.125f;
      s.kc = kc; s.vc = vc; s.kc_w = kc; s.vc_w = vc; s.anc = e->use_anc ? e->anc : nullptr; s.out_bf16 = e->dba; s.pos = e->pos;
      s.H = H; s.D = D; s.Tmax = Tmax;
      if (int rc = launch_self_attn(st, s, Q)) return rc;
    }
    if (int rc = proj(e->dba, D, L.wo, D, &ns)) return rc;
    if (int rc = launch_resid_ln(st, e->dx, e->dpart, ns, (long long)Q * D, L.bo, L.ln2g, L.ln2b, e->dbn, Q, D)) return rc;
    if (int rc = proj(e->dbn, D, L.xwq, D, &ns)) return rc;
    {
      CrossAttnArgs c;
      c.q = e->dpart; c.nsplit = ns; c.split_stride = (long long)Q * D; c.q_bias = L.xbq; c.q_alpha = 0.125f;
      c.kc = e->cross_k + l * cross_layer; c.vc = e->cross_v + l * cross_layer; c.out_bf16 = e->dba;
      c.part_o = e->part_o; c.part_ml = e->part_ml; c.counters = e->xcounters;
      c.S = S; c.H = H; c.D = D; c.G = G; c.pos = e->pos;
      if (e->opts.record_alignment && e->cfg.n_align_heads > 0) {
        c.align = e->align; c.head_slots = e->head_slots + l * H; c.Ha = e->cfg.n_align_heads;
        c.Tcap = e->cfg.max_align_steps; c.step_base = e->opts.begin_index;
      }
      if (int rc = launch_cross_attn(st, c, A)) return rc;
    }
    if (int rc = proj(e->dba, D, L.xwo, D, &ns)) return rc;
    if (int rc = launch_resid_ln(st, e->dx, e->dpart, ns, (long long)Q * D, L.xbo, L.ln3g, L.ln3b, e->dbn, Q, D)) return rc;
    if (int rc = proj(e->dbn, D, L.w1, ffn, &ns)) return rc;
    if (int rc = launch_gelu_bias(st, e->dpart, ns, (long long)Q * ffn, L.b1, e->dbh, Q, ffn)) return rc;
    if (int rc = proj(e->dbh, ffn, L.w2, D, &ns)) return rc;
    pbias = L.b2;
  }
  if (int rc = launch_resid_ln(st, e->dx, e->dpart, ns, (long long)Q * D, pbias, e->dec_lnf_g, e->dec_lnf_b, e->dbn, Q, D)) return rc;
  {  // tied LM head: 406 weight tiles, no split; rows of the embedding beyond V are zero-filled by TMA and not stored
    const DecGemmPlan pl = gemm_dec_plan(Q, e->V, D, e->num_sms, false);
    GemmEpi ep;
    ep.out_f32 = e->logits; ep.row_stride = e->Vp;
    if (int rc = gemm_dec(st, e->dbn, e->embed, Q, e->V, D, e->V, ep, pl, 0)) return rc;
  }
  return 0;
}

// one decoder step for all Q sequences (enqueued on st; captured into a CUDA graph by the caller)
int step_impl(bw_engine* e, cudaStream_t st) {
  const int D = e->D, H = e->H, S = e->S, ffn = e->cfg.ffn, V = e->V, Tmax = e->Tmax, Q = e->Q, A = e->A, G = e->G;
  const long long self_layer0 = (long long)e->cfg.max_audios * e->cfg.max_beams * Tmax * D;
  const long long cross_layer0 = (long long)e->cfg.max_audios * H * S * 64;
  bool mega_done = false, select_done = false;
  if (!e->no_mega && G == 1 && Q <= 8 && (int)e->dec.size() <= MEGA_MAXL) {
    // persistent one-kernel step (decode_mega.cu); falls through to the per-op path when unsupported (-3)
    MegaArgs m{};
    for (size_t l = 0; l < e->dec.size(); ++l) {
      const DecLayer& L = e->dec[l];
      MegaLayer& o = m.layers[l];
      o.ln1g = L.ln1g; o.ln1b = L.ln1b; o.bqkv = L.bqkv; o.bo = L.bo; o.ln2g = L.ln2g; o.ln2b = L.ln2b; o.xbq = L.xbq; o.xbo = L.xbo;
      o.ln3g = L.ln3g; o.ln3b = L.ln3b; o.b1 = L.b1; o.b2 = L.b2;
      o.wqkv = L.wqkv; o.wo = L.wo; o.xwq = L.xwq; o.xwo = L.xwo; o.w1 = L.w1; o.w2 = L.w2;
      o.self_k = e->self_k + l * self_layer0; o.self_v = e->self_v + l * self_layer0;
      o.cross_k = e->cross_k + l * cross_layer0; o.cross_v = e->cross_v + l * cross_layer0;
      o.head_slots = (e->opts.record_alignment && e->cfg.n_align_heads > 0) ? e->head_slots + l * H : nullptr;
    }
    m.L = (int)e->dec.size(); m.D = D; m.H = H; m.ffn = ffn; m.V = V; m.S = S; m.Tmax = Tmax; m.Q = Q;
    m.embed = e->embed; m.dec_pos = e->dec_pos; m.lnf_g = e->dec_lnf_g; m.lnf_b = e->dec_lnf_b;
    m.tokens = e->tokens; m.pos = e->pos; m.ldl = e->Vp;
    m.dx = e->dx; m.dqkv = e->dqkv; m.dattn = e->dattn; m.dq = e->dq; m.dh = e->dh; m.logits = e->logits;
    m.part_o = e->part_o; m.part_ml = e->part_ml; m.xcounters = e->xcounters; m.bar = e->mega_bar;
    int ns = e->num_sms / (Q * H);
    const int ns_min = (S + 255) / 256;
    if (ns < ns_min) ns = ns_min;
    if (ns > XSPLIT) ns = XSPLIT;
    m.nsplit = ns;
    if (e->opts.record_alignment && e->cfg.n_align_heads > 0) {
      m.align = e->align; m.Ha = e->cfg.n_align_heads; m.Tcap = e->cfg.max_align_steps; m.step_base = e->opts.begin_index;
    }
    m.trace = e->mega_trace;
    if (!e->opts.timestamp_rules && !e->no_fused_select) {
      m.fuse_select = 1;
      m.suppress_bits = e->sup_bits; m.begin_suppress_bits = e->bsup_bits; m.begin_index = e->opts.begin_index;
      m.eos = e->opts.eos_token; m.pad = e->opts.pad_token; m.finished = e->finished; m.tokens_rw = e->tokens; m.pos_rw = e->pos;
      m.sel_best = e->sel_best; m.sel_ctr = e->sel_ctr;
    }
    m.flags = e->mega_flags;
    const int rc = launch_decode_mega(st, m, e->num_sms);
    if (rc == 0) {
      mega_done = true;
      select_done = m.fuse_select != 0;
    }
    else if (rc != -3) return rc;
  }
  if (!mega_done && !e->simt && Q >= e->batch_min) {
    if (int rc = step_batched(e, st)) return rc;
    mega_done = true;
  }
  if (!mega_done) {
  if (int rc = launch_embed(st, e->embed, e->dec_pos, e->tokens, e->pos, e->dx, Q, D, Tmax)) return rc;
  const long long self_layer = (long long)e->cfg.max_audios * e->cfg.max_beams * Tmax * D;
  const long long cross_layer = (long long)e->cfg.max_audios * H * S * 64;
  for (size_t l = 0; l < e->dec.size(); ++l) {
    const DecLayer& L = e->dec[l];
    bf16* kc = e->self_k + l * self_layer;
    bf16* vc = e->self_v + l * self_layer;
    for (int m0 = 0; m0 < Q; m0 += Q) {  // (one launch: the kernel walks M in chunks of 8)
       // LN1 + fused QKV projection (+ self-KV append)
      GemvArgs g;
      g.M = Q - m0;
      g.x = e->dx + (long long)m0 * D; g.ldx = D; g.ln_g = L.ln1g; g.ln_b = L.ln1b;
      g.W = L.wqkv; g.N = 3 * D; g.K = D; g.bias = L.bqkv; g.alpha = 0.125f; g.alpha_cols = D;
      g.out = e->dqkv + (long long)m0 * 3 * D; g.ldo = 3 * D;
      g.kc = kc; g.vc = vc; g.D = D; g.Tmax = Tmax; g.seq0 = m0; g.pos = e->pos;
      if (int rc = launch_gemv(st, g)) return rc;
    }
    {
      SelfAttnArgs s;
      s.qkv = e->dqkv; s.kc = kc; s.vc = vc; s.anc = e->use_anc ? e->anc : nullptr; s.out = e->dattn; s.pos = e->pos;
      s.H = H; s.D = D; s.Tmax = Tmax;
      if (int rc = launch_self_attn(st, s, Q)) return rc;
    }
    for (int m0 = 0; m0 < Q; m0 += Q) {  // (one launch: the kernel walks M in chunks of 8)
       // out-proj + residual
      GemvArgs g;
      g.M = Q - m0;
      g.x = e->dattn + (long long)m0 * D; g.ldx = D; g.W = L.wo; g.N = D; g.K = D; g.bias = L.bo;
      g.residual = e->dx + (long long)m0 * D; g.out = e->dx + (long long)m0 * D; g.ldo = D;
      if (int rc = launch_gemv(st, g)) return rc;
    }
    for (int m0 = 0; m0 < Q; m0 += Q) {  // (one launch: the kernel walks M in chunks of 8)
       // LN2 + cross q projection
      GemvArgs g;
      g.M = Q - m0;
      g.x = e->dx + (long long)m0 * D; g.ldx = D; g.ln_g = L.ln2g; g.ln_b = L.ln2b;
      g.W = L.xwq; g.N = D; g.K = D; g.bias = L.xbq; g.alpha = 0.125f; g.alpha_cols = D;
      g.out = e->dq + (long long)m0 * D; g.ldo = D;
      if (int rc = launch_gemv(st, g)) return rc;
    }
    {
      CrossAttnArgs c;
      c.q = e->dq; c.kc = e->cross_k + l * cross_layer; c.vc = e->cross_v + l * cross_layer; c.out = e->dattn;
      c.part_o = e->part_o; c.part_ml = e->part_ml; c.counters = e->xcounters;
      c.S = S; c.H = H; c.D = D; c.G = G; c.pos = e->pos;
      if (e->opts.record_alignment && e->cfg.n_align_heads > 0) {
        c.align = e->align; c.head_slots = e->head_slots + l * H; c.Ha = e->cfg.n_align_heads;
        c.Tcap = e->cfg.max_align_steps; c.step_base = e->opts.begin_index;  // row 0 = first generated token as input
      }
      if (int rc = launch_cross_attn(st, c, A)) return rc;
    }
    for (int m0 = 0; m0 < Q; m0 += Q) {  // (one launch: the kernel walks M in chunks of 8)
       // cross out-proj + residual
      GemvArgs g;
      g.M = Q - m0;
      g.x = e->dattn + (long long)m0 * D; g.ldx = D; g.W = L.xwo; g.N = D; g.K = D; g.bias = L.xbo;
      g.residual = e->dx + (long long)m0 * D; g.out = e->dx + (long long)m0 * D; g.ldo = D;
      if (int rc = launch_gemv(st, g)) return rc;
    }
    for (int m0 = 0; m0 < Q; m0 += Q) {  // (one launch: the kernel walks M in chunks of 8)
       // LN3 + fc1 + GELU
      GemvArgs g;
      g.M = Q - m0;
      g.x = e->dx + (long long)m0 * D; g.ldx = D; g.ln_g = L.ln3g; g.ln_b = L.ln3b;
      g.W = L.w1; g.N = ffn; g.K = D; g.bias = L.b1; g.act = 1;
      g.out = e->dh + (long long)m0 * ffn; g.ldo = ffn;
      if (int rc = launch_gemv(st, g)) return rc;
    }
    for (int m0 = 0; m0 < Q; m0 += Q) {  // (one launch: the kernel walks M in chunks of 8)
       // fc2 + residual
      GemvArgs g;
      g.M = Q - m0;
      g.x = e->dh + (long long)m0 * ffn; g.ldx = ffn; g.W = L.w2; g.N = D; g.K = ffn; g.bias = L.b2;
      g.residual = e->dx + (long long)m0 * D; g.out = e->dx + (long long)m0 * D; g.ldo = D;
      if (int rc = launch_gemv(st, g)) return rc;
    }
  }
  for (int m0 = 0; m0 < Q; m0 += Q) {  // (one launch: the kernel walks M in chunks of 8)
       // final LN + tied LM head
    GemvArgs g;
    g.M = Q - m0;
    g.x = e->dx + (long long)m0 * D; g.ldx = D; g.ln_g = e->dec_lnf_g; g.ln_b = e->dec_lnf_b;
    g.W = e->embed; g.N = V; g.K = D;
    g.out = e->logits + (long long)m0 * e->Vp; g.ldo = e->Vp;
    if (int rc = launch_gemv(st, g)) return rc;
  }
  }  // !mega_done
  if (select_done) return 0;
  SelectArgs s;
  s.logits = e->logits; s.V = V; s.ldl = e->Vp; s.Q = Q; s.Tmax = Tmax; s.tokens = e->tokens; s.finished = e->finished; s.pos = e->pos;
  s.done_ctr = e->done_ctr; s.suppress_bits = e->sup_bits; s.begin_suppress_bits = e->bsup_bits;
  s.begin_index = e->opts.begin_index; s.eos = e->opts.eos_token; s.pad = e->opts.pad_token;
  s.ts_rules = e->opts.timestamp_rules; s.ts_begin = e->opts.timestamp_begin; s.no_ts = e->opts.no_timestamps_token;
  s.max_initial_ts = e->opts.max_initial_timestamp_index; s.out_lse = e->lse;
  if (G > 1) { s.n_cand = 2 * G; s.run_scores = e->run_scores; s.cand_scores = e->cand_scores; s.cand_tokens = e->cand_tokens; }
  return launch_select(st, s);
}

__global__ void mel_to_tm_kernel(const float* __restrict__ mel, bf16* __restrict__ out, int n_mels, int frames) {
  // [B][n_mels][frames] fp32 -> [B][frames+2][n_mels] bf16 (rows 0 and frames+1 zero)
  __shared__ float tile[32][33];
  const int b = blockIdx.z, f0 = blockIdx.x * 32, m0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int i = ty; i < 32; i += 8) {
    const int m = m0 + i, f = f0 + tx;
    tile[i][tx] = (m < n_mels && f < frames) ? mel[((long long)b * n_mels + m) * frames + f] : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int f = f0 + i, m = m0 + tx;
    if (f < frames && m < n_mels) out[((long long)b * (frames + 2) + f + 1) * n_mels + m] = f2e(tile[tx][i]);
  }
}

__global__ void iota_anc_kernel(int* anc, int Q, int Tmax) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < Q * Tmax) anc[i] = i / Tmax;
}

// new sequence i continues old sequence parent[i]: permute block-table rows, overwrite history + newest token
__global__ void reorder_kernel(const int* __restrict__ anc_old, int* __restrict__ anc_new, const int* __restrict__ tok_old,
                               int* __restrict__ tok_new, const int* __restrict__ parent, const int* __restrict__ next_tok,
                               const int* __restrict__ pos_ptr, int Tmax) {
  const int i = blockIdx.x;
  const int p = parent[i];
  const int cur = *pos_ptr;  // tokens [0, cur] are filled; position cur-1 was the last KV written
  for (int s = threadIdx.x; s < Tmax; s += blockDim.x) {
    anc_new[i * Tmax + s] = (s < cur) ? anc_old[p * Tmax + s] : i;
    int t = tok_old[p * Tmax + s];
    if (s == cur) t = next_tok[i];
    tok_new[i * Tmax + s] = t;
  }
}

}  // namespace BW_API_NS
using namespace BW_API_NS;

extern "C" {

const char* bw_last_error(void) { return BW_NS::get_error(); }
int bw_abi_version(void) { return BW_ABI_VERSION; }
int bw_runtime_flags(void) { return (g_mega_coop == 1 ? 1 : 0) | (g_pdl_enabled == 1 ? 2 : 0); }
int bw_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int bw_engine_create(const bw_config* cfg, bw_engine** out) {
  BW_CHECK(cfg && out, "bw_engine_create: null argument");
  BW_CHECK(cfg->d_model == cfg->n_heads * 64, "head_dim must be 64 (d_model=%d, heads=%d)", cfg->d_model, cfg->n_heads);
  BW_CHECK(cfg->d_model % 64 == 0 && cfg->ffn % 64 == 0, "d_model and ffn must be multiples of 64");
  BW_CHECK(cfg->n_mels == 128 || cfg->n_mels == 64, "n_mels=%d unsupported (the conv stem's TMA view needs a multiple of 64)", cfg->n_mels);
  BW_CHECK(cfg->max_beams >= 1 && cfg->max_beams <= MAXG, "max_beams must be in 1..%d", MAXG);
  BW_CHECK(cfg->max_source_positions >= 1 && cfg->max_source_positions <= 1536, "max_source_positions out of range (1..1536)");
  BW_CHECK(bw_device_count() > 0, "no CUDA device: thewhisper_b200 has no CPU fallback");
  bw_engine* e = new bw_engine();
  e->cfg = *cfg;
  e->D = cfg->d_model; e->H = cfg->n_heads; e->S = cfg->max_source_positions; e->F = 2 * e->S; e->V = cfg->vocab;
  e->Tmax = cfg->max_target_positions; e->Spad = (e->S + 7) / 8 * 8;
  e->Vp = (e->V + 31) / 32 * 32;
  {
    const char* bm = getenv("BW_BATCH_MIN");
    if (bm) e->batch_min = atoi(bm);
    const char* g2 = getenv("BW_GEMM2");
    if (g2) e->gemm2 = g2[0] != '0';
    const char* a2 = getenv("BW_ATTN2");
    if (a2) e->attn2 = a2[0] != '0';
    const char* eg = getenv("BW_ENC_GRAPH");
    if (eg) e->enc_graph = eg[0] != '0';
    const char* ep = getenv("BW_ENC_PDL");
    if (ep) e->enc_pdl = ep[0] != '0';
    const char* avd = getenv("BW_ATTN_VDIRECT");
    if (avd) e->attn_vdirect = avd[0] != '0';
    const char* g2r = getenv("BW_GEMM2_MIN_ROWS");
    if (g2r) e->gemm2_min_rows = atoll(g2r);
  }
  const char* ng = getenv("BW_NO_GRAPH");
  e->no_graph = ng && ng[0] == '1';
  const char* nm = getenv("BW_NO_MEGA");
  e->no_mega = nm && nm[0] == '1';
  e->no_fused_select = getenv("BW_NO_FUSED_SELECT") != nullptr;
  {
    const char* fl = getenv("BW_MEGA_FLAGS");
    if (fl) e->mega_flags = atoi(fl);
  }
  {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess) e->num_sms = sms;
  }
  const char* impl = getenv("BW_GEMM_IMPL");
  e->simt = impl && strcmp(impl, "simt") == 0;
  *out = e;
  return 0;
}

void bw_engine_destroy(bw_engine* e) {
  if (!e) return;
  for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second);
  for (auto& kv : e->enc_graphs) cudaGraphExecDestroy(kv.second);
  for (auto& kv : e->buffers) cudaFree(kv.second.first);
  logmel_plan_destroy(e->mel_plan);
  delete e;
}

int bw_engine_set_tensor(bw_engine* e, const char* name, const void* p) {
  BW_CHECK(e && name && p, "bw_engine_set_tensor: null argument");
  BW_CHECK(!e->finalized, "bw_engine_set_tensor after finalize");
  e->tensors[name] = p;
  return 0;
}

int bw_engine_set_mel_filters(bw_engine* e, const float* bank_host) {
  BW_CHECK(e && bank_host, "bw_engine_set_mel_filters: null argument");
  logmel_plan_destroy(e->mel_plan);
  e->mel_plan = nullptr;
  return logmel_plan_create_from_bank(&e->mel_plan, bank_host, e->cfg.n_mels);
}

int bw_engine_set_alignment_heads(bw_engine* e, const int32_t* pairs, int32_t n) {
  BW_CHECK(e && (pairs || n == 0), "bw_engine_set_alignment_heads: null argument");
  BW_CHECK(n == e->cfg.n_align_heads, "alignment heads: got %d pairs, config says %d", n, e->cfg.n_align_heads);
  e->align_pairs.assign(pairs, pairs + 2 * n);
  return 0;
}

int bw_engine_finalize(bw_engine* e) {
  BW_CHECK(e && !e->finalized, "bw_engine_finalize: bad engine");
  const bw_config& c = e->cfg;
  const int D = e->D, S = e->S, F = e->F, H = e->H, V = e->V, Tmax = e->Tmax, A = c.max_audios, Qm = c.max_audios * c.max_beams;
#define NEED(T, field, name) if (int rc = need<T>(e, name, &field)) return rc;
  NEED(bf16, e->conv1_w, "enc.conv1.w") NEED(float, e->conv1_b, "enc.conv1.b")
  NEED(bf16, e->conv2_w, "enc.conv2.w") NEED(float, e->conv2_b, "enc.conv2.b")
  NEED(float, e->enc_pos, "enc.pos") NEED(float, e->enc_lnf_g, "enc.lnf.g") NEED(float, e->enc_lnf_b, "enc.lnf.b")
  NEED(bf16, e->embed, "dec.embed") NEED(float, e->dec_pos, "dec.pos")
  NEED(float, e->dec_lnf_g, "dec.lnf.g") NEED(float, e->dec_lnf_b, "dec.lnf.b")
  e->enc.resize(c.enc_layers);
  for (int i = 0; i < c.enc_layers; ++i) {
    const std::string p = "enc." + std::to_string(i) + ".";
    EncLayer& L = e->enc[i];
    NEED(float, L.ln1g, p + "ln1.g") NEED(float, L.ln1b, p + "ln1.b") NEED(bf16, L.wqkv, p + "wqkv") NEED(float, L.bqkv, p + "bqkv")
    NEED(bf16, L.wo, p + "wo") NEED(float, L.bo, p + "bo") NEED(float, L.ln2g, p + "ln2.g") NEED(float, L.ln2b, p + "ln2.b")
    NEED(bf16, L.w1, p + "w1") NEED(float, L.b1, p + "b1") NEED(bf16, L.w2, p + "w2") NEED(float, L.b2, p + "b2")
  }
  e->dec.resize(c.dec_layers);
  for (int i = 0; i < c.dec_layers; ++i) {
    const std::string p = "dec." + std::to_string(i) + ".";
    DecLayer& L = e->dec[i];
    NEED(float, L.ln1g, p + "ln1.g") NEED(float, L.ln1b, p + "ln1.b") NEED(bf16, L.wqkv, p + "wqkv") NEED(float, L.bqkv, p + "bqkv")
    NEED(bf16, L.wo, p + "wo") NEED(float, L.bo, p + "bo") NEED(float, L.ln2g, p + "ln2.g") NEED(float, L.ln2b, p + "ln2.b")
    NEED(bf16, L.xwq, p + "xwq") NEED(float, L.xbq, p + "xbq") NEED(bf16, L.xwk, p + "xwk") NEED(bf16, L.xwv, p + "xwv")
    NEED(float, L.xbv, p + "xbv") NEED(bf16, L.xwo, p + "xwo") NEED(float, L.xbo, p + "xbo")
    NEED(float, L.ln3g, p + "ln3.g") NEED(float, L.ln3b, p + "ln3.b")
    NEED(bf16, L.w1, p + "w1") NEED(float, L.b1, p + "b1") NEED(bf16, L.w2, p + "w2") NEED(float, L.b2, p + "b2")
  }
#undef NEED
  BW_CHECK(e->mel_plan != nullptr, "mel filter bank not set (bw_engine_set_mel_filters)");
  const size_t BS = (size_t)A * S;
  if (dalloc(e, "mel_tm", &e->mel_tm, (size_t)A * (F + 2) * c.n_mels)) return -1;
  if (dalloc(e, "mel_scratch", &e->mel_scratch, (size_t)A * F * c.n_mels)) return -1;
  if (dalloc(e, "mel_max", &e->mel_max, (size_t)A)) return -1;
  if (dalloc(e, "h1", &e->h1, (size_t)A * (F + 2) * D)) return -1;
  if (dalloc(e, "x_enc", &e->x_enc, BS * D)) return -1;
  if (dalloc(e, "xn", &e->xn, BS * D)) return -1;
  if (dalloc(e, "qkv", &e->qkv, BS * 3 * D)) return -1;
  if (dalloc(e, "vt", &e->vt, (size_t)A * H * 64 * e->Spad)) return -1;
  if (dalloc(e, "ao", &e->ao, BS * D)) return -1;
  if (dalloc(e, "hbuf", &e->hbuf, BS * c.ffn)) return -1;
  if (dalloc(e, "enc_out", &e->enc_out, BS * D)) return -1;
  if (dalloc(e, "cross_k", &e->cross_k, (size_t)c.dec_layers * A * H * S * 64, false)) return -1;
  if (dalloc(e, "cross_v", &e->cross_v, (size_t)c.dec_layers * A * H * S * 64, false)) return -1;
  if (dalloc(e, "self_k", &e->self_k, (size_t)c.dec_layers * Qm * Tmax * D, false)) return -1;
  if (dalloc(e, "self_v", &e->self_v, (size_t)c.dec_layers * Qm * Tmax * D, false)) return -1;
  if (dalloc(e, "tokens", &e->tokens, (size_t)Qm * Tmax)) return -1;
  if (dalloc(e, "tokens_tmp", &e->reorder_tmp, (size_t)Qm * Tmax + 2 * Qm)) return -1;
  if (dalloc(e, "finished", &e->finished, (size_t)Qm)) return -1;
  if (dalloc(e, "pos", &e->pos, 1)) return -1;
  if (dalloc(e, "anc", &e->anc, (size_t)Qm * Tmax)) return -1;
  if (dalloc(e, "anc_tmp", &e->anc_tmp, (size_t)Qm * Tmax)) return -1;
  if (dalloc(e, "done_ctr", &e->done_ctr, 1)) return -1;
  if (dalloc(e, "mega_bar", &e->mega_bar, 1024)) return -1;  // arrival counter [0] + per-CTA flags [32, 32 + SMs)
  {
    const char* tr = getenv("BW_MEGA_TRACE");
    if (tr && tr[0] == '1' && dalloc(e, "mega_trace", &e->mega_trace, (size_t)e->num_sms * MEGA_TRACE_N * 6)) return -1;
  }
  if (dalloc(e, "xcounters", &e->xcounters, (size_t)A * H)) return -1;
  if (dalloc(e, "sel_ctr", &e->sel_ctr, 1)) return -1;
  if (dalloc(e, "sel_best", &e->sel_best, (size_t)Qm)) return -1;
  if (dalloc(e, "sup_bits", &e->sup_bits, (size_t)(V + 31) / 32)) return -1;
  if (dalloc(e, "bsup_bits", &e->bsup_bits, (size_t)(V + 31) / 32)) return -1;
  if (dalloc(e, "dx", &e->dx, (size_t)Qm * D)) return -1;
  if (dalloc(e, "dqkv", &e->dqkv, (size_t)Qm * 3 * D)) return -1;
  if (dalloc(e, "dattn", &e->dattn, (size_t)Qm * D)) return -1;
  if (dalloc(e, "dq", &e->dq, (size_t)Qm * D)) return -1;
  if (dalloc(e, "dh", &e->dh, (size_t)Qm * c.ffn)) return -1;
  if (dalloc(e, "logits", &e->logits, (size_t)Qm * e->Vp)) return -1;
  {
    const size_t qpad = ((size_t)Qm + 127) / 128 * 128;  // whole 128-row TMA boxes
    if (dalloc(e, "dbn", &e->dbn, qpad * D)) return -1;
    if (dalloc(e, "dba", &e->dba, qpad * D)) return -1;
    if (dalloc(e, "dbh", &e->dbh, qpad * c.ffn)) return -1;
    if (dalloc(e, "dpart", &e->dpart, (size_t)Qm * DPART_PER_ROW)) return -1;
  }
  if (dalloc(e, "lse", &e->lse, (size_t)Qm)) return -1;
  if (dalloc(e, "run_scores", &e->run_scores, (size_t)Qm)) return -1;
  if (dalloc(e, "cand_scores", &e->cand_scores, (size_t)Qm * 16)) return -1;
  if (dalloc(e, "cand_tokens", &e->cand_tokens, (size_t)Qm * 16)) return -1;
  if (dalloc(e, "part_o", &e->part_o, (size_t)A * H * XSPLIT * c.max_beams * 64)) return -1;
  if (dalloc(e, "part_ml", &e->part_ml, (size_t)A * H * XSPLIT * c.max_beams * 2)) return -1;
  if (dalloc(e, "head_slots", &e->head_slots, (size_t)c.dec_layers * H)) return -1;
  {
    std::vector<int> hs((size_t)c.dec_layers * H, -1);
    for (int i = 0; i < c.n_align_heads && 2 * i + 1 < (int)e->align_pairs.size(); ++i) {
      const int l = e->align_pairs[2 * i], h = e->align_pairs[2 * i + 1];
      BW_CHECK(l >= 0 && l < c.dec_layers && h >= 0 && h < H, "alignment head (%d,%d) out of range", l, h);
      hs[(size_t)l * H + h] = i;
    }
    BW_CUDA_OK(cudaMemcpy(e->head_slots, hs.data(), hs.size() * sizeof(int), cudaMemcpyHostToDevice));
  }
  if (c.n_align_heads > 0) {
    BW_CHECK((int)e->align_pairs.size() == 2 * c.n_align_heads, "alignment heads not set");
    if (dalloc(e, "align", &e->align, (size_t)Qm * c.n_align_heads * c.max_align_steps * S)) return -1;  // one block per sequence slot
    if (dalloc(e, "ts_map", &e->ts_map, (size_t)A * c.max_align_steps)) return -1;
    if (dalloc(e, "ts_work", &e->ts_work, (size_t)A * word_timestamps_work_floats(c.n_align_heads, c.max_align_steps, S), false)) return -1;
    if (dalloc(e, "ts_out", &e->ts_out, (size_t)A * (c.max_align_steps + 8))) return -1;
    if (dalloc(e, "ts_items", &e->ts_items, (size_t)A * 3)) return -1;
  }
  e->finalized = true;
  return 0;
}

int bw_engine_buffer(bw_engine* e, const char* name, void** p, size_t* bytes) {
  BW_CHECK(e && name && p, "bw_engine_buffer: null argument");
  auto it = e->buffers.find(name);
  BW_CHECK(it != e->buffers.end(), "bw_engine_buffer: unknown buffer '%s'", name);
  *p = it->second.first;
  if (bytes) *bytes = it->second.second;
  return 0;
}

int bw_logmel(bw_engine* e, const float* pcm, int32_t B, int32_t n_samples, float* mel_f32_out, void* stream) {
  BW_CHECK(e && e->finalized && pcm, "bw_logmel: bad arguments");
  BW_CHECK(B >= 1 && B <= e->cfg.max_audios, "bw_logmel: B=%d outside 1..%d", B, e->cfg.max_audios);
  BW_CHECK(n_samples == e->F * 160, "bw_logmel: n_samples=%d, expected %d for this chunk length", n_samples, e->F * 160);
  return logmel(static_cast<cudaStream_t>(stream), e->mel_plan, pcm, B, n_samples, e->F, e->mel_tm, mel_f32_out, e->mel_scratch, e->mel_max);
}

int bw_set_mel(bw_engine* e, const float* mel, int32_t B, void* stream) {
  BW_CHECK(e && e->finalized && mel, "bw_set_mel: bad arguments");
  BW_CHECK(B >= 1 && B <= e->cfg.max_audios, "bw_set_mel: B=%d outside 1..%d", B, e->cfg.max_audios);
  dim3 grid((e->F + 31) / 32, (e->cfg.n_mels + 31) / 32, B);
  mel_to_tm_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(mel, e->mel_tm, e->cfg.n_mels, e->F);
  BW_CUDA_OK(cudaGetLastError());
  return 0;
}

// The encoder pass: ~300 kernels (7 per layer + 64 cross-K/V projections).  At B = 1 they are 5-30 us each and the host's launch cost
// (two cuTensorMapEncode + cudaLaunchKernelEx per GEMM) and the gaps between them are a third of the pass, so from the second call
// with a given batch size on the pass is replayed as ONE CUDA graph whose kernel nodes are chained by programmatic dependent launch
// (the first call runs on the stream: it also sets the kernels' function attributes, which must not happen under capture).
static int encode_pdl(bw_engine* e, int B, cudaStream_t st) {
  if (!e->enc_pdl) return encode_impl(e, B, st);
  if (g_pdl_enabled < 0) {
    const char* ev = getenv("BW_PDL");
    g_pdl_enabled = (ev && ev[0] == '0') ? 0 : 1;
  }
  g_pdl = g_pdl_enabled;
  const int rc = encode_impl(e, B, st);
  g_pdl = 0;
  return rc;
}

int bw_encode(bw_engine* e, int32_t B, void* stream) {
  BW_CHECK(e && e->finalized, "bw_encode: engine not finalized");
  BW_CHECK(B >= 1 && B <= e->cfg.max_audios, "bw_encode: B=%d outside 1..%d", B, e->cfg.max_audios);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (e->no_graph || !e->enc_graph || e->simt) return encode_pdl(e, B, st);
  auto it = e->enc_graphs.find(B);
  if (it == e->enc_graphs.end()) {
    if (e->enc_calls[B]++ == 0) return encode_pdl(e, B, st);
    cudaStream_t cs;
    BW_CUDA_OK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    for (int attempt = 0; attempt < 2 && !exec; ++attempt) {
      BW_CUDA_OK(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
      const int rc = encode_pdl(e, B, cs);
      cudaError_t ce = cudaStreamEndCapture(cs, &graph);
      if (rc == 0 && ce == cudaSuccess) ce = cudaGraphInstantiate(&exec, graph, 0);
      if (graph) cudaGraphDestroy(graph);
      graph = nullptr;
      if (rc == 0 && ce == cudaSuccess) break;
      exec = nullptr;
      cudaGetLastError();
      if (attempt == 0 && g_pdl_enabled == 1) {
        g_pdl_enabled = 0;  // a driver that cannot capture programmatic launches: plain edges
        continue;
      }
      break;
    }
    cudaStreamDestroy(cs);
    if (!exec) {  // no graph on this driver: stream launches from now on
      e->enc_graph = false;
      return encode_pdl(e, B, st);
    }
    it = e->enc_graphs.emplace(B, exec).first;
  }
  BW_CUDA_OK(cudaGraphLaunch(it->second, st));
  return 0;
}

int bw_decode_begin(bw_engine* e, int32_t A, int32_t G, const int32_t* prompt, int32_t plen, const bw_decode_opts* opts, void* stream) {
  BW_CHECK(e && e->finalized && prompt && opts, "bw_decode_begin: bad arguments");
  BW_CHECK(A >= 1 && A <= e->cfg.max_audios && G >= 1 && G <= e->cfg.max_beams, "bw_decode_begin: A=%d G=%d out of range", A, G);
  BW_CHECK(plen >= 1 && plen <= e->Tmax, "bw_decode_begin: prompt_len=%d out of range", plen);
  BW_CHECK(opts->begin_index >= 1 && opts->begin_index <= plen, "bw_decode_begin: begin_index=%d outside 1..prompt_len", opts->begin_index);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  e->A = A; e->G = G; e->Q = A * G; e->opts = *opts; e->use_anc = G > 1;
  const int Q = e->Q, Tmax = e->Tmax, V = e->V;
  std::vector<int> tok((size_t)Q * Tmax, opts->pad_token);
  for (int q = 0; q < Q; ++q) memcpy(&tok[(size_t)q * Tmax], prompt + (size_t)q * plen, sizeof(int) * plen);
  BW_CUDA_OK(cudaMemcpyAsync(e->tokens, tok.data(), tok.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  std::vector<unsigned> bits((V + 31) / 32, 0u), bbits((V + 31) / 32, 0u);
  for (int i = 0; i < opts->n_suppress; ++i) {
    const int t = opts->suppress_tokens[i];
    if (t >= 0 && t < V) bits[t >> 5] |= 1u << (t & 31);
  }
  for (int i = 0; i < opts->n_begin_suppress; ++i) {
    const int t = opts->begin_suppress_tokens[i];
    if (t >= 0 && t < V) bbits[t >> 5] |= 1u << (t & 31);
  }
  BW_CUDA_OK(cudaMemcpyAsync(e->sup_bits, bits.data(), bits.size() * sizeof(unsigned), cudaMemcpyHostToDevice, st));
  BW_CUDA_OK(cudaMemcpyAsync(e->bsup_bits, bbits.data(), bbits.size() * sizeof(unsigned), cudaMemcpyHostToDevice, st));
  BW_CUDA_OK(cudaMemsetAsync(e->finished, 0, sizeof(int) * Q, st));
  BW_CUDA_OK(cudaMemsetAsync(e->pos, 0, sizeof(int), st));
  BW_CUDA_OK(cudaMemsetAsync(e->done_ctr, 0, sizeof(unsigned), st));
  BW_CUDA_OK(cudaMemsetAsync(e->xcounters, 0, sizeof(unsigned) * e->cfg.max_audios * e->H, st));
  iota_anc_kernel<<<(Q * Tmax + 255) / 256, 256, 0, st>>>(e->anc, Q, Tmax);
  BW_CUDA_OK(cudaGetLastError());
  BW_CUDA_OK(cudaStreamSynchronize(st));  // host staging vectors go out of scope
  e->cur_graph = nullptr;
  if (!e->no_graph) {
    GraphKey key{A, G, opts->begin_index, opts->timestamp_rules * 4 + (opts->max_initial_timestamp_index + 1) * 8, opts->record_alignment,
                 e->mega_flags * 4 + (e->no_mega ? 1 : 0) + (e->no_fused_select ? 2 : 0),
                 opts->eos_token, opts->pad_token, opts->timestamp_begin, opts->no_timestamps_token};
    auto it = e->graphs.find(key);
    if (it == e->graphs.end()) {
      cudaStream_t cs;
      BW_CUDA_OK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
      cudaGraph_t graph = nullptr;
      for (int attempt = 0; attempt < 2; ++attempt) {
        BW_CUDA_OK(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
        const int rc = step_impl(e, cs);
        const cudaError_t ce = cudaStreamEndCapture(cs, &graph);
        if (rc == 0 && ce == cudaSuccess) break;
        if (graph) cudaGraphDestroy(graph);
        graph = nullptr;
        cudaGetLastError();
        if (attempt == 0 && (g_mega_coop == 1 || g_pdl_enabled == 1)) {
          // a driver that cannot capture a cooperative / programmatic launch: plain launches, as in round 1
          g_mega_coop = 0;
          g_pdl_enabled = 0;
          continue;
        }
        cudaStreamDestroy(cs);
        if (rc == 0) set_error("cudaStreamEndCapture: %s", cudaGetErrorString(ce));
        return -1;
      }
      int n_kernel_nodes = 0;
      {
        size_t nn = 0;
        if (cudaGraphGetNodes(graph, nullptr, &nn) == cudaSuccess && nn > 0) {
          std::vector<cudaGraphNode_t> nodes(nn);
          if (cudaGraphGetNodes(graph, nodes.data(), &nn) == cudaSuccess) {
            for (size_t i = 0; i < nn; ++i) {
              cudaGraphNodeType ty;
              if (cudaGraphNodeGetType(nodes[i], &ty) == cudaSuccess && ty == cudaGraphNodeTypeKernel) ++n_kernel_nodes;
            }
          }
        }
      }
      cudaGraphExec_t exec = nullptr;
      BW_CUDA_OK(cudaGraphInstantiate(&exec, graph, 0));
      cudaGraphDestroy(graph);
      e->graph_kernels[exec] = n_kernel_nodes;
      cudaStreamDestroy(cs);
      it = e->graphs.emplace(key, exec).first;
    }
    e->cur_graph = it->second;
  }
  return 0;
}

int bw_decode_run(bw_engine* e, int32_t n_steps, void* stream) {
  BW_CHECK(e && e->finalized && e->Q > 0, "bw_decode_run: no decode in progress");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (int i = 0; i < n_steps; ++i) {
    if (e->cur_graph) {
      BW_CUDA_OK(cudaGraphLaunch(e->cur_graph, st));
      e->step_kernel_launches += e->graph_kernels[e->cur_graph];
    } else {
      if (int rc = step_impl(e, st)) return rc;
    }
  }
  return 0;
}

long long bw_decode_kernel_launches(bw_engine* e) { return e ? e->step_kernel_launches : -1; }

int bw_decode_read(bw_engine* e, int32_t* tokens_host, int32_t* finished_host, int32_t* pos_host, void* stream) {
  BW_CHECK(e && e->finalized && e->Q > 0, "bw_decode_read: no decode in progress");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (tokens_host) BW_CUDA_OK(cudaMemcpyAsync(tokens_host, e->tokens, sizeof(int) * e->Q * e->Tmax, cudaMemcpyDeviceToHost, st));
  if (finished_host) BW_CUDA_OK(cudaMemcpyAsync(finished_host, e->finished, sizeof(int) * e->Q, cudaMemcpyDeviceToHost, st));
  if (pos_host) BW_CUDA_OK(cudaMemcpyAsync(pos_host, e->pos, sizeof(int), cudaMemcpyDeviceToHost, st));
  BW_CUDA_OK(cudaStreamSynchronize(st));
  return 0;
}

int bw_decode_reorder(bw_engine* e, const int32_t* parent_host, const int32_t* next_token_host, void* stream) {
  BW_CHECK(e && e->finalized && e->Q > 0 && parent_host && next_token_host, "bw_decode_reorder: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int Q = e->Q, Tmax = e->Tmax;
  int* d_parent = e->reorder_tmp + (size_t)e->cfg.max_audios * e->cfg.max_beams * Tmax;
  int* d_next = d_parent + Q;
  BW_CUDA_OK(cudaMemcpyAsync(d_parent, parent_host, sizeof(int) * Q, cudaMemcpyHostToDevice, st));
  BW_CUDA_OK(cudaMemcpyAsync(d_next, next_token_host, sizeof(int) * Q, cudaMemcpyHostToDevice, st));
  reorder_kernel<<<Q, 128, 0, st>>>(e->anc, e->anc_tmp, e->tokens, e->reorder_tmp, d_parent, d_next, e->pos, Tmax);
  BW_CUDA_OK(cudaGetLastError());
  BW_CUDA_OK(cudaMemcpyAsync(e->anc, e->anc_tmp, sizeof(int) * Q * Tmax, cudaMemcpyDeviceToDevice, st));
  BW_CUDA_OK(cudaMemcpyAsync(e->tokens, e->reorder_tmp, sizeof(int) * Q * Tmax, cudaMemcpyDeviceToDevice, st));
  BW_CUDA_OK(cudaStreamSynchronize(st));
  return 0;
}

int bw_decode_beam_step(bw_engine* e, const float* run_scores_host, float* cand_scores_host, int32_t* cand_tokens_host, void* stream) {
  BW_CHECK(e && e->finalized && e->Q > 0 && e->G > 1, "bw_decode_beam_step: no beam decode in progress");
  BW_CHECK(run_scores_host && cand_scores_host && cand_tokens_host, "bw_decode_beam_step: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int Q = e->Q, nc = 2 * e->G;
  BW_CUDA_OK(cudaMemcpyAsync(e->run_scores, run_scores_host, sizeof(float) * Q, cudaMemcpyHostToDevice, st));
  if (int rc = bw_decode_run(e, 1, stream)) return rc;
  BW_CUDA_OK(cudaMemcpyAsync(cand_scores_host, e->cand_scores, sizeof(float) * Q * nc, cudaMemcpyDeviceToHost, st));
  BW_CUDA_OK(cudaMemcpyAsync(cand_tokens_host, e->cand_tokens, sizeof(int) * Q * nc, cudaMemcpyDeviceToHost, st));
  BW_CUDA_OK(cudaStreamSynchronize(st));
  return 0;
}

static int word_timestamps_impl(bw_engine* e, int32_t n, const int32_t* audio, const int32_t* slot_map, int32_t map_pitch, const int32_t* n_tokens,
                                const int32_t* num_frames, double time_precision, float* out_host, int32_t out_pitch, void* stream) {
  BW_CHECK(e && e->finalized && (audio || slot_map) && n_tokens && num_frames && out_host, "bw_word_timestamps: bad arguments");
  BW_CHECK(e->cfg.n_align_heads > 0 && e->align, "bw_word_timestamps: engine built without alignment heads");
  BW_CHECK(n >= 1 && n <= e->cfg.max_audios, "bw_word_timestamps: n=%d outside 1..%d", n, e->cfg.max_audios);
  const int Tcap = e->cfg.max_align_steps, Qm = e->cfg.max_audios * e->cfg.max_beams;
  std::vector<int> items((size_t)n * 3), map;
  int maxT = 0, maxNF = 0;
  for (int i = 0; i < n; ++i) {
    BW_CHECK(n_tokens[i] >= 1 && n_tokens[i] <= Tcap, "bw_word_timestamps: n_tokens=%d outside 1..%d", n_tokens[i], Tcap);
    BW_CHECK(num_frames[i] >= 1 && num_frames[i] <= e->S, "bw_word_timestamps: num_frames=%d outside 1..%d", num_frames[i], e->S);
    BW_CHECK(out_pitch >= n_tokens[i] + 1, "bw_word_timestamps: out_pitch=%d too small for %d tokens", out_pitch, n_tokens[i]);
    if (audio) BW_CHECK(audio[i] >= 0 && audio[i] < Qm, "bw_word_timestamps: slot index out of range");
    items[3 * i] = audio ? audio[i] : 0; items[3 * i + 1] = n_tokens[i]; items[3 * i + 2] = num_frames[i];
    maxT = n_tokens[i] > maxT ? n_tokens[i] : maxT;
    maxNF = num_frames[i] > maxNF ? num_frames[i] : maxNF;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (slot_map) {
    BW_CHECK(map_pitch >= maxT, "bw_word_timestamps_gather: map_pitch=%d smaller than %d tokens", map_pitch, maxT);
    map.assign((size_t)n * Tcap, 0);
    for (int i = 0; i < n; ++i)
      for (int t = 0; t < n_tokens[i]; ++t) {
        const int sl = slot_map[(size_t)i * map_pitch + t];
        BW_CHECK(sl >= 0 && sl < Qm, "bw_word_timestamps_gather: slot %d out of range", sl);
        map[(size_t)i * Tcap + t] = sl;
      }
    BW_CUDA_OK(cudaMemcpyAsync(e->ts_map, map.data(), map.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  }
  BW_CUDA_OK(cudaMemcpyAsync(e->ts_items, items.data(), items.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  if (int rc = word_timestamps_batch_device(st, e->align, e->cfg.n_align_heads, Tcap, e->S, e->ts_items, slot_map ? e->ts_map : nullptr, Tcap, n, maxT,
                                            maxNF, time_precision, e->ts_work, e->ts_out))
    return rc;
  BW_CUDA_OK(cudaMemcpy2DAsync(out_host, (size_t)out_pitch * sizeof(float), e->ts_out, (size_t)(Tcap + 8) * sizeof(float),
                               (size_t)(maxT + 1) * sizeof(float), n, cudaMemcpyDeviceToHost, st));
  BW_CUDA_OK(cudaStreamSynchronize(st));  // the host staging vectors go out of scope; the caller reads out_host
  return 0;
}

int bw_word_timestamps_batch(bw_engine* e, int32_t n, const int32_t* audio, const int32_t* n_tokens, const int32_t* num_frames,
                             double time_precision, float* out_host, int32_t out_pitch, void* stream) {
  BW_CHECK(audio, "bw_word_timestamps_batch: null argument");
  return word_timestamps_impl(e, n, audio, nullptr, 0, n_tokens, num_frames, time_precision, out_host, out_pitch, stream);
}

int bw_word_timestamps_gather(bw_engine* e, int32_t n, const int32_t* slot_map, int32_t map_pitch, const int32_t* n_tokens,
                              const int32_t* num_frames, double time_precision, float* out_host, int32_t out_pitch, void* stream) {
  BW_CHECK(slot_map, "bw_word_timestamps_gather: null argument");
  return word_timestamps_impl(e, n, nullptr, slot_map, map_pitch, n_tokens, num_frames, time_precision, out_host, out_pitch, stream);
}

int bw_word_timestamps(bw_engine* e, int32_t audio, int32_t n_tokens, int32_t num_frames, double time_precision, float* out_host,
                       void* stream) {
  return bw_word_timestamps_batch(e, 1, &audio, &n_tokens, &num_frames, time_precision, out_host, n_tokens + 1, stream);
}

// ---- single ops -------------------------------------------------------------------------------------------------
int bw_op_gemm(const void* A, const void* W, int32_t M, int32_t N, int32_t K, const float* bias, float alpha, int32_t act,
               const float* residual, void* out, int32_t out_is_f32, int32_t impl, int32_t force_bn, void* stream) {
  BW_CHECK(A && W && out, "bw_op_gemm: null pointer");
  GemmEpi ep = plainEpi(M, N);
  ep.bias = bias; ep.alpha = alpha; ep.act = act; ep.residual = residual;
  if (out_is_f32) ep.out_f32 = static_cast<float*>(out);
  else ep.out_bf16 = static_cast<bf16*>(out);
  const GemmA a = plainA(static_cast<const bf16*>(A), M, K);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (impl == 1) return gemm_simt(st, a, static_cast<const bf16*>(W), 1, M, N, K, ep);
  if (impl == 2) return gemm_tc2(st, static_cast<const bf16*>(A), static_cast<const bf16*>(W), M, N, K, M, ep, force_bn);
  return gemm_tc(st, a, static_cast<const bf16*>(W), 1, M, N, K, ep, force_bn);
}

int bw_op_gemm_splitk(const void* A, const void* W, int32_t M, int32_t N, int32_t K, int32_t n_valid, int32_t ksplit, int32_t force_bn,
                      float* out_partials, int32_t* ksplit_used, void* stream) {
  BW_CHECK(A && W && out_partials && ksplit_used, "bw_op_gemm_splitk: null pointer");
  GemmEpi ep = plainEpi(M, N);
  ep.out_f32 = out_partials;
  ep.n_valid = (n_valid > 0 && n_valid < N) ? n_valid : 0;
  *ksplit_used = gemm_tc_ksplit(K, ksplit);
  return gemm_tc_split(static_cast<cudaStream_t>(stream), plainA(static_cast<const bf16*>(A), M, K), static_cast<const bf16*>(W), 1, M, N, K, ep,
                       force_bn, ksplit, (long long)M * N);
}

int bw_op_gemm_dec(const void* X, const void* W, int32_t Q, int32_t N, int32_t K, int32_t n_valid, int32_t want_split, float* out_partials,
                   int32_t* ksplit_used, void* stream) {
  BW_CHECK(X && W && out_partials && ksplit_used, "bw_op_gemm_dec: null pointer");
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const DecGemmPlan pl = gemm_dec_plan(Q, N, K, sms, want_split != 0);
  *ksplit_used = pl.ksplit;
  GemmEpi ep;
  ep.out_f32 = out_partials; ep.row_stride = N;
  return gemm_dec(static_cast<cudaStream_t>(stream), static_cast<const bf16*>(X), static_cast<const bf16*>(W), Q, N, K, n_valid, ep, pl, (long long)Q * N);
}

int bw_op_gelu_bias(const float* partials, int32_t nsplit, const float* bias, void* h_bf16, int32_t Q, int32_t N, void* stream) {
  BW_CHECK(partials && bias && h_bf16 && nsplit >= 1, "bw_op_gelu_bias: bad arguments");
  return launch_gelu_bias(static_cast<cudaStream_t>(stream), partials, nsplit, (long long)Q * N, bias, static_cast<bf16*>(h_bf16), Q, N);
}

int bw_op_resid_ln(float* x, const float* partials, int32_t nsplit, const float* bias, const float* ln_g, const float* ln_b, void* y_bf16,
                   int32_t Q, int32_t D, void* stream) {
  BW_CHECK(x && (nsplit == 0 || partials) && (!y_bf16 || (ln_g && ln_b)), "bw_op_resid_ln: null pointer");
  return launch_resid_ln(static_cast<cudaStream_t>(stream), x, partials, nsplit, (long long)Q * D, bias, ln_g, ln_b, static_cast<bf16*>(y_bf16), Q, D);
}

int bw_op_attn_enc(const void* qkv, void* vt_scratch, void* out, int32_t B, int32_t S, int32_t H, int32_t impl, void* stream) {
  BW_CHECK(qkv && out, "bw_op_attn_enc: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (impl == 1) return attn_enc_simt(st, static_cast<const bf16*>(qkv), static_cast<bf16*>(out), B, S, H);
  BW_CHECK(vt_scratch, "bw_op_attn_enc: vt_scratch required for the tcgen05 path");
  const int Spad = (S + 7) / 8 * 8;
  if (impl == 3) return attn_enc_tc2(st, static_cast<const bf16*>(qkv), nullptr, static_cast<bf16*>(out), B, S, Spad, H);
  if (int rc = transpose_v(st, static_cast<const bf16*>(qkv), static_cast<bf16*>(vt_scratch), B, S, Spad, H)) return rc;
  if (impl == 2) return attn_enc_tc2(st, static_cast<const bf16*>(qkv), static_cast<const bf16*>(vt_scratch), static_cast<bf16*>(out), B, S, Spad, H);
  return attn_enc_tc(st, static_cast<const bf16*>(qkv), static_cast<const bf16*>(vt_scratch), static_cast<bf16*>(out), B, S, Spad, H);
}

int bw_op_layernorm(const float* x, const float* g, const float* b, void* out, int32_t out_is_f32, int32_t rows, int32_t D, void* stream) {
  BW_CHECK(x && g && b && out, "bw_op_layernorm: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return out_is_f32 ? layernorm_f32(st, x, g, b, static_cast<float*>(out), rows, D)
                    : layernorm_bf16(st, x, g, b, static_cast<bf16*>(out), rows, D);
}

int bw_op_gemv(const float* x, const float* ln_g, const float* ln_b, const void* W, int32_t M, int32_t N, int32_t K, const float* bias,
               float alpha, int32_t act, const float* residual, float* out, void* stream) {
  BW_CHECK(x && W && out, "bw_op_gemv: null pointer");
  GemvArgs g;
  g.x = x; g.ldx = K; g.ln_g = ln_g; g.ln_b = ln_b; g.W = static_cast<const bf16*>(W); g.N = N; g.K = K; g.M = M;
  g.bias = bias; g.alpha = alpha; g.alpha_cols = (alpha != 1.0f) ? N : 0; g.act = act; g.residual = residual; g.out = out; g.ldo = N;
  return launch_gemv(static_cast<cudaStream_t>(stream), g);
}

int bw_op_self_attn(const float* qkv, int32_t nsplit, const float* qkv_bias, float q_alpha, void* kc, void* vc, const int32_t* anc,
                    int32_t append, void* out, int32_t out_is_f32, const int32_t* pos_dev, int32_t Q, int32_t H, int32_t Tmax,
                    int32_t elem_dtype, void* stream) {
  BW_CHECK(qkv && kc && vc && out && pos_dev, "bw_op_self_attn: null pointer");
  BW_CHECK(Q >= 1 && H >= 1 && Tmax >= 1 && nsplit >= 0, "bw_op_self_attn: Q=%d H=%d Tmax=%d nsplit=%d out of range", Q, H, Tmax, nsplit);
  BW_CHECK(elem_dtype == 0 || elem_dtype == 1, "bw_op_self_attn: elem_dtype=%d must be 0 (bf16) or 1 (fp16)", elem_dtype);
  const int D = H * 64;
  SelfAttnArgs s;
  s.qkv = qkv; s.nsplit = nsplit; s.split_stride = (long long)Q * 3 * D; s.qkv_bias = qkv_bias; s.q_alpha = q_alpha;
  s.kc = static_cast<const bf16*>(kc); s.vc = static_cast<const bf16*>(vc); s.anc = anc; s.pos = pos_dev;
  if (append) { s.kc_w = static_cast<bf16*>(kc); s.vc_w = static_cast<bf16*>(vc); }
  if (out_is_f32) s.out = static_cast<float*>(out);
  else s.out_bf16 = static_cast<bf16*>(out);
  s.H = H; s.D = D; s.Tmax = Tmax;
  return launch_self_attn(static_cast<cudaStream_t>(stream), s, Q);
}

int bw_op_cross_attn(const float* q, int32_t nsplit, const float* q_bias, float q_alpha, const void* kc, const void* vc,
                     void* out, int32_t out_is_f32, float* part_o, float* part_ml, uint32_t* counters, int32_t A, int32_t G,
                     int32_t H, int32_t S, float* align, const int32_t* head_slots, int32_t Ha, int32_t Tcap, int32_t step_base,
                     const int32_t* pos_dev, int32_t impl, int32_t elem_dtype, void* stream) {
  BW_CHECK(q && kc && vc && out, "bw_op_cross_attn: null pointer");
  BW_CHECK(impl == 2 || (part_o && part_ml && counters), "bw_op_cross_attn: the split kernel needs part_o, part_ml and counters");
  BW_CHECK(!align || (head_slots && pos_dev && Ha >= 1 && Tcap >= 1), "bw_op_cross_attn: align needs head_slots, pos_dev, Ha and Tcap");
  BW_CHECK(A >= 1 && H >= 1 && S >= 1 && nsplit >= 0, "bw_op_cross_attn: A=%d H=%d S=%d nsplit=%d out of range", A, H, S, nsplit);
  BW_CHECK(elem_dtype == 0 || elem_dtype == 1, "bw_op_cross_attn: elem_dtype=%d must be 0 (bf16) or 1 (fp16)", elem_dtype);
  CrossAttnArgs c;
  c.q = q; c.nsplit = nsplit; c.split_stride = (long long)A * G * H * 64; c.q_bias = q_bias; c.q_alpha = q_alpha;
  c.kc = static_cast<const bf16*>(kc); c.vc = static_cast<const bf16*>(vc);
  if (out_is_f32) c.out = static_cast<float*>(out);
  else c.out_bf16 = static_cast<bf16*>(out);
  c.part_o = part_o; c.part_ml = part_ml; c.counters = counters;
  c.S = S; c.H = H; c.D = H * 64; c.G = G; c.pos = pos_dev;
  c.align = align; c.head_slots = head_slots; c.Ha = Ha; c.Tcap = Tcap; c.step_base = step_base;
  return launch_cross_attn(static_cast<cudaStream_t>(stream), c, A, impl);
}

}  // extern "C"
