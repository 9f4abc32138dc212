// The HBM-streaming kernels of a decoder step (q_len = 1): GEMV with fused LayerNorm / epilogues, causal self-attention
// over the token KV cache, cross-attention over the resident encoder K/V.
//
// At batch 1 every one of these moves only 3-13 MB, i.e. ~20-90 KB per SM: they are bound by DRAM *latency*, not
// bandwidth, unless every byte a CTA needs is requested up front.  So each kernel issues ALL of its 16-byte weight / KV
// loads into registers first (one DRAM round trip), overlaps the x staging + LayerNorm prologue with them, and only
// then computes.  (First version looped load->use with 4-8 loads in flight: 3.0 ms per step, 10% of the HBM roofline;
// see profiles/.)
#include <math.h>

#include "decode.cuh"
#include "kernels.h"

namespace BW_NS {

namespace {

constexpr int GEMV_THREADS = 256;
constexpr int GEMV_WARPS = GEMV_THREADS / 32;

__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  float2 t;
  t = unpack_bf16(u.x); f[0] = t.x; f[1] = t.y;
  t = unpack_bf16(u.y); f[2] = t.x; f[3] = t.y;
  t = unpack_bf16(u.z); f[4] = t.x; f[5] = t.y;
  t = unpack_bf16(u.w); f[6] = t.x; f[7] = t.y;
}

// 16-byte async copy global -> shared (LDGSTS): issued up front at no register cost; ptxas cannot sink it the way it
// sinks ld.global.nc, which is what serialised the K and V fetches of the attention kernels into two DRAM round trips
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// 8 consecutive values of a row that may be stored as nsplit raw split-K partial sums ([split][row][col], split_stride apart):
// summed in split order (deterministic), + bias, * alpha.  The loads of four splits are issued together: a dependent
// load -> add -> load chain costs one L2 round trip per split (96 us for the self-attention kernel at Q = 64: profiles/r2c).
__device__ __forceinline__ void split_sum8(const float* __restrict__ p, long long idx, int nsplit, long long split_stride,
                                           const float* __restrict__ bias, int bias_idx, float alpha, float (&o)[8]) {
  float4 a0 = *reinterpret_cast<const float4*>(p + idx), a1 = *reinterpret_cast<const float4*>(p + idx + 4);
  if (nsplit > 0) {
    int s = 1;
    for (; s + 3 < nsplit; s += 4) {
      float4 b0[4], b1[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        b0[u] = *reinterpret_cast<const float4*>(p + (long long)(s + u) * split_stride + idx);
        b1[u] = *reinterpret_cast<const float4*>(p + (long long)(s + u) * split_stride + idx + 4);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        a0.x += b0[u].x; a0.y += b0[u].y; a0.z += b0[u].z; a0.w += b0[u].w;
        a1.x += b1[u].x; a1.y += b1[u].y; a1.z += b1[u].z; a1.w += b1[u].w;
      }
    }
    for (; s < nsplit; ++s) {
      const float4 b0 = *reinterpret_cast<const float4*>(p + (long long)s * split_stride + idx);
      const float4 b1 = *reinterpret_cast<const float4*>(p + (long long)s * split_stride + idx + 4);
      a0.x += b0.x; a0.y += b0.y; a0.z += b0.z; a0.w += b0.w;
      a1.x += b1.x; a1.y += b1.y; a1.z += b1.z; a1.w += b1.w;
    }
    if (bias) {
      const float4 c0 = *reinterpret_cast<const float4*>(bias + bias_idx), c1 = *reinterpret_cast<const float4*>(bias + bias_idx + 4);
      a0.x += c0.x; a0.y += c0.y; a0.z += c0.z; a0.w += c0.w;
      a1.x += c1.x; a1.y += c1.y; a1.z += c1.z; a1.w += c1.w;
    }
    a0.x *= alpha; a0.y *= alpha; a0.z *= alpha; a0.w *= alpha;
    a1.x *= alpha; a1.y *= alpha; a1.z *= alpha; a1.w *= alpha;
  }
  o[0] = a0.x; o[1] = a0.y; o[2] = a0.z; o[3] = a0.w; o[4] = a1.x; o[5] = a1.y; o[6] = a1.z; o[7] = a1.w;
}

template <int NC, int R>
struct WRegs {
  uint4 w[R][NC];
};

// lane l holds elements [l*8 + i*256, +8) of each row, i < NC  (512 contiguous bytes per warp-load: fully coalesced)
template <int NC, int R>
__device__ __forceinline__ void load_rows(WRegs<NC, R>& wr, const bf16* __restrict__ W, int K, int n, int n_end, int lane) {
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int row = min(n + r, n_end - 1);  // clamp: a duplicate row whose result is discarded
    const bf16* wp = W + (long long)row * K;
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      const int k = lane * 8 + i * 256;
      wr.w[r][i] = (k < K) ? ld_nc_u4(wp + k) : make_uint4(0u, 0u, 0u, 0u);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// out[m, n] = epi( LN?(x[m, :]) . W[n, :] ), m < MB <= 8.  NC = ceil(K / 256) bound, R rows per warp in flight.
// ------------------------------------------------------------------------------------------------
template <int MB, int NC, int R, bool PIPE>
__global__ void __launch_bounds__(GEMV_THREADS) gemv_kernel(const GemvArgs a, const int rows_per_warp) {
  extern __shared__ float xs[];  // [MB][K]
  __shared__ float red[GEMV_WARPS][MB];
  __shared__ float stat[2][MB];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int K = a.K;
  const int gw = blockIdx.x * GEMV_WARPS + warp;
  const int n_begin = gw * rows_per_warp;
  const int n_end = min(a.N, n_begin + rows_per_warp);

  // 1) weight rows of the first pass: requested before anything else so the DRAM latency hides the prologue
  WRegs<NC, R> cur;
  if (n_begin < n_end) load_rows<NC, R>(cur, a.W, K, n_begin, n_end, lane);

  // 2) for every chunk of MB rows of x: stage (+ LayerNorm: two-pass, biased variance, eps 1e-5 like torch.nn.LayerNorm),
  //    then all of this warp's weight rows against the chunk.  M > MB re-uses the weights already in registers, so a
  //    batch streams each weight row from HBM once per launch instead of once per 8 sequences.
  const int pos = a.pos ? *a.pos : 0;
  const bool single_pass = (n_begin + R >= n_end);
  for (int m0 = 0; m0 < a.M; m0 += MB) {
    const int mrows = min(MB, a.M - m0);
    __syncthreads();  // previous chunk's readers are done with xs
    for (int i = threadIdx.x; i < MB * K; i += GEMV_THREADS) {
      const int m = i / K, k = i - m * K;
      xs[i] = (m < mrows) ? a.x[(long long)(m0 + m) * a.ldx + k] : 0.f;
    }
    __syncthreads();
    if (a.ln_g) {
      float part[MB];
#pragma unroll
      for (int m = 0; m < MB; ++m) part[m] = 0.f;
      for (int k = threadIdx.x; k < K; k += GEMV_THREADS) {
#pragma unroll
        for (int m = 0; m < MB; ++m) part[m] += xs[m * K + k];
      }
#pragma unroll
      for (int m = 0; m < MB; ++m) {
        const float s = warp_sum(part[m]);
        if (lane == 0) red[warp][m] = s;
      }
      __syncthreads();
      if (threadIdx.x < MB) {
        float s = 0.f;
        for (int w = 0; w < GEMV_WARPS; ++w) s += red[w][threadIdx.x];
        stat[0][threadIdx.x] = s / (float)K;
      }
      __syncthreads();
#pragma unroll
      for (int m = 0; m < MB; ++m) part[m] = 0.f;
      for (int k = threadIdx.x; k < K; k += GEMV_THREADS) {
#pragma unroll
        for (int m = 0; m < MB; ++m) {
          const float d = xs[m * K + k] - stat[0][m];
          part[m] = fmaf(d, d, part[m]);
        }
      }
#pragma unroll
      for (int m = 0; m < MB; ++m) {
        const float s = warp_sum(part[m]);
        if (lane == 0) red[warp][m] = s;
      }
      __syncthreads();
      if (threadIdx.x < MB) {
        float s = 0.f;
        for (int w = 0; w < GEMV_WARPS; ++w) s += red[w][threadIdx.x];
        stat[1][threadIdx.x] = rsqrtf(s / (float)K + 1e-5f);
      }
      __syncthreads();
      for (int k = threadIdx.x; k < K; k += GEMV_THREADS) {
        const float g = a.ln_g[k], bb = a.ln_b[k];
#pragma unroll
        for (int m = 0; m < MB; ++m) xs[m * K + k] = (xs[m * K + k] - stat[0][m]) * stat[1][m] * g + bb;
      }
      __syncthreads();
    }
    // (multi-pass launches -- the LM head -- are only issued with M <= MB, so `cur` is reloaded per chunk only then)
    if (m0 > 0 && !single_pass && n_begin < n_end) load_rows<NC, R>(cur, a.W, K, n_begin, n_end, lane);
    for (int n = n_begin; n < n_end; n += R) {
      WRegs<NC, R> nxt;
      const bool has_next = (n + R) < n_end;
      if (PIPE && has_next) load_rows<NC, R>(nxt, a.W, K, n + R, n_end, lane);
      float acc[R][MB];
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int m = 0; m < MB; ++m) acc[r][m] = 0.f;
#pragma unroll
      for (int i = 0; i < NC; ++i) {
        const int k = lane * 8 + i * 256;
        if (k < K) {
          float wf[R][8];
#pragma unroll
          for (int r = 0; r < R; ++r) unpack8(cur.w[r][i], wf[r]);
#pragma unroll
          for (int m = 0; m < MB; ++m) {
            const float4 xa = *reinterpret_cast<const float4*>(&xs[m * K + k]);
            const float4 xb = *reinterpret_cast<const float4*>(&xs[m * K + k + 4]);
#pragma unroll
            for (int r = 0; r < R; ++r) {
              float s = acc[r][m];
              s = fmaf(wf[r][0], xa.x, s); s = fmaf(wf[r][1], xa.y, s); s = fmaf(wf[r][2], xa.z, s); s = fmaf(wf[r][3], xa.w, s);
              s = fmaf(wf[r][4], xb.x, s); s = fmaf(wf[r][5], xb.y, s); s = fmaf(wf[r][6], xb.z, s); s = fmaf(wf[r][7], xb.w, s);
              acc[r][m] = s;
            }
          }
        }
      }
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int m = 0; m < MB; ++m) acc[r][m] = warp_sum(acc[r][m]);
      // lanes [16r, 16r + MB) finish row n + r
      const int m = lane & 15, r_sel = lane >> 4;
      const int nn = n + r_sel;
      if (r_sel < R && m < mrows && nn < n_end) {
        float v = 0.f;
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
          for (int mm = 0; mm < MB; ++mm)
            if (r == r_sel && mm == m) v = acc[r][mm];
        const int mg = m0 + m;
        if (a.bias) v += a.bias[nn];
        if (nn < a.alpha_cols) v *= a.alpha;
        if (a.act == 1) v = gelu_erf(v);
        if (a.residual) v += a.residual[(long long)mg * a.ldo + nn];
        a.out[(long long)mg * a.ldo + nn] = v;
        if (a.kc && nn >= a.D) {
          const long long row = ((long long)(a.seq0 + mg) * a.Tmax + pos) * a.D;
          if (nn < 2 * a.D) a.kc[row + nn - a.D] = f2e(v);
          else a.vc[row + nn - 2 * a.D] = f2e(v);
        }
      }
      if (PIPE) {
        if (has_next) cur = nxt;
      } else if (has_next) {
        load_rows<NC, R>(cur, a.W, K, n + R, n_end, lane);
      }
    }
  }
}

__device__ __forceinline__ float block_max4(float v, float* red4) {  // 128 threads
  v = warp_max(v);
  if ((threadIdx.x & 31) == 0) red4[threadIdx.x >> 5] = v;
  __syncthreads();
  const float r = fmaxf(fmaxf(red4[0], red4[1]), fmaxf(red4[2], red4[3]));
  __syncthreads();
  return r;
}
__device__ __forceinline__ float block_sum4(float v, float* red4) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) red4[threadIdx.x >> 5] = v;
  __syncthreads();
  const float r = red4[0] + red4[1] + red4[2] + red4[3];
  __syncthreads();
  return r;
}

// ------------------------------------------------------------------------------------------------
// causal self-attention over cached positions 0..pos of one (sequence, head).  128 threads = 16 key groups x 8 lanes;
// a lane owns 8 of the 64 head dims, so one warp-load covers 4 whole 128-byte K (or V) rows.  Keys are walked in chunks of 128
// with an online softmax: 33 KB of static smem whatever Tmax is (the first version held all Tmax = 448 positions: 116 KB, ONE CTA
// per SM, 43 waves at 320 sequences x 20 heads = 362 us per layer, profiles/r2c_summary.md); all loads of a chunk in flight together.
// ------------------------------------------------------------------------------------------------
constexpr int SCH = 128;

__global__ void __launch_bounds__(128) self_attn_kernel(const SelfAttnArgs a) {
  __shared__ __align__(16) uint8_t sK[SCH * 128];
  __shared__ __align__(16) uint8_t sV[SCH * 128];
  __shared__ float sc[SCH];
  __shared__ float red4[4];
  __shared__ float redo[16][64];
  const int h = blockIdx.x, q = blockIdx.y;
  pdl_wait();
  pdl_launch();
  const int pos = *a.pos;
  const int n = pos + 1;
  const int grp = threadIdx.x >> 3, sub = threadIdx.x & 7;
  // batched path: k / v of this step come from the projection's output (qkv), are rounded to bf16, appended to the cache at
  // position pos (a sequence's newest row lives in its own slot) and attended over; the GEMV path appended them itself
  uint4 kw = make_uint4(0u, 0u, 0u, 0u), vw = kw;
  const bool appender = a.kc_w && grp == (pos & 15);
  if (appender) {
    const long long kidx = (long long)q * 3 * a.D + a.D + h * 64 + sub * 8;
    float kf[8], vf[8];
    split_sum8(a.qkv, kidx, a.nsplit, a.split_stride, a.qkv_bias, a.D + h * 64 + sub * 8, 1.0f, kf);
    split_sum8(a.qkv, kidx + a.D, a.nsplit, a.split_stride, a.qkv_bias, 2 * a.D + h * 64 + sub * 8, 1.0f, vf);
    kw.x = pack_bf16(kf[0], kf[1]); kw.y = pack_bf16(kf[2], kf[3]); kw.z = pack_bf16(kf[4], kf[5]); kw.w = pack_bf16(kf[6], kf[7]);
    vw.x = pack_bf16(vf[0], vf[1]); vw.y = pack_bf16(vf[2], vf[3]); vw.z = pack_bf16(vf[4], vf[5]); vw.w = pack_bf16(vf[6], vf[7]);
    const long long off = ((long long)q * a.Tmax + pos) * a.D + h * 64 + sub * 8;
    *reinterpret_cast<uint4*>(a.kc_w + off) = kw;
    *reinterpret_cast<uint4*>(a.vc_w + off) = vw;
  }
  float qv[8];
  split_sum8(a.qkv, (long long)q * 3 * a.D + h * 64 + sub * 8, a.nsplit, a.split_stride, a.qkv_bias, h * 64 + sub * 8, a.q_alpha, qv);
  float m_run = -INFINITY, l_run = 0.f;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  for (int c0 = 0; c0 < n; c0 += SCH) {
    const int nc = min(SCH, n - c0);
    __syncthreads();  // everybody is done with the previous chunk's rows and probabilities
    for (int s = grp; s < nc; s += 16) {
      const int ks = c0 + s;
      if (a.kc_w && ks == pos) {  // (this thread is the appender: same group, same piece)
        *reinterpret_cast<uint4*>(sK + s * 128 + sub * 16) = kw;
        *reinterpret_cast<uint4*>(sV + s * 128 + sub * 16) = vw;
      } else {
        const int slot = a.anc ? a.anc[q * a.Tmax + ks] : q;
        const long long off = ((long long)slot * a.Tmax + ks) * a.D + h * 64 + sub * 8;
        cp_async16(sK + s * 128 + sub * 16, a.kc + off);
        cp_async16(sV + s * 128 + sub * 16, a.vc + off);
      }
    }
    cp_async_wait_all();  // each thread reads back only the 16-byte pieces it copied (or wrote) itself
    float lmax = -INFINITY;
    for (int sb = 0; sb < nc; sb += 16) {  // uniform trip count: the shuffles need all 32 lanes
      const int s = sb + grp;
      float d = 0.f;
      if (s < nc) {
        float kf[8];
        unpack8(*reinterpret_cast<const uint4*>(sK + s * 128 + sub * 16), kf);
#pragma unroll
        for (int j = 0; j < 8; ++j) d = fmaf(qv[j], kf[j], d);
      }
      d += __shfl_xor_sync(0xffffffffu, d, 1);
      d += __shfl_xor_sync(0xffffffffu, d, 2);
      d += __shfl_xor_sync(0xffffffffu, d, 4);
      if (s < nc) {
        if (sub == 0) sc[s] = d;
        lmax = fmaxf(lmax, d);
      }
    }
    const float m_new = fmaxf(m_run, block_max4(lmax, red4));  // (also orders the sc[] writes before the reads below)
    const float scale = __expf(m_run - m_new);                // first chunk: exp(-inf) = 0
    float lsum = 0.f;
    for (int s = threadIdx.x; s < nc; s += 128) {
      const float e = __expf(sc[s] - m_new);
      sc[s] = e;
      lsum += e;
    }
    l_run = l_run * scale + block_sum4(lsum, red4);
    m_run = m_new;
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] *= scale;
    for (int s = grp; s < nc; s += 16) {
      float vf[8];
      unpack8(*reinterpret_cast<const uint4*>(sV + s * 128 + sub * 16), vf);
      const float p = sc[s];
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = fmaf(p, vf[j], acc[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) redo[grp][sub * 8 + j] = acc[j];
  __syncthreads();
  if (threadIdx.x < 64) {
    float o = 0.f;
#pragma unroll
    for (int g = 0; g < 16; ++g) o += redo[g][threadIdx.x];
    const float r = o / l_run;
    if (a.out_bf16) a.out_bf16[(long long)q * a.D + h * 64 + threadIdx.x] = f2e(r);
    else a.out[(long long)q * a.D + h * 64 + threadIdx.x] = r;
  }
}

// ------------------------------------------------------------------------------------------------
// cross-attention over the encoder K/V of one audio, shared by its G beams.  XSPLIT key splits per (audio, head), at most
// 128 keys per split, so a CTA's whole K and V slice (2 x 16 KB) is requested up front: 16 x 16-byte loads per thread,
// one DRAM round trip.  The last-arriving split block merges the partials (flash-decoding), no extra launch.
// ------------------------------------------------------------------------------------------------
constexpr int XK = 128;

template <int GM>  // compile-time bound on the beams per audio (1 or MAXG)
__global__ void __launch_bounds__(128) cross_attn_kernel(const CrossAttnArgs a) {
  __shared__ float red4[4];
  __shared__ float gm[GM], gl[GM];
  __shared__ unsigned is_last;
  const int split = blockIdx.x, h = blockIdx.y, au = blockIdx.z;
  const int grp = threadIdx.x >> 3, sub = threadIdx.x & 7;
  const int G = (GM == 1) ? 1 : a.G;
  const int ks = (a.S + XSPLIT - 1) / XSPLIT;
  const int s0 = split * ks;
  const int n = max(0, min(a.S, s0 + ks) - s0);
  const bf16* kbase = a.kc + (((long long)au * a.H + h) * a.S + s0) * 64 + sub * 8;
  const bf16* vbase = a.vc + (((long long)au * a.H + h) * a.S + s0) * 64 + sub * 8;

  extern __shared__ __align__(16) uint8_t dyn[];  // K slice [XK][128 B] | V slice [XK][128 B] | sc [GM][XK] | redo [16][GM][64]
  uint8_t* sK = dyn;
  uint8_t* sV = dyn + XK * 128;
  float (*sc)[XK] = reinterpret_cast<float (*)[XK]>(dyn + 2 * XK * 128);
  float (*redo)[GM][64] = reinterpret_cast<float (*)[GM][64]>(dyn + 2 * XK * 128 + GM * XK * sizeof(float));
  // the encoder K/V of an audio are constant during decoding: requested BEFORE the programmatic-launch wait, so under PDL the
  // 32 KB of this CTA are in flight while the previous kernel (the cross-q projection) is still finishing
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int kk = i * 16 + grp;
    if (kk < n) {
      cp_async16(sK + kk * 128 + sub * 16, kbase + (long long)kk * 64);
      cp_async16(sV + kk * 128 + sub * 16, vbase + (long long)kk * 64);
    }
  }
  pdl_wait();
  pdl_launch();
  float qv[GM][8];
#pragma unroll
  for (int g = 0; g < GM; ++g) {
    if (g < G) split_sum8(a.q, (long long)(au * G + g) * a.D + h * 64 + sub * 8, a.nsplit, a.split_stride, a.q_bias, h * 64 + sub * 8, a.q_alpha, qv[g]);
  }
  const int slot = a.head_slots ? a.head_slots[h] : -1;
  float* align_row = nullptr;
  if (slot >= 0 && a.align) {
    const int step = *a.pos - a.step_base;
    // one block of [Ha][Tcap][S] per SEQUENCE slot (au * G + g): beam search gathers a row per step from the slot that was the
    // winner's ancestor at that step (bw_word_timestamps_gather)
    if (step >= 0 && step < a.Tcap) align_row = a.align + (((long long)au * G * a.Ha + slot) * a.Tcap + step) * a.S + s0;
  }
  cp_async_wait_all();  // each thread reads back only the 16-byte pieces it copied itself
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int kk = i * 16 + grp;
    float kf[8];
    if (kk < n) unpack8(*reinterpret_cast<const uint4*>(sK + kk * 128 + sub * 16), kf);
    else {
#pragma unroll
      for (int j = 0; j < 8; ++j) kf[j] = 0.f;
    }
#pragma unroll
    for (int g = 0; g < GM; ++g) {
      if (g < G) {
        float d = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) d = fmaf(qv[g][j], kf[j], d);
        d += __shfl_xor_sync(0xffffffffu, d, 1);
        d += __shfl_xor_sync(0xffffffffu, d, 2);
        d += __shfl_xor_sync(0xffffffffu, d, 4);
        if (sub == 0 && kk < n) {
          sc[g][kk] = d;
          if (align_row) align_row[(long long)g * a.Ha * a.Tcap * a.S + kk] = d;
        }
      }
    }
  }
  __syncthreads();
  for (int g = 0; g < G; ++g) {  // n <= 128: one key per thread
    const float v = (threadIdx.x < n) ? sc[g][threadIdx.x] : -INFINITY;
    const float mx = block_max4(v, red4);
    const float e = (threadIdx.x < n) ? __expf(v - mx) : 0.f;
    if (threadIdx.x < n) sc[g][threadIdx.x] = e;
    const float sum = block_sum4(e, red4);
    if (threadIdx.x == 0) {
      gm[g] = mx;
      gl[g] = sum;
    }
  }
  __syncthreads();
  float acc[GM][8];
#pragma unroll
  for (int g = 0; g < GM; ++g)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[g][j] = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int kk = i * 16 + grp;
    if (kk < n) {
      float vf[8];
      unpack8(*reinterpret_cast<const uint4*>(sV + kk * 128 + sub * 16), vf);
#pragma unroll
      for (int g = 0; g < GM; ++g) {
        if (g < G) {
          const float p = sc[g][kk];
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[g][j] = fmaf(p, vf[j], acc[g][j]);
        }
      }
    }
  }
#pragma unroll
  for (int g = 0; g < GM; ++g)
    if (g < G) {
#pragma unroll
      for (int j = 0; j < 8; ++j) redo[grp][g][sub * 8 + j] = acc[g][j];
    }
  __syncthreads();
  const long long pbase = (((long long)au * a.H + h) * XSPLIT + split) * G;
  if (threadIdx.x < 64) {
    for (int g = 0; g < G; ++g) {
      float o = 0.f;
#pragma unroll
      for (int r = 0; r < 16; ++r) o += redo[r][g][threadIdx.x];
      a.part_o[(pbase + g) * 64 + threadIdx.x] = o;
    }
  }
  if (threadIdx.x < G) {
    a.part_ml[(pbase + threadIdx.x) * 2 + 0] = gm[threadIdx.x];
    a.part_ml[(pbase + threadIdx.x) * 2 + 1] = gl[threadIdx.x];
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned prev = atomicAdd(&a.counters[au * a.H + h], 1u);
    is_last = (prev == XSPLIT - 1) ? 1u : 0u;
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  if (threadIdx.x < 64) {
    const int d = threadIdx.x;
    const long long hb = ((long long)au * a.H + h) * XSPLIT * G;
    for (int g = 0; g < G; ++g) {
      float M = -INFINITY;
      for (int sp = 0; sp < XSPLIT; ++sp) {
        const float l = __ldcg(&a.part_ml[(hb + (long long)sp * G + g) * 2 + 1]);
        if (l > 0.f) M = fmaxf(M, __ldcg(&a.part_ml[(hb + (long long)sp * G + g) * 2 + 0]));
      }
      float L = 0.f, o = 0.f;
      for (int sp = 0; sp < XSPLIT; ++sp) {
        const float l = __ldcg(&a.part_ml[(hb + (long long)sp * G + g) * 2 + 1]);
        if (l > 0.f) {
          const float w = __expf(__ldcg(&a.part_ml[(hb + (long long)sp * G + g) * 2 + 0]) - M);
          L = fmaf(l, w, L);
          o = fmaf(__ldcg(&a.part_o[(hb + (long long)sp * G + g) * 64 + d]), w, o);
        }
      }
      if (a.out_bf16) a.out_bf16[(long long)(au * G + g) * a.D + h * 64 + d] = f2e(o / L);
      else a.out[(long long)(au * G + g) * a.D + h * 64 + d] = o / L;
    }
  }
  if (threadIdx.x == 0) a.counters[au * a.H + h] = 0u;
}


// ------------------------------------------------------------------------------------------------
// Cross-attention for large batches: ONE CTA streams all S keys of one (audio, head) through a double-buffered smem ring with an
// online softmax -- no key splits, so no partial results, no atomics, no __threadfence and no merge pass (the split kernel above
// spends ~45 % of its issue slots on those and on block reductions at A = 64: profiles/r2a_summary.md, 0.68 of the HBM peak).
// Chosen when A * H CTAs fill the machine at least twice; small batches keep the split kernel (more CTAs per byte).
//   QK : thread t owns key t of the 128-key tile: its 128-byte K row sits in smem with the 16-byte pieces XOR-swizzled by (row & 7),
//        so a row-per-thread LDS.128 is conflict-free; 64 FMAs per beam, no shuffles
//   PV : thread (t / 16, t % 16) owns 4 of the 64 output dims for every 8th key; the 8 key slices are folded once at the very end
// One tile (16 KB K + 16 KB V) is in flight per CTA while the previous one is processed; 64 KB smem -> 3 CTAs per SM.
// ------------------------------------------------------------------------------------------------
constexpr int XT = 128;  // keys per tile

template <int GM>
__global__ void __launch_bounds__(128) cross_attn_stream_kernel(const CrossAttnArgs a) {
  extern __shared__ __align__(128) uint8_t dyn[];  // K [2][XT][128 B] | V [2][XT][128 B] | sp [GM][XT] | sq [GM][64] | red [GM][4] | fold [8][GM][64]
  uint8_t* sK = dyn;
  uint8_t* sV = dyn + 2 * XT * 128;
  float* sp = reinterpret_cast<float*>(dyn + 4 * XT * 128);
  float* sq = sp + GM * XT;
  float* red = sq + GM * 64;
  float* fold = red + GM * 4;
  const int h = blockIdx.x, au = blockIdx.y;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int G = (GM < MAXG) ? GM : a.G;  // exact instantiation for 1..5 beams; the MAXG one handles 6..8 with predicates
  const int S = a.S;
  const int ntiles = (S + XT - 1) / XT;
  const bf16* kbase = a.kc + ((long long)au * a.H + h) * S * 64;
  const bf16* vbase = a.vc + ((long long)au * a.H + h) * S * 64;

  auto issue_tile = [&](int tile, int stage) {
    const int r0 = tile * XT;
    const int nrows = min(XT, S - r0);
    uint8_t* dk = sK + stage * XT * 128;
    uint8_t* dv = sV + stage * XT * 128;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int i = t + 128 * j;  // 16-byte piece of the tile: row i / 8, piece i % 8 (global: contiguous)
      const int row = i >> 3, c = i & 7;
      if (row < nrows) {
        cp_async16(dk + row * 128 + ((c ^ (row & 7)) << 4), kbase + (long long)(r0 + row) * 64 + c * 8);
        cp_async16(dv + row * 128 + (c << 4), vbase + (long long)(r0 + row) * 64 + c * 8);
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  // the encoder K/V are constant during decoding: the first tile is requested before the programmatic-launch wait
  issue_tile(0, 0);
  pdl_wait();
  pdl_launch();
  if (t < G * 8) {  // 8 values per thread: beam t / 8, dims (t % 8) * 8 ...
    float qf[8];
    split_sum8(a.q, (long long)(au * G + (t >> 3)) * a.D + h * 64 + (t & 7) * 8, a.nsplit, a.split_stride, a.q_bias, h * 64 + (t & 7) * 8, a.q_alpha, qf);
#pragma unroll
    for (int i = 0; i < 8; ++i) sq[(t >> 3) * 64 + (t & 7) * 8 + i] = qf[i];
  }
  const int slot = a.head_slots ? a.head_slots[h] : -1;
  float* align_base = nullptr;
  if (slot >= 0 && a.align) {
    const int step = *a.pos - a.step_base;
    if (step >= 0 && step < a.Tcap) align_base = a.align + (((long long)au * G * a.Ha + slot) * a.Tcap + step) * S;
  }
  float m_run[GM], l_part[GM], o[GM][4];
#pragma unroll
  for (int g = 0; g < GM; ++g) {
    m_run[g] = -INFINITY;
    l_part[g] = 0.f;
#pragma unroll
    for (int d = 0; d < 4; ++d) o[g][d] = 0.f;
  }
  const int kg = t >> 4, dg = t & 15;
  for (int tile = 0; tile < ntiles; ++tile) {
    const int stage = tile & 1;
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();  // tile landed for everybody; everybody is done with the other stage, sp and red of the previous tile
    if (tile + 1 < ntiles) issue_tile(tile + 1, stage ^ 1);
    const int r0 = tile * XT;
    const bool valid = r0 + t < S;
    // ---- scores of key t for every beam
    float sc[GM];
#pragma unroll
    for (int g = 0; g < GM; ++g) sc[g] = 0.f;
    {
      const uint8_t* krow = sK + stage * XT * 128 + t * 128;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        float kf[8];
        unpack8(*reinterpret_cast<const uint4*>(krow + ((c ^ (t & 7)) << 4)), kf);
#pragma unroll
        for (int g = 0; g < GM; ++g) {
          if (g < G) {
            const float4 q0 = *reinterpret_cast<const float4*>(sq + g * 64 + c * 8);
            const float4 q1 = *reinterpret_cast<const float4*>(sq + g * 64 + c * 8 + 4);
            float s0 = sc[g];
            s0 = fmaf(q0.x, kf[0], s0); s0 = fmaf(q0.y, kf[1], s0); s0 = fmaf(q0.z, kf[2], s0); s0 = fmaf(q0.w, kf[3], s0);
            s0 = fmaf(q1.x, kf[4], s0); s0 = fmaf(q1.y, kf[5], s0); s0 = fmaf(q1.z, kf[6], s0); s0 = fmaf(q1.w, kf[7], s0);
            sc[g] = s0;
          }
        }
      }
    }
    if (align_base && valid) {
#pragma unroll
      for (int g = 0; g < GM; ++g)
        if (g < G) align_base[(long long)g * a.Ha * a.Tcap * S + r0 + t] = sc[g];
    }
#pragma unroll
    for (int g = 0; g < GM; ++g) {
      if (g < G) {
        const float v = warp_max(valid ? sc[g] : -INFINITY);
        if (lane == 0) red[g * 4 + warp] = v;
      }
    }
    __syncthreads();
    float scale[GM];
#pragma unroll
    for (int g = 0; g < GM; ++g) {
      scale[g] = 1.f;
      if (g < G) {
        const float mt = fmaxf(fmaxf(red[g * 4], red[g * 4 + 1]), fmaxf(red[g * 4 + 2], red[g * 4 + 3]));
        const float m_new = fmaxf(m_run[g], mt);  // finite: every tile holds at least one valid key
        scale[g] = __expf(m_run[g] - m_new);      // first tile: exp(-inf) = 0
        const float p = valid ? __expf(sc[g] - m_new) : 0.f;
        l_part[g] = l_part[g] * scale[g] + p;
        sp[g * XT + t] = p;
        m_run[g] = m_new;
      }
    }
    __syncthreads();
    // ---- P.V: this thread's 4 dims over keys kg, kg + 8, ...
    {
      const uint8_t* vt = sV + stage * XT * 128 + dg * 8;
#pragma unroll
      for (int g = 0; g < GM; ++g)
        if (g < G) {
#pragma unroll
          for (int d = 0; d < 4; ++d) o[g][d] *= scale[g];
        }
#pragma unroll 4
      for (int j = 0; j < XT / 8; ++j) {
        const int k = kg + 8 * j;
        const uint2 vv = *reinterpret_cast<const uint2*>(vt + k * 128);
        const float2 v01 = unpack_bf16(vv.x), v23 = unpack_bf16(vv.y);
#pragma unroll
        for (int g = 0; g < GM; ++g) {
          if (g < G) {
            const float p = sp[g * XT + k];  // 0 for the rows beyond S (their V bytes are stale smem: multiplied by 0 ... but NaN-safe?)
            if (p != 0.f) {
              o[g][0] = fmaf(p, v01.x, o[g][0]); o[g][1] = fmaf(p, v01.y, o[g][1]);
              o[g][2] = fmaf(p, v23.x, o[g][2]); o[g][3] = fmaf(p, v23.y, o[g][3]);
            }
          }
        }
      }
    }
  }
  // ---- fold: sum of exp over the 128 key owners, outputs over the 8 key slices
  __syncthreads();
#pragma unroll
  for (int g = 0; g < GM; ++g) {
    if (g < G) {
      const float v = warp_sum(l_part[g]);
      if (lane == 0) red[g * 4 + warp] = v;
#pragma unroll
      for (int d = 0; d < 4; ++d) fold[(kg * GM + g) * 64 + dg * 4 + d] = o[g][d];
    }
  }
  __syncthreads();
  for (int i = t; i < G * 64; i += 128) {
    const int g = i >> 6, d = i & 63;
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) acc += fold[(j * GM + g) * 64 + d];
    const float l = (red[g * 4] + red[g * 4 + 1]) + (red[g * 4 + 2] + red[g * 4 + 3]);
    const float r = acc / l;
    const long long off = (long long)(au * G + g) * a.D + h * 64 + d;
    if (a.out_bf16) a.out_bf16[off] = f2e(r);
    else a.out[off] = r;
  }
}

template <int MB, int NC, int R, bool PIPE>
int launch_gemv_t(cudaStream_t st, const GemvArgs& a, int grid, int rpw, size_t smem) {
  static bool attr = false;
  if (!attr) {
    BW_CUDA_OK(cudaFuncSetAttribute(gemv_kernel<MB, NC, R, PIPE>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr = true;
  }
  gemv_kernel<MB, NC, R, PIPE><<<grid, GEMV_THREADS, smem, st>>>(a, rpw);
  BW_CUDA_OK(cudaGetLastError());
  return 0;
}

template <int MB>
int launch_gemv_mb(cudaStream_t st, const GemvArgs& a) {
  const size_t smem = (size_t)MB * a.K * sizeof(float);
  if (a.K <= 1280) {
    // two rows per warp in flight; ~2 CTAs per SM for small N, software-pipelined row pairs for the LM head
    int rpw = (a.N + 296 * GEMV_WARPS - 1) / (296 * GEMV_WARPS);
    rpw = (rpw + 1) & ~1;
    if (rpw < 2) rpw = 2;
    const int grid = (a.N + rpw * GEMV_WARPS - 1) / (rpw * GEMV_WARPS);
    return launch_gemv_t<MB, 5, 2, true>(st, a, grid, rpw, smem);
  }
  // long rows (fc2, K = 4*D): one row per warp, all 20 loads of the row in flight
  int rpw = (a.N + 592 * GEMV_WARPS - 1) / (592 * GEMV_WARPS);
  if (rpw < 1) rpw = 1;
  const int grid = (a.N + rpw * GEMV_WARPS - 1) / (rpw * GEMV_WARPS);
  return launch_gemv_t<MB, 20, 1, false>(st, a, grid, rpw, smem);
}

}  // namespace

int launch_gemv(cudaStream_t st, const GemvArgs& a) {
  BW_CHECK(a.M >= 1, "gemv: M=%d must be >= 1", a.M);
  BW_CHECK(a.K % 8 == 0 && a.K <= 5120, "gemv: K=%d must be a multiple of 8 and <= 5120", a.K);
  if (a.M <= 1) return launch_gemv_mb<1>(st, a);
  if (a.M <= 2) return launch_gemv_mb<2>(st, a);
  if (a.M <= 4) return launch_gemv_mb<4>(st, a);
  return launch_gemv_mb<8>(st, a);  // M > 8: the kernel walks the rows in chunks of 8 with the weights held in registers
}

int launch_self_attn(cudaStream_t st, const SelfAttnArgs& a, int Q) {
  BW_CUDA_OK(launch_k(self_attn_kernel, dim3(a.H, Q), dim3(128), 0, st, a));
  return 0;
}

int launch_cross_attn(cudaStream_t st, const CrossAttnArgs& a, int A, int impl) {
  BW_CHECK(a.G >= 1 && a.G <= MAXG, "cross_attn: G=%d must be in 1..%d", a.G, MAXG);
  BW_CHECK(a.S <= XSPLIT * XK, "cross_attn: S=%d exceeds %d", a.S, XSPLIT * XK);
  BW_CHECK(impl >= 0 && impl <= 2, "cross_attn: impl=%d must be 0 (policy), 1 (split) or 2 (streaming)", impl);
  constexpr size_t smem1 = 2 * XK * 128 + (size_t)(1 * XK + 16 * 1 * 64) * sizeof(float);
  constexpr size_t smemG = 2 * XK * 128 + (size_t)(MAXG * XK + 16 * MAXG * 64) * sizeof(float);
  static bool attr = false;
  if (!attr) {
    BW_CUDA_OK(cudaFuncSetAttribute(cross_attn_kernel<MAXG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemG));
    attr = true;
  }
  {  // large batches: one CTA per (audio, head) streams all keys (no splits / partials / merge)
    // CTAs (A * H) from which the streaming kernel is used; 0 = never.  (Read per launch: launches happen at graph capture only.)
    const char* ev = getenv("BW_XATTN_STREAM_MIN");
    const int stream_min = ev ? atoi(ev) : 296;
    const bool stream = impl == 2 || (impl == 0 && stream_min > 0 && A * a.H >= stream_min);
    if (stream) {
      auto smem_of = [](int gm) { return (size_t)4 * XT * 128 + (size_t)(gm * XT + gm * 64 + gm * 4 + 8 * gm * 64) * sizeof(float); };
      // instantiated for the exact beam count (a bound of 8 with g < G predicates issued 8 / 5 of the instructions at beam 5)
#define BW_XSTREAM(GMV)                                                                                                   \
  {                                                                                                                       \
    static bool attr_##GMV = false;                                                                                        \
    if (!attr_##GMV) {                                                                                                     \
      BW_CUDA_OK(cudaFuncSetAttribute(cross_attn_stream_kernel<GMV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_of(GMV))); \
      attr_##GMV = true;                                                                                                   \
    }                                                                                                                     \
    BW_CUDA_OK(launch_k(cross_attn_stream_kernel<GMV>, dim3(a.H, A), dim3(128), smem_of(GMV), st, a));                     \
  }
      switch (a.G) {
        case 1: BW_XSTREAM(1) break;
        case 2: BW_XSTREAM(2) break;
        case 3: BW_XSTREAM(3) break;
        case 4: BW_XSTREAM(4) break;
        case 5: BW_XSTREAM(5) break;
        default: BW_XSTREAM(8) break;
      }
#undef BW_XSTREAM
      return 0;
    }
  }
  if (a.G == 1) BW_CUDA_OK(launch_k(cross_attn_kernel<1>, dim3(XSPLIT, a.H, A), dim3(128), smem1, st, a));
  else BW_CUDA_OK(launch_k(cross_attn_kernel<MAXG>, dim3(XSPLIT, a.H, A), dim3(128), smemG, st, a));
  return 0;
}

}  // namespace bw
