// Attention with FEW queries (the perceiver resampler, models/brainformer.py:175-219 CausalCrossAttention with <= 64
// learnable-query tokens against the encoder's S = 4096 context tokens, and the 32-token self-attention Block that
// follows it, :247-268) -- SURVEY section 8f row N2.  head_dim 16 / 32 / 64, no mask (the reference passes None), optional
// RoPE on q and k (apply_rope, :70-91, for the self-attention Block).
//
// With <= 64 queries the score matrix of one (trial, head) is at most 64 x S: the work (4.3 GFLOP forward at cfg 4) is far
// below what K and V cost to read (134 MB), so these are bandwidth-bound CUDA-core kernels, split over the key axis:
//
//   small_attn_fwd_kernel      (optionally only the first k_len[b] keys of trial b: a cache whose trials hold different
//                              numbers of tokens; chunks past that write the empty partial)
//                              one CTA = (256-key chunk, head, trial): thread j owns key j (its K and V rows live in
//                              registers), scores against every query (Q in shared memory) -> chunk maximum / sum per
//                              query -> P in shared memory -> thread (query, 4 dims) sums P V over the chunk's keys
//                              -> partial (m, l, O) of the chunk
//   small_attn_combine_kernel  merges the chunks' partials in chunk order (deterministic) -> O (bf16), lse
//   small_attn_bwd_kernel      same decomposition: thread j forms P and dS for its key against every query, accumulates
//                              dK[j], dV[j] in registers (written once, no atomics); dS goes to shared memory and thread
//                              (query, 4 dims) sums dS K over the chunk -> partial dQ of the chunk
//   small_attn_dq_kernel       sums the chunks' partial dQ in chunk order, rotates back (RoPE), writes bf16
#include "common.cuh"
#include "fk_b200.h"

namespace fk {

constexpr int kSaKeys = 256;         // keys per CTA = threads per CTA
constexpr int kSaMaxQ = 64;

struct SaParams {
  const __nv_bfloat16 *q, *k, *v;    // [B, Tq, H, HD] / [B, S, H, HD] with row strides (elements)
  long long q_bs, q_ts, k_bs, k_ts, v_bs, v_ts;
  int B, H, Tq, S, n_chunks;
  float scale_log2;                  // softmax scale * log2(e)
  const float2* rope;                // [P][HD / 2] (cos, sin) or null
  int rope_q0, rope_k0;              // position of query 0 / key 0 in the table
};

template <int HD>
__device__ __forceinline__ void load_row(const __nv_bfloat16* p, float (&x)[HD]) {
#pragma unroll
  for (int i = 0; i < HD / 8; ++i) {
    const uint4 w = *reinterpret_cast<const uint4*>(p + i * 8);
    const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      x[i * 8 + 2 * e] = __uint_as_float(ww[e] << 16);
      x[i * 8 + 2 * e + 1] = __uint_as_float(ww[e] & 0xffff0000u);
    }
  }
}
template <int HD>
__device__ __forceinline__ void rotate(float (&x)[HD], const float2* cs, bool inverse) {
  // pairs of adjacent elements, as apply_rope's reshape(..., -1, 2) (brainformer.py:87); the rotated value is rounded
  // to bf16 like the tensor the reference hands to SDPA (`.type_as(x)`)
#pragma unroll
  for (int i = 0; i < HD / 2; ++i) {
    const float2 c = cs[i];
    const float a = x[2 * i], b = x[2 * i + 1];
    const float sn = inverse ? -c.y : c.y;
    x[2 * i] = a * c.x - b * sn;
    x[2 * i + 1] = a * sn + b * c.x;
  }
}
template <int HD>
__device__ __forceinline__ void round_bf16(float (&x)[HD]) {
#pragma unroll
  for (int i = 0; i < HD; ++i) x[i] = __bfloat162float(__float2bfloat16_rn(x[i]));
}
template <int HD>
__device__ __forceinline__ void store_row_bf16(__nv_bfloat16* p, const float (&x)[HD]) {
#pragma unroll
  for (int i = 0; i < HD / 8; ++i) {
    uint32_t w[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      __nv_bfloat162 t = __floats2bfloat162_rn(x[i * 8 + 2 * e], x[i * 8 + 2 * e + 1]);
      w[e] = *reinterpret_cast<uint32_t*>(&t);
    }
    *reinterpret_cast<uint4*>(p + i * 8) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// queries of one (trial, head) -> shared memory as fp32 [Tq][HD] (rotated if RoPE is on)
template <int HD>
__device__ __forceinline__ void stage_queries(const SaParams& p, int b, int h, float* qs) {
  for (int t = threadIdx.x; t < p.Tq; t += blockDim.x) {
    float x[HD];
    load_row<HD>(p.q + b * p.q_bs + static_cast<long long>(t) * p.q_ts + h * HD, x);
    if (p.rope != nullptr) { rotate<HD>(x, p.rope + static_cast<long long>(p.rope_q0 + t) * (HD / 2), false); round_bf16<HD>(x); }
#pragma unroll
    for (int d = 0; d < HD; ++d) qs[t * HD + d] = x[d];
  }
}

// max / sum over the 256 threads of the CTA for each of Tq values held one per (thread, t) in smem column form
template <int HD>
__global__ void __launch_bounds__(kSaKeys)
small_attn_fwd_kernel(const SaParams p, const int* __restrict__ k_len, float* __restrict__ part_o, float* __restrict__ part_ml) {
  extern __shared__ float sm[];
  float* qs = sm;                                   // [max(Tq, kSaKeys)][HD]: queries, later the chunk's V rows
  float* ps = qs + kSaKeys * HD;                    // [Tq][kSaKeys + 1]
  float* red = ps + kSaMaxQ * (kSaKeys + 1);        // [8 warps][Tq]
  float* mrow = red + 8 * kSaMaxQ;                  // [Tq] chunk maximum, then reused for the sum
  const int chunk = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int j = chunk * kSaKeys + threadIdx.x;
  const int S = k_len == nullptr ? p.S : min(p.S, k_len[b]);     // keys of this trial that take part
  const long long pbase = ((static_cast<long long>(b) * p.H + h) * p.n_chunks + chunk) * p.Tq;
  if (chunk * kSaKeys >= S) {
    // no key of the chunk takes part: the empty partial (m = -inf, l = 0, O = 0), which the combine merges as a no-op
    for (int o = threadIdx.x; o < p.Tq * HD; o += kSaKeys) part_o[pbase * HD + o] = 0.f;
    for (int t = threadIdx.x; t < p.Tq; t += kSaKeys) {
      part_ml[(pbase + t) * 2] = -INFINITY;
      part_ml[(pbase + t) * 2 + 1] = 0.f;
    }
    return;
  }
  const bool ok = j < S;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  stage_queries<HD>(p, b, h, qs);
  float kr[HD], vr[HD];
  if (ok) {
    load_row<HD>(p.k + b * p.k_bs + static_cast<long long>(j) * p.k_ts + h * HD, kr);
    load_row<HD>(p.v + b * p.v_bs + static_cast<long long>(j) * p.v_ts + h * HD, vr);
    if (p.rope != nullptr) { rotate<HD>(kr, p.rope + static_cast<long long>(p.rope_k0 + j) * (HD / 2), false); round_bf16<HD>(kr); }
  }
  __syncthreads();
  // ---- scores of this key against every query (log2 domain), warp maxima ----
  for (int t = 0; t < p.Tq; ++t) {
    float s = -INFINITY;
    if (ok) {
      s = 0.f;
#pragma unroll
      for (int d = 0; d < HD; ++d) s = fmaf(qs[t * HD + d], kr[d], s);
      s *= p.scale_log2;
    }
    ps[t * (kSaKeys + 1) + threadIdx.x] = s;
    const float m = warp_max(s);
    if (lane == 0) red[warp * kSaMaxQ + t] = m;
  }
  __syncthreads();
  if (threadIdx.x < p.Tq) {
    float m = red[threadIdx.x];
#pragma unroll
    for (int w = 1; w < 8; ++w) m = fmaxf(m, red[w * kSaMaxQ + threadIdx.x]);
    mrow[threadIdx.x] = m;
  }
  __syncthreads();
  // ---- P = 2^(s - m) in place, warp sums ----
  for (int t = 0; t < p.Tq; ++t) {
    const float m = mrow[t];
    const float s = ps[t * (kSaKeys + 1) + threadIdx.x];
    const float e = (m == -INFINITY) ? 0.f : exp2f(s - m);
    ps[t * (kSaKeys + 1) + threadIdx.x] = e;
    const float sum = warp_sum(e);
    if (lane == 0) red[warp * kSaMaxQ + t] = sum;
  }
  // V rows of the chunk -> shared memory (over the query tile, which is no longer needed after the barrier)
  __syncthreads();
  float* vs = qs;
#pragma unroll
  for (int d = 0; d < HD; ++d) vs[threadIdx.x * HD + d] = ok ? vr[d] : 0.f;
  if (threadIdx.x < p.Tq) {
    float l = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) l += red[w * kSaMaxQ + threadIdx.x];
    part_ml[(pbase + threadIdx.x) * 2] = mrow[threadIdx.x];
    part_ml[(pbase + threadIdx.x) * 2 + 1] = l;
  }
  __syncthreads();
  // ---- O partial: thread (t, 4 dims) sums over the chunk's keys ----
  constexpr int DG = HD / 4;
  for (int o = threadIdx.x; o < p.Tq * DG; o += kSaKeys) {
    const int t = o / DG, d0 = (o % DG) * 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    const float* pr = ps + t * (kSaKeys + 1);
    for (int jj = 0; jj < kSaKeys; ++jj) {
      const float e = pr[jj];
      const float4 v4 = *reinterpret_cast<const float4*>(vs + jj * HD + d0);
      acc.x = fmaf(e, v4.x, acc.x); acc.y = fmaf(e, v4.y, acc.y); acc.z = fmaf(e, v4.z, acc.z); acc.w = fmaf(e, v4.w, acc.w);
    }
    *reinterpret_cast<float4*>(part_o + (pbase + t) * HD + d0) = acc;
  }
}

template <int HD>
__global__ void __launch_bounds__(256)
small_attn_combine_kernel(const float* __restrict__ part_o, const float* __restrict__ part_ml, int n_chunks, int Tq, int H, int B,
                          __nv_bfloat16* __restrict__ out, long long o_bs, long long o_ts, float* __restrict__ lse) {
  // one thread per (trial, head, query, dim)
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(B) * H * Tq * HD) return;
  const int d = static_cast<int>(i % HD);
  const int t = static_cast<int>((i / HD) % Tq);
  const int h = static_cast<int>((i / (static_cast<long long>(HD) * Tq)) % H);
  const int b = static_cast<int>(i / (static_cast<long long>(HD) * Tq * H));
  const long long base = (static_cast<long long>(b) * H + h) * n_chunks;
  float m = -INFINITY;
  for (int c = 0; c < n_chunks; ++c) m = fmaxf(m, part_ml[((base + c) * Tq + t) * 2]);
  float l = 0.f, o = 0.f;
  for (int c = 0; c < n_chunks; ++c) {
    const float mc = part_ml[((base + c) * Tq + t) * 2];
    const float w = (mc == -INFINITY) ? 0.f : exp2f(mc - m);
    l = fmaf(w, part_ml[((base + c) * Tq + t) * 2 + 1], l);
    o = fmaf(w, part_o[((base + c) * Tq + t) * HD + d], o);
  }
  out[b * o_bs + static_cast<long long>(t) * o_ts + h * HD + d] = __float2bfloat16_rn(l > 0.f ? o / l : 0.f);
  if (d == 0) lse[(static_cast<long long>(b) * H + h) * Tq + t] = (l > 0.f) ? m + log2f(l) : INFINITY;
}

struct SaBwdParams {
  const __nv_bfloat16 *dout, *out;   // [B, Tq, H, HD], row stride o_ts
  long long o_bs, o_ts, do_bs, do_ts;
  const float* lse;                  // [B, H, Tq] (log2 domain)
  __nv_bfloat16 *dk, *dv;            // [B, S, H, HD] with the strides of k / v
  float* part_dq;                    // [B, H, n_chunks, Tq, HD]
  float scale;
};

template <int HD>
__global__ void __launch_bounds__(kSaKeys)
small_attn_bwd_kernel(const SaParams p, const SaBwdParams g) {
  extern __shared__ float sm[];
  float* qs = sm;                                   // [max(Tq, kSaKeys)][HD]: queries, later the chunk's K rows
  float* ds = qs + kSaKeys * HD;                    // [Tq][kSaKeys + 1]
  float* dos = ds + kSaMaxQ * (kSaKeys + 1);        // [Tq][HD]
  float* st = dos + kSaMaxQ * HD;                   // [Tq] lse | [Tq] delta
  const int chunk = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int j = chunk * kSaKeys + threadIdx.x;
  const bool ok = j < p.S;
  stage_queries<HD>(p, b, h, qs);
  for (int t = threadIdx.x; t < p.Tq; t += blockDim.x) {
    float x[HD], o[HD];
    load_row<HD>(g.dout + b * g.do_bs + static_cast<long long>(t) * g.do_ts + h * HD, x);
    load_row<HD>(g.out + b * g.o_bs + static_cast<long long>(t) * g.o_ts + h * HD, o);
    float dl = 0.f;
#pragma unroll
    for (int d = 0; d < HD; ++d) { dos[t * HD + d] = x[d]; dl = fmaf(x[d], o[d], dl); }
    st[t] = g.lse[(static_cast<long long>(b) * p.H + h) * p.Tq + t];
    st[kSaMaxQ + t] = dl;
  }
  float kr[HD], vr[HD], dkr[HD], dvr[HD];
#pragma unroll
  for (int d = 0; d < HD; ++d) { kr[d] = 0.f; vr[d] = 0.f; dkr[d] = 0.f; dvr[d] = 0.f; }
  if (ok) {
    load_row<HD>(p.k + b * p.k_bs + static_cast<long long>(j) * p.k_ts + h * HD, kr);
    load_row<HD>(p.v + b * p.v_bs + static_cast<long long>(j) * p.v_ts + h * HD, vr);
    if (p.rope != nullptr) { rotate<HD>(kr, p.rope + static_cast<long long>(p.rope_k0 + j) * (HD / 2), false); round_bf16<HD>(kr); }
  }
  __syncthreads();
  for (int t = 0; t < p.Tq; ++t) {
    float s = 0.f, dp = 0.f;
#pragma unroll
    for (int d = 0; d < HD; ++d) { s = fmaf(qs[t * HD + d], kr[d], s); dp = fmaf(dos[t * HD + d], vr[d], dp); }
    const float pe = ok ? exp2f(s * p.scale_log2 - st[t]) : 0.f;
    const float dsv = pe * (dp - st[kSaMaxQ + t]);
#pragma unroll
    for (int d = 0; d < HD; ++d) { dvr[d] = fmaf(pe, dos[t * HD + d], dvr[d]); dkr[d] = fmaf(dsv, qs[t * HD + d], dkr[d]); }
    ds[t * (kSaKeys + 1) + threadIdx.x] = dsv;
  }
  if (ok) {
#pragma unroll
    for (int d = 0; d < HD; ++d) dkr[d] *= g.scale;
    if (p.rope != nullptr) rotate<HD>(dkr, p.rope + static_cast<long long>(p.rope_k0 + j) * (HD / 2), true);
    store_row_bf16<HD>(g.dk + b * p.k_bs + static_cast<long long>(j) * p.k_ts + h * HD, dkr);
    store_row_bf16<HD>(g.dv + b * p.v_bs + static_cast<long long>(j) * p.v_ts + h * HD, dvr);
  }
  __syncthreads();                                    // every thread is done with the queries: K rows take their place
#pragma unroll
  for (int d = 0; d < HD; ++d) qs[threadIdx.x * HD + d] = kr[d];
  __syncthreads();
  constexpr int DG = HD / 4;
  const long long pbase = ((static_cast<long long>(b) * p.H + h) * p.n_chunks + chunk) * p.Tq;
  for (int o = threadIdx.x; o < p.Tq * DG; o += kSaKeys) {
    const int t = o / DG, d0 = (o % DG) * 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    const float* dr = ds + t * (kSaKeys + 1);
    for (int jj = 0; jj < kSaKeys; ++jj) {
      const float e = dr[jj];
      const float4 k4 = *reinterpret_cast<const float4*>(qs + jj * HD + d0);
      acc.x = fmaf(e, k4.x, acc.x); acc.y = fmaf(e, k4.y, acc.y); acc.z = fmaf(e, k4.z, acc.z); acc.w = fmaf(e, k4.w, acc.w);
    }
    *reinterpret_cast<float4*>(g.part_dq + (pbase + t) * HD + d0) = acc;
  }
}

template <int HD>
__global__ void __launch_bounds__(128)
small_attn_dq_kernel(const float* __restrict__ part_dq, int n_chunks, int Tq, int H, int B, float scale, const float2* rope,
                     int rope_q0, __nv_bfloat16* __restrict__ dq, long long q_bs, long long q_ts) {
  // one thread per (trial, head, query): sums the chunk partials in chunk order, rotates back, writes the row
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(B) * H * Tq) return;
  const int t = static_cast<int>(i % Tq);
  const int h = static_cast<int>((i / Tq) % H);
  const int b = static_cast<int>(i / (static_cast<long long>(Tq) * H));
  float acc[HD];
#pragma unroll
  for (int d = 0; d < HD; ++d) acc[d] = 0.f;
  const long long base = (static_cast<long long>(b) * H + h) * n_chunks;
  for (int c = 0; c < n_chunks; ++c) {
    const float* src = part_dq + ((base + c) * Tq + t) * HD;
#pragma unroll
    for (int d = 0; d < HD; d += 4) {
      const float4 v = *reinterpret_cast<const float4*>(src + d);
      acc[d] += v.x; acc[d + 1] += v.y; acc[d + 2] += v.z; acc[d + 3] += v.w;
    }
  }
#pragma unroll
  for (int d = 0; d < HD; ++d) acc[d] *= scale;
  if (rope != nullptr) rotate<HD>(acc, rope + static_cast<long long>(rope_q0 + t) * (HD / 2), true);
  store_row_bf16<HD>(dq + b * q_bs + static_cast<long long>(t) * q_ts + h * HD, acc);
}

template <int HD>
static int small_attn_smem_fwd() { return (kSaKeys * HD + kSaMaxQ * (kSaKeys + 1) + 8 * kSaMaxQ + kSaMaxQ) * 4; }
template <int HD>
static int small_attn_smem_bwd() { return (kSaKeys * HD + kSaMaxQ * (kSaKeys + 1) + kSaMaxQ * HD + 2 * kSaMaxQ) * 4; }

}  // namespace fk

using namespace fk;

#define FK_API extern "C" __attribute__((visibility("default")))

static bool sa_common_ok(const void* q, const void* k, const void* v, int B, int H, int Tq, int S, int hd, long long q_ts,
                         long long k_ts, long long v_ts) {
  return q && k && v && B > 0 && H > 0 && Tq > 0 && Tq <= kSaMaxQ && S > 0 && (hd == 16 || hd == 32 || hd == 64) &&
         q_ts % 8 == 0 && k_ts % 8 == 0 && v_ts % 8 == 0 && B <= 65535 && H <= 65535;
}

FK_API int fk_small_attn_chunks(int S) { return S > 0 ? (S + kSaKeys - 1) / kSaKeys : FK_ERR_BAD_ARG; }

template <int HD>
static int sa_forward(const SaParams& p, const int* k_len, float* part_o, float* part_ml, __nv_bfloat16* out, long long o_bs,
                      long long o_ts, float* lse, cudaStream_t stream) {
  static bool done[FK_MAX_DEVICES];
  const int dev = fk_device_ordinal();
  const int smem = small_attn_smem_fwd<HD>();
  if (!done[dev]) {
    if (cudaFuncSetAttribute(small_attn_fwd_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) {
      fk_set_last_error("cudaFuncSetAttribute(max dynamic smem) failed", __FILE__, __LINE__);
      return FK_ERR_CUDA;
    }
    done[dev] = true;
  }
  const dim3 grid(static_cast<unsigned>(p.n_chunks), static_cast<unsigned>(p.H), static_cast<unsigned>(p.B));
  small_attn_fwd_kernel<HD><<<grid, kSaKeys, smem, stream>>>(p, k_len, part_o, part_ml);
  FK_CHECK_LAUNCH();
  const long long n = static_cast<long long>(p.B) * p.H * p.Tq * HD;
  small_attn_combine_kernel<HD><<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(part_o, part_ml, p.n_chunks, p.Tq, p.H, p.B,
                                                                                           out, o_bs, o_ts, lse);
  FK_CHECK_LAUNCH();
  fk_count_launch(2);
  return FK_OK;
}

FK_API int fk_small_attn_forward(const void* q, long long q_bs, long long q_ts, const void* k, long long k_bs, long long k_ts,
                                 const void* v, long long v_bs, long long v_ts, void* out, long long o_bs, long long o_ts,
                                 float* lse, int B, int H, int Tq, int S, int head_dim, float scale, const float* rope_table,
                                 int rope_len, int rope_q0, int rope_k0, float* part_o, float* part_ml, const int* k_len,
                                 void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(sa_common_ok(q, k, v, B, H, Tq, S, head_dim, q_ts, k_ts, v_ts) && out && lse && part_o && part_ml && o_ts % 8 == 0,
             "fk_small_attn_forward: bad argument (<= 64 queries, head_dim 16 / 32 / 64, 16-byte aligned rows)");
  FK_REQUIRE(rope_table == nullptr || (rope_q0 >= 0 && rope_k0 >= 0 && rope_q0 + Tq <= rope_len && rope_k0 + S <= rope_len),
             "fk_small_attn_forward: token positions fall outside the rope table");
  SaParams p = {};
  p.q = static_cast<const __nv_bfloat16*>(q); p.k = static_cast<const __nv_bfloat16*>(k); p.v = static_cast<const __nv_bfloat16*>(v);
  p.q_bs = q_bs; p.q_ts = q_ts; p.k_bs = k_bs; p.k_ts = k_ts; p.v_bs = v_bs; p.v_ts = v_ts;
  p.B = B; p.H = H; p.Tq = Tq; p.S = S; p.n_chunks = (S + kSaKeys - 1) / kSaKeys;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.rope = reinterpret_cast<const float2*>(rope_table); p.rope_q0 = rope_q0; p.rope_k0 = rope_k0;
  __nv_bfloat16* o = static_cast<__nv_bfloat16*>(out);
  if (head_dim == 16) return sa_forward<16>(p, k_len, part_o, part_ml, o, o_bs, o_ts, lse, stream);
  if (head_dim == 32) return sa_forward<32>(p, k_len, part_o, part_ml, o, o_bs, o_ts, lse, stream);
  return sa_forward<64>(p, k_len, part_o, part_ml, o, o_bs, o_ts, lse, stream);
}

template <int HD>
static int sa_backward(const SaParams& p, const SaBwdParams& g, __nv_bfloat16* dq, cudaStream_t stream) {
  static bool done[FK_MAX_DEVICES];
  const int dev = fk_device_ordinal();
  const int smem = small_attn_smem_bwd<HD>();
  if (!done[dev]) {
    if (cudaFuncSetAttribute(small_attn_bwd_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) {
      fk_set_last_error("cudaFuncSetAttribute(max dynamic smem) failed", __FILE__, __LINE__);
      return FK_ERR_CUDA;
    }
    done[dev] = true;
  }
  const dim3 grid(static_cast<unsigned>(p.n_chunks), static_cast<unsigned>(p.H), static_cast<unsigned>(p.B));
  small_attn_bwd_kernel<HD><<<grid, kSaKeys, smem, stream>>>(p, g);
  FK_CHECK_LAUNCH();
  const long long n = static_cast<long long>(p.B) * p.H * p.Tq;
  small_attn_dq_kernel<HD><<<static_cast<unsigned>((n + 127) / 128), 128, 0, stream>>>(g.part_dq, p.n_chunks, p.Tq, p.H, p.B, g.scale, p.rope,
                                                                                      p.rope_q0, dq, p.q_bs, p.q_ts);
  FK_CHECK_LAUNCH();
  fk_count_launch(2);
  return FK_OK;
}

FK_API int fk_small_attn_backward(const void* q, long long q_bs, long long q_ts, const void* k, long long k_bs, long long k_ts,
                                  const void* v, long long v_bs, long long v_ts, const void* out, long long o_bs, long long o_ts,
                                  const void* dout, long long do_bs, long long do_ts, const float* lse, void* dq, void* dk,
                                  void* dv, int B, int H, int Tq, int S, int head_dim, float scale, const float* rope_table,
                                  int rope_len, int rope_q0, int rope_k0, float* part_dq, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(sa_common_ok(q, k, v, B, H, Tq, S, head_dim, q_ts, k_ts, v_ts) && out && dout && lse && dq && dk && dv && part_dq &&
                 o_ts % 8 == 0 && do_ts % 8 == 0,
             "fk_small_attn_backward: bad argument (<= 64 queries, head_dim 16 / 32 / 64, 16-byte aligned rows)");
  FK_REQUIRE(rope_table == nullptr || (rope_q0 >= 0 && rope_k0 >= 0 && rope_q0 + Tq <= rope_len && rope_k0 + S <= rope_len),
             "fk_small_attn_backward: token positions fall outside the rope table");
  SaParams p = {};
  p.q = static_cast<const __nv_bfloat16*>(q); p.k = static_cast<const __nv_bfloat16*>(k); p.v = static_cast<const __nv_bfloat16*>(v);
  p.q_bs = q_bs; p.q_ts = q_ts; p.k_bs = k_bs; p.k_ts = k_ts; p.v_bs = v_bs; p.v_ts = v_ts;
  p.B = B; p.H = H; p.Tq = Tq; p.S = S; p.n_chunks = (S + kSaKeys - 1) / kSaKeys;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.rope = reinterpret_cast<const float2*>(rope_table); p.rope_q0 = rope_q0; p.rope_k0 = rope_k0;
  SaBwdParams g = {};
  g.dout = static_cast<const __nv_bfloat16*>(dout); g.out = static_cast<const __nv_bfloat16*>(out);
  g.o_bs = o_bs; g.o_ts = o_ts; g.do_bs = do_bs; g.do_ts = do_ts; g.lse = lse;
  g.dk = static_cast<__nv_bfloat16*>(dk); g.dv = static_cast<__nv_bfloat16*>(dv); g.part_dq = part_dq; g.scale = scale;
  __nv_bfloat16* dqp = static_cast<__nv_bfloat16*>(dq);
  if (head_dim == 16) return sa_backward<16>(p, g, dqp, stream);
  if (head_dim == 32) return sa_backward<32>(p, g, dqp, stream);
  return sa_backward<64>(p, g, dqp, stream);
}
