// Flash-style attention forward / backward with an ANALYTIC mask, head_dim 32 (the reference's
// head_dim in every config: models/brainformer.py:27,49, franky_baseline_gpt2.ipynb cell 5).
//
// Replaces F.scaled_dot_product_attention(q, k, v, attn_mask=<bool tensor>) at
// models/brainformer.py:168 / :215 and models/simple_mae CausalSelfAttention.  The reference passes a
// dense bool mask ([S,S] block-causal buffer, a gathered [B,1,s,s] sub-mask in MAE, or a [B,1,T,T]
// padding mask in simple_mae), which makes SDPA ineligible for its flash kernel and materialises
// B*s*s booleans.  All three masks are instances of ONE rule on per-token integer labels:
//        key j is visible to query i   <=>   kid[b][j] <= qid[b][i]
//   block-causal (brainformer.py:93-111): qid = kid = position / n_electrodes
//   MAE sub-mask (brainformer.py:392-413): the same labels gathered at the kept positions
//   padding      (simple_mae:349-352)    : kid = padded ? INT_MAX : 0,  qid = padded ? -1 : 0
//   no mask                              : qid = kid = null
// so no mask tensor is ever read.  Per-tile label ranges (qmin/qmax/kmin/kmax) skip fully masked
// tiles and drop the per-element compare on fully visible ones.  A query with no visible key yields
// a zero output row (the reference's math path would produce NaN there).
//
// Q/K/V/O are addressed as [batch][token][head][32] with arbitrary token / batch strides, so the
// kernels read q, k, v straight out of the fused QKV projection buffer and write O in the layout the
// output projection consumes: no head transposes.  Scores use bf16 tensor-core MMAs (mma.sync
// m16n8k16, fp32 accumulate) -- at head_dim 32 the kernel is bound by the exp2/softmax work per score,
// not by the MMA rate -- with cp.async double-buffered K/V tiles and an XOR-swizzled smem layout that
// keeps ldmatrix conflict-free.  RoPE (brainformer.py:70-91) is a separate in-place pass (fk_rope).
//
// Backward = three kernels: delta = rowsum(dO * O); dK/dV (one CTA per key tile, loops over query
// tiles, transposed products so nothing is transposed through memory and no atomics are used); dQ
// (one CTA per query tile, loops over key tiles).
#include <climits>

#include "common.cuh"

namespace fk {

constexpr int kHD = 32;            // head dim
constexpr int kTQ = 128;           // rows per CTA (8 warps x 16)
constexpr int kTK = 64;            // streamed tile
constexpr int kAttnThreads = 256;
constexpr float kLog2e = 1.4426950408889634f;

struct AttnParams {
  const __nv_bfloat16 *q, *k, *v, *o, *d_o;   // o/d_o: forward output and its gradient (backward only reads them)
  __nv_bfloat16 *out, *dq, *dk, *dv;
  float *lse;            // [B, H, Sq]  log2-domain logsumexp of the scaled scores
  float *delta;          // [B, H, Sq]
  const int *qid, *kid;  // [B, Sq], [B, Sk] or null
  const int *qmin, *qmax, *kmin, *kmax;   // per 64-token tile label ranges [B, ceil(S/64)] (null when ids are null)
  long long q_bs, q_ts, k_bs, k_ts, v_bs, v_ts, o_bs, o_ts;       // batch / token strides in elements (head stride = 32)
  long long dq_bs, dq_ts, dk_bs, dk_ts, dv_bs, dv_ts, do_bs, do_ts;
  int B, H, Sq, Sk;
  float scale_log2;      // softmax scale * log2(e)
  float scale;
};

// ---- smem tile of [rows][32] bf16 (64 B per row), 16-byte chunks XOR-swizzled by (row>>1)&3 -------------
__device__ __forceinline__ uint32_t tile_off(int row, int chunk) { return row * 64 + ((chunk ^ ((row >> 1) & 3)) << 4); }

__device__ __forceinline__ void cp_async16(uint32_t saddr, const void* g, bool valid) {
  const int sz = valid ? 16 : 0;     // src-size 0 => zero fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(saddr), "l"(g), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// load `rows` x 32 bf16 (row r -> token tok0 + r, zero beyond ntok) into a swizzled tile
template <int ROWS>
__device__ __forceinline__ void load_tile_async(uint32_t sbase, const __nv_bfloat16* g, long long tstride, int tok0, int ntok) {
  for (int i = threadIdx.x; i < ROWS * 4; i += kAttnThreads) {
    const int r = i >> 2, c = i & 3;
    const bool ok = (tok0 + r) < ntok;
    const __nv_bfloat16* src = g + static_cast<long long>(ok ? tok0 + r : 0) * tstride + c * 8;
    cp_async16(sbase + tile_off(r, c), src, ok);
  }
}

__device__ __forceinline__ void ldsm_x4(uint32_t saddr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(saddr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t saddr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(saddr));
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// 2^x on the SFU (ex2.approx.ftz): one MUFU, no range fix-up code around it
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}

// A fragments (16 rows x 32 k) of this warp's rows [row0, row0+16) from a swizzled tile: a[kstep][4]
__device__ __forceinline__ void load_a_frags(uint32_t sbase, int row0, uint32_t (&a)[2][4]) {
  const int lane = threadIdx.x & 31;
  const int r = row0 + (lane & 7) + ((lane >> 3) & 1) * 8;
#pragma unroll
  for (int ks = 0; ks < 2; ++ks) ldsm_x4(sbase + tile_off(r, ks * 2 + (lane >> 4)), a[ks][0], a[ks][1], a[ks][2], a[ks][3]);
}

// acc[nt][4] (16 x 64) = A(16 x 32, registers) * T^T where the tile T is stored [n = 64 rows][k = 32]
__device__ __forceinline__ void mma_a_tileT(float (&acc)[8][4], const uint32_t (&a)[2][4], uint32_t sbase) {
  const int lane = threadIdx.x & 31;
  const int nr = (lane & 7) + (lane >> 4) * 8, kc = (lane >> 3) & 1;
#pragma unroll
  for (int np = 0; np < 4; ++np) {
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
      uint32_t b0, b1, b2, b3;
      ldsm_x4(sbase + tile_off(np * 16 + nr, ks * 2 + kc), b0, b1, b2, b3);
      mma16816(acc[np * 2], a[ks], b0, b1);
      mma16816(acc[np * 2 + 1], a[ks], b2, b3);
    }
  }
}

// out[dt][4] (16 x 32) += P(16 x 64, fp32 accumulators converted to bf16 A fragments) * T where T is stored [k = 64 rows][n = 32]
__device__ __forceinline__ void mma_p_tile(float (&out)[4][4], const float (&pacc)[8][4], uint32_t sbase) {
  const int lane = threadIdx.x & 31;
  const int kr = (lane & 7) + ((lane >> 3) & 1) * 8, nc = lane >> 4;
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    uint32_t a[4];
    a[0] = pack_bf16(pacc[2 * ks][0], pacc[2 * ks][1]);
    a[1] = pack_bf16(pacc[2 * ks][2], pacc[2 * ks][3]);
    a[2] = pack_bf16(pacc[2 * ks + 1][0], pacc[2 * ks + 1][1]);
    a[3] = pack_bf16(pacc[2 * ks + 1][2], pacc[2 * ks + 1][3]);
#pragma unroll
    for (int np = 0; np < 2; ++np) {
      uint32_t b0, b1, b2, b3;
      ldsm_x4_t(sbase + tile_off(ks * 16 + kr, np * 2 + nc), b0, b1, b2, b3);
      mma16816(out[np * 2], a, b0, b1);
      mma16816(out[np * 2 + 1], a, b2, b3);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// forward.  grid = (ceil(Sq/128), H, B)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kAttnThreads, 3)
attn_fwd_kernel(const AttnParams p) {
  __shared__ __align__(128) uint8_t sQ[kTQ * 64];
  __shared__ __align__(128) uint8_t sK[2][kTK * 64];
  __shared__ __align__(128) uint8_t sV[2][kTK * 64];
  __shared__ int sKid[2][kTK];
  const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t4 = lane & 3;
  const int q0 = qt * kTQ;
  const __nv_bfloat16* qg = p.q + b * p.q_bs + h * kHD;
  const __nv_bfloat16* kg = p.k + b * p.k_bs + h * kHD;
  const __nv_bfloat16* vg = p.v + b * p.v_bs + h * kHD;
  const bool masked = p.qid != nullptr;
  const int nkt = (p.Sk + kTK - 1) / kTK, nqt64 = (p.Sq + 63) / 64, nkt64 = nkt;

  // label range of this CTA's 128 queries (two 64-token tiles)
  int tq_min = 0, tq_max = 0;
  if (masked) {
    const int i0 = qt * 2, i1 = min(qt * 2 + 1, nqt64 - 1);
    tq_min = min(p.qmin[b * nqt64 + i0], p.qmin[b * nqt64 + i1]);
    tq_max = max(p.qmax[b * nqt64 + i0], p.qmax[b * nqt64 + i1]);
  }
  auto tile_visible = [&](int kt) { return !masked || p.kmin[b * nkt64 + kt] <= tq_max; };

  const uint32_t sQa = smem_u32(sQ);
  load_tile_async<kTQ>(sQa, qg, p.q_ts, q0, p.Sq);
  cp_async_commit();
  // first visible key tile
  int kt = 0;
  while (kt < nkt && !tile_visible(kt)) ++kt;
  auto issue = [&](int tile, int buf) {
    load_tile_async<kTK>(smem_u32(sK[buf]), kg, p.k_ts, tile * kTK, p.Sk);
    load_tile_async<kTK>(smem_u32(sV[buf]), vg, p.v_ts, tile * kTK, p.Sk);
    if (masked && threadIdx.x < kTK) {
      const int j = tile * kTK + threadIdx.x;
      sKid[buf][threadIdx.x] = (j < p.Sk) ? p.kid[static_cast<long long>(b) * p.Sk + j] : 0;   // (j >= Sk: masked by position)
    }
    cp_async_commit();
  };
  if (kt < nkt) issue(kt, 0);

  cp_async_wait<1>();
  __syncthreads();
  uint32_t qa[2][4];
  load_a_frags(sQa, warp * 16, qa);

  const int r0 = q0 + warp * 16 + g, r1 = r0 + 8;
  int qid0 = 0, qid1 = 0;
  if (masked) {
    qid0 = (r0 < p.Sq) ? p.qid[static_cast<long long>(b) * p.Sq + r0] : -0x7fffffff;
    qid1 = (r1 < p.Sq) ? p.qid[static_cast<long long>(b) * p.Sq + r1] : -0x7fffffff;
  }
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
  float oacc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) oacc[i][j] = 0.f;

  int buf = 0;
  while (kt < nkt) {
    int nxt = kt + 1;
    while (nxt < nkt && !tile_visible(nxt)) ++nxt;
    if (nxt < nkt) issue(nxt, buf ^ 1);
    if (nxt < nkt) cp_async_wait<1>(); else cp_async_wait<0>();
    __syncthreads();

    float s[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) s[i][j] = 0.f;
    mma_a_tileT(s, qa, smem_u32(sK[buf]));

    const bool need_mask = (masked && p.kmax[b * nkt64 + kt] > tq_min) || (kt * kTK + kTK > p.Sk);
    if (need_mask) {           // warp-uniform: only tiles that straddle a label boundary (or the ragged tail) pay for it
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int col = nt * 8 + t4 * 2 + (e & 1);
          const int kid = masked ? sKid[buf][col] : 0;
          const int qid = masked ? ((e & 2) ? qid1 : qid0) : 0;
          // keys past Sk are masked by position: no label value may stand for them, a query labelled INT32_MAX sees every key
          if (kid > qid || kt * kTK + col >= p.Sk) s[nt][e] = -INFINITY;
        }
      }
    }
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      mx0 = fmaxf(mx0, fmaxf(s[nt][0], s[nt][1]));
      mx1 = fmaxf(mx1, fmaxf(s[nt][2], s[nt][3]));
    }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    // running maxima live in the scaled log2 domain; the raw scores are scaled inside the exp2 FFMA
    const float mn0 = fmaxf(m0, mx0 * p.scale_log2), mn1 = fmaxf(m1, mx1 * p.scale_log2);
    const float ms0 = (mn0 == -INFINITY) ? 0.f : mn0, ms1 = (mn1 == -INFINITY) ? 0.f : mn1;
    const float al0 = fast_exp2(m0 - ms0), al1 = fast_exp2(m1 - ms1);
    float rs0 = 0.f, rs1 = 0.f;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      s[nt][0] = fast_exp2(fmaf(s[nt][0], p.scale_log2, -ms0)); s[nt][1] = fast_exp2(fmaf(s[nt][1], p.scale_log2, -ms0));
      s[nt][2] = fast_exp2(fmaf(s[nt][2], p.scale_log2, -ms1)); s[nt][3] = fast_exp2(fmaf(s[nt][3], p.scale_log2, -ms1));
      rs0 += s[nt][0] + s[nt][1];
      rs1 += s[nt][2] + s[nt][3];
    }
    l0 = l0 * al0 + rs0; l1 = l1 * al1 + rs1;
    m0 = mn0; m1 = mn1;
#pragma unroll
    for (int dt = 0; dt < 4; ++dt) { oacc[dt][0] *= al0; oacc[dt][1] *= al0; oacc[dt][2] *= al1; oacc[dt][3] *= al1; }
    mma_p_tile(oacc, s, smem_u32(sV[buf]));
    __syncthreads();          // everyone is done with buf before it is refilled
    kt = nxt;
    buf ^= 1;
  }
  // ---- epilogue: normalise, write O (bf16) and the log2-domain LSE ----
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float inv0 = (l0 > 0.f) ? 1.f / l0 : 0.f, inv1 = (l1 > 0.f) ? 1.f / l1 : 0.f;
  __nv_bfloat16* og = p.out + b * p.o_bs + h * kHD;
#pragma unroll
  for (int dt = 0; dt < 4; ++dt) {
    const int col = dt * 8 + t4 * 2;
    if (r0 < p.Sq) *reinterpret_cast<uint32_t*>(og + static_cast<long long>(r0) * p.o_ts + col) = pack_bf16(oacc[dt][0] * inv0, oacc[dt][1] * inv0);
    if (r1 < p.Sq) *reinterpret_cast<uint32_t*>(og + static_cast<long long>(r1) * p.o_ts + col) = pack_bf16(oacc[dt][2] * inv1, oacc[dt][3] * inv1);
  }
  if (t4 == 0 && p.lse != nullptr) {
    float* lg = p.lse + (static_cast<long long>(b) * p.H + h) * p.Sq;
    if (r0 < p.Sq) lg[r0] = (l0 > 0.f) ? m0 + log2f(l0) : INFINITY;
    if (r1 < p.Sq) lg[r1] = (l1 > 0.f) ? m1 + log2f(l1) : INFINITY;
  }
}

// ------------------------------------------------------------------------------------------------
// delta[b,h,i] = sum_d dO[b,i,h,d] * O[b,i,h,d].   one warp per (b, i): lanes = 16 heads x 2 halves
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
attn_delta_kernel(const AttnParams p) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;   // (b, i, h)
  const long long total = static_cast<long long>(p.B) * p.Sq * p.H;
  if (idx >= total) return;
  const int h = static_cast<int>(idx % p.H);
  const long long bi = idx / p.H;
  const int i = static_cast<int>(bi % p.Sq), b = static_cast<int>(bi / p.Sq);
  const uint4* o = reinterpret_cast<const uint4*>(p.o + b * p.o_bs + static_cast<long long>(i) * p.o_ts + h * kHD);
  const uint4* d = reinterpret_cast<const uint4*>(p.d_o + b * p.do_bs + static_cast<long long>(i) * p.do_ts + h * kHD);
  float acc = 0.f;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const uint4 a = o[c], e = d[c];
    const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, ew[4] = {e.x, e.y, e.z, e.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __nv_bfloat162 x = *reinterpret_cast<const __nv_bfloat162*>(&aw[j]);
      const __nv_bfloat162 y = *reinterpret_cast<const __nv_bfloat162*>(&ew[j]);
      acc += __bfloat162float(x.x) * __bfloat162float(y.x) + __bfloat162float(x.y) * __bfloat162float(y.y);
    }
  }
  p.delta[(static_cast<long long>(b) * p.H + h) * p.Sq + i] = acc;
}

// ------------------------------------------------------------------------------------------------
// dQ.  grid = (ceil(Sq/128), H, B); same loop structure as the forward.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kAttnThreads, 2)
attn_bwd_dq_kernel(const AttnParams p) {
  __shared__ __align__(128) uint8_t sQ[kTQ * 64];
  __shared__ __align__(128) uint8_t sDO[kTQ * 64];
  __shared__ __align__(128) uint8_t sK[2][kTK * 64];
  __shared__ __align__(128) uint8_t sV[2][kTK * 64];
  __shared__ int sKid[2][kTK];
  const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t4 = lane & 3;
  const int q0 = qt * kTQ;
  const __nv_bfloat16* qg = p.q + b * p.q_bs + h * kHD;
  const __nv_bfloat16* kg = p.k + b * p.k_bs + h * kHD;
  const __nv_bfloat16* vg = p.v + b * p.v_bs + h * kHD;
  const __nv_bfloat16* dog = p.d_o + b * p.do_bs + h * kHD;
  const bool masked = p.qid != nullptr;
  const int nkt = (p.Sk + kTK - 1) / kTK, nqt64 = (p.Sq + 63) / 64, nkt64 = nkt;
  int tq_min = 0, tq_max = 0;
  if (masked) {
    const int i0 = qt * 2, i1 = min(qt * 2 + 1, nqt64 - 1);
    tq_min = min(p.qmin[b * nqt64 + i0], p.qmin[b * nqt64 + i1]);
    tq_max = max(p.qmax[b * nqt64 + i0], p.qmax[b * nqt64 + i1]);
  }
  auto tile_visible = [&](int kt) { return !masked || p.kmin[b * nkt64 + kt] <= tq_max; };

  load_tile_async<kTQ>(smem_u32(sQ), qg, p.q_ts, q0, p.Sq);
  load_tile_async<kTQ>(smem_u32(sDO), dog, p.do_ts, q0, p.Sq);
  cp_async_commit();
  int kt = 0;
  while (kt < nkt && !tile_visible(kt)) ++kt;
  auto issue = [&](int tile, int buf) {
    load_tile_async<kTK>(smem_u32(sK[buf]), kg, p.k_ts, tile * kTK, p.Sk);
    load_tile_async<kTK>(smem_u32(sV[buf]), vg, p.v_ts, tile * kTK, p.Sk);
    if (masked && threadIdx.x < kTK) {
      const int j = tile * kTK + threadIdx.x;
      sKid[buf][threadIdx.x] = (j < p.Sk) ? p.kid[static_cast<long long>(b) * p.Sk + j] : 0x7fffffff;
    }
    cp_async_commit();
  };
  if (kt < nkt) issue(kt, 0);
  cp_async_wait<1>();
  __syncthreads();
  uint32_t qa[2][4], doa[2][4];
  load_a_frags(smem_u32(sQ), warp * 16, qa);
  load_a_frags(smem_u32(sDO), warp * 16, doa);

  const int r0 = q0 + warp * 16 + g, r1 = r0 + 8;
  int qid0 = 0, qid1 = 0;
  if (masked) {
    qid0 = (r0 < p.Sq) ? p.qid[static_cast<long long>(b) * p.Sq + r0] : -0x7fffffff;
    qid1 = (r1 < p.Sq) ? p.qid[static_cast<long long>(b) * p.Sq + r1] : -0x7fffffff;
  }
  const float* lg = p.lse + (static_cast<long long>(b) * p.H + h) * p.Sq;
  const float* dg = p.delta + (static_cast<long long>(b) * p.H + h) * p.Sq;
  const float lse0 = (r0 < p.Sq) ? lg[r0] : INFINITY, lse1 = (r1 < p.Sq) ? lg[r1] : INFINITY;
  const float dl0 = (r0 < p.Sq) ? dg[r0] : 0.f, dl1 = (r1 < p.Sq) ? dg[r1] : 0.f;
  float dq[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) dq[i][j] = 0.f;

  int buf = 0;
  while (kt < nkt) {
    int nxt = kt + 1;
    while (nxt < nkt && !tile_visible(nxt)) ++nxt;
    if (nxt < nkt) issue(nxt, buf ^ 1);
    if (nxt < nkt) cp_async_wait<1>(); else cp_async_wait<0>();
    __syncthreads();

    float s[8][4], dp[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) { s[i][j] = 0.f; dp[i][j] = 0.f; }
    mma_a_tileT(s, qa, smem_u32(sK[buf]));
    mma_a_tileT(dp, doa, smem_u32(sV[buf]));
    const bool need_mask = (masked && p.kmax[b * nkt64 + kt] > tq_min) || (kt * kTK + kTK > p.Sk);
    if (need_mask) {
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int col = nt * 8 + t4 * 2 + (e & 1);
          const int kid = masked ? sKid[buf][col] : ((kt * kTK + col < p.Sk) ? 0 : 0x7fffffff);
          const int qid = masked ? ((e & 2) ? qid1 : qid0) : 0;
          if (kid > qid) s[nt][e] = -INFINITY;                 // exp2(-inf) = 0
        }
      }
    }
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      // dS / scale = P * (dP - delta); the softmax scale is applied once to the dQ accumulators at the end
      s[nt][0] = fast_exp2(fmaf(s[nt][0], p.scale_log2, -lse0)) * (dp[nt][0] - dl0);
      s[nt][1] = fast_exp2(fmaf(s[nt][1], p.scale_log2, -lse0)) * (dp[nt][1] - dl0);
      s[nt][2] = fast_exp2(fmaf(s[nt][2], p.scale_log2, -lse1)) * (dp[nt][2] - dl1);
      s[nt][3] = fast_exp2(fmaf(s[nt][3], p.scale_log2, -lse1)) * (dp[nt][3] - dl1);
    }
    mma_p_tile(dq, s, smem_u32(sK[buf]));
    __syncthreads();
    kt = nxt;
    buf ^= 1;
  }
  __nv_bfloat16* og = p.dq + b * p.dq_bs + h * kHD;
#pragma unroll
  for (int dt = 0; dt < 4; ++dt) {
    const int col = dt * 8 + t4 * 2;
    if (r0 < p.Sq) *reinterpret_cast<uint32_t*>(og + static_cast<long long>(r0) * p.dq_ts + col) = pack_bf16(dq[dt][0] * p.scale, dq[dt][1] * p.scale);
    if (r1 < p.Sq) *reinterpret_cast<uint32_t*>(og + static_cast<long long>(r1) * p.dq_ts + col) = pack_bf16(dq[dt][2] * p.scale, dq[dt][3] * p.scale);
  }
}

// ------------------------------------------------------------------------------------------------
// dK, dV.  grid = (ceil(Sk/128), H, B): the CTA owns 128 keys (8 warps x 16) and streams 64-query
// tiles.  Everything is computed transposed (S^T = K Q^T), so P^T and dS^T are already A operands.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kAttnThreads, 2)
attn_bwd_dkv_kernel(const AttnParams p) {
  __shared__ __align__(128) uint8_t sK[kTQ * 64];
  __shared__ __align__(128) uint8_t sV[kTQ * 64];
  __shared__ __align__(128) uint8_t sQ[2][kTK * 64];
  __shared__ __align__(128) uint8_t sDO[2][kTK * 64];
  __shared__ int sQid[2][kTK];
  __shared__ __align__(8) float sLse[2][kTK], sDelta[2][kTK];
  const int kt128 = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t4 = lane & 3;
  const int k0 = kt128 * kTQ;
  const __nv_bfloat16* qg = p.q + b * p.q_bs + h * kHD;
  const __nv_bfloat16* kg = p.k + b * p.k_bs + h * kHD;
  const __nv_bfloat16* vg = p.v + b * p.v_bs + h * kHD;
  const __nv_bfloat16* dog = p.d_o + b * p.do_bs + h * kHD;
  const float* lg = p.lse + (static_cast<long long>(b) * p.H + h) * p.Sq;
  const float* dg = p.delta + (static_cast<long long>(b) * p.H + h) * p.Sq;
  const bool masked = p.qid != nullptr;
  const int nqt = (p.Sq + kTK - 1) / kTK, nkt64 = (p.Sk + 63) / 64;
  int tk_min = 0, tk_max = 0;
  if (masked) {
    const int i0 = kt128 * 2, i1 = min(kt128 * 2 + 1, nkt64 - 1);
    tk_min = min(p.kmin[b * nkt64 + i0], p.kmin[b * nkt64 + i1]);
    tk_max = max(p.kmax[b * nkt64 + i0], p.kmax[b * nkt64 + i1]);
  }
  auto tile_visible = [&](int qt) { return !masked || p.qmax[b * nqt + qt] >= tk_min; };

  load_tile_async<kTQ>(smem_u32(sK), kg, p.k_ts, k0, p.Sk);
  load_tile_async<kTQ>(smem_u32(sV), vg, p.v_ts, k0, p.Sk);
  cp_async_commit();
  int qt = 0;
  while (qt < nqt && !tile_visible(qt)) ++qt;
  auto issue = [&](int tile, int buf) {
    load_tile_async<kTK>(smem_u32(sQ[buf]), qg, p.q_ts, tile * kTK, p.Sq);
    load_tile_async<kTK>(smem_u32(sDO[buf]), dog, p.do_ts, tile * kTK, p.Sq);
    if (threadIdx.x < kTK) {
      const int i = tile * kTK + threadIdx.x;
      const bool ok = i < p.Sq;
      sQid[buf][threadIdx.x] = masked ? (ok ? p.qid[static_cast<long long>(b) * p.Sq + i] : -0x7fffffff) : (ok ? 0 : -0x7fffffff);
      sLse[buf][threadIdx.x] = ok ? lg[i] : INFINITY;
      sDelta[buf][threadIdx.x] = ok ? dg[i] : 0.f;
    }
    cp_async_commit();
  };
  if (qt < nqt) issue(qt, 0);
  cp_async_wait<1>();
  __syncthreads();
  uint32_t ka[2][4], va[2][4];
  load_a_frags(smem_u32(sK), warp * 16, ka);
  load_a_frags(smem_u32(sV), warp * 16, va);
  const int kr0 = k0 + warp * 16 + g, kr1 = kr0 + 8;
  int kid0 = 0x7fffffff, kid1 = 0x7fffffff;
  if (kr0 < p.Sk) kid0 = masked ? p.kid[static_cast<long long>(b) * p.Sk + kr0] : 0;
  if (kr1 < p.Sk) kid1 = masked ? p.kid[static_cast<long long>(b) * p.Sk + kr1] : 0;
  float dk[4][4], dv[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) { dk[i][j] = 0.f; dv[i][j] = 0.f; }

  int buf = 0;
  while (qt < nqt) {
    int nxt = qt + 1;
    while (nxt < nqt && !tile_visible(nxt)) ++nxt;
    if (nxt < nqt) issue(nxt, buf ^ 1);
    if (nxt < nqt) cp_async_wait<1>(); else cp_async_wait<0>();
    __syncthreads();

    float st[8][4], dpt[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) { st[i][j] = 0.f; dpt[i][j] = 0.f; }
    mma_a_tileT(st, ka, smem_u32(sQ[buf]));        // S^T[key, q]
    mma_a_tileT(dpt, va, smem_u32(sDO[buf]));      // dP^T[key, q] = V dO^T
    // label compare only where the tile pair straddles a boundary; out-of-range queries have lse = +inf (P = 0),
    // out-of-range keys only produce rows that are never stored
    const bool need_mask = masked && (tk_max > p.qmin[b * nqt + qt]);
    if (need_mask) {
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int col = nt * 8 + t4 * 2 + (e & 1);
          if (((e & 2) ? kid1 : kid0) > sQid[buf][col]) st[nt][e] = -INFINITY;
        }
      }
    }
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const int col = nt * 8 + t4 * 2;
      const float2 ls = *reinterpret_cast<const float2*>(&sLse[buf][col]);
      const float2 dl = *reinterpret_cast<const float2*>(&sDelta[buf][col]);
      st[nt][0] = fast_exp2(fmaf(st[nt][0], p.scale_log2, -ls.x));       // P^T
      st[nt][1] = fast_exp2(fmaf(st[nt][1], p.scale_log2, -ls.y));
      st[nt][2] = fast_exp2(fmaf(st[nt][2], p.scale_log2, -ls.x));
      st[nt][3] = fast_exp2(fmaf(st[nt][3], p.scale_log2, -ls.y));
      dpt[nt][0] = st[nt][0] * (dpt[nt][0] - dl.x);                      // dS^T / scale
      dpt[nt][1] = st[nt][1] * (dpt[nt][1] - dl.y);
      dpt[nt][2] = st[nt][2] * (dpt[nt][2] - dl.x);
      dpt[nt][3] = st[nt][3] * (dpt[nt][3] - dl.y);
    }
    mma_p_tile(dv, st, smem_u32(sDO[buf]));        // dV += P^T dO
    mma_p_tile(dk, dpt, smem_u32(sQ[buf]));        // dK += dS^T Q
    __syncthreads();
    qt = nxt;
    buf ^= 1;
  }
  __nv_bfloat16* dkg = p.dk + b * p.dk_bs + h * kHD;
  __nv_bfloat16* dvg = p.dv + b * p.dv_bs + h * kHD;
#pragma unroll
  for (int dt = 0; dt < 4; ++dt) {
    const int col = dt * 8 + t4 * 2;
    if (kr0 < p.Sk) {
      *reinterpret_cast<uint32_t*>(dkg + static_cast<long long>(kr0) * p.dk_ts + col) = pack_bf16(dk[dt][0] * p.scale, dk[dt][1] * p.scale);
      *reinterpret_cast<uint32_t*>(dvg + static_cast<long long>(kr0) * p.dv_ts + col) = pack_bf16(dv[dt][0], dv[dt][1]);
    }
    if (kr1 < p.Sk) {
      *reinterpret_cast<uint32_t*>(dkg + static_cast<long long>(kr1) * p.dk_ts + col) = pack_bf16(dk[dt][2] * p.scale, dk[dt][3] * p.scale);
      *reinterpret_cast<uint32_t*>(dvg + static_cast<long long>(kr1) * p.dv_ts + col) = pack_bf16(dv[dt][2], dv[dt][3]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// per 64-token tile min / max of the labels
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(64)
attn_label_range_kernel(const int* __restrict__ ids, int B, int S, int* __restrict__ tmin, int* __restrict__ tmax) {
  const int tile = blockIdx.x, b = blockIdx.y, nt = (S + 63) / 64;
  const int i = tile * 64 + threadIdx.x;
  int lo = 0x7fffffff, hi = -0x7fffffff - 1;         // INT32_MAX / INT32_MIN: both are valid labels
  if (i < S) lo = hi = ids[static_cast<long long>(b) * S + i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  __shared__ int slo[2], shi[2];
  if ((threadIdx.x & 31) == 0) { slo[threadIdx.x >> 5] = lo; shi[threadIdx.x >> 5] = hi; }
  __syncthreads();
  if (threadIdx.x == 0) {
    tmin[b * nt + tile] = min(slo[0], slo[1]);
    tmax[b * nt + tile] = max(shi[0], shi[1]);
  }
}

// ------------------------------------------------------------------------------------------------
// Positions of a streaming step whose trials sit at different positions (fk_stream_positions): thread (i, b) handles new
// token i of trial b at position p = len_in[b] + i.  qid is nondecreasing in i, so a 64-token tile's range is the labels of
// its first and last token.  With per-trial counts (cnt non-null) only the first c = cnt[b] slots are new tokens; a slot
// at or past c gets the query label INT_MIN, which no key label (>= 0) satisfies, a RoPE position inside the table and
// the scratch cache row B * cap, outside every trial's window.  The new slots are a prefix of the trial's slots, so a tile
// holding a padded slot has qmin = INT_MIN and qmax = the label of its last new slot (INT_MIN if it has none).
// ------------------------------------------------------------------------------------------------
constexpr int kNoLabel = INT_MIN;

__global__ void __launch_bounds__(256)
stream_positions_kernel(const int* __restrict__ len_in, const int* __restrict__ cnt, int* __restrict__ len_out, int n_new,
                        int per_label, int cap, int* __restrict__ qid, int* __restrict__ qmin, int* __restrict__ qmax,
                        int* __restrict__ pos, long long* __restrict__ rows) {
  const int b = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_new) return;
  const int L = len_in[b];
  const int c = cnt == nullptr ? n_new : min(max(cnt[b], 0), n_new);
  const int p = L + i;
  const long long o = static_cast<long long>(b) * n_new + i;
  const bool live = i < c;
  qid[o] = live ? p / per_label : kNoLabel;
  pos[o] = min(p, cap - 1);
  rows[o] = static_cast<long long>(live ? b : gridDim.y) * cap + (live ? p : 0);
  if ((i & 63) == 0) {
    const int t = b * ((n_new + 63) >> 6) + (i >> 6);
    const int last = min(i + 63, n_new - 1);
    qmin[t] = last < c ? p / per_label : kNoLabel;
    qmax[t] = live ? (L + min(last, c - 1)) / per_label : kNoLabel;
  }
  if (i == 0) len_out[b] = L + c;
}

// ------------------------------------------------------------------------------------------------
// Positions of a sliding streaming step over ring caches of `cap` tokens (fk_stream_ring_positions): one CTA per trial b.
// New slot i < c = cnt[b] holds the token at the absolute position p = len_in[b] + i (64-bit, unbounded): query label
// p / per_label, cache row b * cap + p mod cap, and the same label as key label of that ring slot.  Slots at or past c get
// kNoLabel, the scratch row B * cap and the RoPE row of position 0.  Once the labels are written, the key tile ranges of
// every 64-slot tile the step wrote are recomputed from the ring.  The RoPE (cos, sin) rows are formed in fp64, from the
// model's fp32 inverse frequencies, and rounded: an fp32 angle p * w loses accuracy past a few thousand tokens.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
stream_ring_positions_kernel(const long long* __restrict__ len_in, const int* __restrict__ cnt, long long* __restrict__ len_out,
                             int n_new, int per_label, int cap, int* __restrict__ qid, int* __restrict__ qmin,
                             int* __restrict__ qmax, long long* __restrict__ rows, int* __restrict__ kid,
                             int* __restrict__ kmin, int* __restrict__ kmax, const float* __restrict__ inv_freq, int half,
                             float2* __restrict__ rope) {
  const int b = blockIdx.x;
  const long long L = len_in[b];
  const int c = cnt == nullptr ? n_new : min(max(cnt[b], 0), n_new);
  const int s0 = static_cast<int>(L % cap);
  for (int i = threadIdx.x; i < n_new; i += blockDim.x) {
    const long long p = L + i;
    const long long o = static_cast<long long>(b) * n_new + i;
    const bool live = i < c;
    const int slot = static_cast<int>(p % cap);
    const int label = static_cast<int>(p / per_label);
    qid[o] = live ? label : kNoLabel;
    rows[o] = live ? static_cast<long long>(b) * cap + slot : static_cast<long long>(gridDim.x) * cap;
    if (live) kid[static_cast<long long>(b) * cap + slot] = label;
    if ((i & 63) == 0) {
      const int t = b * ((n_new + 63) >> 6) + (i >> 6);
      const int last = min(i + 63, n_new - 1);
      qmin[t] = last < c ? label : kNoLabel;
      qmax[t] = live ? static_cast<int>((L + min(last, c - 1)) / per_label) : kNoLabel;
    }
  }
  for (int e = threadIdx.x; e < n_new * half; e += blockDim.x) {
    const int i = e / half, j = e - i * half;
    const double ang = static_cast<double>(i < c ? L + i : 0) * static_cast<double>(inv_freq[j]);
    double sn, cs;
    sincos(ang, &sn, &cs);
    rope[(static_cast<long long>(b) * n_new + i) * half + j] = make_float2(static_cast<float>(cs), static_cast<float>(sn));
  }
  __syncthreads();                                     // the ring's new key labels are visible to the whole CTA
  // a tile [a, a + 64) holds a written slot iff it holds s0 or (a - s0) mod cap < c: the c slots from s0 on, mod cap
  const int ntk = (cap + 63) >> 6, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int t = warp; t < ntk && c > 0; t += blockDim.x >> 5) {
    const int a = t * 64;
    if (!((s0 >= a && s0 < a + 64) || (a - s0 + cap) % cap < c)) continue;
    const int* ring = kid + static_cast<long long>(b) * cap;
    int lo = INT_MAX, hi = INT_MIN;
    for (int x = a + lane; x < min(a + 64, cap); x += 32) {
      lo = min(lo, ring[x]);
      hi = max(hi, ring[x]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
      hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if (lane == 0) {
      kmin[b * ntk + t] = lo;
      kmax[b * ntk + t] = hi;
    }
  }
  if (threadIdx.x == 0) len_out[b] = L + c;
}

// ------------------------------------------------------------------------------------------------
// RoPE (brainformer.py:70-91): adjacent pairs rotated by the cached complex exponentials, fp32 math,
// in place on bf16 [B, S, H, HD] (HD = 16, 32 or 64) with arbitrary token / batch strides.  inverse = conjugate (backward).
// table: [P, HD / 2] float2 (cos, sin); position of token (b, s) = pos ? pos[b*S+s] : s + pos_offset.
// ------------------------------------------------------------------------------------------------
template <int HD>
__global__ void __launch_bounds__(256)
rope_kernel(__nv_bfloat16* __restrict__ x, long long bs, long long ts, int B, int S, int H, const float2* __restrict__ table,
            int P, const int* __restrict__ pos, int pos_offset, int inverse) {
  // one thread = 8 consecutive elements (4 pairs) = one 16-byte chunk, HD / 8 chunks per head
  constexpr int kChunks = HD / 8;
  constexpr int kShift = HD == 16 ? 1 : HD == 32 ? 2 : 3;     // log2(kChunks)
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(B) * S * H * kChunks;
  if (idx >= total) return;
  const int c = static_cast<int>(idx & (kChunks - 1));
  const int h = static_cast<int>((idx >> kShift) % H);
  const long long bsidx = (idx >> kShift) / H;
  const int s = static_cast<int>(bsidx % S), b = static_cast<int>(bsidx / S);
  int ps = pos ? pos[static_cast<long long>(b) * S + s] : s + pos_offset;
  ps = min(max(ps, 0), P - 1);
  uint4* ptr = reinterpret_cast<uint4*>(x + b * bs + static_cast<long long>(s) * ts + h * HD + c * 8);
  uint4 raw = *ptr;
  uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
  const float2* tb = table + static_cast<long long>(ps) * (HD / 2) + c * 4;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162*>(&w[j]);
    const float a = __bfloat162float(v.x), bb = __bfloat162float(v.y);
    const float2 cs = tb[j];
    const float sn = inverse ? -cs.y : cs.y;
    w[j] = pack_bf16(a * cs.x - bb * sn, a * sn + bb * cs.x);
  }
  *ptr = make_uint4(w[0], w[1], w[2], w[3]);
}

}  // namespace fk

using namespace fk;

#define FK_API extern "C" __attribute__((visibility("default")))

static int fill_common(AttnParams& p, int B, int H, int Sq, int Sk, float scale) {
  p.B = B; p.H = H; p.Sq = Sq; p.Sk = Sk;
  p.scale = scale;
  p.scale_log2 = scale * kLog2e;
  return 0;
}

FK_API int fk_attn_label_ranges(const int* ids, int B, int S, int* tmin, int* tmax, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(ids && tmin && tmax && B > 0 && S > 0, "fk_attn_label_ranges: bad argument");
  attn_label_range_kernel<<<dim3((S + 63) / 64, B), 64, 0, stream>>>(ids, B, S, tmin, tmax);
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}

FK_API int fk_stream_positions_counts(const int* len_in, const int* counts, int* len_out, int B, int n_new,
                                      int tokens_per_label, int cap, int* qid, int* qmin, int* qmax, int* pos, long long* rows,
                                      void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(len_in && len_out && len_in != len_out && counts != len_out && qid && qmin && qmax && pos && rows,
             "fk_stream_positions: a buffer is missing, or len_out aliases len_in or counts");
  FK_REQUIRE(B > 0 && B <= 65535 && n_new > 0 && n_new <= cap && tokens_per_label > 0,
             "fk_stream_positions: bad sizes (B in [1, 65535], n_new in [1, cap], tokens_per_label >= 1)");
  stream_positions_kernel<<<dim3((n_new + 255) / 256, B), 256, 0, stream>>>(len_in, counts, len_out, n_new, tokens_per_label,
                                                                             cap, qid, qmin, qmax, pos, rows);
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}

FK_API int fk_stream_ring_positions(const long long* len_in, const int* counts, long long* len_out, int B, int n_new,
                                    int tokens_per_label, int cap, int* qid, int* qmin, int* qmax, long long* rows, int* kid,
                                    int* kmin, int* kmax, const float* inv_freq, int half, float* rope, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(len_in && len_out && len_in != len_out && qid && qmin && qmax && rows && kid && kmin && kmax && inv_freq && rope,
             "fk_stream_ring_positions: a buffer is missing, or len_out aliases len_in");
  FK_REQUIRE(B > 0 && B <= 65535 && n_new > 0 && n_new <= cap && tokens_per_label > 0 && half > 0,
             "fk_stream_ring_positions: bad sizes (B in [1, 65535], n_new in [1, cap], tokens_per_label >= 1, half >= 1)");
  stream_ring_positions_kernel<<<B, 256, 0, stream>>>(len_in, counts, len_out, n_new, tokens_per_label, cap, qid, qmin, qmax,
                                                      rows, kid, kmin, kmax, inv_freq, half, reinterpret_cast<float2*>(rope));
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}

FK_API int fk_stream_positions(const int* len_in, int* len_out, int B, int n_new, int tokens_per_label, int cap, int* qid,
                               int* qmin, int* qmax, int* pos, long long* rows, void* stream_) {
  return fk_stream_positions_counts(len_in, nullptr, len_out, B, n_new, tokens_per_label, cap, qid, qmin, qmax, pos, rows,
                                    stream_);
}

FK_API int fk_attn_forward(const void* q, const void* k, const void* v, void* out, float* lse, int B, int H, int Sq, int Sk,
                           int head_dim, long long q_bs, long long q_ts, long long k_bs, long long k_ts, long long v_bs,
                           long long v_ts, long long o_bs, long long o_ts, const int* qid, const int* kid, const int* qmin,
                           const int* qmax, const int* kmin, const int* kmax, float scale, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(head_dim == kHD, "fk_attn_forward: only head_dim 32 is built");
  FK_REQUIRE(q && k && v && out && B > 0 && H > 0 && Sq > 0 && Sk > 0, "fk_attn_forward: bad argument");
  FK_REQUIRE((qid == nullptr) == (kid == nullptr), "fk_attn_forward: qid and kid go together");
  FK_REQUIRE(qid == nullptr || (qmin && qmax && kmin && kmax), "fk_attn_forward: label ranges missing");
  FK_REQUIRE(q_ts % 8 == 0 && k_ts % 8 == 0 && v_ts % 8 == 0 && o_ts % 2 == 0, "fk_attn_forward: strides must keep 16-byte alignment");
  AttnParams p = {};
  fill_common(p, B, H, Sq, Sk, scale);
  p.q = static_cast<const __nv_bfloat16*>(q); p.k = static_cast<const __nv_bfloat16*>(k); p.v = static_cast<const __nv_bfloat16*>(v);
  p.out = static_cast<__nv_bfloat16*>(out); p.lse = lse;
  p.q_bs = q_bs; p.q_ts = q_ts; p.k_bs = k_bs; p.k_ts = k_ts; p.v_bs = v_bs; p.v_ts = v_ts; p.o_bs = o_bs; p.o_ts = o_ts;
  p.qid = qid; p.kid = kid; p.qmin = qmin; p.qmax = qmax; p.kmin = kmin; p.kmax = kmax;
  attn_fwd_kernel<<<dim3((Sq + kTQ - 1) / kTQ, H, B), kAttnThreads, 0, stream>>>(p);
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}

FK_API int fk_attn_backward(const void* q, const void* k, const void* v, const void* o, const void* d_o, const float* lse,
                            float* delta, void* dq, void* dk, void* dv, int B, int H, int Sq, int Sk, int head_dim,
                            long long q_bs, long long q_ts, long long k_bs, long long k_ts, long long v_bs, long long v_ts,
                            long long o_bs, long long o_ts, long long do_bs, long long do_ts, long long dq_bs, long long dq_ts,
                            long long dk_bs, long long dk_ts, long long dv_bs, long long dv_ts, const int* qid, const int* kid,
                            const int* qmin, const int* qmax, const int* kmin, const int* kmax, float scale, int parts, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(head_dim == kHD, "fk_attn_backward: only head_dim 32 is built");
  FK_REQUIRE(parts > 0 && parts < 8, "fk_attn_backward: parts is a bitmask of 1 (delta), 2 (dK/dV), 4 (dQ)");
  FK_REQUIRE(q && k && v && o && d_o && lse && delta && dq && dk && dv && B > 0 && H > 0 && Sq > 0 && Sk > 0, "fk_attn_backward: bad argument");
  FK_REQUIRE((qid == nullptr) == (kid == nullptr), "fk_attn_backward: qid and kid go together");
  FK_REQUIRE(qid == nullptr || (qmin && qmax && kmin && kmax), "fk_attn_backward: label ranges missing");
  FK_REQUIRE(q_ts % 8 == 0 && k_ts % 8 == 0 && v_ts % 8 == 0 && o_ts % 8 == 0 && do_ts % 8 == 0, "fk_attn_backward: strides must keep 16-byte alignment");
  AttnParams p = {};
  fill_common(p, B, H, Sq, Sk, scale);
  p.q = static_cast<const __nv_bfloat16*>(q); p.k = static_cast<const __nv_bfloat16*>(k); p.v = static_cast<const __nv_bfloat16*>(v);
  p.o = static_cast<const __nv_bfloat16*>(o); p.d_o = static_cast<const __nv_bfloat16*>(d_o);
  p.lse = const_cast<float*>(lse); p.delta = delta;
  p.dq = static_cast<__nv_bfloat16*>(dq); p.dk = static_cast<__nv_bfloat16*>(dk); p.dv = static_cast<__nv_bfloat16*>(dv);
  p.q_bs = q_bs; p.q_ts = q_ts; p.k_bs = k_bs; p.k_ts = k_ts; p.v_bs = v_bs; p.v_ts = v_ts; p.o_bs = o_bs; p.o_ts = o_ts;
  p.do_bs = do_bs; p.do_ts = do_ts; p.dq_bs = dq_bs; p.dq_ts = dq_ts; p.dk_bs = dk_bs; p.dk_ts = dk_ts; p.dv_bs = dv_bs; p.dv_ts = dv_ts;
  p.qid = qid; p.kid = kid; p.qmin = qmin; p.qmax = qmax; p.kmin = kmin; p.kmax = kmax;
  const long long nd = static_cast<long long>(B) * Sq * H;
  int n = 0;
  if (parts & 1) {
    attn_delta_kernel<<<static_cast<unsigned>((nd + 255) / 256), 256, 0, stream>>>(p);
    FK_CHECK_LAUNCH();
    ++n;
  }
  if (parts & 2) {
    attn_bwd_dkv_kernel<<<dim3((Sk + kTQ - 1) / kTQ, H, B), kAttnThreads, 0, stream>>>(p);
    FK_CHECK_LAUNCH();
    ++n;
  }
  if (parts & 4) {
    attn_bwd_dq_kernel<<<dim3((Sq + kTQ - 1) / kTQ, H, B), kAttnThreads, 0, stream>>>(p);
    FK_CHECK_LAUNCH();
    ++n;
  }
  fk_count_launch(n);
  return FK_OK;
}

FK_API int fk_rope(void* x, long long bs, long long ts, int B, int S, int H, int head_dim, const float* table, int P,
                   const int* pos, int pos_offset, int inverse, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(head_dim == 16 || head_dim == 32 || head_dim == 64, "fk_rope: head_dim must be 16, 32 or 64");
  FK_REQUIRE(x && table && B > 0 && S > 0 && H > 0 && P > 0, "fk_rope: bad argument");
  FK_REQUIRE(ts % 8 == 0 && bs % 8 == 0, "fk_rope: strides must keep 16-byte alignment");
  // positions s + pos_offset must lie inside the table (e.g. more tokens than the rope cache holds would make the
  // reference's rope[-T:] slice fail too); explicit positions are the caller's contract ([0, P)) and are clamped
  FK_REQUIRE(pos != nullptr || (pos_offset >= 0 && static_cast<long long>(pos_offset) + S <= P),
             "fk_rope: token positions pos_offset .. pos_offset + S - 1 fall outside the rope table");
  const long long total = static_cast<long long>(B) * S * H * (head_dim / 8);
  auto kern = head_dim == 64 ? rope_kernel<64> : head_dim == 16 ? rope_kernel<16> : rope_kernel<32>;
  kern<<<static_cast<unsigned>((total + 255) / 256), 256, 0, stream>>>(
      static_cast<__nv_bfloat16*>(x), bs, ts, B, S, H, reinterpret_cast<const float2*>(table), P, pos, pos_offset, inverse);
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}
