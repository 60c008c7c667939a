// Bandwidth-bound fused kernels of the transformer blocks: LayerNorm / RMSNorm forward + backward and
// the SwiGLU gate.  One warp per row, 16-byte accesses, fp32 statistics; roofline = HBM.
//
// Reference ops: nn.LayerNorm (models/brainformer.py:237-239,287; eps 1e-5, affine) which the
// reference runs as ATen native_layer_norm; RMSNorm (models/simple_mae:181-192: fp32
// x * rsqrt(mean(x^2) + 1e-6), cast back, times weight -- five eager launches in the reference);
// MLP gate silu(w1 x) * (w3 x) (models/brainformer.py:123-124).
#include "common.cuh"

namespace fk {

constexpr int kNormWarps = 8;

template <typename T> struct Vec4;
template <> struct Vec4<float> {
  static __device__ __forceinline__ void load(const float* p, float (&v)[4]) {
    const float4 t = *reinterpret_cast<const float4*>(p); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  static __device__ __forceinline__ void store(float* p, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};
template <> struct Vec4<__nv_bfloat16> {
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&v)[4]) {
    const uint2 t = *reinterpret_cast<const uint2*>(p);
    const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&t.x), b = *reinterpret_cast<const __nv_bfloat162*>(&t.y);
    v[0] = __bfloat162float(a.x); v[1] = __bfloat162float(a.y); v[2] = __bfloat162float(b.x); v[3] = __bfloat162float(b.y);
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&v)[4]) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
    uint2 t; t.x = *reinterpret_cast<uint32_t*>(&a); t.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(p) = t;
  }
};

// ------------------------------------------------------------------------------------------------
// forward: y = (x - mean) * rstd * w + b   (rms: y = x * rstd * w, rstd = rsqrt(mean(x^2) + eps))
// MAXV = ceil(D / 128) float4 groups per lane (D <= 128 * MAXV)
// ------------------------------------------------------------------------------------------------
template <typename TIn, typename TOut, int MAXV>
__global__ void __launch_bounds__(kNormWarps * 32)
norm_fwd_kernel(const TIn* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias, TOut* __restrict__ y,
                float* __restrict__ mean_out, float* __restrict__ rstd_out, long long M, int D, float eps, int rms,
                const __nv_bfloat16* __restrict__ delta = nullptr, float* __restrict__ x_out = nullptr, long long x_period = 0) {
  // delta / x_out (fp32 residual stream only): x_new = x + delta is written to x_out and normalised, fusing the
  // residual add of the transformer block into the norm that follows it.  x_period > 0: x has only x_period rows
  // and is broadcast over the batch (row % x_period) -- the positional / electrode embedding added to the patch
  // embedding (models/brainformer.py:343) without materialising the sum first.
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * kNormWarps + (threadIdx.x >> 5);
  if (row >= M) return;
  const TIn* xr = x + (x_period > 0 ? row % x_period : row) * D;
  float v[MAXV][4];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int d = (i * 32 + lane) * 4;
    if (d < D) {
      Vec4<TIn>::load(xr + d, v[i]);
      if (delta != nullptr) {
        float dl[4];
        Vec4<__nv_bfloat16>::load(delta + row * D + d, dl);
#pragma unroll
        for (int j = 0; j < 4; ++j) v[i][j] += dl[j];
        Vec4<float>::store(x_out + row * D + d, v[i]);
      }
      s += v[i][0] + v[i][1] + v[i][2] + v[i][3];
    } else { v[i][0] = v[i][1] = v[i][2] = v[i][3] = 0.f; }
  }
  float mean = 0.f;
  if (!rms) mean = warp_sum(s) / D;
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int d = (i * 32 + lane) * 4;
    if (d < D) {
#pragma unroll
      for (int j = 0; j < 4; ++j) { const float c = v[i][j] - mean; ss += c * c; }
    }
  }
  const float rstd = rsqrtf(warp_sum(ss) / D + eps);
  if (lane == 0) {
    if (mean_out) mean_out[row] = mean;
    rstd_out[row] = rstd;
  }
  TOut* yr = y + row * D;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int d = (i * 32 + lane) * 4;
    if (d < D) {
      float wv[4], bv[4] = {0.f, 0.f, 0.f, 0.f}, o[4];
      Vec4<float>::load(w + d, wv);
      if (bias) Vec4<float>::load(bias + d, bv);
#pragma unroll
      for (int j = 0; j < 4; ++j) o[j] = (v[i][j] - mean) * rstd * wv[j] + bv[j];
      Vec4<TOut>::store(yr + d, o);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// backward: dx = rstd * (gw - mean(gw) - xhat * mean(gw * xhat))   (rms: no mean(gw) term)
// dw / db partial sums per CTA -> [gridDim.x, D]; the caller sums the partials.
// Persistent CTAs: each warp strides over rows and keeps its dw/db partials in registers.
// ------------------------------------------------------------------------------------------------
// Software pipelined: a warp issues the loads of its NEXT row (x, dy and the residual-path gradient) before it reduces
// and stores the current one, so every warp keeps a full row (5 KB at D = 512) in flight all the time -- with the loads
// of one row at a time and the residual gradient fetched after the reduction (two dependent DRAM round trips per row)
// the kernel sat at half of the HBM peak.  One CTA of kNormBwdWarps warps per SM, up to 168 registers per thread.
// AHEAD = false (D > 512): the next row's registers, the current row and the dw/db accumulators of MAXV = 8 do not fit
// in 168 registers, so the warp loads its current row at the top of the iteration instead (from L2 when the row is a
// multiple of 16 bytes: the bulk prefetch below puts it there).
constexpr int kNormBwdWarps = 12;
#ifndef FK_NORM_BWD_AHEAD
#define FK_NORM_BWD_AHEAD 2
#endif
constexpr int kNormBwdAhead = FK_NORM_BWD_AHEAD;     // rows per warp in flight (1 in registers, the rest on their way into L2)

template <typename TIn, typename TG, typename TDx, int MAXV, bool AHEAD = true>
__global__ void __launch_bounds__(kNormBwdWarps * 32, 1)
norm_bwd_kernel(const TIn* __restrict__ x, const TG* __restrict__ g, const float* __restrict__ w, const float* __restrict__ mean_in,
                const float* __restrict__ rstd_in, TDx* __restrict__ dx, float* __restrict__ dw_part, float* __restrict__ db_part,
                long long M, int D, int rms, const float* __restrict__ g_res = nullptr, __nv_bfloat16* __restrict__ dx_bf16 = nullptr) {
  // g_res: gradient that reaches x through the residual path (added to dx); dx_bf16: second copy of dx for the
  // bf16 branch of the fused residual add (x_new = x + delta  =>  d delta = d x = dx)
  extern __shared__ float sm[];        // [D] weight, then [kNormBwdWarps][D] for the final reduction
  float* w_s = sm;
  float* red = sm + D;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int d = threadIdx.x; d < D; d += blockDim.x) w_s[d] = w[d];
  __syncthreads();
  float dw[MAXV][4], db[MAXV][4];
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
#pragma unroll
    for (int j = 0; j < 4; ++j) { dw[i][j] = 0.f; db[i][j] = 0.f; }
  }
  const long long stride = static_cast<long long>(gridDim.x) * kNormBwdWarps;
  long long row = static_cast<long long>(blockIdx.x) * kNormBwdWarps + warp;
  const bool has_res = g_res != nullptr;
  float nx[MAXV][4], ng[MAXV][4], nr[MAXV][4], nmean = 0.f, nrstd = 0.f;
  auto clear = [&]() {
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
#pragma unroll
      for (int j = 0; j < 4; ++j) { nx[i][j] = 0.f; ng[i][j] = 0.f; nr[i][j] = 0.f; }
    }
  };
  auto fetch = [&](long long r) {
    nmean = rms ? 0.f : mean_in[r];
    nrstd = rstd_in[r];
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int d = (i * 32 + lane) * 4;
      if (d < D) {
        Vec4<TIn>::load(x + r * D + d, nx[i]);
        Vec4<TG>::load(g + r * D + d, ng[i]);
        if (has_res) Vec4<float>::load(g_res + r * D + d, nr[i]);
      }
    }
  };
  clear();
  // rows further ahead are pulled into L2 by bulk prefetches (one lane, no registers), so that the register loads of the
  // next row find them there: kNormBwdAhead rows per warp on their way from DRAM at any time
  const bool pf_ok = (D * sizeof(TIn)) % 16 == 0 && (D * sizeof(TG)) % 16 == 0;
  auto prefetch_l2 = [&](long long r) {
    if (!pf_ok || r >= M || lane != 0) return;
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(x + r * D), "r"(static_cast<uint32_t>(D * sizeof(TIn))) : "memory");
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(g + r * D), "r"(static_cast<uint32_t>(D * sizeof(TG))) : "memory");
    if (has_res)
      asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(g_res + r * D), "r"(static_cast<uint32_t>(D * sizeof(float))) : "memory");
  };
  if (AHEAD && row < M) fetch(row);
#pragma unroll
  for (int a = 1; a < kNormBwdAhead; ++a) prefetch_l2(row + a * stride);
  for (; row < M; row += stride) {
    prefetch_l2(row + kNormBwdAhead * stride);
    if (!AHEAD) { clear(); fetch(row); }      // (cleared here, so that no register carries over from the last row)
    float xh[MAXV][4], gv[MAXV][4], gr[MAXV][4];
    const float mean = nmean, rstd = nrstd;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
#pragma unroll
      for (int j = 0; j < 4; ++j) { xh[i][j] = nx[i][j]; gv[i][j] = ng[i][j]; gr[i][j] = nr[i][j]; }
    }
    if (AHEAD && row + stride < M) fetch(row + stride);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int d = (i * 32 + lane) * 4;
      if (d < D) {
        float wv[4];
        Vec4<float>::load(w_s + d, wv);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          xh[i][j] = (xh[i][j] - mean) * rstd;
          dw[i][j] += gv[i][j] * xh[i][j];
          db[i][j] += gv[i][j];
          gv[i][j] *= wv[j];                       // gw
          s1 += gv[i][j];
          s2 += gv[i][j] * xh[i][j];
        }
      }
    }
    s1 = rms ? 0.f : warp_sum(s1) / D;
    s2 = warp_sum(s2) / D;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int d = (i * 32 + lane) * 4;
      if (d < D) {
        float o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          o[j] = rstd * (gv[i][j] - s1 - xh[i][j] * s2);
          if (has_res) o[j] += gr[i][j];
        }
        Vec4<TDx>::store(dx + row * D + d, o);
        if (dx_bf16 != nullptr) Vec4<__nv_bfloat16>::store(dx_bf16 + row * D + d, o);
      }
    }
  }
  // CTA reduction of the parameter-gradient partials (dweight, then dbias, through one [warps][D] buffer)
#pragma unroll
  for (int pass = 0; pass < 2; ++pass) {
    if (pass == 1 && db_part == nullptr) break;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int d = (i * 32 + lane) * 4;
      if (d < D) Vec4<float>::store(red + warp * D + d, pass == 0 ? dw[i] : db[i]);
    }
    __syncthreads();
    float* out = pass == 0 ? dw_part : db_part;
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
      float a = 0.f;
#pragma unroll
      for (int wi = 0; wi < kNormBwdWarps; ++wi) a += red[wi * D + d];
      out[static_cast<long long>(blockIdx.x) * D + d] = a;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// SwiGLU gate on the fused [M, 2H] projection (columns [0,H) = w1 x, [H,2H) = w3 x), bf16.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 swiglu8(const uint4 a, const uint4 b) {
  const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
  uint32_t ow[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const __nv_bfloat162 av = *reinterpret_cast<const __nv_bfloat162*>(&aw[j]), bv = *reinterpret_cast<const __nv_bfloat162*>(&bw[j]);
    const float a0 = __bfloat162float(av.x), a1 = __bfloat162float(av.y);
    // silu is rounded to bf16 before the product, as the reference's two separate bf16 ops do
    // (__fdividef: 2-ulp division, one MUFU.RCP instead of the IEEE division sequence; the result is rounded to bf16)
    const float s0 = __bfloat162float(__float2bfloat16_rn(__fdividef(a0, 1.f + __expf(-a0))));
    const float s1 = __bfloat162float(__float2bfloat16_rn(__fdividef(a1, 1.f + __expf(-a1))));
    __nv_bfloat162 o = __floats2bfloat162_rn(s0 * __bfloat162float(bv.x), s1 * __bfloat162float(bv.y));
    ow[j] = *reinterpret_cast<uint32_t*>(&o);
  }
  return make_uint4(ow[0], ow[1], ow[2], ow[3]);
}

__global__ void __launch_bounds__(256)
swiglu_fwd_kernel(const __nv_bfloat16* __restrict__ h13, __nv_bfloat16* __restrict__ y, long long M, int H) {
  const long long idx = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) * 8;
  if (idx >= M * H) return;
  const long long row = idx / H;
  const int c = static_cast<int>(idx % H);
  const uint4 a = *reinterpret_cast<const uint4*>(h13 + row * 2 * H + c);
  const uint4 b = *reinterpret_cast<const uint4*>(h13 + row * 2 * H + H + c);
  *reinterpret_cast<uint4*>(y + idx) = swiglu8(a, b);
}

__global__ void __launch_bounds__(256)
swiglu_bwd_kernel(const __nv_bfloat16* __restrict__ h13, const __nv_bfloat16* __restrict__ gy, __nv_bfloat16* __restrict__ dh13,
                  long long M, int H, int blk) {
  // blk = H: columns [0,H) = w1 x, [H,2H) = w3 x; blk < H: blocks of blk hidden units stored as [w1 block | w3 block]
  // (the layout the fused w1 | w3 GEMM of gemm.cu writes)
  const long long idx = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) * 8;
  if (idx >= M * H) return;
  const long long row = idx / H;
  const int cu = static_cast<int>(idx % H);
  const int c = (cu / blk) * 2 * blk + (cu % blk);
  const int H3 = blk;                       // distance from a unit's w1 column to its w3 column
  const uint4 a = *reinterpret_cast<const uint4*>(h13 + row * 2 * H + c);
  const uint4 b = *reinterpret_cast<const uint4*>(h13 + row * 2 * H + H3 + c);
  const uint4 g = *reinterpret_cast<const uint4*>(gy + idx);
  const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w}, gw[4] = {g.x, g.y, g.z, g.w};
  uint32_t da[4], db[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const __nv_bfloat162 av = *reinterpret_cast<const __nv_bfloat162*>(&aw[j]), bv = *reinterpret_cast<const __nv_bfloat162*>(&bw[j]);
    const __nv_bfloat162 gv = *reinterpret_cast<const __nv_bfloat162*>(&gw[j]);
    float ra[2], rb[2];
    const float aa[2] = {__bfloat162float(av.x), __bfloat162float(av.y)}, bb[2] = {__bfloat162float(bv.x), __bfloat162float(bv.y)};
    const float gg[2] = {__bfloat162float(gv.x), __bfloat162float(gv.y)};
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const float sig = __fdividef(1.f, 1.f + __expf(-aa[e]));
      const float silu = aa[e] * sig;
      ra[e] = gg[e] * bb[e] * sig * (1.f + aa[e] * (1.f - sig));
      rb[e] = gg[e] * silu;
    }
    __nv_bfloat162 oa = __floats2bfloat162_rn(ra[0], ra[1]), ob = __floats2bfloat162_rn(rb[0], rb[1]);
    da[j] = *reinterpret_cast<uint32_t*>(&oa);
    db[j] = *reinterpret_cast<uint32_t*>(&ob);
  }
  *reinterpret_cast<uint4*>(dh13 + row * 2 * H + c) = make_uint4(da[0], da[1], da[2], da[3]);
  *reinterpret_cast<uint4*>(dh13 + row * 2 * H + H3 + c) = make_uint4(db[0], db[1], db[2], db[3]);
}

template <typename TIn, typename TOut>
static int launch_norm_fwd(const void* x, const float* w, const float* b, void* y, float* mean, float* rstd, long long M, int D,
                           float eps, int rms, cudaStream_t stream, const __nv_bfloat16* delta = nullptr, float* x_out = nullptr,
                           long long x_period = 0) {
  const unsigned grid = static_cast<unsigned>((M + kNormWarps - 1) / kNormWarps);
  const TIn* xi = static_cast<const TIn*>(x);
  TOut* yo = static_cast<TOut*>(y);
  if (D <= 128) norm_fwd_kernel<TIn, TOut, 1><<<grid, kNormWarps * 32, 0, stream>>>(xi, w, b, yo, mean, rstd, M, D, eps, rms, delta, x_out, x_period);
  else if (D <= 256) norm_fwd_kernel<TIn, TOut, 2><<<grid, kNormWarps * 32, 0, stream>>>(xi, w, b, yo, mean, rstd, M, D, eps, rms, delta, x_out, x_period);
  else if (D <= 512) norm_fwd_kernel<TIn, TOut, 4><<<grid, kNormWarps * 32, 0, stream>>>(xi, w, b, yo, mean, rstd, M, D, eps, rms, delta, x_out, x_period);
  else if (D <= 1024) norm_fwd_kernel<TIn, TOut, 8><<<grid, kNormWarps * 32, 0, stream>>>(xi, w, b, yo, mean, rstd, M, D, eps, rms, delta, x_out, x_period);
  else return FK_ERR_UNSUPPORTED;
  return FK_OK;
}

template <typename TIn, typename TG, typename TDx>
static int launch_norm_bwd(const void* x, const void* g, const float* w, const float* mean, const float* rstd, void* dx,
                           float* dwp, float* dbp, long long M, int D, int rms, int grid, cudaStream_t stream,
                           const float* g_res = nullptr, __nv_bfloat16* dx_bf16 = nullptr) {
  const TIn* xi = static_cast<const TIn*>(x);
  const TG* gi = static_cast<const TG*>(g);
  TDx* dxo = static_cast<TDx*>(dx);
  const size_t smem = static_cast<size_t>(kNormBwdWarps + 1) * D * sizeof(float);
  if (D <= 128) norm_bwd_kernel<TIn, TG, TDx, 1><<<grid, kNormBwdWarps * 32, smem, stream>>>(xi, gi, w, mean, rstd, dxo, dwp, dbp, M, D, rms, g_res, dx_bf16);
  else if (D <= 256) norm_bwd_kernel<TIn, TG, TDx, 2><<<grid, kNormBwdWarps * 32, smem, stream>>>(xi, gi, w, mean, rstd, dxo, dwp, dbp, M, D, rms, g_res, dx_bf16);
  else if (D <= 512) norm_bwd_kernel<TIn, TG, TDx, 4><<<grid, kNormBwdWarps * 32, smem, stream>>>(xi, gi, w, mean, rstd, dxo, dwp, dbp, M, D, rms, g_res, dx_bf16);
  else if (D <= 1024) {
    // above D = 944 the shared memory exceeds the default 48 KB limit of a launch: opt in once per device
    static bool done[FK_MAX_DEVICES];
    const int dev = fk_device_ordinal();
    if (!done[dev]) {
      if (cudaFuncSetAttribute(norm_bwd_kernel<TIn, TG, TDx, 8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (kNormBwdWarps + 1) * 1024 * static_cast<int>(sizeof(float))) != cudaSuccess) {
        fk_set_last_error("cudaFuncSetAttribute(max dynamic smem) failed", __FILE__, __LINE__);
        return FK_ERR_CUDA;
      }
      done[dev] = true;
    }
    norm_bwd_kernel<TIn, TG, TDx, 8, false><<<grid, kNormBwdWarps * 32, smem, stream>>>(xi, gi, w, mean, rstd, dxo, dwp, dbp, M, D, rms, g_res, dx_bf16);
  } else return FK_ERR_UNSUPPORTED;
  return FK_OK;
}

}  // namespace fk

using namespace fk;

#define FK_API extern "C" __attribute__((visibility("default")))

// dtype codes: 0 = f32, 1 = bf16
FK_API int fk_norm_forward(const void* x, int x_dtype, const float* weight, const float* bias, void* y, int y_dtype,
                           float* mean, float* rstd, long long M, int D, float eps, int rms, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(x && weight && y && rstd && M > 0 && D > 0 && D % 4 == 0, "fk_norm_forward: bad argument (D % 4 == 0)");
  FK_REQUIRE(rms || mean, "fk_norm_forward: LayerNorm needs the mean buffer");
  int rc = FK_ERR_UNSUPPORTED;
  if (x_dtype == 0 && y_dtype == 1) rc = launch_norm_fwd<float, __nv_bfloat16>(x, weight, bias, y, mean, rstd, M, D, eps, rms, stream);
  else if (x_dtype == 0 && y_dtype == 0) rc = launch_norm_fwd<float, float>(x, weight, bias, y, mean, rstd, M, D, eps, rms, stream);
  else if (x_dtype == 1 && y_dtype == 1) rc = launch_norm_fwd<__nv_bfloat16, __nv_bfloat16>(x, weight, bias, y, mean, rstd, M, D, eps, rms, stream);
  if (rc != FK_OK) { fk_set_last_error("fk_norm_forward: unsupported dtype combination or D > 1024", __FILE__, __LINE__); return rc; }
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}

FK_API int fk_norm_backward_grid(void) { return 148; }

// dweight / dbias = column sums of the per-block partials [nb, D] of fk_norm_backward / fk_add_norm_backward: both in ONE
// launch, rows added in a fixed order (deterministic).
__global__ void __launch_bounds__(256)
norm_partials_reduce_kernel(const float* __restrict__ dw_part, const float* __restrict__ db_part, int nb, int D,
                            float* __restrict__ dw, float* __restrict__ db) {
  // block = 8 columns x 32 row groups (D / 8 blocks: enough CTAs in flight for a 2.4 MB read)
  __shared__ float red[2][32][9];
  const int cl = threadIdx.x & 7, rg = threadIdx.x >> 3;
  const int c = blockIdx.x * 8 + cl;
  float a = 0.f, b = 0.f;
  if (c < D) {
    for (int r = rg; r < nb; r += 32) {
      a += dw_part[static_cast<long long>(r) * D + c];
      if (db_part != nullptr) b += db_part[static_cast<long long>(r) * D + c];
    }
  }
  red[0][rg][cl] = a;
  red[1][rg][cl] = b;
  __syncthreads();
  if (rg == 0 && c < D) {
    float sa = 0.f, sb = 0.f;
#pragma unroll 8
    for (int g = 0; g < 32; ++g) { sa += red[0][g][cl]; sb += red[1][g][cl]; }
    dw[c] = sa;
    if (db_part != nullptr) db[c] = sb;
  }
}

FK_API int fk_norm_reduce_partials(const float* dw_part, const float* db_part, int nb, int D, float* dw, float* db, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(dw_part && dw && nb > 0 && D > 0 && (db_part == nullptr || db != nullptr), "fk_norm_reduce_partials: bad argument");
  norm_partials_reduce_kernel<<<static_cast<unsigned>((D + 7) / 8), 256, 0, stream>>>(dw_part, db_part, nb, D, dw, db);
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}

FK_API int fk_norm_backward(const void* x, int x_dtype, const void* g, int g_dtype, const float* weight, const float* mean,
                            const float* rstd, void* dx, int dx_dtype, float* dw_part, float* db_part, long long M, int D,
                            int rms, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(x && g && weight && rstd && dx && dw_part && M > 0 && D > 0 && D % 4 == 0, "fk_norm_backward: bad argument");
  FK_REQUIRE(rms || mean, "fk_norm_backward: LayerNorm needs the mean buffer");
  const int grid = fk_norm_backward_grid();
  int rc = FK_ERR_UNSUPPORTED;
  if (x_dtype == 0 && g_dtype == 1 && dx_dtype == 0) rc = launch_norm_bwd<float, __nv_bfloat16, float>(x, g, weight, mean, rstd, dx, dw_part, db_part, M, D, rms, grid, stream);
  else if (x_dtype == 0 && g_dtype == 0 && dx_dtype == 0) rc = launch_norm_bwd<float, float, float>(x, g, weight, mean, rstd, dx, dw_part, db_part, M, D, rms, grid, stream);
  else if (x_dtype == 1 && g_dtype == 1 && dx_dtype == 1) rc = launch_norm_bwd<__nv_bfloat16, __nv_bfloat16, __nv_bfloat16>(x, g, weight, mean, rstd, dx, dw_part, db_part, M, D, rms, grid, stream);
  if (rc == FK_ERR_UNSUPPORTED) fk_set_last_error("fk_norm_backward: unsupported dtype combination or D > 1024", __FILE__, __LINE__);
  if (rc != FK_OK) return rc;
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}

FK_API int fk_swiglu_forward(const void* h13, void* y, long long M, int H, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(h13 && y && M > 0 && H > 0 && H % 8 == 0, "fk_swiglu_forward: bad argument (H % 8 == 0)");
  const long long n = M * H / 8;
  swiglu_fwd_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(h13),
                                                                                static_cast<__nv_bfloat16*>(y), M, H);
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}

FK_API int fk_swiglu_backward(const void* h13, const void* gy, void* dh13, long long M, int H, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(h13 && gy && dh13 && M > 0 && H > 0 && H % 8 == 0, "fk_swiglu_backward: bad argument (H % 8 == 0)");
  const long long n = M * H / 8;
  swiglu_bwd_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(
      static_cast<const __nv_bfloat16*>(h13), static_cast<const __nv_bfloat16*>(gy), static_cast<__nv_bfloat16*>(dh13), M, H, H);
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}

// Same on the block-interleaved projection the fused w1 | w3 GEMM (fk_gemm_nt, epilogue 2) writes: blocks of `block` hidden
// units stored as [w1 block | w3 block]; gy [M, H] is in plain hidden-unit order.
FK_API int fk_swiglu_backward_blocked(const void* h13, const void* gy, void* dh13, long long M, int H, int block, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(h13 && gy && dh13 && M > 0 && H > 0 && block > 0 && block % 8 == 0 && H % block == 0,
             "fk_swiglu_backward_blocked: bad argument (block % 8 == 0, H % block == 0)");
  const long long n = M * H / 8;
  swiglu_bwd_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(
      static_cast<const __nv_bfloat16*>(h13), static_cast<const __nv_bfloat16*>(gy), static_cast<__nv_bfloat16*>(dh13), M, H, block);
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}

// Fused residual add + norm (fp32 residual stream): x_new = x + delta (bf16), y = norm(x_new).  Replaces the pair
// `x = x + branch(...)` ; `ln(x)` of models/brainformer.py:243-244 (one pass over the residual stream instead of two).
// x_period > 0: x holds x_period rows and is broadcast over the batch (embedding + patch projection, brainformer.py:343).
FK_API int fk_add_norm_forward(const float* x, const void* delta_bf16, const float* weight, const float* bias, float* x_out,
                               void* y, int y_dtype, float* mean, float* rstd, long long M, int D, float eps, int rms,
                               long long x_period, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(x && delta_bf16 && weight && x_out && y && rstd && M > 0 && D > 0 && D % 4 == 0, "fk_add_norm_forward: bad argument");
  FK_REQUIRE(rms || mean, "fk_add_norm_forward: LayerNorm needs the mean buffer");
  FK_REQUIRE(x_period >= 0 && (x_period == 0 || M % x_period == 0), "fk_add_norm_forward: M must be a multiple of x_period");
  const __nv_bfloat16* dl = static_cast<const __nv_bfloat16*>(delta_bf16);
  int rc = FK_ERR_UNSUPPORTED;
  if (y_dtype == 1) rc = launch_norm_fwd<float, __nv_bfloat16>(x, weight, bias, y, mean, rstd, M, D, eps, rms, stream, dl, x_out, x_period);
  else if (y_dtype == 0) rc = launch_norm_fwd<float, float>(x, weight, bias, y, mean, rstd, M, D, eps, rms, stream, dl, x_out, x_period);
  if (rc != FK_OK) { fk_set_last_error("fk_add_norm_forward: unsupported dtype or D > 1024", __FILE__, __LINE__); return rc; }
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}

// Backward of the fused op: dx = norm_backward(g_y) + g_res (g_res nullable: gradient arriving at x_new through the
// residual path); writes dx as fp32 (gradient of x) and, if dx_bf16 != NULL, a bf16 copy (gradient of delta).
FK_API int fk_add_norm_backward(const float* x_new, const void* g_y, int g_dtype, const float* g_res, const float* weight,
                                const float* mean, const float* rstd, float* dx, void* dx_bf16, float* dw_part, float* db_part,
                                long long M, int D, int rms, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(x_new && g_y && weight && rstd && dx && dw_part && M > 0 && D > 0 && D % 4 == 0, "fk_add_norm_backward: bad argument");
  FK_REQUIRE(rms || mean, "fk_add_norm_backward: LayerNorm needs the mean buffer");
  const int grid = fk_norm_backward_grid();
  __nv_bfloat16* db16 = static_cast<__nv_bfloat16*>(dx_bf16);
  int rc = FK_ERR_UNSUPPORTED;
  if (g_dtype == 1) rc = launch_norm_bwd<float, __nv_bfloat16, float>(x_new, g_y, weight, mean, rstd, dx, dw_part, db_part, M, D, rms, grid, stream, g_res, db16);
  else if (g_dtype == 0) rc = launch_norm_bwd<float, float, float>(x_new, g_y, weight, mean, rstd, dx, dw_part, db_part, M, D, rms, grid, stream, g_res, db16);
  if (rc == FK_ERR_UNSUPPORTED) fk_set_last_error("fk_add_norm_backward: unsupported dtype or D > 1024", __FILE__, __LINE__);
  if (rc != FK_OK) return rc;
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}
