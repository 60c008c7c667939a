// Helpers of the implicit-GEMM convolutions (conv.py; reference: models/vq_brain.py:22-45 CausalConv1d /
// CausalConvTranspose1d -- `F.pad` on the time axis, and the bias gradients of the convolutions and of nn.Linear):
//
//   pad_rows_kernel         [B, T, C] (fp32 or bf16, row-strided) -> the zero-padded bf16 signal [(B * rpt + slack), C] that the
//                           convolution's TMA reads as overlapping im2col rows: ONE pass that writes the padding zeros and
//                           the data (replaces a memset + a generic strided torch copy that ran at 1.5 TB/s)
//   colsum_partials_kernel  column sums of a bf16 [M, N] matrix (bias gradient = dY^T 1): per-CTA partials [nb, N] in a fixed
//                           order; the caller reduces them with fk_norm_reduce_partials (deterministic)
//   stream_rows_kernel      the GEMM input rows of one STREAMED causal convolution (SoundStream.stream): per trial the h
//                           history rows of the previous step, then act(x + r) for the n new rows (the ELU between layers
//                           and the ResidualUnit's `x + layers(x)`, rounded as the offline bf16 ops round), then zeros;
//                           also writes the next step's history (the last h rows of [history | new rows]); with
//                           per-trial counts of new rows, rows past a trial's count are zeros and never read from x
//
// All HBM-bound: 16-byte accesses, persistent grids of 148 * k CTAs.
#include "common.cuh"
#include "fk_b200.h"

namespace fk {

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}

// one thread = 8 channels of one output row
template <bool kF32>
__global__ void __launch_bounds__(256)
pad_rows_kernel(const void* __restrict__ x_, long long sb, long long st, long long B, long long T, int C8, long long rpt,
                long long left, long long total_rows, __nv_bfloat16* __restrict__ out) {
  const long long n = total_rows * C8;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / C8;
    const int c = static_cast<int>(i - r * C8) * 8;
    const long long b = r / rpt, t = r - b * rpt - left;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (b < B && t >= 0 && t < T) {
      if (kF32) {
        const float* p = static_cast<const float*>(x_) + b * sb + t * st + c;
        const float4 a = *reinterpret_cast<const float4*>(p), d = *reinterpret_cast<const float4*>(p + 4);
        v = make_uint4(pack_bf16x2(a.x, a.y), pack_bf16x2(a.z, a.w), pack_bf16x2(d.x, d.y), pack_bf16x2(d.z, d.w));
      } else {
        v = *reinterpret_cast<const uint4*>(static_cast<const __nv_bfloat16*>(x_) + b * sb + t * st + c);
      }
    }
    *reinterpret_cast<uint4*>(out + r * (C8 * 8ll) + c) = v;
  }
}

__device__ __forceinline__ void load8_f32(const void* base, int f32, long long off, float (&v)[8]) {
  if (f32) {
    const float* p = static_cast<const float*>(base) + off;
    const float4 a = *reinterpret_cast<const float4*>(p), d = *reinterpret_cast<const float4*>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = d.x; v[5] = d.y; v[6] = d.z; v[7] = d.w;
  } else {
    const uint4 q = *reinterpret_cast<const uint4*>(static_cast<const __nv_bfloat16*>(base) + off);
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      v[2 * j] = __uint_as_float(w[j] << 16);
      v[2 * j + 1] = __uint_as_float(w[j] & 0xffff0000u);
    }
  }
}

// new row t of trial b: act(x + r) as bf16.  With r the sum is rounded to bf16 first (torch's bf16 add); ELU (alpha 1) is
// torch's formula, x > 0 ? x : expm1(x) in fp32, so the row equals F.elu of the offline bf16 tensor bit for bit.
__device__ __forceinline__ uint4 stream_new_row(const void* x, int x_f32, long long x_sb, long long x_st,
                                                const __nv_bfloat16* r, long long r_sb, long long r_st, int elu, long long b,
                                                long long t, int c) {
  float v[8];
  load8_f32(x, x_f32, b * x_sb + t * x_st + c, v);
  if (r != nullptr) {
    float a[8];
    load8_f32(r, 0, b * r_sb + t * r_st + c, a);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __bfloat162float(__float2bfloat16_rn(v[j] + a[j]));
  }
  if (elu) {
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = v[j] > 0.f ? v[j] : expm1f(v[j]);
  }
  return make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
}

// one thread = 8 channels of one row; items [0, total_rows * C8) are rows of out, the next B * h * C8 rows of hist_out.
// cnt (nullable): trial b's new rows are its first cnt[b] rows of x; the rest of x is never read, its GEMM rows are zeros
// and the history advances by cnt[b] rows only (cnt[b] = 0 carries it over unchanged).
__global__ void __launch_bounds__(256)
stream_rows_kernel(const void* __restrict__ x, int x_f32, long long x_sb, long long x_st, const __nv_bfloat16* __restrict__ r,
                   long long r_sb, long long r_st, const __nv_bfloat16* __restrict__ hist_in, __nv_bfloat16* __restrict__ hist_out,
                   const int* __restrict__ cnt, long long B, long long n, int h, int C8, int elu, long long rpt,
                   long long total_rows, __nv_bfloat16* __restrict__ out) {
  const long long n_out = total_rows * C8, n_all = n_out + B * h * C8;
  const long long C = C8 * 8ll;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_all;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    long long row, b, t;                       // t = row of trial b in [history | new rows]
    __nv_bfloat16* dst;
    if (i < n_out) {
      row = i / C8;
      b = row / rpt;
      t = row - b * rpt;
      dst = out + row * C;
    } else {
      row = (i - n_out) / C8;                  // hist_out row (b, j) takes row n_b + j of [history | new rows]
      b = row / h;
      t = row - b * h;
      dst = hist_out + row * C;
    }
    const long long nb = (cnt != nullptr && b < B) ? min(max(static_cast<long long>(cnt[b]), 0ll), n) : n;
    if (i >= n_out) t += nb;
    const int c = static_cast<int>(i % C8) * 8;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (b < B && t < h)
      v = *reinterpret_cast<const uint4*>(hist_in + (b * h + t) * C + c);
    else if (b < B && t < h + nb)
      v = stream_new_row(x, x_f32, x_sb, x_st, r, r_sb, r_st, elu, b, t - h, c);
    *reinterpret_cast<uint4*>(dst + c) = v;
  }
}

constexpr int kColsumThreads = 256;

// CTA = (N / 8 column groups, capped at 256) x row groups; rows strided over the grid; partial [blockIdx.x, N]
__global__ void __launch_bounds__(kColsumThreads)
colsum_partials_kernel(const __nv_bfloat16* __restrict__ g, long long M, int N, long long ld, float* __restrict__ part) {
  extern __shared__ float red[];                      // [row groups][N]
  const int n8 = N / 8;
  const int cgs = n8 < kColsumThreads ? n8 : kColsumThreads;          // column groups handled at once
  const int rgs = kColsumThreads / cgs;                                // row groups
  const int cg = threadIdx.x % cgs, rg = threadIdx.x / cgs;
  for (int c0 = 0; c0 < n8; c0 += cgs) {
    const int c = (c0 + cg) * 8;
    float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (rg < rgs && c < N) {
      for (long long r = static_cast<long long>(blockIdx.x) * rgs + rg; r < M; r += static_cast<long long>(gridDim.x) * rgs) {
        const uint4 v = *reinterpret_cast<const uint4*>(g + r * ld + c);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          a[2 * j] += __uint_as_float(w[j] << 16);
          a[2 * j + 1] += __uint_as_float(w[j] & 0xffff0000u);
        }
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) red[rg * (cgs * 8) + cg * 8 + j] = a[j];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < cgs * 8 && c0 * 8 + i < N; i += kColsumThreads) {
      float s = 0.f;
      for (int q = 0; q < rgs; ++q) s += red[q * (cgs * 8) + i];
      part[static_cast<long long>(blockIdx.x) * N + c0 * 8 + i] = s;
    }
    __syncthreads();
  }
}

}  // namespace fk

using namespace fk;

#define FK_API extern "C" __attribute__((visibility("default")))

FK_API int fk_pad_rows(const void* x, int x_dtype, long long B, long long T, int C, long long stride_b, long long stride_t,
                       void* out, long long rows_per_trial, long long left, long long total_rows, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(x && out && B > 0 && T > 0 && C > 0 && C % 8 == 0, "fk_pad_rows: bad argument (C % 8 == 0)");
  FK_REQUIRE(x_dtype == 0 || x_dtype == 1, "fk_pad_rows: x must be f32 (0) or bf16 (1)");
  FK_REQUIRE(rows_per_trial >= left + T && left >= 0 && total_rows >= B * rows_per_trial, "fk_pad_rows: the padded layout does not hold the data");
  FK_REQUIRE(stride_b % 8 == 0 && stride_t % 8 == 0 && stride_t >= C, "fk_pad_rows: row strides must be multiples of 8 elements");
  FK_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0, "fk_pad_rows: 16-byte aligned buffers");
  const long long n = total_rows * (C / 8);
  long long blocks = (n + 255) / 256;
  const long long cap = static_cast<long long>(fk_sm_count()) * 16;
  if (blocks > cap) blocks = cap;
  if (x_dtype == 0)
    pad_rows_kernel<true><<<static_cast<unsigned>(blocks), 256, 0, stream>>>(x, stride_b, stride_t, B, T, C / 8, rows_per_trial, left, total_rows,
                                                                           static_cast<__nv_bfloat16*>(out));
  else
    pad_rows_kernel<false><<<static_cast<unsigned>(blocks), 256, 0, stream>>>(x, stride_b, stride_t, B, T, C / 8, rows_per_trial, left, total_rows,
                                                                            static_cast<__nv_bfloat16*>(out));
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}

FK_API int fk_conv_stream_rows_counts(const void* x, int x_dtype, long long x_sb, long long x_st, const void* r,
                                      long long r_sb, long long r_st, const void* hist_in, void* hist_out, const int* counts,
                                      long long B, long long n, int h, int C, int act, void* out, long long rows_per_trial,
                                      long long total_rows, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(x && out && B > 0 && n > 0 && h >= 0 && C > 0 && C % 8 == 0, "fk_conv_stream_rows: bad argument (n >= 1, C % 8 == 0)");
  FK_REQUIRE(x_dtype == 0 || x_dtype == 1, "fk_conv_stream_rows: x must be f32 (0) or bf16 (1)");
  FK_REQUIRE(act == 0 || act == 1, "fk_conv_stream_rows: act must be 0 (none) or 1 (ELU)");
  FK_REQUIRE(h == 0 || (hist_in && hist_out && hist_in != hist_out), "fk_conv_stream_rows: h > 0 needs two distinct history buffers");
  FK_REQUIRE(rows_per_trial >= h + n && total_rows >= B * rows_per_trial, "fk_conv_stream_rows: the row layout does not hold history and new rows");
  FK_REQUIRE(x_sb % 8 == 0 && x_st % 8 == 0 && x_st >= C && (!r || (r_sb % 8 == 0 && r_st % 8 == 0 && r_st >= C)),
             "fk_conv_stream_rows: row strides must be multiples of 8 elements and >= C");
  FK_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(r) | reinterpret_cast<uintptr_t>(hist_in) |
               reinterpret_cast<uintptr_t>(hist_out) | reinterpret_cast<uintptr_t>(out)) & 15) == 0,
             "fk_conv_stream_rows: 16-byte aligned buffers");
  const long long items = (total_rows + B * h) * (C / 8);
  long long blocks = (items + 255) / 256;
  const long long cap = static_cast<long long>(fk_sm_count()) * 16;
  if (blocks > cap) blocks = cap;
  stream_rows_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(
      x, x_dtype == 0, x_sb, x_st, static_cast<const __nv_bfloat16*>(r), r_sb, r_st, static_cast<const __nv_bfloat16*>(hist_in),
      static_cast<__nv_bfloat16*>(hist_out), counts, B, n, h, C / 8, act, rows_per_trial, total_rows,
      static_cast<__nv_bfloat16*>(out));
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}

FK_API int fk_conv_stream_rows(const void* x, int x_dtype, long long x_sb, long long x_st, const void* r, long long r_sb,
                               long long r_st, const void* hist_in, void* hist_out, long long B, long long n, int h, int C,
                               int act, void* out, long long rows_per_trial, long long total_rows, void* stream_) {
  return fk_conv_stream_rows_counts(x, x_dtype, x_sb, x_st, r, r_sb, r_st, hist_in, hist_out, nullptr, B, n, h, C, act, out,
                                    rows_per_trial, total_rows, stream_);
}

FK_API int fk_colsum_grid(void) { return fk_sm_count() * 4; }

FK_API int fk_colsum_partials(const void* g, long long M, int N, long long ld, float* part, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(g && part && M > 0 && N > 0 && N % 8 == 0 && ld >= N && ld % 8 == 0, "fk_colsum_partials: bad argument (N % 8 == 0, ld % 8 == 0)");
  FK_REQUIRE((reinterpret_cast<uintptr_t>(g) & 15) == 0, "fk_colsum_partials: g must be 16-byte aligned");
  const int n8 = N / 8;
  const int cgs = n8 < kColsumThreads ? n8 : kColsumThreads;
  const int rgs = kColsumThreads / cgs;
  const size_t smem = static_cast<size_t>(rgs) * cgs * 8 * sizeof(float);
  FK_REQUIRE(smem <= 48 * 1024, "fk_colsum_partials: internal staging exceeds 48 KB");
  colsum_partials_kernel<<<fk_colsum_grid(), kColsumThreads, smem, stream>>>(static_cast<const __nv_bfloat16*>(g), M, N, ld, part);
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}
