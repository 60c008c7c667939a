// Dense bf16 GEMMs of the transformer blocks on the 5th-gen tensor cores (tcgen05.mma, fp32 accumulators in TMEM,
// operands staged by TMA), with the elementwise work that follows each projection fused into the epilogue.
//
// Replaces (reference call sites, models/brainformer.py): the bias-free Linears qw / kw / vw (:141-143, one fused
// projection) with apply_rope (:70-91, :156-158) in the epilogue; project (:171); the SwiGLU MLP w1 / w3 (:119-124, one
// fused projection whose epilogue forms silu(w1 x) * (w3 x)) and w2; and their autograd: dX = dY W (same kernel on a
// transposed weight copy) and dW = dY^T X (fk_gemm_tn, both operands read MN-major straight from the row-major
// activations, split over the token dimension).
//
// Three kernels, all persistent (one CTA per SM), warp-specialised like vq_search.cu: warp 0 = TMA producer,
// warp 1 = MMA issuer (whole-warp loop, one elected lane issues), warp 2 = TMEM allocator, warps 4-11 = epilogue.
//
//   gemm_res_kernel   C[M,N] = A[M,K] B[N,K]^T, K <= 512.  The A row block (128 rows x K) stays RESIDENT in shared memory
//                     for all N tiles of the block, only B streams (256-column tiles, 32 KB k-slabs through an mbarrier
//                     ring), accumulators double buffered in TMEM (2 x 256 columns) so the epilogue of tile j overlaps the
//                     MMAs of tile j+1.  The next block's A slabs are loaded one by one as the last tile releases them.
//   gemm_stream_kernel  same product for long K: 256 x 256 tiles (two M=128 halves share each B slab), both operands
//                     streamed, the 512 TMEM columns hold one tile (the epilogue is exposed once per long K loop).
//   gemm_tn_kernel    out[Na,Nb] (fp32) = A[M,Na]^T B[M,Nb] over a range of rows: 256 x 256 tiles, both operands MN-major
//                     (64-column chunks of 64 rows, 128-byte swizzle), partial sums per row range written to a workspace
//                     and added up in a fixed order by gemm_tn_reduce_kernel (deterministic, no atomics).
//
// L2 -> SM traffic bounds these shapes as much as the tensor pipe does (K is only 512..4096): a 128-row resident block or
// a 256 x 256 streamed tile needs one operand byte per 128 flops, about what the L2 fabric delivers at the bf16 peak.
#include "common.cuh"
#include "fk_b200.h"
#include "tma_host.cuh"

namespace fk {

constexpr int kGemmThreads = 384;          // 4 control warps + 8 epilogue warps
constexpr int kASlabBytes = 128 * 128;     // 128 rows x 64 bf16
constexpr int kBSlabBytes = 256 * 128;     // 256 rows x 64 bf16
constexpr int kGemmSmemLimit = 232448 - 1024;

// (epilogue 3 was a SwiGLU backward in the epilogue, removed; the numbers of the others are part of the C ABI)
enum { EPI_STORE = 0, EPI_ROPE = 1, EPI_SWIGLU = 2, EPI_ROPE64 = 4, EPI_ROPE16 = 5 };
// (cos, sin) pairs one epilogue thread holds for its row: one head of 32 columns, of 64 columns (EPI_ROPE64) or of 16
// columns (EPI_ROPE16)
template <int EPI> constexpr int rope_pairs() { return EPI == EPI_ROPE64 ? 32 : EPI == EPI_ROPE16 ? 8 : 16; }
template <int EPI> constexpr bool is_rope() { return EPI == EPI_ROPE || EPI == EPI_ROPE64 || EPI == EPI_ROPE16; }

struct GemmParams {
  __nv_bfloat16* C;          // [M, N] (EPI_SWIGLU: the fused projection h13)
  long long ldc;
  __nv_bfloat16* C2;         // EPI_SWIGLU: gated [M, N/2]
  long long ldc2;
  const float* bias;         // [N] or null (EPI_STORE)
  const float2* rope_table;  // EPI_ROPE: [rope_len][16] (cos, sin); EPI_ROPE64: [rope_len][32]; EPI_ROPE16: [rope_len][8]
  const int* rope_pos;       // [M] or null: position of row m = rope_pos ? rope_pos[m] : (m % rope_S) + rope_offset
  int rope_len, rope_offset, rope_cols, rope_S;
  long long M;
  int N, K, nslab, ntile, nstage;
};

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float bf16_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }

__device__ __forceinline__ void tmem_wait_ld32(uint32_t (&a)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]),
                 "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]),
                 "+r"(a[16]), "+r"(a[17]), "+r"(a[18]), "+r"(a[19]), "+r"(a[20]), "+r"(a[21]), "+r"(a[22]), "+r"(a[23]),
                 "+r"(a[24]), "+r"(a[25]), "+r"(a[26]), "+r"(a[27]), "+r"(a[28]), "+r"(a[29]), "+r"(a[30]), "+r"(a[31])
               :: "memory");
}

// MN-major operand tile written by TMA with the 128-byte swizzle as [chunk][64 k-rows][64 elements]: the canonical
// layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units -- LBO = distance between 64-element chunks along M/N,
// SBO = distance between 8-row groups along K (1024 B).  A K step of 16 rows adds 2048 B to the start address.
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t saddr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// 32 fp32 accumulator columns of one row -> 32 bf16 (64 bytes) at dst (16-byte aligned)
__device__ __forceinline__ void store32_bf16(__nv_bfloat16* dst, const float (&v)[32]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    *reinterpret_cast<uint4*>(dst + i * 8) =
        make_uint4(pack_bf16(v[i * 8], v[i * 8 + 1]), pack_bf16(v[i * 8 + 2], v[i * 8 + 3]),
                   pack_bf16(v[i * 8 + 4], v[i * 8 + 5]), pack_bf16(v[i * 8 + 6], v[i * 8 + 7]));
  }
}
__device__ __forceinline__ void load32_bf16(const __nv_bfloat16* src, float (&v)[32]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint4 w = *reinterpret_cast<const uint4*>(src + i * 8);
    v[i * 8] = bf16_lo(w.x); v[i * 8 + 1] = bf16_hi(w.x); v[i * 8 + 2] = bf16_lo(w.y); v[i * 8 + 3] = bf16_hi(w.y);
    v[i * 8 + 4] = bf16_lo(w.z); v[i * 8 + 5] = bf16_hi(w.z); v[i * 8 + 6] = bf16_lo(w.w); v[i * 8 + 7] = bf16_hi(w.w);
  }
}
__device__ __forceinline__ void to_f32(const uint32_t (&r)[32], float (&v)[32]) {
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
// (__fdividef: one MUFU.RCP + multiply instead of the IEEE division sequence -- the gate epilogue is bound by the length of
//  each epilogue warp's instruction stream, not by any pipe)
__device__ __forceinline__ float sigmoidf_fast(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }

// ---- coalesced epilogue stores through a per-warp 2 KB staging tile (16 rows x 128 bytes, two passes per 32 rows) -------
// An accumulator row belongs to one thread (TMEM lane = row), so direct stores are 32 rows x 16 bytes per instruction:
// 32 half-used sectors -- measured, that store path (not the tensor pipe, not L2 reads) paced the A-resident kernel at
// ~1.9 TB/s of output.  Instead each pass writes 16 rows into the staging tile and the TMA store engine writes the tile
// out in full 128-byte lines.  16-byte pieces are XOR-swizzled with (row & 7), which IS the 128-byte TMA swizzle and keeps
// the row-wise writes conflict free; rows / columns outside the tensor are clipped by the hardware.
// Lane l holds columns 0..63 of row (row0 + l) as 32 packed bf16 pairs.
// A warp's staging area holds `tiles` (1 or 2) such tiles used round-robin (`cnt` = passes so far): with two, the store of
// one pass is still reading its tile while the next pass fills the other.
__device__ __forceinline__ void warp_store_32x64_tma(uint8_t* stg0, int tiles, uint32_t& cnt, int lane, const uint32_t (&w)[32],
                                                     const CUtensorMap* tm, int col, long long row0) {
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    uint8_t* stg = stg0 + ((tiles == 2) ? (cnt & 1u) * 2048u : 0u);
    ++cnt;
    if (lane == 0) {                                                                   // the store that last used this tile has read it
      if (tiles == 2) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      else asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
    __syncwarp();
    if ((lane >> 4) == half) {
      const int r = lane & 15;
#pragma unroll
      for (int pc = 0; pc < 8; ++pc)
        *reinterpret_cast<uint4*>(stg + r * 128 + ((pc ^ (r & 7)) << 4)) = make_uint4(w[4 * pc], w[4 * pc + 1], w[4 * pc + 2], w[4 * pc + 3]);
    }
    fence_proxy_async();                            // generic-proxy writes -> visible to the async proxy (TMA)
    __syncwarp();
    if (lane == 0) {
      asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];"
                   ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(col), "r"(static_cast<int>(row0) + half * 16), "r"(smem_u32(stg))
                   : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
  }
}
// One 128 x 256 accumulator tile of the A-resident kernels: this warp's 32 rows (TMEM lane quarter) x 128 columns (half ch).
template <int EPI, int NCS, class Release>
__device__ __forceinline__ void res_epilogue_tile(const GemmParams& p, const CUtensorMap& tm_c, const CUtensorMap& tm_c2, uint8_t* stg,
                                                  int stg_tiles, uint32_t& stg_cnt, int lane, int ch, uint32_t taddr, int n0,
                                                  long long row0, const float2 (&cs)[NCS], uint64_t* full_bar, uint32_t full_parity,
                                                  Release release) {
    if (EPI == EPI_STORE || is_rope<EPI>()) {
      mbar_wait(full_bar, full_parity);
      tc_fence_after();
#pragma unroll
      for (int dc = 0; dc < 2; ++dc) {               // two 64-column halves of this warp's 128 columns
        uint32_t r0[32], r1[32];
        tmem_ld32(taddr + ch * 128 + dc * 64, r0);
        tmem_ld32(taddr + ch * 128 + dc * 64 + 32, r1);
        tmem_wait_ld32(r0);
        tmem_wait_ld32(r1);
        if (dc == 1) release();
        const int col = n0 + ch * 128 + dc * 64;
        uint32_t w[32];
#pragma unroll
        for (int hc = 0; hc < 2; ++hc) {
          float v[32];
          if (hc == 0) to_f32(r0, v); else to_f32(r1, v);
          if (is_rope<EPI>()) {
            if (col + hc * 32 < p.rope_cols) {
              const int c0 = (EPI == EPI_ROPE64) ? hc * 16 : 0;     // a 64-column head spans both 32-column halves
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const int ci = (EPI == EPI_ROPE16) ? (i & 7) : c0 + i;   // two 16-column heads per 32-column half
                const float x0 = v[2 * i], x1 = v[2 * i + 1];
                v[2 * i] = x0 * cs[ci].x - x1 * cs[ci].y;
                v[2 * i + 1] = x0 * cs[ci].y + x1 * cs[ci].x;
              }
            }
          } else if (p.bias != nullptr && col + hc * 32 < p.N) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + col + hc * 32) + i);
              v[4 * i] += b4.x; v[4 * i + 1] += b4.y; v[4 * i + 2] += b4.z; v[4 * i + 3] += b4.w;
            }
          }
#pragma unroll
          for (int i = 0; i < 16; ++i) w[hc * 16 + i] = pack_bf16(v[2 * i], v[2 * i + 1]);
        }
        if (col < p.N) warp_store_32x64_tma(stg, stg_tiles, stg_cnt, lane, w, &tm_c, col, row0);
      }
    } else {   // EPI_SWIGLU
      // tile columns: [0,128) = w1 block, [128,256) = w3 block of the same 128 hidden units (weights interleaved by the
      // host in blocks of 128).  This warp: hidden units ch*64 .. ch*64+63 of the block.
      mbar_wait(full_bar, full_parity);
      tc_fence_after();
      uint32_t wa[32], wb[32];
      {
        uint32_t r0[32], r1[32];
        tmem_ld32(taddr + ch * 64, r0);
        tmem_ld32(taddr + ch * 64 + 32, r1);
        tmem_wait_ld32(r0);
        tmem_wait_ld32(r1);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          wa[i] = pack_bf16(__uint_as_float(r0[2 * i]), __uint_as_float(r0[2 * i + 1]));
          wa[16 + i] = pack_bf16(__uint_as_float(r1[2 * i]), __uint_as_float(r1[2 * i + 1]));
        }
        tmem_ld32(taddr + 128 + ch * 64, r0);
        tmem_ld32(taddr + 128 + ch * 64 + 32, r1);
        tmem_wait_ld32(r0);
        tmem_wait_ld32(r1);
        release();
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          wb[i] = pack_bf16(__uint_as_float(r0[2 * i]), __uint_as_float(r0[2 * i + 1]));
          wb[16 + i] = pack_bf16(__uint_as_float(r1[2 * i]), __uint_as_float(r1[2 * i + 1]));
        }
      }
      const int ca = n0 + ch * 64;                            // column of the w1 part inside h13
      if (ca < p.N) {
        warp_store_32x64_tma(stg, stg_tiles, stg_cnt, lane, wa, &tm_c, ca, row0);
        warp_store_32x64_tma(stg, stg_tiles, stg_cnt, lane, wb, &tm_c, ca + 128, row0);
        // the saved h13 is bf16: gate from the ROUNDED values, so that backward (which reads h13) sees the same function
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const float a0 = bf16_lo(wa[i]), a1 = bf16_hi(wa[i]), b0 = bf16_lo(wb[i]), b1 = bf16_hi(wb[i]);
          wa[i] = pack_bf16(a0 * sigmoidf_fast(a0) * b0, a1 * sigmoidf_fast(a1) * b1);
        }
        warp_store_32x64_tma(stg, stg_tiles, stg_cnt, lane, wa, &tm_c2, (n0 >> 1) + ch * 64, row0);
      }
    }
}

// ================================================================================================
// A-resident kernels (K <= 512)
// ================================================================================================
constexpr int kBStageBytes = 256 * 64;     // 256 rows x 32 bf16 (64-byte rows, SWIZZLE_64B)
constexpr int kStageTileBytes = 2048;      // per epilogue warp: 16 rows x 128 bytes

// Epilogue warps (4-11) of both A-resident kernels: row block grp * ctas + rank of every group grp0, grp0 + grp_step, ...
// below n_groups (blocks beyond M: clipped stores), all N tiles of each, the two TMEM accumulator stages in turn.  Each warp
// owns stg_tiles staging tiles of the CTA's area Stg.  Lane 0 calls arrive(as) once every TMEM read of accumulator stage
// `as` by this warp has completed.
template <int EPI, class Arrive>
__device__ __forceinline__ void res_epilogue_warp(const GemmParams& p, const CUtensorMap& tm_c, const CUtensorMap& tm_c2, uint8_t* Stg,
                                                  int stg_tiles, uint32_t tmem_base, uint64_t* tmem_full, int grp0, int n_groups,
                                                  int grp_step, int ctas, int rank, Arrive arrive) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = warp - 4;
  const int q = warp & 3;          // TMEM lane quarter this warp may read
  const int ch = e >> 2;           // column half of the 256-column tile
  uint8_t* stg = Stg + e * stg_tiles * kStageTileBytes;
  uint32_t tc = 0, stg_cnt = 0;
  for (int grp = grp0; grp < n_groups; grp += grp_step) {
    const int blk = grp * ctas + rank;
    const long long row0 = static_cast<long long>(blk) * 128 + q * 32;     // first row of this warp
    const long long row = row0 + lane;
    constexpr int kCs = rope_pairs<EPI>();
    float2 cs[kCs];
    if (is_rope<EPI>()) {
      int ps = 0;
      if (row < p.M) ps = p.rope_pos ? p.rope_pos[row] : static_cast<int>(row % p.rope_S) + p.rope_offset;
      ps = min(max(ps, 0), p.rope_len - 1);
#pragma unroll
      for (int i = 0; i < kCs; ++i) cs[i] = __ldg(p.rope_table + static_cast<long long>(ps) * kCs + i);
    }
    for (int t = 0; t < p.ntile; ++t, ++tc) {
      const uint32_t as = tc & 1;
      const int n0 = t * 256;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * 256;
      auto release = [&]() {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) arrive(as);
      };
      res_epilogue_tile<EPI>(p, tm_c, tm_c2, stg, stg_tiles, stg_cnt, lane, ch, taddr, n0, row0, cs, &tmem_full[as], (tc >> 1) & 1, release);
    }
  }
  if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");      // all bulk stores of this warp have completed
}

// Single CTA per row block: used when the problem has fewer than 4 row blocks (or the device an odd number of SMs).
template <int EPI>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_res_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                const __grid_constant__ CUtensorMap tm_c, const __grid_constant__ CUtensorMap tm_c2, const GemmParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  uint8_t* As = smem;                                        // nslab x 16 KB (64-wide k-slabs, SWIZZLE_128B)
  uint8_t* Bs = As + p.nslab * kASlabBytes;                  // nstage x 16 KB (32-wide k-slabs, SWIZZLE_64B)
  uint8_t* Stg = Bs + p.nstage * kBStageBytes;               // 8 x 2 KB epilogue staging tiles
  uint64_t* bars = reinterpret_cast<uint64_t*>(Stg + 8 * kStageTileBytes);
  uint64_t* a_full = bars;            // [8]
  uint64_t* a_empty = bars + 8;       // [8]
  uint64_t* b_full = bars + 16;       // [8]
  uint64_t* b_empty = bars + 24;      // [8]
  uint64_t* tmem_full = bars + 32;    // [2]
  uint64_t* tmem_empty = bars + 34;   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 36);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tm_a); tma_prefetch_desc(&tm_b); tma_prefetch_desc(&tm_c); tma_prefetch_desc(&tm_c2); }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < 8; ++i) {
      mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1);
      mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 8); }
    fence_mbar_init();
  }
  if (warp == 2) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int n_blocks = static_cast<int>((p.M + 127) / 128);
  const int nkb = (p.K + 31) / 32;          // 32-wide k-slabs of B; A slab of k-slab j = j / 2

  if (warp == 0) {
    // ================================ TMA producer ================================
    int stage = 0;
    uint32_t phase = 0, it = 0;
    for (int blk = blockIdx.x; blk < n_blocks; blk += gridDim.x, ++it) {
      for (int t = 0; t < p.ntile; ++t) {
        for (int j = 0; j < nkb; ++j) {
          if (t == 0 && (j & 1) == 0) {
            // A slab j/2 of this block: free once the last tile of the previous block has consumed it
            const int ks = j >> 1;
            mbar_wait(&a_empty[ks], (it & 1) ^ 1);
            if (elect_one()) {
              mbar_expect_tx(&a_full[ks], kASlabBytes);
              tma_load_2d(As + ks * kASlabBytes, &tm_a, &a_full[ks], ks * 64, blk * 128);
            }
            __syncwarp();
          }
          mbar_wait(&b_empty[stage], phase ^ 1);
          if (elect_one()) {
            mbar_expect_tx(&b_full[stage], kBStageBytes);
            tma_load_2d(Bs + stage * kBStageBytes, &tm_b, &b_full[stage], j * 32, t * 256);
          }
          __syncwarp();
          if (++stage == p.nstage) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ================================
    constexpr uint32_t idesc = umma_idesc_bf16(128, 256);
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t as_addr = smem_u32(As), bs_addr = smem_u32(Bs);
    int stage = 0;
    uint32_t phase = 0, it = 0, tc = 0;
    // (the loop body is kept minimal: one issuing warp has to turn a 16 KB stage around in the 256 cycles its two MMAs
    //  take -- every integer division, diagnostic branch or descriptor rebuild in here showed up in the GEMM's time)
    const uint64_t adesc0 = umma_desc_sw128(as_addr), bdesc0 = umma_desc_sw64(bs_addr);
    for (int blk = blockIdx.x; blk < n_blocks; blk += gridDim.x, ++it) {
      for (int t = 0; t < p.ntile; ++t, ++tc) {
        const uint32_t as = tc & 1;
        mbar_wait(&tmem_empty[as], ((tc >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_u + as * 256;
        const bool first_tile = t == 0, last_tile = t == p.ntile - 1;
        uint64_t adesc = adesc0;      // 64-byte half (j & 1) of slab j / 2: +4 within a slab, + slab size - 4 to the next
        for (int j = 0; j < nkb; ++j) {
          if (first_tile && (j & 1) == 0) mbar_wait(&a_full[j >> 1], it & 1);
          mbar_wait(&b_full[stage], phase);
          tc_fence_after();
          const uint64_t bdesc = bdesc0 + static_cast<uint64_t>(stage * (kBStageBytes >> 4));
          if (elect_one()) {
            umma_bf16(d_tmem, adesc, bdesc, idesc, j != 0);
            umma_bf16(d_tmem, adesc + 2, bdesc + 2, idesc, 1u);
            umma_commit(&b_empty[stage]);
            if (last_tile && ((j & 1) == 1 || j == nkb - 1)) umma_commit(&a_empty[j >> 1]);
          }
          __syncwarp();
          adesc += (j & 1) ? static_cast<uint64_t>((kASlabBytes >> 4) - 4) : 4ull;
          if (++stage == p.nstage) { stage = 0; phase ^= 1; }
        }
        if (elect_one()) umma_commit(&tmem_full[as]);
        __syncwarp();
      }
    }
  } else if (warp >= 4) {
    // ================================ epilogue ================================
    res_epilogue_warp<EPI>(p, tm_c, tm_c2, Stg, 1, tmem_base, tmem_full, static_cast<int>(blockIdx.x), n_blocks,
                           static_cast<int>(gridDim.x), 1, 0, [&](uint32_t as) { mbar_arrive(&tmem_empty[as]); });
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

// ================================================================================================
// A-resident kernel on CTA PAIRS (cta_group::2): two SMs of one TPC own two adjacent 128-row blocks (both resident) and
// work on ONE 256 x 256 tile at a time.  Each CTA streams only HALF of every weight stage (128 of the 256 weight rows,
// 8 KB instead of 16 KB) -- the tensor cores of both SMs read both halves -- so the same 80 KB next to the resident block
// hold 10 stages instead of 5: twice the look-ahead, which is what bounds the single-CTA kernel (profiles/r02_gemm_experiments.txt).
// The leader CTA (cluster rank 0) issues every MMA; both CTAs run their own TMA producer (completion bytes go to the
// LEADER's full barriers) and their own epilogue on their own TMEM (rows 0-127 / 128-255 of the tile).
// ================================================================================================
constexpr int kB2StageBytes = 128 * 64;    // this CTA's half of a weight stage: 128 rows x 32 bf16

template <int EPI>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_res2_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                 const __grid_constant__ CUtensorMap tm_c, const __grid_constant__ CUtensorMap tm_c2, const GemmParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  uint8_t* As = smem;                                        // nslab x 16 KB
  uint8_t* Bs = As + p.nslab * kASlabBytes;                  // nstage x 8 KB
  uint8_t* Stg = Bs + p.nstage * kB2StageBytes;              // 8 warps x 2 x 2 KB epilogue staging tiles (double buffered)
  uint64_t* bars = reinterpret_cast<uint64_t*>(Stg + 16 * kStageTileBytes);
  uint64_t* a_full = bars;            // [8]   (waited on in the leader only)
  uint64_t* a_empty = bars + 8;       // [8]
  uint64_t* b_full = bars + 16;       // [16]  (leader only)
  uint64_t* b_empty = bars + 32;      // [16]
  uint64_t* tmem_full = bars + 48;    // [2]
  uint64_t* tmem_empty = bars + 50;   // [2]   (leader only: 8 epilogue warps of each CTA arrive)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 52);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tm_a); tma_prefetch_desc(&tm_b); tma_prefetch_desc(&tm_c); tma_prefetch_desc(&tm_c2); }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < 8; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < 16; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 16); }
    fence_mbar_init();
  }
  if (warp == 2) { tmem_alloc_2sm(tmem_slot, 512); tmem_relinquish_2sm(); }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                       // both CTAs' barriers and TMEM exist before anything crosses the pair
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int n_blocks = static_cast<int>((p.M + 127) / 128);
  const int n_groups = (n_blocks + 1) / 2;
  const int n_pairs = static_cast<int>(gridDim.x / 2), pair_id = static_cast<int>(blockIdx.x / 2);
  const int nkb = (p.K + 31) / 32;

  if (warp == 0) {
    // ================================ TMA producer (both CTAs) ================================
    int stage = 0;
    uint32_t phase = 0, it = 0;
    for (int grp = pair_id; grp < n_groups; grp += n_pairs, ++it) {
      const int blk = grp * 2 + static_cast<int>(rank);
      for (int t = 0; t < p.ntile; ++t) {
        for (int j = 0; j < nkb; ++j) {
          if (t == 0 && (j & 1) == 0) {
            const int ks = j >> 1;
            mbar_wait(&a_empty[ks], (it & 1) ^ 1);
            if (elect_one()) {
              if (leader) mbar_expect_tx(&a_full[ks], 2 * kASlabBytes);          // this CTA's slab + the peer's
              tma_load_2d_2sm(As + ks * kASlabBytes, &tm_a, mapa_shared(smem_u32(&a_full[ks]), 0), ks * 64, blk * 128);
            }
            __syncwarp();
          }
          mbar_wait(&b_empty[stage], phase ^ 1);
          if (elect_one()) {
            if (leader) mbar_expect_tx(&b_full[stage], 2 * kB2StageBytes);
            tma_load_2d_2sm(Bs + stage * kB2StageBytes, &tm_b, mapa_shared(smem_u32(&b_full[stage]), 0), j * 32,
                            t * 256 + static_cast<int>(rank) * 128);
          }
          __syncwarp();
          if (++stage == p.nstage) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1 && leader) {
    // ================================ MMA issuer (leader CTA) ================================
    constexpr uint32_t idesc = umma_idesc_bf16(256, 256);
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint64_t adesc0 = umma_desc_sw128(smem_u32(As)), bdesc0 = umma_desc_sw64(smem_u32(Bs));
    int stage = 0;
    uint32_t phase = 0, it = 0, tc = 0;
    for (int grp = pair_id; grp < n_groups; grp += n_pairs, ++it) {
      for (int t = 0; t < p.ntile; ++t, ++tc) {
        const uint32_t as = tc & 1;
        mbar_wait(&tmem_empty[as], ((tc >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_u + as * 256;
        const bool first_tile = t == 0, last_tile = t == p.ntile - 1;
        uint64_t adesc = adesc0;
        for (int j = 0; j < nkb; ++j) {
          if (first_tile && (j & 1) == 0) mbar_wait(&a_full[j >> 1], it & 1);
          mbar_wait(&b_full[stage], phase);
          tc_fence_after();
          const uint64_t bdesc = bdesc0 + static_cast<uint64_t>(stage * (kB2StageBytes >> 4));
          if (elect_one()) {
            umma_bf16_2sm(d_tmem, adesc, bdesc, idesc, j != 0);
            umma_bf16_2sm(d_tmem, adesc + 2, bdesc + 2, idesc, 1u);
            umma_commit_2sm(&b_empty[stage], 3);
            if (last_tile && ((j & 1) == 1 || j == nkb - 1)) umma_commit_2sm(&a_empty[j >> 1], 3);
          }
          __syncwarp();
          adesc += (j & 1) ? static_cast<uint64_t>((kASlabBytes >> 4) - 4) : 4ull;
          if (++stage == p.nstage) { stage = 0; phase ^= 1; }
        }
        if (elect_one()) umma_commit_2sm(&tmem_full[as], 3);
        __syncwarp();
      }
    }
  } else if (warp >= 4) {
    // ================================ epilogue (both CTAs, own TMEM) ================================
    // (the epilogue warps of both CTAs free an accumulator stage on the leader's barrier)
    res_epilogue_warp<EPI>(p, tm_c, tm_c2, Stg, 2, tmem_base, tmem_full, pair_id, n_groups, n_pairs, 2, static_cast<int>(rank),
                           [&](uint32_t as) {
                             if (leader) mbar_arrive(&tmem_empty[as]);
                             else mbar_arrive_cluster(mapa_shared(smem_u32(&tmem_empty[as]), 0));
                           });
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) { tc_fence_after(); tmem_dealloc_2sm(tmem_base, 512); }
}

// ================================================================================================
// Streaming kernel (long K): 256 x 256 tiles, EPI_STORE (+ bias)
// ================================================================================================
constexpr int kStreamStageBytes = 2 * kASlabBytes + kBSlabBytes;     // 64 KB: A rows 0-255 | B rows 0-255

__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_stream_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, const GemmParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.nstage * kStreamStageBytes);
  uint64_t* full = bars;              // [4]
  uint64_t* empty = bars + 4;         // [4]
  uint64_t* tmem_full = bars + 8;     // [1]
  uint64_t* tmem_empty = bars + 9;    // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 10);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tm_a); tma_prefetch_desc(&tm_b); }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < 4; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(tmem_full, 1);
    mbar_init(tmem_empty, 8);
    fence_mbar_init();
  }
  if (warp == 2) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const long long n_rb = (p.M + 255) / 256;
  const long long n_units = n_rb * p.ntile;     // unit u: row block u / ntile, column tile u % ntile

  if (warp == 0) {
    int stage = 0;
    uint32_t phase = 0;
    for (long long u = blockIdx.x; u < n_units; u += gridDim.x) {
      const int rb = static_cast<int>(u / p.ntile), t = static_cast<int>(u % p.ntile);
      for (int ks = 0; ks < p.nslab; ++ks) {
        mbar_wait(&empty[stage], phase ^ 1);
        if (elect_one()) {
          uint8_t* st = smem + stage * kStreamStageBytes;
          mbar_expect_tx(&full[stage], kStreamStageBytes);
          tma_load_2d(st, &tm_a, &full[stage], ks * 64, rb * 256);                       // box 64 x 256 rows
          tma_load_2d(st + 2 * kASlabBytes, &tm_b, &full[stage], ks * 64, t * 256);
        }
        __syncwarp();
        if (++stage == p.nstage) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = umma_idesc_bf16(128, 256);
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t s_addr = smem_u32(smem);
    int stage = 0;
    uint32_t phase = 0, uc = 0;
    for (long long u = blockIdx.x; u < n_units; u += gridDim.x, ++uc) {
      mbar_wait(tmem_empty, (uc & 1) ^ 1);
      tc_fence_after();
      for (int ks = 0; ks < p.nslab; ++ks) {
        mbar_wait(&full[stage], phase);
        tc_fence_after();
        const uint32_t st = s_addr + stage * kStreamStageBytes;
        const uint64_t a0 = umma_desc_sw128(st), a1 = umma_desc_sw128(st + kASlabBytes);
        const uint64_t bdesc = umma_desc_sw128(st + 2 * kASlabBytes);
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) umma_bf16(tmem_u, a0 + 2 * kk, bdesc + 2 * kk, idesc, (ks | kk) != 0);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) umma_bf16(tmem_u + 256, a1 + 2 * kk, bdesc + 2 * kk, idesc, (ks | kk) != 0);
          umma_commit(&empty[stage]);
        }
        __syncwarp();
        if (++stage == p.nstage) { stage = 0; phase ^= 1; }
      }
      if (elect_one()) umma_commit(tmem_full);
      __syncwarp();
    }
  } else if (warp >= 4) {
    const int e = warp - 4;
    const int q = warp & 3, h = e >> 2;           // lane quarter, row half
    uint32_t uc = 0;
    for (long long u = blockIdx.x; u < n_units; u += gridDim.x, ++uc) {
      const int rb = static_cast<int>(u / p.ntile), t = static_cast<int>(u % p.ntile);
      const long long row = static_cast<long long>(rb) * 256 + h * 128 + q * 32 + lane;
      const bool row_ok = row < p.M;
      mbar_wait(tmem_full, uc & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + h * 256;
      uint32_t r[2][32];
      tmem_ld32(taddr, r[0]);
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        tmem_wait_ld32(r[c & 1]);
        if (c < 7) {
          tmem_ld32(taddr + (c + 1) * 32, r[(c + 1) & 1]);
        } else {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(tmem_empty);
        }
        const int col = t * 256 + c * 32;
        float v[32];
        to_f32(r[c & 1], v);
        if (p.bias != nullptr) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] += (col + i < p.N) ? __ldg(p.bias + col + i) : 0.f;
        }
        if (row_ok && col < p.N) store32_bf16(p.C + row * p.ldc + col, v);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

// ================================================================================================
// TN kernel: out[Na, Nb] = A[M, Na]^T B[M, Nb] (fp32 partial sums per row range)
// ================================================================================================
struct TnParams {
  float* ws;                 // [splits][Na][Nb]
  long long M;
  int Na, Nb, ta, tb, splits, nstage;
  long long rows_per_split;  // multiple of krows
  int krows;                 // rows of the contraction per pipeline stage (64; the patch size for the patch embedding)
  // patch-embedding mode (fk_patch_embed_forward): every row range is one (trial, time patch) and its [Na, Nb] product IS
  // the projection of that patch's Na tokens -- written as bf16 rows with the bias (and the electrode embedding) added
  __nv_bfloat16* out_bf16;   // [splits * Na, Nb] or null
  const float* bias;         // [Nb] or null
  const float* emb;          // [Na, Nb] or null
};

__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tn_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, const TnParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  constexpr int kStage = 2 * kBSlabBytes;      // A: 4 chunks x 8 KB | B: 4 chunks x 8 KB
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.nstage * kStage);
  uint64_t* full = bars;
  uint64_t* empty = bars + 4;
  uint64_t* tmem_full = bars + 8;
  uint64_t* tmem_empty = bars + 9;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 10);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tm_a); tma_prefetch_desc(&tm_b); }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < 4; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(tmem_full, 1);
    mbar_init(tmem_empty, 8);
    fence_mbar_init();
  }
  if (warp == 2) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // unit u -> (split, tile): consecutive CTAs work on the SAME row range and different output tiles, so a row range of
  // the activations is fetched from HBM once and served to the other tiles from L2
  const int n_tiles = p.ta * p.tb;
  const long long n_units = static_cast<long long>(n_tiles) * p.splits;
  auto k_range = [&](int split, long long& k0, long long& k1) {
    k0 = split * p.rows_per_split;
    k1 = min(p.M, k0 + p.rows_per_split);
  };

  if (warp == 0) {
    int stage = 0;
    uint32_t phase = 0;
    for (long long u = blockIdx.x; u < n_units; u += gridDim.x) {
      const int split = static_cast<int>(u / n_tiles), tile = static_cast<int>(u % n_tiles);
      const int ia = tile / p.tb, ib = tile % p.tb;
      long long k0, k1;
      k_range(split, k0, k1);
      for (long long k = k0; k < k1; k += p.krows) {
        mbar_wait(&empty[stage], phase ^ 1);
        if (elect_one()) {
          uint8_t* st = smem + stage * kStage;
          mbar_expect_tx(&full[stage], static_cast<uint32_t>(2 * 4 * p.krows * 128));
          tma_load_3d(st, &tm_a, &full[stage], 0, static_cast<int>(k), ia * 4);              // box 64 x krows rows x 4 chunks
          // (patch-embedding mode: B = W^T [patch, dim] is the same for every row range -> row coordinate within the range)
          tma_load_3d(st + kBSlabBytes, &tm_b, &full[stage], 0, static_cast<int>(p.out_bf16 ? k - k0 : k), ib * 4);
        }
        __syncwarp();
        if (++stage == p.nstage) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = umma_idesc_bf16(128, 256) | (1u << 15) | (1u << 16);     // A and B MN-major
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t s_addr = smem_u32(smem);
    int stage = 0;
    uint32_t phase = 0, uc = 0;
    for (long long u = blockIdx.x; u < n_units; u += gridDim.x, ++uc) {
      const int split = static_cast<int>(u / n_tiles);
      long long k0, k1;
      k_range(split, k0, k1);
      mbar_wait(tmem_empty, (uc & 1) ^ 1);
      tc_fence_after();
      bool first = true;
      const uint32_t chunk_bytes = static_cast<uint32_t>(p.krows) * 128u;      // one 64-column chunk of a stage
      const int nkk = p.krows >> 4;
      for (long long k = k0; k < k1; k += p.krows) {
        mbar_wait(&full[stage], phase);
        tc_fence_after();
        const uint32_t st = s_addr + stage * kStage;
        const uint64_t a0 = umma_desc_mn_sw128(st, chunk_bytes), a1 = umma_desc_mn_sw128(st + 2 * chunk_bytes, chunk_bytes);
        const uint64_t bdesc = umma_desc_mn_sw128(st + kBSlabBytes, chunk_bytes);
        if (elect_one()) {
          // a K step of 16 rows = 2048 B = +128 in the (address >> 4) field
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            if (kk < nkk) umma_bf16(tmem_u, a0 + 128 * kk, bdesc + 128 * kk, idesc, !(first && kk == 0));
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            if (kk < nkk) umma_bf16(tmem_u + 256, a1 + 128 * kk, bdesc + 128 * kk, idesc, !(first && kk == 0));
          umma_commit(&empty[stage]);
        }
        __syncwarp();
        first = false;
        if (++stage == p.nstage) { stage = 0; phase ^= 1; }
      }
      if (elect_one()) umma_commit(tmem_full);
      __syncwarp();
    }
  } else if (warp >= 4) {
    const int e = warp - 4;
    const int q = warp & 3, h = e >> 2;
    uint32_t uc = 0;
    for (long long u = blockIdx.x; u < n_units; u += gridDim.x, ++uc) {
      const int split = static_cast<int>(u / n_tiles), tile = static_cast<int>(u % n_tiles);
      const int ia = tile / p.tb, ib = tile % p.tb;
      long long k0, k1;
      k_range(split, k0, k1);
      const int row = ia * 256 + h * 128 + q * 32 + lane;        // index along Na
      const bool row_ok = row < p.Na;
      float* dst = p.ws + (static_cast<long long>(split) * p.Na + row) * p.Nb + ib * 256;
      // (the host never creates an empty row range: fk_gemm_tn_splits drops splits that would be empty)
      mbar_wait(tmem_full, uc & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + h * 256;
      uint32_t r[2][32];
      tmem_ld32(taddr, r[0]);
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        tmem_wait_ld32(r[c & 1]);
        if (c < 7) {
          tmem_ld32(taddr + (c + 1) * 32, r[(c + 1) & 1]);
        } else {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(tmem_empty);
        }
        if (row_ok && ib * 256 + c * 32 < p.Nb) {
          if (p.out_bf16 != nullptr) {
            const int col = ib * 256 + c * 32;
            float v[32];
            to_f32(r[c & 1], v);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              float4 add = p.bias ? __ldg(reinterpret_cast<const float4*>(p.bias + col) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
              if (p.emb != nullptr) {
                const float4 e4 = __ldg(reinterpret_cast<const float4*>(p.emb + static_cast<long long>(row) * p.Nb + col) + i);
                add.x += e4.x; add.y += e4.y; add.z += e4.z; add.w += e4.w;
              }
              v[4 * i] += add.x; v[4 * i + 1] += add.y; v[4 * i + 2] += add.z; v[4 * i + 3] += add.w;
            }
            store32_bf16(p.out_bf16 + (static_cast<long long>(split) * p.Na + row) * p.Nb + col, v);
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i)
              *reinterpret_cast<uint4*>(dst + c * 32 + i * 4) =
                  make_uint4(r[c & 1][i * 4], r[c & 1][i * 4 + 1], r[c & 1][i * 4 + 2], r[c & 1][i * 4 + 3]);
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

__global__ void __launch_bounds__(256)
gemm_tn_reduce_kernel(const float* __restrict__ ws, float* __restrict__ out, long long n4, int splits) {
  const long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
  if (i >= n4) return;
  float4 acc = *reinterpret_cast<const float4*>(ws + i * 4);
  for (int s = 1; s < splits; ++s) {
    const float4 v = ldg_nc_f4(ws + (static_cast<long long>(s) * n4 + i) * 4);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  *reinterpret_cast<float4*>(out + i * 4) = acc;
}

}  // namespace fk

using namespace fk;

#define FK_API extern "C" __attribute__((visibility("default")))

template <class Kern>
static int set_smem_attr(Kern* kern, bool& done, int bytes) {
  if (done) return FK_OK;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) != cudaSuccess) {
    fk_set_last_error("cudaFuncSetAttribute(max dynamic smem) failed", __FILE__, __LINE__);
    return FK_ERR_CUDA;
  }
  done = true;
  return FK_OK;
}

// One A-resident launch: gemm_res2_kernel<EPI> on clusters of 2 CTAs (pair) or gemm_res_kernel<EPI>.
template <int EPI>
static int launch_res(bool pair, unsigned grid, int smem_bytes, cudaStream_t stream, const CUtensorMap& ta, const CUtensorMap& tb,
                      const CUtensorMap& tc, const CUtensorMap& tc2, const GemmParams& p) {
  static bool done[2][FK_MAX_DEVICES];      // shared-memory opt-in of gemm_res_kernel<EPI> / gemm_res2_kernel<EPI> per device
  auto* kern = pair ? gemm_res2_kernel<EPI> : gemm_res_kernel<EPI>;
  const int rc = set_smem_attr(kern, done[pair][fk_device_ordinal()], kGemmSmemLimit);
  if (rc != FK_OK) return rc;
  if (!pair) {
    kern<<<grid, kGemmThreads, smem_bytes, stream>>>(ta, tb, tc, tc2, p);
    return FK_OK;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid, 1, 1);
  cfg.blockDim = dim3(kGemmThreads, 1, 1);
  cfg.dynamicSmemBytes = static_cast<size_t>(smem_bytes);
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  const cudaError_t le = cudaLaunchKernelEx(&cfg, kern, ta, tb, tc, tc2, p);
  if (le != cudaSuccess) { fk_set_last_error(cudaGetErrorString(le), __FILE__, __LINE__); return FK_ERR_CUDA; }
  return FK_OK;
}

FK_API int fk_gemm_nt(const void* A, long long lda, const void* B, long long ldb, void* C, long long ldc, long long M, int N,
                      int K, const float* bias, int epilogue, void* C2, long long ldc2, const float* rope_table, int rope_len,
                      const int* rope_pos, int rope_offset, int rope_cols, int rope_S, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(A && B && M > 0 && N > 0 && K > 0, "fk_gemm_nt: bad argument");
  FK_REQUIRE(M < (1ll << 31) - 256, "fk_gemm_nt: too many rows");
  // (lda < K is allowed: rows of A may overlap -- the im2col rows of a channels-last convolution are read as a view)
  FK_REQUIRE(K % 8 == 0 && lda % 8 == 0 && ldb % 8 == 0 && lda > 0 && ldb >= K, "fk_gemm_nt: K and the leading dimensions must be multiples of 8 (16-byte rows)");
  FK_REQUIRE(N % 32 == 0, "fk_gemm_nt: N must be a multiple of 32");
  FK_REQUIRE((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(B) & 15) == 0, "fk_gemm_nt: operands must be 16-byte aligned");
  FK_REQUIRE(epilogue != 3, "fk_gemm_nt: epilogue 3 (SwiGLU backward) was removed; use epilogue 0 for d gated and fk_swiglu_backward_blocked");
  FK_REQUIRE(epilogue >= EPI_STORE && epilogue <= EPI_ROPE16, "fk_gemm_nt: unknown epilogue");
  GemmParams p = {};
  p.C = static_cast<__nv_bfloat16*>(C); p.ldc = ldc;
  p.C2 = static_cast<__nv_bfloat16*>(C2); p.ldc2 = ldc2;
  p.bias = bias;
  p.rope_table = reinterpret_cast<const float2*>(rope_table); p.rope_pos = rope_pos; p.rope_len = rope_len;
  p.rope_offset = rope_offset; p.rope_cols = rope_cols; p.rope_S = rope_S;
  p.M = M; p.N = N; p.K = K;
  p.nslab = (K + 63) / 64;
  p.ntile = (N + 255) / 256;
  FK_REQUIRE(C && ldc % 8 == 0 && ldc >= N && (reinterpret_cast<uintptr_t>(C) & 15) == 0, "fk_gemm_nt: C must be 16-byte aligned with ldc % 8 == 0");
  if (epilogue == EPI_ROPE || epilogue == EPI_ROPE64 || epilogue == EPI_ROPE16) {
    FK_REQUIRE(rope_table && rope_len > 0 && rope_cols % (epilogue == EPI_ROPE64 ? 64 : 32) == 0 && rope_cols <= N && (rope_pos || rope_S > 0),
               "fk_gemm_nt: bad rope arguments");
    FK_REQUIRE(rope_pos != nullptr || (rope_offset >= 0 && static_cast<long long>(rope_offset) + (M < rope_S ? M : rope_S) <= rope_len),
               "fk_gemm_nt: token positions fall outside the rope table");
  }
  if (epilogue == EPI_SWIGLU)
    FK_REQUIRE(N % 256 == 0 && C2 && ldc2 % 8 == 0 && ldc2 >= N / 2 && bias == nullptr, "fk_gemm_nt: SwiGLU epilogue needs N % 256 == 0 and the gated output");
  FK_REQUIRE(bias == nullptr || epilogue == EPI_STORE, "fk_gemm_nt: bias goes with the plain epilogue");

  CUtensorMap ta, tb;
  const int G = fk_sm_count();
  if (K <= 512) {
    // CTA pairs (gemm_res2_kernel) hold twice the weight look-ahead of single CTAs (gemm_res_kernel), which are left with
    // the problems of fewer than 4 row blocks and devices with an odd number of SMs
    const long long n_blocks = (M + 127) / 128;
    const bool pair = n_blocks >= 4 && G % 2 == 0;
    int rc = make_tmap_bf16_2d(&ta, A, static_cast<uint64_t>(M), static_cast<uint64_t>(K), static_cast<uint64_t>(lda), 128);
    rc |= make_tmap_bf16_2d_sw64(&tb, B, static_cast<uint64_t>(N), static_cast<uint64_t>(K), static_cast<uint64_t>(ldb), pair ? 128 : 256);
    // outputs go through the TMA store engine: 16-row x 64-column boxes, 128-byte swizzle
    CUtensorMap tc, tc2;
    rc |= make_tmap_bf16_2d(&tc, C, static_cast<uint64_t>(M), static_cast<uint64_t>(N), static_cast<uint64_t>(ldc), 16);
    tc2 = tc;
    if (epilogue == EPI_SWIGLU)
      rc |= make_tmap_bf16_2d(&tc2, C2, static_cast<uint64_t>(M), static_cast<uint64_t>(N / 2), static_cast<uint64_t>(ldc2), 16);
    if (rc != FK_OK) { fk_set_last_error("cuTensorMapEncodeTiled failed", __FILE__, __LINE__); return FK_ERR_DRIVER; }
    // every weight stage that fits next to the resident block and the staging tiles (2 per epilogue warp on pairs)
    const int stg_bytes = (pair ? 16 : 8) * kStageTileBytes;
    const int stage_bytes = pair ? kB2StageBytes : kBStageBytes;
    const int max_stages = pair ? 16 : 8;
    int nstage = (kGemmSmemLimit - 512 - stg_bytes - p.nslab * kASlabBytes) / stage_bytes;
    if (nstage > max_stages) nstage = max_stages;
    p.nstage = nstage;
    const int smem_bytes = p.nslab * kASlabBytes + nstage * stage_bytes + stg_bytes + 512;
    const long long n_groups = pair ? (n_blocks + 1) / 2 : n_blocks;     // row blocks per CTA pair / CTA
    const long long max_groups = pair ? G / 2 : G;
    const unsigned grid = static_cast<unsigned>((n_groups < max_groups ? n_groups : max_groups) * (pair ? 2 : 1));
    switch (epilogue) {
      case EPI_STORE: rc = launch_res<EPI_STORE>(pair, grid, smem_bytes, stream, ta, tb, tc, tc2, p); break;
      case EPI_ROPE: rc = launch_res<EPI_ROPE>(pair, grid, smem_bytes, stream, ta, tb, tc, tc2, p); break;
      case EPI_SWIGLU: rc = launch_res<EPI_SWIGLU>(pair, grid, smem_bytes, stream, ta, tb, tc, tc2, p); break;
      case EPI_ROPE64: rc = launch_res<EPI_ROPE64>(pair, grid, smem_bytes, stream, ta, tb, tc, tc2, p); break;
      default: rc = launch_res<EPI_ROPE16>(pair, grid, smem_bytes, stream, ta, tb, tc, tc2, p); break;
    }
    if (rc != FK_OK) return rc;
  } else {
    FK_REQUIRE(epilogue == EPI_STORE, "fk_gemm_nt: fused epilogues need K <= 512 (the A-resident kernel)");
    int rc = make_tmap_bf16_2d(&ta, A, static_cast<uint64_t>(M), static_cast<uint64_t>(K), static_cast<uint64_t>(lda), 256);
    rc |= make_tmap_bf16_2d(&tb, B, static_cast<uint64_t>(N), static_cast<uint64_t>(K), static_cast<uint64_t>(ldb), 256);
    if (rc != FK_OK) { fk_set_last_error("cuTensorMapEncodeTiled failed", __FILE__, __LINE__); return FK_ERR_DRIVER; }
    p.nstage = 3;
    const int smem_bytes = p.nstage * kStreamStageBytes + 512;
    const long long n_units = ((M + 255) / 256) * p.ntile;
    const unsigned grid = static_cast<unsigned>(n_units < G ? n_units : G);
    static bool done[FK_MAX_DEVICES];
    const int r2 = set_smem_attr(gemm_stream_kernel, done[fk_device_ordinal()], kGemmSmemLimit);
    if (r2 != FK_OK) return r2;
    gemm_stream_kernel<<<grid, kGemmThreads, smem_bytes, stream>>>(ta, tb, p);
  }
  FK_CHECK_LAUNCH();
  fk_count_launch(1);
  return FK_OK;
}

// number of row ranges fk_gemm_tn splits the contraction into (workspace = splits * Na * Nb floats)
FK_API int fk_gemm_tn_splits(long long M, int Na, int Nb, int max_ctas) {
  if (M <= 0 || Na <= 0 || Nb <= 0) return FK_ERR_BAD_ARG;
  const long long tiles = static_cast<long long>((Na + 255) / 256) * ((Nb + 255) / 256);
  long long G = max_ctas;
  if (G <= 0) G = fk_sm_count();
  if (G <= 0) G = 148;
  const long long max_splits = (M + 63) / 64;
  long long best = 1;
  double best_eff = 0.0;
  for (int w = 1; w <= 3; ++w) {
    long long s = (G * w) / tiles;
    if (s < 1) s = 1;
    if (s > max_splits) s = max_splits;
    if (s > 64) s = 64;
    const long long units = tiles * s;
    const double eff = static_cast<double>(units) / (static_cast<double>((units + G - 1) / G) * G);
    if (eff > best_eff + 1e-9) { best_eff = eff; best = s; }
  }
  // rows per split are rounded up to 64: drop splits that would be empty
  const long long rps = ((M + best - 1) / best + 63) / 64 * 64;
  return static_cast<int>((M + rps - 1) / rps);
}

FK_API int fk_gemm_tn(const void* A, long long lda, const void* B, long long ldb, float* out, long long M, int Na, int Nb,
                      float* ws, int splits, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(A && B && out && ws && M > 0 && Na > 0 && Nb > 0, "fk_gemm_tn: bad argument");
  FK_REQUIRE(M < (1ll << 31) - 64, "fk_gemm_tn: too many rows");
  // (ld < N is allowed: overlapping rows, see fk_gemm_nt)
  FK_REQUIRE(Na % 64 == 0 && Nb % 64 == 0 && lda % 8 == 0 && ldb % 8 == 0 && lda > 0 && ldb > 0,
             "fk_gemm_tn: Na and Nb must be multiples of 64, leading dimensions multiples of 8");
  FK_REQUIRE((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(B) & 15) == 0 &&
             (reinterpret_cast<uintptr_t>(out) & 15) == 0 && (reinterpret_cast<uintptr_t>(ws) & 15) == 0, "fk_gemm_tn: pointers must be 16-byte aligned");
  const int G = fk_sm_count();
  FK_REQUIRE(G > 0 && splits == fk_gemm_tn_splits(M, Na, Nb, G), "fk_gemm_tn: split count does not match fk_gemm_tn_splits");
  CUtensorMap ta, tb;
  int rc = make_tmap_bf16_chunks(&ta, A, static_cast<uint64_t>(M), static_cast<uint64_t>(Na), static_cast<uint64_t>(lda), 64);
  rc |= make_tmap_bf16_chunks(&tb, B, static_cast<uint64_t>(M), static_cast<uint64_t>(Nb), static_cast<uint64_t>(ldb), 64);
  if (rc != FK_OK) { fk_set_last_error("cuTensorMapEncodeTiled failed", __FILE__, __LINE__); return FK_ERR_DRIVER; }
  TnParams p = {};
  p.ws = ws; p.M = M; p.Na = Na; p.Nb = Nb; p.ta = (Na + 255) / 256; p.tb = (Nb + 255) / 256; p.splits = splits;
  p.rows_per_split = ((M + splits - 1) / splits + 63) / 64 * 64;
  p.krows = 64;
  p.nstage = 3;
  const int smem_bytes = p.nstage * 2 * kBSlabBytes + 512;
  const long long n_units = static_cast<long long>(p.ta) * p.tb * splits;
  const unsigned grid = static_cast<unsigned>(n_units < G ? n_units : G);
  static bool done[FK_MAX_DEVICES];
  const int r2 = set_smem_attr(gemm_tn_kernel, done[fk_device_ordinal()], kGemmSmemLimit);
  if (r2 != FK_OK) return r2;
  gemm_tn_kernel<<<grid, kGemmThreads, smem_bytes, stream>>>(ta, tb, p);
  FK_CHECK_LAUNCH();
  const long long n4 = static_cast<long long>(Na) * Nb / 4;
  gemm_tn_reduce_kernel<<<static_cast<unsigned>((n4 + 255) / 256), 256, 0, stream>>>(ws, out, n4, splits);
  FK_CHECK_LAUNCH();
  fk_count_launch(2);
  return FK_OK;
}

// Patch embedding of brainformer.Encoder (models/brainformer.py:282 `to_patches` 'b (t p1) c -> b (t c) p1', :285 / :338-343
// Linear(p1 -> dim) with bias, + the electrode embedding): token (trial b, patch t, electrode c) = x[b, t p1 .. t p1 + p1, c].
// With x viewed as the row-major matrix [B T, E], the p1 rows of one (b, t) ARE the transposed patch matrix of that
// patch's E tokens, so the projection of those tokens is the TN product  x_bt[p1, E]^T  Wt[p1, dim]: the gemm_tn kernel
// with one row range per patch, both operands read MN-major by TMA straight from x and W^T -- the patch tensor
// [B, S, p1] of the reference (a transposed copy) never exists.  Epilogue: + bias (+ emb [E, dim]) -> bf16 [B S, dim].
FK_API int fk_patch_embed_forward(const void* x_bf16, long long ldx, const void* wt_bf16, const float* bias, const float* emb,
                                  void* out_bf16, long long n_rows, int E, int patch, int dim, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(x_bf16 && wt_bf16 && out_bf16 && n_rows > 0 && E > 0 && patch > 0 && dim > 0, "fk_patch_embed_forward: bad argument");
  FK_REQUIRE(patch % 16 == 0 && patch <= 64 && n_rows % patch == 0, "fk_patch_embed_forward: patch size must be 16, 32, 48 or 64 and divide the rows");
  FK_REQUIRE(E % 64 == 0 && dim % 64 == 0 && ldx % 8 == 0 && ldx >= E, "fk_patch_embed_forward: electrodes and dim must be multiples of 64");
  FK_REQUIRE(n_rows < (1ll << 31) - 64, "fk_patch_embed_forward: too many rows");
  FK_REQUIRE((reinterpret_cast<uintptr_t>(x_bf16) & 15) == 0 && (reinterpret_cast<uintptr_t>(wt_bf16) & 15) == 0 &&
             (reinterpret_cast<uintptr_t>(out_bf16) & 15) == 0, "fk_patch_embed_forward: pointers must be 16-byte aligned");
  const int G = fk_sm_count();
  FK_REQUIRE(G > 0, "fk_patch_embed_forward: no device");
  CUtensorMap ta, tb;
  // A = x: rows = (trial, bin), Na = electrodes.  B = W^T [patch, dim]: the same rows for every row range (the producer
  // gives B the row coordinate within the range).
  int rc = make_tmap_bf16_chunks(&ta, x_bf16, static_cast<uint64_t>(n_rows), static_cast<uint64_t>(E), static_cast<uint64_t>(ldx),
                                 static_cast<uint32_t>(patch));
  rc |= make_tmap_bf16_chunks(&tb, wt_bf16, static_cast<uint64_t>(patch), static_cast<uint64_t>(dim), static_cast<uint64_t>(dim),
                              static_cast<uint32_t>(patch));
  if (rc != FK_OK) { fk_set_last_error("cuTensorMapEncodeTiled failed", __FILE__, __LINE__); return FK_ERR_DRIVER; }
  TnParams p = {};
  p.ws = nullptr; p.M = n_rows; p.Na = E; p.Nb = dim; p.ta = (E + 255) / 256; p.tb = (dim + 255) / 256;
  p.splits = static_cast<int>(n_rows / patch);
  p.rows_per_split = patch; p.krows = patch; p.nstage = 3;
  p.out_bf16 = static_cast<__nv_bfloat16*>(out_bf16); p.bias = bias; p.emb = emb;
  const int smem_bytes = p.nstage * 2 * kBSlabBytes + 512;
  const long long n_units = static_cast<long long>(p.ta) * p.tb * p.splits;
  const unsigned grid = static_cast<unsigned>(n_units < G ? n_units : G);
  static bool done[FK_MAX_DEVICES];
  const int r2 = set_smem_attr(gemm_tn_kernel, done[fk_device_ordinal()], kGemmSmemLimit);
  if (r2 != FK_OK) return r2;
  gemm_tn_kernel<<<grid, kGemmThreads, smem_bytes, stream>>>(ta, tb, p);
  FK_CHECK_LAUNCH();
  fk_count_launch(1);
  return FK_OK;
}
