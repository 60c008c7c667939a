// Attention backward on the 5th-gen tensor cores (tcgen05.mma + TMEM + TMA), head_dim 32, label masks.  Head_dim 16 runs
// the head_dim-32 kernels instantiated with HD = 16 (16-column heads, 32-byte rows and the 32-byte swizzle), on the default
// path only: folded statistics, MN-major accumulate operands.  The forward and the statistics kernel are instantiated at
// HD = 64 as well (128-byte rows, the 128-byte swizzle); the head_dim-64 backward is a kernel of its own
// (attn_bwd_tc64_kernel), after the forward.
//
// Same math and mask rule as attention.cu (reference: F.scaled_dot_product_attention backward at
// models/brainformer.py:168), restructured for Blackwell: every matmul is a tcgen05.mma issued by one thread,
// score tiles live in TMEM, and each compute thread owns one resident row, so the per-row statistics never
// need a shuffle.  Two launches of one kernel template:
//
//   MODE_DKV  CTA owns 128 keys (resident K, V), streams 64-query tiles (Q, dO):
//             S^T = K Q^T, dP^T = V dO^T  (TMEM)  ->  P^T = 2^(S^T c - lse[q]),  dS^T = P^T (dP^T - delta[q])
//             -> bf16 operands in TMEM  ->  dV += P^T dO,  dK += dS^T Q  (TMEM accumulators, 32 columns each)
//   MODE_DQ   CTA owns 128 queries (resident Q, dO), streams 64-key tiles (K, V):
//             S = Q K^T, dP = dO V^T  ->  P, dS  ->  dQ += dS K
//
// Pipeline per CTA (512 threads): warp 0 = TMA producer (8-stage ring of streamed tiles), warp 1 = MMA issuer
// of the score products, warp 2 = TMEM allocator, warp 3 = builds the list of visible tiles, then issues the
// accumulate MMAs, warps 4-15 = three compute warpgroups, one per TMEM score stage (tile j belongs to warpgroup
// j % 3), so three tiles are in flight.  P / dS never touch shared memory: a compute thread packs its row to bf16 and
// writes it back IN PLACE over the fp32 score columns it has already consumed (tcgen05.st), and the accumulate MMAs
// read that as their A operand straight from TMEM (TS mode); their B operand is the streamed [tokens][32] tile itself,
// read MN-major (K = tokens), the same tile that served the score MMA as a K-major operand (K = head dim).  Tiles are
// TMA-loaded with the 64-byte swizzle.  The smem data pipe, which bounds an SS-mode version of this kernel, only
// carries the streamed operands.
#include <algorithm>
#include <type_traits>

#include "common.cuh"
#include "fk_b200.h"
#include "tma_host.cuh"

namespace fk {

constexpr int kRows = 128;        // resident rows per CTA (UMMA M)
constexpr int kCols = 64;         // streamed tile (UMMA N of the score MMAs, K of the accumulate MMAs)
constexpr int kNST = 8;           // streamed smem stages
constexpr int kNG = 3;            // score stages in TMEM = tiles in flight = compute warpgroups (tile j belongs to j % kNG)
// TMEM map (512 columns): score stage g at g*128 (S 64 | dP 64 fp32 columns).  The compute warpgroup overwrites its
// stage IN PLACE with the bf16 operands of the accumulate MMAs (P pairs at +0..31, dS pairs at +64..95), so no separate
// operand buffers exist and three tiles fit; accumulators at 384 (dV) and 416 (dK / dQ).
constexpr int kSub = kCols / 16;              // 16-column sub-chunks per tile
constexpr int kTcThreads = 128 + 128 * kNG;
constexpr int kAccCol = 128 * kNG;
// Resident operands of the score MMAs in TMEM (TS mode: a tcgen05.mma with its A operand in TMEM costs N/2 = 32 cycles at
// N = 64, against the 48-cycle floor of the shared-memory form): columns 448.. hold the two resident tiles as packed bf16
// pairs (16 columns each), the two constant ones tiles of the folded statistics (8 each) and, for the dQ kernel, the
// resident queries' statistics rows (8).
constexpr int kResCol = kAccCol + 64;         // 448: resident A (K / Q), +16: resident B (V / dO)
constexpr int kOnesCol = kResCol + 32;        // 480: ones(cols 0-2), +8: ones(cols 3-5)
constexpr int kAugCol = kOnesCol + 16;        // 496: DQ statistics rows
constexpr int kMaxTiles = 2048;   // streamed tiles per sequence (S <= 131072); entries carry a flag in bit 15
constexpr int MODE_DKV = 0, MODE_DQ = 1;

struct TcParams {
  const int *row_id, *col_id;                          // labels of the resident / streamed side, or null
  const int *row_min, *row_max, *col_min, *col_max;    // per-64-token tile label ranges
  const float *lse, *delta;                            // [B, H, Sq]
  __nv_bfloat16 *out0, *out1;                          // DKV: dV, dK.  DQ: (unused), dQ
  long long o0_bs, o0_ts, o1_bs, o1_ts;
  int B, H, S_row, S_col, Sq;
  float scale, scale_log2;
  const float2* rope_table;                            // [rope_len][hd/2] (cos, sin) or null: inverse RoPE fused into the
  const int* rope_pos;                                 // store of dK / dQ (position of row = rope_pos ? rope_pos[b][row]
  int rope_len, rope_offset;                           //  : row + rope_offset), replacing two fk_rope passes per layer
  long long* prof;                                     // kProf instantiation: [n_ctas][16] cycle counters
  unsigned int* items;                                 // caller-owned hand-out counters of THIS launch: [0] next item,
                                                       // [1] CTAs finished; zero on entry, zeroed again by the last CTA out
  int fold;                                            // 1: lse and delta arrive as an extra K step of the score MMAs (tm_aug):
                                                       //    S' = S - lse / c, dP' = dP - delta come out of the tensor core
  int mn_major;                                        // 1: the accumulate MMAs read their B operand (Q / dO / K tile,
                                                       // [64 tokens][32 dims]) MN-major from the score stage itself;
                                                       // 0: K-major from transposed copies (tm_tA / tm_tB)
};

// Diagnosis only (scripts/gpu_attn_stalls.py): fk_attn_backward_tc_profile launches the stall-accounting
// instantiation, which writes per CTA: 0 lifetime, 1 setup, 2 tiles, 3 first score stage ready, 4 sum wait sdp_full,
// 5 (unused), 6 sum named barrier, 7 sum compute, 8 last p_ready, 9 accumulators complete, 10 stores done,
// 11 score issuer wait st_full, 12 score issuer wait stage_free, 13 acc issuer wait p_ready, 14 producer wait st_empty
// (3..10 by warpgroup 0, warp 4, lane 0; times since CTA start).

template <int kProf>
__device__ __forceinline__ void wait_acc(uint64_t* bar, uint32_t phase, long long& acc) {
  if constexpr (kProf == 1) {
    if (mbar_test_wait(bar, phase)) return;
    const long long t = clock64();
    mbar_wait(bar, phase);
    acc += clock64() - t;
  } else {
    mbar_wait(bar, phase);
  }
}

struct TcSmem {
  // offsets from the 1024-aligned dynamic smem base
  static constexpr int resA = 0;                       // 128 x 64 B; second buffer (next item, prefetched) at + 16384
  static constexpr int resB = 8192;
  static constexpr int stream = 32768;                 // kNST x 16 KB: stA | stB | tA | tB (4 KB each)
  static constexpr int stats = stream + kNST * 16384;  // [2 wg][2 buffers][lse | delta | id][64] x 4 B           // [2 wg][lse | delta | id][64] x 4 B
  static constexpr int tiles = stats + kNG * 2 * 3 * 64 * 4; // uint16 visible-tile list
  // folded statistics (TcParams::fold): two constant [128][16] operand tiles (ones in columns 0-2 / 3-5) and, for the dQ
  // kernel, the resident queries' statistics rows (two buffers, like the resident tiles); 32-byte rows, SWIZZLE_32B
  static constexpr int ones = (tiles + 2 * kMaxTiles * 2 + 1023) / 1024 * 1024;   // two lists: the next item's is built while this one runs
  static constexpr int aug_res = ones + 8192;
  static constexpr int bars = aug_res + 8192;
  static constexpr int total = bars + 512;
};

// FK_ATTN_EXP (diagnosis builds only, results are WRONG): 1 = no MUFU, 2 = no TMEM operand stores, 3 = no stats LDS,
// 4 = no math at all between the TMEM loads and stores, 5 = no delta subtraction (and no delta LDS),
// 6 = neither delta nor lse (P = ex2(S * c)), 7 = 6 + no statistics staging / named barrier and no scale multiply
// (P = ex2(S)): the upper bound of folding lse, delta and the softmax scale into the score MMAs.
#ifndef FK_ATTN_EXP
#define FK_ATTN_EXP 0
#endif
__device__ __forceinline__ float fast_ex2(float x) {
#if FK_ATTN_EXP == 1
  return x * 0.25f;
#else
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
#endif
}
// (F2FP.BF16.PACK_AB runs at full rate, 126 pairs/clk/SM, and MUFU.EX2 at 16/clk/SM: scripts/microbench/xu_rate.cu)
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ void tmem_ld32_dep(uint32_t taddr, uint32_t (&r)[32]) { tmem_ld32(taddr, r); }
__device__ __forceinline__ void tmem_wait2(uint32_t (&a)[32], uint32_t (&b)[32]) {
  // wait::ld with both destination arrays as in/out operands so no use is scheduled above the wait
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]),
                 "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]),
                 "+r"(a[16]), "+r"(a[17]), "+r"(a[18]), "+r"(a[19]), "+r"(a[20]), "+r"(a[21]), "+r"(a[22]), "+r"(a[23]),
                 "+r"(a[24]), "+r"(a[25]), "+r"(a[26]), "+r"(a[27]), "+r"(a[28]), "+r"(a[29]), "+r"(a[30]), "+r"(a[31])
               :: "memory");
  asm volatile("" : "+r"(b[0]), "+r"(b[1]), "+r"(b[2]), "+r"(b[3]), "+r"(b[4]), "+r"(b[5]), "+r"(b[6]), "+r"(b[7]),
                    "+r"(b[8]), "+r"(b[9]), "+r"(b[10]), "+r"(b[11]), "+r"(b[12]), "+r"(b[13]), "+r"(b[14]), "+r"(b[15]),
                    "+r"(b[16]), "+r"(b[17]), "+r"(b[18]), "+r"(b[19]), "+r"(b[20]), "+r"(b[21]), "+r"(b[22]), "+r"(b[23]),
                    "+r"(b[24]), "+r"(b[25]), "+r"(b[26]), "+r"(b[27]), "+r"(b[28]), "+r"(b[29]), "+r"(b[30]), "+r"(b[31])
               :: "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_wait2_16(uint32_t (&a)[16], uint32_t (&b)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]),
                 "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]),
                 "+r"(b[0]), "+r"(b[1]), "+r"(b[2]), "+r"(b[3]), "+r"(b[4]), "+r"(b[5]), "+r"(b[6]), "+r"(b[7]),
                 "+r"(b[8]), "+r"(b[9]), "+r"(b[10]), "+r"(b[11]), "+r"(b[12]), "+r"(b[13]), "+r"(b[14]), "+r"(b[15])
               :: "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}

__device__ __forceinline__ void tmem_wait1_16(uint32_t (&a)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]),
                 "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15])
               :: "memory");
}
__device__ __forceinline__ void tmem_wait1_32(uint32_t (&a)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]),
                 "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]),
                 "+r"(a[16]), "+r"(a[17]), "+r"(a[18]), "+r"(a[19]), "+r"(a[20]), "+r"(a[21]), "+r"(a[22]), "+r"(a[23]),
                 "+r"(a[24]), "+r"(a[25]), "+r"(a[26]), "+r"(a[27]), "+r"(a[28]), "+r"(a[29]), "+r"(a[30]), "+r"(a[31])
               :: "memory");
}

// Head width HD of the templated kernels: a [tokens][HD] bf16 row is 2 HD bytes, TMA-loaded with the swizzle of that
// width (SWIZZLE_32B at 16, SWIZZLE_64B at 32, SWIZZLE_128B at 64).  A K step of 16 rows of an MN-major tile adds 2 HD in
// the descriptor's (address >> 4) field.
template <int HD>
__device__ __forceinline__ uint64_t umma_desc_rows(uint32_t saddr) {
  if constexpr (HD == 16) return umma_desc_sw32(saddr);
  else if constexpr (HD == 32) return umma_desc_sw64(saddr);
  else return umma_desc_sw128(saddr);
}
template <int N>
__device__ __forceinline__ void tmem_ld_wait(uint32_t taddr, uint32_t (&r)[N]) {
  if constexpr (N == 16) { tmem_ld16(taddr, r); tmem_wait1_16(r); }
  else { tmem_ld32(taddr, r); tmem_wait1_32(r); }
}
template <int N>
__device__ __forceinline__ void tmem_st_cols(uint32_t taddr, const uint32_t (&r)[N]) {
  if constexpr (N == 16) tmem_st16(taddr, r);
  else tmem_st32(taddr, r);
}

// Work-item hand-out of the persistent kernels: p.items[0] = next item, p.items[1] = CTAs that have finished; the last
// CTA to finish puts both back to zero, so no host-side reset (and no extra launch) is needed.  The two words belong
// to the caller (one pair per launch in flight: launches on different streams must be given different pairs), so the
// library holds no device-side state and is re-entrant per stream.

// HD = 16 is instantiated on the default path only (kProf 0, folded statistics, MN-major accumulate operands): the
// resident tiles take 8 packed TMEM columns each, the score MMAs one K step, the accumulate MMAs N = 16.
template <int MODE, int kProf, bool kFold, int HD = 32>
__global__ void __launch_bounds__(kTcThreads, 1)
attn_bwd_tc_kernel(const __grid_constant__ CUtensorMap tm_resA, const __grid_constant__ CUtensorMap tm_resB,
                   const __grid_constant__ CUtensorMap tm_stA, const __grid_constant__ CUtensorMap tm_stB,
                   const __grid_constant__ CUtensorMap tm_tA, const __grid_constant__ CUtensorMap tm_tB,
                   const __grid_constant__ CUtensorMap tm_aug, const TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + TcSmem::bars);
  uint64_t* res_full = bars;               // [2]    resident tiles of item n in buffer n & 1
  uint64_t* list_ready = bars + 2;         // [1]    warp 2 has written the id and the tile list of the next item
  uint64_t* st_full = bars + 3;            // [kNST]
  uint64_t* st_empty = bars + 3 + kNST;    // [kNST]
  uint64_t* sdp_full = bars + 3 + 2 * kNST;   // [kNG]  score stage g written by the tensor core
  uint64_t* stage_free = sdp_full + kNG;   // [kNG]  the accumulate MMAs that read stage g (as P / dS) have retired
  uint64_t* p_ready = stage_free + kNG;    // [kNG]  P / dS written in place into stage g (4 warps arrive)
  uint64_t* acc_full = p_ready + kNG;      // [1]
  uint64_t* dp_full = acc_full + 1;        // [kNG]  fold: dP of stage g written (sdp_full then announces S alone, so the
                                           //        exponentials of a tile start while its dP MMAs still run)
  uint64_t* res_tmem = dp_full + kNG;      // [1]    warpgroup 0 has copied the item's resident tiles into TMEM (4 warps arrive)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_tmem + 1);
  int* n_tiles_slot = reinterpret_cast<int*>(res_tmem + 1) + 1;   // [2]
  int* item_slot = reinterpret_cast<int*>(res_tmem + 1) + 3;      // [2]: item ids handed to this CTA, double buffered
  uint16_t* tile_lists = reinterpret_cast<uint16_t*>(smem + TcSmem::tiles);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr bool kFull = kProf == 1;
  const bool masked = p.row_id != nullptr;
  const int n_col_tiles = (p.S_col + kCols - 1) / kCols;
  const int n_row_tiles64 = (p.S_row + 63) / 64;
  const int n_row_tiles = (p.S_row + kRows - 1) / kRows;
  const int n_items = n_row_tiles * p.H * p.B;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_resA); tma_prefetch_desc(&tm_resB); tma_prefetch_desc(&tm_stA);
    tma_prefetch_desc(&tm_stB); tma_prefetch_desc(&tm_tB);
    if (MODE == MODE_DKV) tma_prefetch_desc(&tm_tA);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(&res_full[0], 1);
    mbar_init(&res_full[1], 1);
    mbar_init(list_ready, 1);
    for (int i = 0; i < kNST; ++i) { mbar_init(&st_full[i], 1); mbar_init(&st_empty[i], 1); }
    for (int i = 0; i < kNG; ++i) {
      mbar_init(&sdp_full[i], 1);
      mbar_init(&stage_free[i], 1);
      mbar_init(&p_ready[i], 4);
      mbar_init(&dp_full[i], 1);
    }
    mbar_init(acc_full, 1);
    mbar_init(res_tmem, 4);
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  constexpr bool fold = kFold;                     // (compile time: the folded and the staged hot loops share no registers)
  if (fold && warp >= 4) {
    // constant operand tiles of the statistics K step: row r = 16 bf16, ones in columns 0-2 (picks -lse / c) resp. 3-5
    // (picks -delta), written in the SWIZZLE_32B pattern (the two 16-byte halves of a row swap when bit 2 of r is set)
    for (int i = threadIdx.x - 128; i < 2 * 128 * 2; i += kTcThreads - 128) {
      const int tile = i >> 8, r = (i >> 1) & 127, pc = i & 1;
      const int c = pc ^ ((r >> 2) & 1);
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (c == 0) v = tile == 0 ? make_uint4(0x3F803F80u, 0x00003F80u, 0u, 0u) : make_uint4(0u, 0x3F800000u, 0x3F803F80u, 0u);
      *reinterpret_cast<uint4*>(smem + TcSmem::ones + tile * 4096 + r * 32 + pc * 16) = v;
    }
    fence_proxy_async();                           // generic-proxy writes -> visible to the tensor core's (async proxy) reads
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (fold && MODE == MODE_DKV && warp >= 4 && warp < 8) {
    // constant A operands of the statistics K step, one row per thread: 16 bf16 = 8 packed columns
    const uint32_t t0 = tmem_base + (static_cast<uint32_t>((warp & 3) * 32) << 16) + kOnesCol;
    const uint32_t os[8] = {0x3F803F80u, 0x00003F80u, 0u, 0u, 0u, 0u, 0u, 0u};      // ones in elements 0-2
    const uint32_t od[8] = {0u, 0x3F800000u, 0x3F803F80u, 0u, 0u, 0u, 0u, 0u};      // ones in elements 3-5
    tmem_st8(t0, os);
    tmem_st8(t0 + 8, od);
    tmem_wait_st();
    tc_fence_before();
  }
  __syncthreads();
  tc_fence_after();

  // ---- persistent loop over work items (row tile, head, batch): barriers, TMEM and the smem rings live across items,
  //      which removes the 1-1.6 us launch gap between consecutive CTAs of an SM and the per-CTA setup.  All barrier
  //      parities below run on counters that continue across items (`base` = streamed tiles of the earlier items). ----
  int base = 0;                 // streamed tiles consumed by earlier items of this CTA
  uint32_t item_n = 0;          // items done by this CTA (parity of the once-per-item barriers)
  int pstage = 0;               // producer ring position (continues across items)
  uint32_t pphase = 0;
  int pre_cnt = -1;             // producer: streamed tiles of THIS item already requested during the previous item
                                // (-1: nothing, not even the resident tiles)
  // dynamic hand-out (items differ a lot in their number of visible tiles).  Warp 2, idle after the TMEM allocation,
  // works one item ahead: it fetches the id of the next item and builds that item's list of visible tiles while the
  // current item runs, so neither the atomic's round trip nor the list build is on anybody's critical path.
  auto build_list = [&](int it, int buf) {       // whole warp
    const int rt_ = it % n_row_tiles, b_ = it / (n_row_tiles * p.H);
    uint16_t* list = tile_lists + buf * kMaxTiles;
    // label range of the resident rows (two 64-token range entries)
    int row_lo = 0, row_hi = 0;
    if (masked) {
      const int i0 = rt_ * 2, i1 = min(rt_ * 2 + 1, n_row_tiles64 - 1);
      row_lo = min(p.row_min[b_ * n_row_tiles64 + i0], p.row_min[b_ * n_row_tiles64 + i1]);
      row_hi = max(p.row_max[b_ * n_row_tiles64 + i0], p.row_max[b_ * n_row_tiles64 + i1]);
    }
    // visible streamed tiles, in order (DKV: q tiles with qmax >= kmin(rows); DQ: k tiles with kmin <= qmax(rows)).
    // bit 15 of an entry = the tile needs the per-element label compare (it straddles a label boundary, or it is
    // the ragged tail of the key axis), so the compute warps never touch the range arrays in global memory.
    int cnt = 0;
    for (int cb = 0; cb < n_col_tiles; cb += 32) {
      const int t = cb + lane;
      bool vis = t < n_col_tiles, nm = false;
      if (vis) {
        int cmin = 0, cmax = 0;
        if (masked) { cmin = p.col_min[b_ * n_col_tiles + t]; cmax = p.col_max[b_ * n_col_tiles + t]; }
        if (MODE == MODE_DKV) {
          vis = !masked || cmax >= row_lo;
          nm = masked && (row_hi > cmin);
        } else {
          vis = !masked || cmin <= row_hi;
          nm = (masked && (cmax > row_lo)) || (t * kCols + kCols > p.S_col);
        }
      }
      const unsigned m = __ballot_sync(0xffffffffu, vis);
      if (vis) list[cnt + __popc(m & ((1u << lane) - 1u))] = static_cast<uint16_t>(t | (nm ? 0x8000 : 0));
      cnt += __popc(m);
    }
    if (lane == 0) n_tiles_slot[buf] = cnt;
  };
  if (warp == 2) {
    int first = 0;
    if (lane == 0) first = static_cast<int>(atomicAdd(&p.items[0], 1u));
    first = __shfl_sync(0xffffffffu, first, 0);
    if (lane == 0) item_slot[0] = first;
    if (first < n_items) build_list(first, 0);
  }
  __syncthreads();
  for (int item = item_slot[0]; item < n_items; item = item_slot[(item_n + 1) & 1], ++item_n) {
  const int rt = item % n_row_tiles, h = (item / n_row_tiles) % p.H, b = item / (n_row_tiles * p.H);
  const int r0 = rt * kRows;
  const long long t_start = kProf ? clock64() : 0;
  unsigned long long g_start = 0;
  if (kProf == 2 && threadIdx.x == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g_start));
  long long* prof = kProf ? p.prof + static_cast<long long>(item) * 24 : nullptr;
  // per-tile event stamps of the first item of CTA 0 (kFull only): trace[event][tile], after the counters
  long long* trace = (kFull && blockIdx.x == 0 && item_n == 0) ? p.prof + static_cast<long long>(n_items) * 24 : nullptr;
  const uint16_t* tile_list = tile_lists + (item_n & 1) * kMaxTiles;     // made visible by the previous item's final barrier
  const int T = n_tiles_slot[item_n & 1];
  if (kFull && threadIdx.x == 0) { prof[1] = clock64() - t_start; prof[2] = T; }

  if (warp == 2) {
    int nxt = 0;
    if (lane == 0) nxt = static_cast<int>(atomicAdd(&p.items[0], 1u));
    nxt = __shfl_sync(0xffffffffu, nxt, 0);
    if (lane == 0) item_slot[(item_n + 1) & 1] = nxt;
    if (nxt < n_items) build_list(nxt, (item_n + 1) & 1);
    __syncwarp();
    if (lane == 0) mbar_arrive(list_ready);      // phase item_n: the producer may now run ahead into the next item
  }

  constexpr uint32_t kStageBytes = (MODE == MODE_DKV) ? 16384u : 12288u;
  constexpr uint32_t kResBytes = 2u * kRows * HD * 2u;       // resident A | B tiles
  constexpr uint32_t kTileBytes = 2u * kCols * HD * 2u;      // streamed A | B tiles

  if (warp == 0) {
    // ================================ TMA producer ================================
    // Control warps run their loops with the WHOLE warp (uniform control flow; barrier waits by all lanes) and issue
    // the asynchronous operation from one elected lane: operands then live in uniform registers and ptxas emits bare
    // UTMALDG / UTCHMMA / UTCBAR instructions.  Under a `lane == 0` branch every such instruction became a divergence
    // waterfall (ELECT + R2UR.BROADCAST chain + branch, ~115 cycles per MMA issue -- scripts/gpu_search_stalls.py).
    {
      const int T_u = __shfl_sync(0xffffffffu, T, 0);
      long long w_se = 0;
      auto load_resident = [&](int h_, int r0_, int b_, int buf) {
        if (elect_one()) {
          mbar_expect_tx(&res_full[buf], (MODE == MODE_DQ && fold) ? kResBytes + 4096u : kResBytes);
          tma_load_4d(smem + TcSmem::resA + buf * 16384, &tm_resA, &res_full[buf], 0, h_, r0_, b_);
          tma_load_4d(smem + TcSmem::resB + buf * 16384, &tm_resB, &res_full[buf], 0, h_, r0_, b_);
          if (MODE == MODE_DQ && fold) tma_load_4d(smem + TcSmem::aug_res + buf * 4096, &tm_aug, &res_full[buf], 0, r0_, h_, b_);
        }
        __syncwarp();
      };
      auto load_tile = [&](int t, int h_, int b_) {
        uint8_t* st = smem + TcSmem::stream + pstage * 16384;
        wait_acc<kProf>(&st_empty[pstage], pphase ^ 1, w_se);
        if (elect_one()) {
          mbar_expect_tx(&st_full[pstage], (HD == 16 || p.mn_major) ? ((MODE == MODE_DKV && fold) ? kTileBytes + 2048u : kTileBytes) : kStageBytes);
          tma_load_4d(st, &tm_stA, &st_full[pstage], 0, h_, t * kCols, b_);
          tma_load_4d(st + 4096, &tm_stB, &st_full[pstage], 0, h_, t * kCols, b_);
          if (MODE == MODE_DKV && fold) tma_load_4d(st + 8192, &tm_aug, &st_full[pstage], 0, t * kCols, h_, b_);   // statistics rows of the tile's queries
          if (HD == 32 && !p.mn_major) {
            if (MODE == MODE_DKV) tma_load_2d(st + 8192, &tm_tA, &st_full[pstage], t * kCols, (b_ * p.H + h_) * 32);
            tma_load_2d(st + 12288, &tm_tB, &st_full[pstage], t * kCols, (b_ * p.H + h_) * 32);
          }
        }
        __syncwarp();
        if (++pstage == kNST) { pstage = 0; pphase ^= 1; }
      };
      // this item: whatever the previous item's run-ahead has not requested yet
      if (pre_cnt < 0) { load_resident(h, r0, b, item_n & 1); pre_cnt = 0; }
      for (int j = pre_cnt; j < T_u; ++j) load_tile(__shfl_sync(0xffffffffu, tile_list[j] & 0x7fff, 0), h, b);
      // run ahead into the next item while this one drains: its resident tiles (other buffer) and as many of its first
      // streamed tiles as the ring takes without waiting on this item's last consumers for long (half the ring)
      mbar_wait(list_ready, item_n & 1);
      const int nxt = __shfl_sync(0xffffffffu, item_slot[(item_n + 1) & 1], 0);
      pre_cnt = -1;
      if (nxt < n_items) {
        const int rt2 = nxt % n_row_tiles, h2 = (nxt / n_row_tiles) % p.H, b2 = nxt / (n_row_tiles * p.H);
        const uint16_t* list2 = tile_lists + ((item_n + 1) & 1) * kMaxTiles;
        const int T2 = __shfl_sync(0xffffffffu, n_tiles_slot[(item_n + 1) & 1], 0);
        load_resident(h2, rt2 * kRows, b2, (item_n + 1) & 1);
        pre_cnt = 0;
        const int ahead = T2 < kNST / 2 ? T2 : kNST / 2;
        for (int j = 0; j < ahead; ++j, ++pre_cnt) load_tile(__shfl_sync(0xffffffffu, list2[j] & 0x7fff, 0), h2, b2);
      }
      if (kFull && lane == 0) prof[14] = w_se;
    }
  } else if (warp == 1) {
    // ================================ score-MMA issuer ================================
    // (the score MMAs and the accumulate MMAs are issued by two different warps so that neither waits behind the other's
    //  barrier; issuing both from one thread, back to back without a barrier between the reader and the overwriter of
    //  a stage, was measured 13 % slower -- DESIGN.md section 4.2)
    {
      constexpr uint32_t idesc_score = umma_idesc_bf16(kRows, kCols);
      const int T_u = __shfl_sync(0xffffffffu, T, 0);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t stream = smem_u32(smem + TcSmem::stream);
      mbar_wait(res_tmem, item_n & 1);                // the resident tiles of this item sit in TMEM (copied by warpgroup 0)
      tc_fence_after();
      const uint32_t tA = tmem_u + kResCol, tB = tmem_u + kResCol + 16;
      long long w_sf = 0, w_free = 0;
      for (int js = 0; js < T_u; ++js) {
        const int gt = base + js;                    // tile counter across items
        const int stage = gt % kNST, g = gt % kNG, n = gt / kNG;
        // (operands of the MMAs are formed BEFORE the waits: ~50 uniform-datapath instructions that would otherwise sit
        //  on the critical path stage_free -> score MMAs)
        uint64_t dS = umma_desc_rows<HD>(stream + stage * 16384), dD = umma_desc_rows<HD>(stream + stage * 16384 + 4096);
        uint32_t d_s = tmem_u + g * 128, d_dp = tmem_u + g * 128 + 64;
        uint64_t* const bar_full = &sdp_full[g];
        // statistics K step (fold): DKV  A = constant ones tile (keys), B = the tile's query statistics;
        //                           DQ   A = the resident queries' statistics, B = constant ones tile (keys)
        uint64_t fB_s = 0, fB_d = 0;
        if constexpr (fold) {
          // B operands of the statistics K step (its A operands are in TMEM): DKV the tile's statistics rows, DQ the ones tiles
          fB_s = fB_d = umma_desc_sw32(stream + stage * 16384 + 8192);
          if (MODE == MODE_DQ) {
            fB_s = umma_desc_sw32(smem_u32(smem + TcSmem::ones));
            fB_d = umma_desc_sw32(smem_u32(smem + TcSmem::ones + 4096));
          }
          asm volatile("" : "+l"(fB_s), "+l"(fB_d));
        }
        {
          // pin the values here: without this the compiler sinks the whole address arithmetic below the waits again
          asm volatile("" : "+l"(dS), "+l"(dD), "+r"(d_s), "+r"(d_dp));
        }
        wait_acc<kProf>(&st_full[stage], (gt / kNST) & 1, w_sf);
        wait_acc<kProf>(&stage_free[g], (n & 1) ^ 1, w_free);
        if (kFull && trace && lane == 0 && js < 128) trace[2 * 128 + js] = clock64();
        tc_fence_after();
        if (elect_one()) {
          // a K step of 16 bf16 = 32 bytes = +2 in the descriptor's (address >> 4) field
          // TS mode: A = the resident tile in TMEM (K step of 16 elements = 8 packed columns)
          umma_bf16_ts(d_s, tA, dS, idesc_score, 0u);
          if (HD == 32) umma_bf16_ts(d_s, tA + 8, dS + 2, idesc_score, 1u);
          if (fold) {
            umma_bf16_ts(d_s, MODE == MODE_DKV ? tmem_u + kOnesCol : tmem_u + kAugCol, fB_s, idesc_score, 1u);
            umma_commit(bar_full);                         // S' complete: the warpgroup starts on the exponentials
          }
          umma_bf16_ts(d_dp, tB, dD, idesc_score, 0u);
          if (HD == 32) umma_bf16_ts(d_dp, tB + 8, dD + 2, idesc_score, 1u);
          if (fold) {
            umma_bf16_ts(d_dp, MODE == MODE_DKV ? tmem_u + kOnesCol + 8 : tmem_u + kAugCol, fB_d, idesc_score, 1u);
            umma_commit(&dp_full[g]);
          } else {
            umma_commit(bar_full);
          }
        }
        __syncwarp();
        if (kFull && trace && lane == 0 && js < 128) trace[3 * 128 + js] = clock64();
      }
      if (kFull && lane == 0) { prof[11] = w_sf; prof[12] = w_free; }
    }
  } else if (warp == 3) {
    // ================================ accumulate-MMA issuer ================================
    {
      constexpr uint32_t idesc_acc = umma_idesc_bf16(kRows, HD);
      const int T_u = __shfl_sync(0xffffffffu, T, 0);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t stream = smem_u32(smem + TcSmem::stream);
      long long w_pr = 0;
      for (int ia = 0; ia < T_u; ++ia) {
        const int gt = base + ia;                    // tile counter across items
        const int stage = gt % kNST, g = gt % kNG, n = gt / kNG;
        // (operands formed before the wait, see the score issuer)
        uint32_t ta = tmem_u + g * 128;                   // P pairs at +0..31, dS pairs at +64..95 (written in place)
        uint64_t dMA = umma_desc_rows<HD>(stream + stage * 16384 + 4096), dMB = umma_desc_rows<HD>(stream + stage * 16384);
        uint64_t* const bar_free = &stage_free[g];
        uint64_t* const bar_empty = &st_empty[stage];
        asm volatile("" : "+l"(dMA), "+l"(dMB), "+r"(ta));      // pin (see the score issuer)
        wait_acc<kProf>(&p_ready[g], n & 1, w_pr);
        if (kFull && trace && lane == 0 && ia < 128) trace[0 * 128 + ia] = clock64();
        tc_fence_after();
        if (HD == 16 || p.mn_major) {
          // B operand straight from the score stage: tile [64 tokens][32 dims], 64-byte rows, SWIZZLE_64B = the canonical
          // MN-major layout (N = 32 dims contiguous, 8-token groups 512 B apart); a K step of 16 tokens = 1024 B.  (At
          // head_dim 16: [64 tokens][16 dims], 32-byte rows, SWIZZLE_32B, 8-token groups 256 B apart, K step 512 B.)
          // DKV: dV += P^T dO (stB), dK += dS^T Q (stA).  DQ: dQ += dS K (stA).
          if (elect_one()) {
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              if (MODE == MODE_DKV) umma_bf16_ts(tmem_u + kAccCol, ta + kk * 8, dMA + 2 * HD * kk, idesc_acc | (1u << 16), (ia > 0 || kk > 0) ? 1u : 0u);
              umma_bf16_ts(tmem_u + kAccCol + 32, ta + 64 + kk * 8, dMB + 2 * HD * kk, idesc_acc | (1u << 16), (ia > 0 || kk > 0) ? 1u : 0u);
            }
            umma_commit(bar_free);
            umma_commit(bar_empty);
          }
        } else {
          const uint64_t dTA = umma_desc_sw128(stream + stage * 16384 + 8192), dTB = umma_desc_sw128(stream + stage * 16384 + 12288);
          if (elect_one()) {
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              if (MODE == MODE_DKV) umma_bf16_ts(tmem_u + kAccCol, ta + kk * 8, dTA + 2 * kk, idesc_acc, (ia > 0 || kk > 0) ? 1u : 0u);
              umma_bf16_ts(tmem_u + kAccCol + 32, ta + 64 + kk * 8, dTB + 2 * kk, idesc_acc, (ia > 0 || kk > 0) ? 1u : 0u);
            }
            umma_commit(&stage_free[g]);
            umma_commit(&st_empty[stage]);
          }
        }
        __syncwarp();
        if (kFull && trace && lane == 0 && ia < 128) trace[1 * 128 + ia] = clock64();
      }
      if (elect_one()) umma_commit(acc_full);
      __syncwarp();
      if (kFull && lane == 0) prof[13] = w_pr;
    }
  } else if (warp >= 4) {
    // ================================ compute warpgroups ================================
    // kNG warpgroups, one per score stage: warpgroup g owns the tiles j with j % kNG == g, reads S / dP of its stage and
    // writes P / dS back in place.
    const int g = (warp - 4) >> 2;               // warpgroup = score stage
    const int q4 = warp & 3;                     // TMEM lane quarter
    const int r = q4 * 32 + lane;                // resident row owned by this thread
    const int tid = r;                           // index within the warpgroup
    const int row = r0 + r;
    const bool row_ok = row < p.S_row;
    float* stats_base = reinterpret_cast<float*>(smem + TcSmem::stats) + g * 384;
    const float* lse_g = p.lse + (static_cast<long long>(b) * p.H + h) * p.Sq;
    const float* delta_g = p.delta + (static_cast<long long>(b) * p.H + h) * p.Sq;
    const int my_id = masked ? (row_ok ? p.row_id[static_cast<long long>(b) * p.S_row + row]
                                       : (MODE == MODE_DKV ? 0x7fffffff : -0x7fffffff))
                             : 0;
    float my_lse = INFINITY, my_delta = 0.f;     // DQ: per-row statistics
    if (MODE == MODE_DQ && row_ok && !fold) { my_lse = lse_g[row]; my_delta = delta_g[row]; }
    if (g == 0) {
      // resident tiles of this item: shared memory (TMA, 64-byte rows, SWIZZLE_64B) -> this thread's TMEM lane as packed
      // bf16 pairs, the A operand layout of a TS-mode MMA.  (Every MMA of the previous item has retired: the item loop
      // ends with a CTA-wide barrier behind acc_full.)
      mbar_wait(&res_full[item_n & 1], (item_n >> 1) & 1);
      const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16);
      if constexpr (HD == 16) {
        // 32-byte rows, SWIZZLE_32B (the halves swap when bit 2 of r is set): 8 packed columns per tile
        const int s1 = (r >> 2) & 1;
#pragma unroll
        for (int t2 = 0; t2 < 2; ++t2) {
          const uint8_t* rowp = smem + (t2 ? TcSmem::resB : TcSmem::resA) + (item_n & 1) * 16384 + r * 32;
          const uint4 w0 = *reinterpret_cast<const uint4*>(rowp + ((0 ^ s1) << 4));
          const uint4 w1 = *reinterpret_cast<const uint4*>(rowp + ((1 ^ s1) << 4));
          const uint32_t v8[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
          tmem_st8(lane_addr + kResCol + t2 * 16, v8);
        }
      } else {
      const int sw = (r >> 1) & 3;
#pragma unroll
      for (int t2 = 0; t2 < 2; ++t2) {
        const uint8_t* rowp = smem + (t2 ? TcSmem::resB : TcSmem::resA) + (item_n & 1) * 16384 + r * 64;
        uint32_t v[16];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const uint4 w = *reinterpret_cast<const uint4*>(rowp + ((c ^ sw) << 4));
          v[4 * c] = w.x; v[4 * c + 1] = w.y; v[4 * c + 2] = w.z; v[4 * c + 3] = w.w;
        }
        tmem_st16(lane_addr + kResCol + t2 * 16, v);
      }
      }
      if (fold && MODE == MODE_DQ) {
        // statistics rows of the resident queries (32-byte rows, SWIZZLE_32B: the halves swap when bit 2 of r is set)
        const uint8_t* rowp = smem + TcSmem::aug_res + (item_n & 1) * 4096 + r * 32;
        const int s1 = (r >> 2) & 1;
        const uint4 w0 = *reinterpret_cast<const uint4*>(rowp + ((0 ^ s1) << 4));
        const uint4 w1 = *reinterpret_cast<const uint4*>(rowp + ((1 ^ s1) << 4));
        const uint32_t a8[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
        tmem_st8(lane_addr + kAugCol, a8);
      }
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(res_tmem);
    }

    // column statistics of a streamed tile, fetched one own-tile ahead
    float pre_f = 0.f;
    int pre_i = 0;
    auto prefetch = [&](int j) {
      if (j >= T) return;
      const int c = (tile_list[j] & 0x7fff) * kCols + (tid & 63);
      const bool ok = c < p.S_col;
      if (fold) {
        // only the labels are still needed, and only by tiles that straddle a label boundary
        if ((tile_list[j] & 0x8000) && tid < 64)
          pre_i = ok ? (masked ? p.col_id[static_cast<long long>(b) * p.S_col + c] : 0) : (MODE == MODE_DKV ? -0x7fffffff : 0x7fffffff);
        return;
      }
      if (MODE == MODE_DKV) {
        if (tid < 64) {
          pre_f = ok ? lse_g[c] : INFINITY;
          pre_i = masked ? (ok ? p.col_id[static_cast<long long>(b) * p.S_col + c] : -0x7fffffff) : 0;
        } else {
          pre_f = ok ? delta_g[c] : 0.f;
        }
      } else if (tid < 64) {
        pre_i = ok ? (masked ? p.col_id[static_cast<long long>(b) * p.S_col + c] : 0) : 0x7fffffff;
      }
    };
    const int j0 = (g + kNG - base % kNG) % kNG;      // first tile of this item that belongs to stage g
    prefetch(j0);
    long long w_full = 0, w_bar = 0, w_comp = 0;
    const bool prof_me = kFull && warp == 4 && lane == 0;
    for (int j = j0; j < T; j += kNG) {
      const int n = (base + j) / kNG;                  // use count of stage g across items
      const bool need_mask = (tile_list[j] & 0x8000) != 0;
      // column statistics: double buffered per warpgroup, so one barrier per tile (write -> barrier -> read; the
      // previous tile's readers use the other buffer)
      float* s_lse = stats_base + (n & 1) * 192;
      float* s_delta = s_lse + 64;
      int* s_id = reinterpret_cast<int*>(s_lse + 128);
#if FK_ATTN_EXP != 7
      if (fold) {
        // no per-tile staging: the statistics come out of the score MMAs.  Labels only for boundary tiles (two barriers:
        // the buffer is shared by consecutive masked tiles of this warpgroup)
        if (need_mask) {
          named_bar_sync(1 + g, 128);
          if (tid < 64) s_id[tid] = pre_i;
          named_bar_sync(1 + g, 128);
        }
      } else {
        if (MODE == MODE_DKV) {
          if (tid < 64) { s_lse[tid] = pre_f; s_id[tid] = pre_i; } else { s_delta[tid - 64] = pre_f; }
        } else if (tid < 64) {
          s_id[tid] = pre_i;
        }
        const long long tb0 = kFull ? clock64() : 0;
        named_bar_sync(1 + g, 128);
        if (kFull) w_bar += clock64() - tb0;
      }
      prefetch(j + kNG);
#endif
      wait_acc<kProf>(&sdp_full[g], n & 1, w_full);
      if (prof_me && j == j0) prof[3] = clock64() - t_start;
      if (kFull && trace && q4 == 0 && lane == 0 && j < 128) trace[4 * 128 + j] = clock64();
      const long long tc0 = kFull ? clock64() : 0;
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16) + g * 128;
      // kSub sub-chunks of 16 columns, software pipelined: the TMEM loads of sub-chunk i+1 are in flight while
      // sub-chunk i is computed and its bf16 pairs are stored over columns this thread has already consumed
      // (sub-chunk i occupies fp32 columns 16 i .. 16 i + 15, its pairs go to 8 i .. 8 i + 7)
      uint32_t sv[2][16], dv[2][16];
      if constexpr (fold) {
        // folded statistics: sv = S - lse / c and dv = dP - delta leave the tensor core.  P of sub-chunk i + 1 is formed
        // one step ahead, and the first one before dP is even waited for (its MMAs run behind the S MMAs).
        float pf[16];
        auto expo = [&](uint32_t (&s16)[16], int i) {
          if (need_mask) {
#pragma unroll
            for (int e = 0; e < 16; ++e) {
              const int cid = s_id[i * 16 + e];
              const bool hide = (MODE == MODE_DKV) ? (my_id > cid) : (cid > my_id);
              if (hide) s16[e] = 0xff800000u;
            }
          }
#pragma unroll
          for (int e = 0; e < 16; ++e) pf[e] = fast_ex2(__uint_as_float(s16[e]) * p.scale_log2);
        };
        tmem_ld16(taddr, sv[0]);
        tmem_wait1_16(sv[0]);
        tmem_ld16(taddr + 16, sv[1]);
        expo(sv[0], 0);
        mbar_wait(&dp_full[g], n & 1);
        tc_fence_after();
        tmem_ld16(taddr + 64, dv[0]);
#pragma unroll
        for (int i = 0; i < kSub; ++i) {
          const int cur = i & 1;
          if (i < kSub - 1) tmem_wait2_16(dv[cur], sv[cur ^ 1]); else tmem_wait1_16(dv[cur]);
          if (i < kSub - 1) tmem_ld16(taddr + 64 + (i + 1) * 16, dv[cur ^ 1]);
          if (i < kSub - 2) tmem_ld16(taddr + (i + 2) * 16, sv[cur]);
          uint32_t pw[8], dw[8];
#pragma unroll
          for (int e2 = 0; e2 < 8; ++e2) {
            const float s0 = pf[2 * e2] * __uint_as_float(dv[cur][2 * e2]);
            const float s1 = pf[2 * e2 + 1] * __uint_as_float(dv[cur][2 * e2 + 1]);
            if (MODE == MODE_DKV) pw[e2] = pack2(pf[2 * e2], pf[2 * e2 + 1]);
            dw[e2] = pack2(s0, s1);
          }
          if (MODE == MODE_DKV) tmem_st8(taddr + i * 8, pw);
          tmem_st8(taddr + 64 + i * 8, dw);
          if (i < kSub - 1) expo(sv[cur ^ 1], i + 1);
        }
      } else {
      tmem_ld16(taddr, sv[0]);
      tmem_ld16(taddr + 64, dv[0]);
#pragma unroll
      for (int i = 0; i < kSub; ++i) {
        const int cur = i & 1;
        tmem_wait2_16(sv[cur], dv[cur]);
        if (i < kSub - 1) {
          tmem_ld16(taddr + (i + 1) * 16, sv[cur ^ 1]);
          tmem_ld16(taddr + 64 + (i + 1) * 16, dv[cur ^ 1]);
        }
        if (need_mask) {          // tile-level (warp-uniform) branch: only tiles that straddle a label boundary
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            const int cid = s_id[i * 16 + e];
            const bool hide = (MODE == MODE_DKV) ? (my_id > cid) : (cid > my_id);
            if (hide) sv[cur][e] = 0xff800000u;              // -inf -> P = 0
          }
        }
        uint32_t pw[8], dw[8];
#pragma unroll
        for (int g8 = 0; g8 < 2; ++g8) {
          float lse8[8], dl8[8];
          if (MODE == MODE_DKV && !fold && FK_ATTN_EXP != 3 && FK_ATTN_EXP != 7) {
            const float4 l0 = *reinterpret_cast<const float4*>(s_lse + i * 16 + g8 * 8);
            const float4 l1 = *reinterpret_cast<const float4*>(s_lse + i * 16 + g8 * 8 + 4);
            const float4 d0 = *reinterpret_cast<const float4*>(s_delta + i * 16 + g8 * 8);
            const float4 d1 = *reinterpret_cast<const float4*>(s_delta + i * 16 + g8 * 8 + 4);
            lse8[0] = l0.x; lse8[1] = l0.y; lse8[2] = l0.z; lse8[3] = l0.w; lse8[4] = l1.x; lse8[5] = l1.y; lse8[6] = l1.z; lse8[7] = l1.w;
            dl8[0] = d0.x; dl8[1] = d0.y; dl8[2] = d0.z; dl8[3] = d0.w; dl8[4] = d1.x; dl8[5] = d1.y; dl8[6] = d1.z; dl8[7] = d1.w;
          } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) { lse8[e] = my_lse; dl8[e] = my_delta; }
          }
#pragma unroll
          for (int e2 = 0; e2 < 4; ++e2) {
            const int i0 = g8 * 8 + e2 * 2;
#if FK_ATTN_EXP == 4
            pw[g8 * 4 + e2] = sv[cur][i0] ^ sv[cur][i0 + 1];
            dw[g8 * 4 + e2] = dv[cur][i0] ^ dv[cur][i0 + 1];
            continue;
#endif
#if FK_ATTN_EXP == 6
            const float p0 = fast_ex2(__uint_as_float(sv[cur][i0]) * p.scale_log2);
            const float p1 = fast_ex2(__uint_as_float(sv[cur][i0 + 1]) * p.scale_log2);
#elif FK_ATTN_EXP == 7
            const float p0 = fast_ex2(__uint_as_float(sv[cur][i0]));
            const float p1 = fast_ex2(__uint_as_float(sv[cur][i0 + 1]));
#else
            // fold: sv = S - lse / c  ->  P = 2^(c sv); otherwise P = 2^(c S - lse)
            const float p0 = fast_ex2(fold ? __uint_as_float(sv[cur][i0]) * p.scale_log2
                                           : fmaf(__uint_as_float(sv[cur][i0]), p.scale_log2, -lse8[e2 * 2]));
            const float p1 = fast_ex2(fold ? __uint_as_float(sv[cur][i0 + 1]) * p.scale_log2
                                           : fmaf(__uint_as_float(sv[cur][i0 + 1]), p.scale_log2, -lse8[e2 * 2 + 1]));
#endif
#if FK_ATTN_EXP == 5 || FK_ATTN_EXP == 6 || FK_ATTN_EXP == 7
            const float s0 = p0 * __uint_as_float(dv[cur][i0]);           // what folding delta into the dP MMA would leave
            const float s1 = p1 * __uint_as_float(dv[cur][i0 + 1]);
#else
            // fold: dv = dP - delta already
            const float s0 = p0 * (fold ? __uint_as_float(dv[cur][i0]) : __uint_as_float(dv[cur][i0]) - dl8[e2 * 2]);
            const float s1 = p1 * (fold ? __uint_as_float(dv[cur][i0 + 1]) : __uint_as_float(dv[cur][i0 + 1]) - dl8[e2 * 2 + 1]);
#endif
            if (MODE == MODE_DKV) pw[g8 * 4 + e2] = pack2(p0, p1);
            dw[g8 * 4 + e2] = pack2(s0, s1);
          }
        }
        // bf16 pairs back into the stage (A operand of the accumulate MMAs, TS mode): 8 packed columns each
#if FK_ATTN_EXP == 2
        if (pw[0] == 0x12345678u && dw[0] == 0x9abcdef0u) tmem_st8(taddr + i * 8, pw);     // keep the math alive
#else
        if (MODE == MODE_DKV) tmem_st8(taddr + i * 8, pw);
        tmem_st8(taddr + 64 + i * 8, dw);
#endif
      }
      }   // staged statistics
#if FK_ATTN_EXP == 8
      // cost probe for a single-pass backward: the dQ partial of this tile ([64 queries x 32] fp32) reduced into global
      // memory with vector reds, 4 per thread (targets: the dV / dK output rows of the tile's queries -- results are WRONG)
      if (MODE == MODE_DKV) {
        const int qrow = (tile_list[j] & 0x7fff) * kCols + (tid & 63);
        if (qrow < p.S_col) {
          __nv_bfloat16* base16 = ((tid >> 6) ? p.out1 + b * p.o1_bs + static_cast<long long>(qrow) * p.o1_ts
                                              : p.out0 + b * p.o0_bs + static_cast<long long>(qrow) * p.o0_ts) + h * 32;
          float* dst = reinterpret_cast<float*>(base16);
#pragma unroll
          for (int v4 = 0; v4 < 4; ++v4)
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + v4 * 4), "f"(0.f), "f"(0.f), "f"(0.f), "f"(0.f) : "memory");
        }
      }
#endif
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_ready[g]);
      if (kFull && trace && q4 == 0 && lane == 0 && j < 128) trace[5 * 128 + j] = clock64();
      if (kFull) w_comp += clock64() - tc0;
    }
    if (prof_me) { prof[4] = w_full; prof[6] = w_bar; prof[7] = w_comp; prof[8] = clock64() - t_start; }
    // ---- epilogue: accumulators -> bf16 -> global ----
    mbar_wait(acc_full, item_n & 1);
    if (prof_me) prof[9] = clock64() - t_start;
    tc_fence_after();
    const bool writes = (MODE == MODE_DKV) ? (g < 2) : (g == 1);     // warp-uniform: wg0 -> acc0 (dV), wg1 -> acc1 (dK / dQ)
    if (writes) {
      const int which = (MODE == MODE_DKV) ? g : 1;
      uint32_t acc[HD];
      if (T > 0) {                                        // uniform: the whole warp executes the aligned TMEM load
        tmem_ld_wait<HD>(tmem_base + (static_cast<uint32_t>(q4 * 32) << 16) + kAccCol + which * 32, acc);
      } else {
#pragma unroll
        for (int i = 0; i < HD; ++i) acc[i] = 0u;
      }
      if (row_ok) {
        const float sc = (which == 1) ? p.scale : 1.f;
        __nv_bfloat16* dst = (which == 0 ? p.out0 + b * p.o0_bs + static_cast<long long>(row) * p.o0_ts
                                         : p.out1 + b * p.o1_bs + static_cast<long long>(row) * p.o1_ts) + h * HD;
        // gradient of a rotated operand (dK / dQ): rotate back (conjugate), as fk_rope(inverse = 1) would afterwards
        const float2* tb = nullptr;
        if (which == 1 && p.rope_table != nullptr) {
          int ps = p.rope_pos ? p.rope_pos[static_cast<long long>(b) * p.S_row + row] : row + p.rope_offset;
          ps = min(max(ps, 0), p.rope_len - 1);
          tb = p.rope_table + static_cast<long long>(ps) * (HD / 2);
        }
#pragma unroll
        for (int c4 = 0; c4 < HD / 8; ++c4) {
          uint32_t w[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float a0 = __uint_as_float(acc[c4 * 8 + e * 2]) * sc, a1 = __uint_as_float(acc[c4 * 8 + e * 2 + 1]) * sc;
            if (tb != nullptr) {
              const float2 cs = tb[c4 * 4 + e];
              const float r0 = a0 * cs.x + a1 * cs.y, r1 = a1 * cs.x - a0 * cs.y;
              a0 = r0; a1 = r1;
            }
            w[e] = pack2(a0, a1);
          }
          *reinterpret_cast<uint4*>(dst + c4 * 8) = make_uint4(w[0], w[1], w[2], w[3]);
        }
      }
    }
    if (prof_me) prof[10] = clock64() - t_start;
  }

  // ---- end of the item: every role has drained (accumulators read, all MMAs retired, tile list no longer needed) ----
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  base += T;
  if (kProf && threadIdx.x == 0) {
    prof[0] = clock64() - t_start;
    if (kProf == 2) {
      unsigned long long g_end;
      unsigned smid;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g_end));
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      prof[20] = static_cast<long long>(g_start); prof[21] = static_cast<long long>(g_end); prof[22] = smid; prof[2] = T;
    }
  }
  }   // item loop

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
  if (threadIdx.x == 0) {
    // the last CTA out re-arms the hand-out for the next launch
    if (atomicAdd(&p.items[1], 1u) == gridDim.x - 1) {
      p.items[0] = 0u;
      p.items[1] = 0u;
      __threadfence();
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Row statistics of the backward as tensor-core operands: delta[b,h,i] = sum_d dO O (as attn_delta_kernel) and the
// statistics row aug[b][h][i][16] (bf16) = (-lse / c split into three bf16 terms | -delta split into three | 0 ...): the
// score MMAs of the backward kernels take it as one more K step, so that S - lse / c and dP - delta leave the tensor core
// ready for P = 2^(c (S - lse / c)) and dS = P (dP - delta).  Three bf16 terms carry 24 mantissa bits.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void split3(float x, float& hi, float& mid, float& lo) {
  hi = __bfloat162float(__float2bfloat16_rn(x));
  const float r1 = x - hi;
  mid = __bfloat162float(__float2bfloat16_rn(r1));
  lo = __bfloat162float(__float2bfloat16_rn(r1 - mid));
}

template <int HD>      // 16, 32 or 64
__global__ void __launch_bounds__(256)
attn_aug_kernel(const __nv_bfloat16* __restrict__ o, const __nv_bfloat16* __restrict__ d_o, const float* __restrict__ lse,
                float* __restrict__ delta, __nv_bfloat16* __restrict__ aug, int B, int H, int S, long long o_bs, long long o_ts,
                long long do_bs, long long do_ts, float inv_scale_log2) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;   // (b, i, h)
  if (idx >= static_cast<long long>(B) * S * H) return;
  const int h = static_cast<int>(idx % H);
  const long long bi = idx / H;
  const int i = static_cast<int>(bi % S), b = static_cast<int>(bi / S);
  const uint4* op = reinterpret_cast<const uint4*>(o + b * o_bs + static_cast<long long>(i) * o_ts + h * HD);
  const uint4* dp = reinterpret_cast<const uint4*>(d_o + b * do_bs + static_cast<long long>(i) * do_ts + h * HD);
  float acc = 0.f;
#pragma unroll
  for (int c = 0; c < HD / 8; ++c) {
    const uint4 a = op[c], e = dp[c];
    const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, ew[4] = {e.x, e.y, e.z, e.w};
#pragma unroll
    for (int j = 0; j < 4; ++j)
      acc += __uint_as_float(aw[j] << 16) * __uint_as_float(ew[j] << 16) +
             __uint_as_float(aw[j] & 0xffff0000u) * __uint_as_float(ew[j] & 0xffff0000u);
  }
  const long long row = (static_cast<long long>(b) * H + h) * S + i;
  delta[row] = acc;
  // a row with no visible key has lse = +inf: a large finite value keeps the three-term split free of inf - inf
  const float l = lse[row];
  const float nl = (l < 3.0e38f) ? -l * inv_scale_log2 : -1.0e30f;
  float v[6];
  split3(nl, v[0], v[1], v[2]);
  split3(-acc, v[3], v[4], v[5]);
  uint4 w;
  w.x = pack2(v[0], v[1]); w.y = pack2(v[2], v[3]); w.z = pack2(v[4], v[5]); w.w = 0u;
  uint4* dst = reinterpret_cast<uint4*>(aug + row * 16);
  dst[0] = w;
  dst[1] = make_uint4(0u, 0u, 0u, 0u);
}

// ------------------------------------------------------------------------------------------------
// [B][S][H][32] (strided) -> [B][H][32][Sp] (zero padded beyond S): the K-major operand for contractions over tokens
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
attn_transpose_kernel(const __nv_bfloat16* __restrict__ x, long long bs, long long ts, int S, int H, int Sp,
                      __nv_bfloat16* __restrict__ xt) {
  __shared__ __nv_bfloat16 tile[64][34];
  const int t0 = blockIdx.x * 64, h = blockIdx.y, b = blockIdx.z;
  // load 64 tokens x 32 dims: 4 threads per token, 16 bytes each
  {
    const int tok = threadIdx.x >> 2, c = threadIdx.x & 3;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (t0 + tok < S) v = *reinterpret_cast<const uint4*>(x + b * bs + static_cast<long long>(t0 + tok) * ts + h * 32 + c * 8);
    const __nv_bfloat16* e = reinterpret_cast<const __nv_bfloat16*>(&v);
#pragma unroll
    for (int i = 0; i < 8; ++i) tile[tok][c * 8 + i] = e[i];
  }
  __syncthreads();
  // store 32 rows (d) x 64 tokens: 8 threads per row, 8 tokens (16 bytes) each
  {
    const int d = threadIdx.x >> 3, c = threadIdx.x & 7;
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 pr;
      pr.x = tile[c * 8 + 2 * i][d];
      pr.y = tile[c * 8 + 2 * i + 1][d];
      w[i] = *reinterpret_cast<uint32_t*>(&pr);
    }
    if (t0 + c * 8 < Sp)
      *reinterpret_cast<uint4*>(xt + ((static_cast<long long>(b) * H + h) * 32 + d) * Sp + t0 + c * 8) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// ================================================================================================
// Forward on tcgen05: persistent CTAs; work item = 256 queries of one (head, trial) (two warpgroups, 128 rows each, one
// thread per row), streaming 128-key tiles (K and V both as [keys][HD] tiles with the swizzle of their row width; the P V
// MMAs read V MN-major).  Per tile and warpgroup g:
//   S_g = Q_g K^T (HD / 16 MMAs, N = 128) -> TMEM;  thread: ONE sweep P = 2^(S c - m) against the stale running maximum m,
//   row sum, bf16 pairs -> operand buffer in TMEM;  O_g += P V (8 TS-mode MMAs, N = HD) accumulating in TMEM.
// The reference m is only re-established (row maximum pass, O / l rescaled) for the first visible tile of a row and when
// the row sum shows that it has gone stale -- O / l is independent of the m that was used.
// TMEM map: S_g at g*128 (128), P_g at 256 + g*64 (64), O_g at 384 + g*32 (32) at head_dim 16 / 32 and at 384 + g*64 (64)
// at head_dim 64, which fills the 512 columns.
// ================================================================================================
constexpr int kFwdTileK = 128;
constexpr int kFwdThreads = 384;
constexpr float kRescaleSlack = 8.f;
// an optimistic sweep whose row sum exceeds this has met scores above its stale reference (every 2^(s - m) <= 1 sums to
// at most 128): the tile is redone with its true maximum
constexpr float kStaleSum = 256.f;

// Shared memory of the forward at head width HD.  Tile rows are laid out 64 B apart at head_dim 16 and 32 (a 16-wide row
// fills the first 32 B of its slot) and 128 B apart at 64.  The K | V ring holds 128 KB: 8 stages at 16 / 32, 4 at 64.
template <int HD>
struct FwdSmem {
  static constexpr int row_bytes = HD == 64 ? 128 : 64;
  static constexpr int q_tile = 128 * row_bytes;        // one warpgroup's Q tile
  static constexpr int stage = 2 * kFwdTileK * row_bytes;    // K tile | V tile
  static constexpr int n_stages = 131072 / stage;
  static constexpr int q = 0;                           // 2 buffers (item n in buffer n & 1) x 2 groups x q_tile
  static constexpr int stream = 4 * q_tile;             // n_stages x stage
  static constexpr int ids = stream + n_stages * stage; // [2 wg][2 buffers][128] int
  static constexpr int tiles = ids + 2 * 2 * 128 * 4;
  static constexpr int bars = tiles + 2 * kMaxTiles * 2;     // two lists: the next item's is built while this one runs
  static constexpr int total = bars + 256;
};
static_assert(FwdSmem<64>::total <= 232448, "attn_fwd_tc_kernel<64>: shared memory");


struct FwdParams {
  const int *qid, *kid;
  const int *qmin, *qmax, *kmin, *kmax;                 // per-64-token tile label ranges
  __nv_bfloat16* out;
  float* lse;
  long long o_bs, o_ts;
  int B, H, Sq, Sk;
  float scale_log2;
  unsigned int* items;                                  // caller-owned hand-out counters (see TcParams::items)
};

// Key-axis split (kPart instantiations, fk_attn_forward_kv_tc): a work item is (256-query block, key chunk, head, trial);
// chunk c covers key tiles [c * chunk_tiles, (c + 1) * chunk_tiles).  Instead of O / l the item writes its unnormalised
// partial O (relative to its reference m) to part_o [B][H][n_chunks][Sq][HD] and (m, l) to part_ml [B][H][n_chunks][Sq][2]
// (log2 domain; m = -inf, l = 0 for a row that saw no key of the chunk); attn_kv_combine_kernel merges them.  A separate
// struct keeps the parameter block of the unsplit kernels as it was.
//
// band (split kernels only, fk_attn_forward_kv_band_tc): key j is visible to query i iff kid <= qid and qid - kid < band,
// the difference taken in 64 bits (every int32 is a valid label).  kNoBand exceeds every such difference: no band.
constexpr long long kNoBand = 1ll << 32;
struct FwdKvParams : FwdParams {
  float* part_o;
  float* part_ml;
  int n_chunks, chunk_tiles;
  long long band;
};
template <bool kPart>
using FwdArgs = std::conditional_t<kPart, FwdKvParams, FwdParams>;

__device__ __forceinline__ long long part_row(const FwdKvParams& p, int b, int h, int chunk, int row) {
  return ((static_cast<long long>(b) * p.H + h) * p.n_chunks + chunk) * p.Sq + row;
}
// N fp32 columns of a partial O row: O * alpha (the reference raise still owed to O after the last tile)
template <int N>
__device__ __forceinline__ void store_part_o(float* dst, const uint32_t (&ov)[N], float alpha) {
#pragma unroll
  for (int c4 = 0; c4 < N / 4; ++c4)
    *reinterpret_cast<float4*>(dst + c4 * 4) =
        make_float4(__uint_as_float(ov[c4 * 4]) * alpha, __uint_as_float(ov[c4 * 4 + 1]) * alpha,
                    __uint_as_float(ov[c4 * 4 + 2]) * alpha, __uint_as_float(ov[c4 * 4 + 3]) * alpha);
}
__device__ __forceinline__ void store_part_ml(float* dst, float m, float l) {
  *reinterpret_cast<float2*>(dst) = make_float2(l > 0.f ? m : -INFINITY, l);
}

// HD = 32: Q / K / V rows of 64 B (SWIZZLE_64B), two score K steps, P V MMAs N = 32.
// HD = 16: rows of 32 B (SWIZZLE_32B), one score K step, P V MMAs N = 16; O_g uses the first 16 of its 32 TMEM columns.
// HD = 64: rows of 128 B (SWIZZLE_128B), four score K steps, P V MMAs N = 64; O_g is rescaled and read out in two
// 32-column halves.
template <int HD, bool kPart = false>
__global__ void __launch_bounds__(kFwdThreads, 1)
attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k,
                   const __grid_constant__ CUtensorMap tm_v, const FwdArgs<kPart> p) {
  using Smem = FwdSmem<HD>;
  constexpr int kStages = Smem::n_stages;
  constexpr int kOCols = HD == 64 ? 64 : 32;        // TMEM columns of O_g
  constexpr int kOChunk = HD == 16 ? 16 : 32;       // O_g columns per TMEM load / store: HD / kOChunk chunks
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Smem::bars);
  uint64_t* q_full = bars;                  // [2]     Q tiles of item n in buffer n & 1
  uint64_t* list_ready = bars + 2;          // [1]     warp 2 has written the id and the tile list of the next item
  uint64_t* st_full = bars + 3;             // [kStages]
  uint64_t* st_empty = st_full + kStages;   // [kStages]  two arrivals: the P V MMAs of both warpgroups
  uint64_t* s_full = st_empty + kStages;    // [2]     S_g written by the tensor core
  uint64_t* s_free = s_full + 2;            // [2]     S_g read out (4 warps)
  uint64_t* p_ready = s_free + 2;           // [2]     P_g written (4 warps)
  uint64_t* p_free = p_ready + 2;           // [2]     P V MMAs of warpgroup g retired (O_g quiescent, P_g reusable)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(p_free + 2);
  int* n_tiles_slot = reinterpret_cast<int*>(p_free + 2) + 1;   // [2]
  int* item_slot = reinterpret_cast<int*>(p_free + 2) + 3;      // [2]
  uint16_t* tile_lists = reinterpret_cast<uint16_t*>(smem + Smem::tiles);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool masked = p.qid != nullptr;
  const int n_k_tiles = (p.Sk + kFwdTileK - 1) / kFwdTileK;
  const int nq64 = (p.Sq + 63) / 64, nk64 = (p.Sk + 63) / 64;
  const int n_q_tiles = (p.Sq + 255) / 256;
  int n_units = n_q_tiles;                        // work units per (head, trial): query blocks (x key chunks when split)
  if constexpr (kPart) n_units *= p.n_chunks;
  const int n_items = n_units * p.H * p.B;

  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tm_q); tma_prefetch_desc(&tm_k); tma_prefetch_desc(&tm_v); }
  if (warp == 1 && lane == 0) {
    mbar_init(&q_full[0], 1);
    mbar_init(&q_full[1], 1);
    mbar_init(list_ready, 1);
    for (int i = 0; i < kStages; ++i) { mbar_init(&st_full[i], 1); mbar_init(&st_empty[i], 2); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&s_free[i], 4);
      mbar_init(&p_ready[i], 4);
      mbar_init(&p_free[i], 1);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // key tiles visible to at least one of the item's rows; bits 14 / 15 = warpgroup 0 / 1 must compare labels
  auto build_list = [&](int it, int buf) {       // whole warp
    const int u_ = it % n_units, b_ = it / (n_units * p.H);
    const int qt_ = kPart ? u_ % n_q_tiles : u_;
    int t_lo = 0, t_hi = n_k_tiles;              // key tiles of the item (its chunk when split)
    if constexpr (kPart) {
      t_lo = (u_ / n_q_tiles) * p.chunk_tiles;
      t_hi = min(t_lo + p.chunk_tiles, n_k_tiles);
    }
    uint16_t* list = tile_lists + buf * kMaxTiles;
    // label ranges of the two warpgroups' rows (two 64-row entries each)
    int wq_lo[2] = {0, 0}, wq_hi[2] = {0, 0};
    if (masked) {
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        const int i0 = min(qt_ * 4 + g * 2, nq64 - 1), i1 = min(qt_ * 4 + g * 2 + 1, nq64 - 1);
        wq_lo[g] = min(p.qmin[b_ * nq64 + i0], p.qmin[b_ * nq64 + i1]);
        wq_hi[g] = max(p.qmax[b_ * nq64 + i0], p.qmax[b_ * nq64 + i1]);
      }
    }
    const int cta_hi = max(wq_hi[0], wq_hi[1]);
    int cnt = 0;
    for (int cb = t_lo; cb < t_hi; cb += 32) {
      const int t = cb + lane;
      bool vis = t < t_hi;
      int flags = 0;
      if (vis) {
        int kmn = 0, kmx = 0;
        if (masked) {
          const int i0 = min(t * 2, nk64 - 1), i1 = min(t * 2 + 1, nk64 - 1);
          kmn = min(p.kmin[b_ * nk64 + i0], p.kmin[b_ * nk64 + i1]);
          kmx = max(p.kmax[b_ * nk64 + i0], p.kmax[b_ * nk64 + i1]);
          vis = kmn <= cta_hi;
          // banded: skipped as well when every key lies band or more labels below every row
          if constexpr (kPart) vis = vis && static_cast<long long>(min(wq_lo[0], wq_lo[1])) - kmx < p.band;
        }
        const bool tail = t * kFwdTileK + kFwdTileK > p.Sk;
        if ((masked && kmx > wq_lo[0]) || tail) flags |= 0x4000;
        if ((masked && kmx > wq_lo[1]) || tail) flags |= 0x8000;
        if constexpr (kPart) {
          // banded: fully visible to a warpgroup only if no row of it lies band or more labels above a key
          if (masked && static_cast<long long>(wq_hi[0]) - kmn >= p.band) flags |= 0x4000;
          if (masked && static_cast<long long>(wq_hi[1]) - kmn >= p.band) flags |= 0x8000;
        }
      }
      const unsigned m = __ballot_sync(0xffffffffu, vis);
      if (vis) list[cnt + __popc(m & ((1u << lane) - 1u))] = static_cast<uint16_t>(t | flags);
      cnt += __popc(m);
    }
    if (lane == 0) n_tiles_slot[buf] = cnt;
  };

  // ---- persistent loop over work items (256-query block, head, trial), as in the backward kernel: dynamic hand-out,
  //      warp 2 prepares the next item's id and tile list one item ahead, the producer runs ahead into the next item,
  //      barrier parities run on counters that continue across items (`base` = key tiles of the earlier items) ----
  int base = 0;
  uint32_t item_n = 0;
  int pstage = 0;
  uint32_t pphase = 0;
  int pre_cnt = -1;
  if (warp == 2) {
    int first = 0;
    if (lane == 0) first = static_cast<int>(atomicAdd(&p.items[0], 1u));
    first = __shfl_sync(0xffffffffu, first, 0);
    if (lane == 0) item_slot[0] = first;
    if (first < n_items) build_list(first, 0);
  }
  __syncthreads();
  for (int item = item_slot[0]; item < n_items; item = item_slot[(item_n + 1) & 1], ++item_n) {
  const int u = item % n_units, h = (item / n_units) % p.H, b = item / (n_units * p.H);
  const int qt = kPart ? u % n_q_tiles : u;
  const int q0 = qt * 256;
  const uint16_t* tile_list = tile_lists + (item_n & 1) * kMaxTiles;
  const int T = n_tiles_slot[item_n & 1];

  if (warp == 2) {
    int nxt = 0;
    if (lane == 0) nxt = static_cast<int>(atomicAdd(&p.items[0], 1u));
    nxt = __shfl_sync(0xffffffffu, nxt, 0);
    if (lane == 0) item_slot[(item_n + 1) & 1] = nxt;
    if (nxt < n_items) build_list(nxt, (item_n + 1) & 1);
    __syncwarp();
    if (lane == 0) mbar_arrive(list_ready);
  }

  if (warp == 0) {
    // ================================ TMA producer ================================
    // (whole-warp loops with one elected issuing lane: see the backward kernel)
    {
      const int T_u = __shfl_sync(0xffffffffu, T, 0);
      auto load_q = [&](int h_, int q0_, int b_, int buf) {
        if (elect_one()) {
          mbar_expect_tx(&q_full[buf], 2 * 128 * HD * 2);
          tma_load_4d(smem + Smem::q + buf * 2 * Smem::q_tile, &tm_q, &q_full[buf], 0, h_, q0_, b_);
          tma_load_4d(smem + Smem::q + buf * 2 * Smem::q_tile + Smem::q_tile, &tm_q, &q_full[buf], 0, h_, q0_ + 128, b_);
        }
        __syncwarp();
      };
      auto load_tile = [&](int t, int h_, int b_) {
        uint8_t* st = smem + Smem::stream + pstage * Smem::stage;
        mbar_wait(&st_empty[pstage], pphase ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&st_full[pstage], 2 * kFwdTileK * HD * 2);
          tma_load_4d(st, &tm_k, &st_full[pstage], 0, h_, t * kFwdTileK, b_);
          tma_load_4d(st + Smem::stage / 2, &tm_v, &st_full[pstage], 0, h_, t * kFwdTileK, b_);   // V tile [128 keys][HD]
        }
        __syncwarp();
        if (++pstage == kStages) { pstage = 0; pphase ^= 1; }
      };
      if (pre_cnt < 0) { load_q(h, q0, b, item_n & 1); pre_cnt = 0; }
      for (int j = pre_cnt; j < T_u; ++j) load_tile(__shfl_sync(0xffffffffu, tile_list[j] & 0x3fff, 0), h, b);
      // run ahead into the next item while this one drains
      mbar_wait(list_ready, item_n & 1);
      const int nxt = __shfl_sync(0xffffffffu, item_slot[(item_n + 1) & 1], 0);
      pre_cnt = -1;
      if (nxt < n_items) {
        const int u2 = nxt % n_units, h2 = (nxt / n_units) % p.H, b2 = nxt / (n_units * p.H);
        const int qt2 = kPart ? u2 % n_q_tiles : u2;
        const uint16_t* list2 = tile_lists + ((item_n + 1) & 1) * kMaxTiles;
        const int T2 = __shfl_sync(0xffffffffu, n_tiles_slot[(item_n + 1) & 1], 0);
        load_q(h2, qt2 * 256, b2, (item_n + 1) & 1);
        pre_cnt = 0;
        const int ahead = T2 < kStages / 2 ? T2 : kStages / 2;
        for (int j = 0; j < ahead; ++j, ++pre_cnt) load_tile(__shfl_sync(0xffffffffu, list2[j] & 0x3fff, 0), h2, b2);
      }
    }
  } else if (warp == 1) {
    // ================================ score-MMA issuer ================================
    {
      constexpr uint32_t idesc = umma_idesc_bf16(128, kFwdTileK);
      const int T_u = __shfl_sync(0xffffffffu, T, 0);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint8_t* q_buf = smem + Smem::q + (item_n & 1) * 2 * Smem::q_tile;
      const uint64_t dQ[2] = {umma_desc_rows<HD>(smem_u32(q_buf)), umma_desc_rows<HD>(smem_u32(q_buf + Smem::q_tile))};
      const uint32_t stream = smem_u32(smem + Smem::stream);
      mbar_wait(&q_full[item_n & 1], (item_n >> 1) & 1);
      tc_fence_after();
      for (int j = 0; j < T_u; ++j) {
        const int gj = base + j;                     // key-tile counter across items
        const int stage = gj % kStages;
        mbar_wait(&st_full[stage], (gj / kStages) & 1);
        const uint64_t dK = umma_desc_rows<HD>(stream + stage * Smem::stage);
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          mbar_wait(&s_free[g], (gj & 1) ^ 1);
          tc_fence_after();
          if (elect_one()) {
            // a K step of 16 dims = 32 B = +2 in the descriptors' (address >> 4) field
            umma_bf16(tmem_u + g * 128, dQ[g], dK, idesc, 0u);
#pragma unroll
            for (int kk = 1; kk < HD / 16; ++kk) umma_bf16(tmem_u + g * 128, dQ[g] + 2 * kk, dK + 2 * kk, idesc, 1u);
            umma_commit(&s_full[g]);
          }
          __syncwarp();
        }
      }
    }
  } else if (warp == 3) {
    // ================================ P V MMA issuer ================================
    {
      constexpr uint32_t idesc = umma_idesc_bf16(128, HD);
      const int T_u = __shfl_sync(0xffffffffu, T, 0);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t stream = smem_u32(smem + Smem::stream);
      for (int j = 0; j < T_u; ++j) {
        const int gj = base + j;
        const int stage = gj % kStages;
        // V tile [128 keys][32 dims] (64-byte rows, SWIZZLE_64B) read MN-major: N = dims contiguous, K = keys, a K step of
        // 16 keys = 1024 B -- no transposed copy of V exists (head_dim 16: 32-byte rows, SWIZZLE_32B, K step 512 B;
        // head_dim 64: 128-byte rows, SWIZZLE_128B, N = 64 dims in one swizzle atom, K step 2048 B)
        const uint64_t dV = umma_desc_rows<HD>(stream + stage * Smem::stage + Smem::stage / 2);
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          mbar_wait(&p_ready[g], gj & 1);
          tc_fence_after();
          const uint32_t pa = tmem_u + 256 + g * 64, oa = tmem_u + 384 + g * kOCols;
          if (elect_one()) {
#pragma unroll
            for (int kk = 0; kk < 8; ++kk)
              umma_bf16_ts(oa, pa + kk * 8, dV + 2 * HD * kk, idesc | (1u << 16), (j > 0 || kk > 0) ? 1u : 0u);
            umma_commit(&p_free[g]);
            umma_commit(&st_empty[stage]);
          }
          __syncwarp();
        }
      }
    }
  } else if (warp >= 4) {
    // ================================ softmax warpgroups ================================
    const int g = (warp - 4) >> 2;
    const int q4 = warp & 3;
    const int r = q4 * 32 + lane;
    const int tid = (warp - 4 - g * 4) * 32 + lane;
    const int row = q0 + g * 128 + r;
    const bool row_ok = row < p.Sq;
    const int my_id = masked ? (row_ok ? p.qid[static_cast<long long>(b) * p.Sq + row] : -0x7fffffff) : 0;
    // banded: the lowest visible key label, my_id - band + 1 clamped to INT_MIN (qid - kid < band <=> kid >= my_lo)
    [[maybe_unused]] int my_lo = INT_MIN;
    if constexpr (kPart) my_lo = static_cast<int>(max(static_cast<long long>(my_id) - p.band + 1, static_cast<long long>(INT_MIN)));
    int* ids_base = reinterpret_cast<int*>(smem + Smem::ids) + g * 256;
    const uint32_t lane_base = static_cast<uint32_t>(q4 * 32) << 16;
    const uint32_t s_addr = tmem_base + lane_base + g * 128;
    const uint32_t p_addr = tmem_base + lane_base + 256 + g * 64;
    const uint32_t o_addr = tmem_base + lane_base + 384 + g * kOCols;
    float m_run = -INFINITY, l_run = 0.f, alpha_pend = 1.f;
    int pre_i = 0;
    // key labels of a tile are only fetched and staged for tiles that need the per-element compare (warp-group uniform
    // flag from the tile list): fully visible tiles -- every tile of the block-causal mask when the electrode count is a
    // multiple of the tile sizes -- cost neither the global load nor the warpgroup barrier
    const uint16_t my_flag = (g == 0) ? 0x4000 : 0x8000;
    auto prefetch = [&](int j) {
      if (j >= T || !(tile_list[j] & my_flag)) return;
      const int c = (tile_list[j] & 0x3fff) * kFwdTileK + tid;
      pre_i = (masked && c < p.Sk) ? p.kid[static_cast<long long>(b) * p.Sk + c] : 0;   // (c >= Sk: masked by position)
    };
    prefetch(0);
    for (int j = 0; j < T; ++j) {
      const int gj = base + j;                       // key-tile counter across items (barrier parities)
      const bool need_mask = (tile_list[j] & my_flag) != 0;
      // keys of this tile that exist: < kFwdTileK only in the ragged tail, which always carries the compare flag.  The
      // columns past Sk are masked by position, not by a sentinel label: every int32 is a valid query label.
      const int n_valid = p.Sk - (tile_list[j] & 0x3fff) * kFwdTileK;
      int* s_id = ids_base;
      if (need_mask) {
        named_bar_sync(1 + g, 128);                  // the previous masked tile's readers are done with the buffer
        s_id[tid] = pre_i;
        named_bar_sync(1 + g, 128);
      }
      prefetch(j + 1);
      mbar_wait(&s_full[g], gj & 1);
      tc_fence_after();
      uint32_t sv[2][32];
      auto mask_chunk = [&](uint32_t (&v)[32], int c) {
        if (need_mask) {
          if constexpr (kPart) {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const int kid = s_id[c * 32 + i];
              if (kid > my_id || kid < my_lo) v[i] = 0xff800000u;
            }
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (s_id[c * 32 + i] > my_id) v[i] = 0xff800000u;
          }
          if (n_valid < kFwdTileK) {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (c * 32 + i >= n_valid) v[i] = 0xff800000u;
          }
        }
      };
      // O_g *= alpha_pend (rare, warp-uniform): only legal once the previous tile's P V MMAs have retired
      auto apply_pending = [&]() {
        if (__any_sync(0xffffffffu, alpha_pend != 1.f)) {
#pragma unroll
          for (int hf = 0; hf < HD / kOChunk; ++hf) {
            uint32_t ov[kOChunk];
            tmem_ld_wait<kOChunk>(o_addr + hf * 32, ov);
#pragma unroll
            for (int i = 0; i < kOChunk; ++i) ov[i] = __float_as_uint(__uint_as_float(ov[i]) * alpha_pend);
            tmem_st_cols<kOChunk>(o_addr + hf * 32, ov);
          }
          alpha_pend = 1.f;
        }
      };
      // one sweep over the 128 scores of this row: P = 2^(S c - m_use) -> bf16 pairs into the operand buffer and the row
      // sum; TMEM loads double buffered.  The optimistic sweep does not even track the row maximum (one instruction per
      // score less): a reference that has gone stale shows up in the row sum instead -- sum > kStaleSum means some
      // 2^(s - m) > 2, +inf means overflow -- and only then is the tile redone with its true maximum.
      float rs = 0.f;
      bool released = false, redo = false;
      auto release_scores = [&]() {                      // S_g fully consumed: the next tile's scores may land
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&s_free[g]);
        released = true;
      };
      auto exp_sweep = [&](float m_use, bool optimistic) {
        rs = 0.f;
        if (optimistic) tmem_ld32(s_addr, sv[0]);        // (otherwise chunk 0 was requested by the maximum pass)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int cur = c & 1;
          tmem_wait1_32(sv[cur]);
          if (c < 3) tmem_ld32(s_addr + (c + 1) * 32, sv[cur ^ 1]);
          mask_chunk(sv[cur], c);
          if (c == 3 && !optimistic) release_scores();   // every score is in registers and no redo can follow
          uint32_t pw[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const float p0 = fast_ex2(fmaf(__uint_as_float(sv[cur][2 * i]), p.scale_log2, -m_use));
            const float p1 = fast_ex2(fmaf(__uint_as_float(sv[cur][2 * i + 1]), p.scale_log2, -m_use));
            rs += p0 + p1;
            pw[i] = pack2(p0, p1);
          }
          if (c == 0 && optimistic) {
            // P_g is reusable and O_g quiescent once the previous tile's P V MMAs have retired
            mbar_wait(&p_free[g], (gj & 1) ^ 1);
            tc_fence_after();
            apply_pending();
          }
          tmem_st16(p_addr + c * 16, pw);
        }
      };
      const bool two_pass = __any_sync(0xffffffffu, m_run == -INFINITY);
      if (!two_pass) {
        // ---- optimistic single sweep against the stale running maximum (softmax is shift invariant; the reference
        //      only has to keep 2^(s - m) inside the fp32 / bf16 exponent range) ----
        exp_sweep(m_run, true);
        redo = __any_sync(0xffffffffu, !(rs <= kStaleSum));        // (also true for +inf / NaN)
        if (!redo) {
          release_scores();
          l_run += rs;
        }
      }
      if (two_pass || redo) {
        // ---- first visible tile of a row (no reference yet) or a jump the stale reference cannot absorb:
        //      row maximum first, then the sweep ----
        float mx1 = -INFINITY;
        tmem_ld32(s_addr, sv[0]);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int cur = c & 1;
          tmem_wait1_32(sv[cur]);
          tmem_ld32(s_addr + ((c + 1) & 3) * 32, sv[cur ^ 1]);      // c == 3: chunk 0 again, for the sweep
          mask_chunk(sv[cur], c);
#pragma unroll
          for (int i = 0; i < 32; i += 2) mx1 = fmaxf(mx1, fmaxf(__uint_as_float(sv[cur][i]), __uint_as_float(sv[cur][i + 1])));
        }
        const float m_tile = mx1 * p.scale_log2;
        // (after a stale-reference redo every increase is taken, otherwise the next tile would trip the same check)
        const bool raise = m_tile > m_run + (redo ? 0.f : kRescaleSlack) || m_run == -INFINITY;
        const float m_new = raise ? fmaxf(m_run, m_tile) : m_run;
        const float m_use = (m_new == -INFINITY) ? 0.f : m_new;
        const float alpha = (raise && m_run != -INFINITY) ? fast_ex2(m_run - m_use) : 1.f;
        if (two_pass) {                                  // (a redone optimistic sweep already waited for p_free)
          mbar_wait(&p_free[g], (gj & 1) ^ 1);
          tc_fence_after();
          apply_pending();
        }
        l_run *= alpha;
        alpha_pend = alpha;
        apply_pending();                                 // O_g *= alpha before this tile accumulates
        m_run = m_new;
        redo = false;
        exp_sweep(m_use, false);
        l_run += rs;
      }
      if (!released) release_scores();
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_ready[g]);
    }
    // ---- epilogue: O / l -> bf16, LSE ----
    if (T > 0) {
      mbar_wait(&p_free[g], ((base + T) & 1) ^ 1);     // the last P V MMAs have retired
      tc_fence_after();
    }
    // 1 / l (a reference raise after the last tile is still owed to O) and the output row.  At head_dim 64, where O is
    // read out in two chunks, they are formed before the first one: formed between the chunks they cost 8 more bytes of
    // spill loads (ptxas -v).
    float inv = 0.f;
    __nv_bfloat16* dst = nullptr;
    auto out_row = [=, &inv, &dst]() {
      inv = (l_run > 0.f) ? alpha_pend / l_run : 0.f;
      dst = row_ok ? p.out + b * p.o_bs + static_cast<long long>(row) * p.o_ts + h * HD : nullptr;
    };
    if constexpr (HD == 64) out_row();
#pragma unroll
    for (int hf = 0; hf < HD / kOChunk; ++hf) {
      uint32_t ov[kOChunk];
      if (T > 0) {
        tmem_ld_wait<kOChunk>(o_addr + hf * 32, ov);
      } else {
#pragma unroll
        for (int i = 0; i < kOChunk; ++i) ov[i] = 0u;
      }
      if constexpr (kPart) {
        if (row_ok) store_part_o<kOChunk>(p.part_o + part_row(p, b, h, u / n_q_tiles, row) * HD + hf * 32, ov, alpha_pend);
      } else if (row_ok) {
        if constexpr (HD != 64) out_row();
#pragma unroll
        for (int c4 = 0; c4 < kOChunk / 8; ++c4) {
          uint32_t w[4];
#pragma unroll
          for (int e = 0; e < 4; ++e)
            w[e] = pack2(__uint_as_float(ov[c4 * 8 + e * 2]) * inv, __uint_as_float(ov[c4 * 8 + e * 2 + 1]) * inv);
          *reinterpret_cast<uint4*>(dst + hf * 32 + c4 * 8) = make_uint4(w[0], w[1], w[2], w[3]);
        }
      }
    }
    if constexpr (kPart) {
      if (row_ok) store_part_ml(p.part_ml + part_row(p, b, h, u / n_q_tiles, row) * 2, m_run, l_run);
    } else if (row_ok && p.lse != nullptr) {
      p.lse[(static_cast<long long>(b) * p.H + h) * p.Sq + row] = (l_run > 0.f) ? m_run + log2f(l_run) : INFINITY;
    }
  }

  // ---- end of the item: every role has drained (O read out, all MMAs retired, tile list no longer needed) ----
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  base += T;
  }   // item loop

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
  if (threadIdx.x == 0) {
    // the last CTA out re-arms the hand-out for the next launch
    if (atomicAdd(&p.items[1], 1u) == gridDim.x - 1) {
      p.items[0] = 0u;
      p.items[1] = 0u;
      __threadfence();
    }
  }
}

// ================================================================================================
// Backward at head_dim 64 (the forward at 64 is attn_fwd_tc_kernel<64>).  Same work split, label-mask / tile-skip rules,
// persistent hand-out and softmax as the head_dim-32 backward above; [tokens][64] bf16 rows are 128 B, so every tile is
// TMA-loaded with the 128-byte swizzle.
//
// attn_bwd_tc64_kernel: three score stages (3 x 128 columns) + dV 64 + dK / dQ 64 fill the 512 TMEM columns, so
// the resident tiles cannot sit in TMEM as at head_dim 32: the score MMAs read both operands from shared memory (SS mode,
// 4 K steps of 16 + the folded statistics step).  P / dS are still written in place over the consumed score columns and
// read by the accumulate MMAs from TMEM (TS mode, N = 64, B operand MN-major straight from the streamed tile).  One path
// only: statistics folded (fk_attn_aug), MN-major accumulate operands.
// ================================================================================================
constexpr int kNST64 = 6;                     // streamed stages: tile A 8 KB | tile B 8 KB | statistics rows 2 KB (DKV)
constexpr int kStage64 = 18432;
constexpr int kAcc64 = 128 * kNG;             // 384: dV (64 columns), 448: dK / dQ (64 columns)

struct TcSmem64 {
  static constexpr int resA = 0;                                  // 2 buffers x [128][64] bf16 (16 KB each)
  static constexpr int resB = 32768;
  static constexpr int stream = 65536;
  static constexpr int ids = stream + kNST64 * kStage64;         // [kNG wg][2 buffers][64] int column labels
  static constexpr int tiles = ids + kNG * 2 * 64 * 4;           // two uint16 visible-tile lists
  static constexpr int ones = (tiles + 2 * kMaxTiles * 2 + 1023) / 1024 * 1024;   // [2][128][16] bf16, SWIZZLE_32B
  static constexpr int aug_res = ones + 8192;                    // DQ: 2 buffers x [128][16] statistics rows
  static constexpr int bars = aug_res + 8192;
  static constexpr int total = bars + 512;
};
static_assert(TcSmem64::total <= 232448, "attn_bwd_tc64_kernel: shared memory");

template <int MODE>
__global__ void __launch_bounds__(kTcThreads, 1)
attn_bwd_tc64_kernel(const __grid_constant__ CUtensorMap tm_resA, const __grid_constant__ CUtensorMap tm_resB,
                     const __grid_constant__ CUtensorMap tm_stA, const __grid_constant__ CUtensorMap tm_stB,
                     const __grid_constant__ CUtensorMap tm_aug, const TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + TcSmem64::bars);
  uint64_t* res_full = bars;               // [2]      resident tiles (+ DQ statistics rows) of item n in buffer n & 1
  uint64_t* list_ready = bars + 2;         // [1]
  uint64_t* st_full = bars + 3;            // [kNST64]
  uint64_t* st_empty = st_full + kNST64;   // [kNST64]
  uint64_t* sdp_full = st_empty + kNST64;  // [kNG]    S' of stage g written
  uint64_t* dp_full = sdp_full + kNG;      // [kNG]    dP' of stage g written
  uint64_t* stage_free = dp_full + kNG;    // [kNG]    the accumulate MMAs reading stage g have retired
  uint64_t* p_ready = stage_free + kNG;    // [kNG]    P / dS written in place into stage g (4 warps arrive)
  uint64_t* acc_full = p_ready + kNG;      // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);
  int* n_tiles_slot = reinterpret_cast<int*>(acc_full + 1) + 1;   // [2]
  int* item_slot = reinterpret_cast<int*>(acc_full + 1) + 3;      // [2]
  uint16_t* tile_lists = reinterpret_cast<uint16_t*>(smem + TcSmem64::tiles);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool masked = p.row_id != nullptr;
  const int n_col_tiles = (p.S_col + kCols - 1) / kCols;
  const int n_row_tiles64 = (p.S_row + 63) / 64;
  const int n_row_tiles = (p.S_row + kRows - 1) / kRows;
  const int n_items = n_row_tiles * p.H * p.B;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_resA); tma_prefetch_desc(&tm_resB); tma_prefetch_desc(&tm_stA);
    tma_prefetch_desc(&tm_stB); tma_prefetch_desc(&tm_aug);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(&res_full[0], 1);
    mbar_init(&res_full[1], 1);
    mbar_init(list_ready, 1);
    for (int i = 0; i < kNST64; ++i) { mbar_init(&st_full[i], 1); mbar_init(&st_empty[i], 1); }
    for (int i = 0; i < kNG; ++i) {
      mbar_init(&sdp_full[i], 1);
      mbar_init(&dp_full[i], 1);
      mbar_init(&stage_free[i], 1);
      mbar_init(&p_ready[i], 4);
    }
    mbar_init(acc_full, 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  if (warp >= 4) {
    // constant operand tiles of the statistics K step (as in attn_bwd_tc_kernel): row r = 16 bf16, ones in columns 0-2
    // (picks -lse / c) resp. 3-5 (picks -delta), SWIZZLE_32B pattern.  DKV: A operand (128 key rows); DQ: B operand
    // (first 64 rows)
    for (int i = threadIdx.x - 128; i < 2 * 128 * 2; i += kTcThreads - 128) {
      const int tile = i >> 8, r = (i >> 1) & 127, pc = i & 1;
      const int c = pc ^ ((r >> 2) & 1);
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (c == 0) v = tile == 0 ? make_uint4(0x3F803F80u, 0x00003F80u, 0u, 0u) : make_uint4(0u, 0x3F800000u, 0x3F803F80u, 0u);
      *reinterpret_cast<uint4*>(smem + TcSmem64::ones + tile * 4096 + r * 32 + pc * 16) = v;
    }
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  int base = 0;
  uint32_t item_n = 0;
  int pstage = 0;
  uint32_t pphase = 0;
  int pre_cnt = -1;
  auto build_list = [&](int it, int buf) {       // whole warp (see attn_bwd_tc_kernel)
    const int rt_ = it % n_row_tiles, b_ = it / (n_row_tiles * p.H);
    uint16_t* list = tile_lists + buf * kMaxTiles;
    int row_lo = 0, row_hi = 0;
    if (masked) {
      const int i0 = rt_ * 2, i1 = min(rt_ * 2 + 1, n_row_tiles64 - 1);
      row_lo = min(p.row_min[b_ * n_row_tiles64 + i0], p.row_min[b_ * n_row_tiles64 + i1]);
      row_hi = max(p.row_max[b_ * n_row_tiles64 + i0], p.row_max[b_ * n_row_tiles64 + i1]);
    }
    int cnt = 0;
    for (int cb = 0; cb < n_col_tiles; cb += 32) {
      const int t = cb + lane;
      bool vis = t < n_col_tiles, nm = false;
      if (vis) {
        int cmin = 0, cmax = 0;
        if (masked) { cmin = p.col_min[b_ * n_col_tiles + t]; cmax = p.col_max[b_ * n_col_tiles + t]; }
        if (MODE == MODE_DKV) {
          vis = !masked || cmax >= row_lo;
          nm = masked && (row_hi > cmin);
        } else {
          vis = !masked || cmin <= row_hi;
          nm = (masked && (cmax > row_lo)) || (t * kCols + kCols > p.S_col);
        }
      }
      const unsigned m = __ballot_sync(0xffffffffu, vis);
      if (vis) list[cnt + __popc(m & ((1u << lane) - 1u))] = static_cast<uint16_t>(t | (nm ? 0x8000 : 0));
      cnt += __popc(m);
    }
    if (lane == 0) n_tiles_slot[buf] = cnt;
  };
  if (warp == 2) {
    int first = 0;
    if (lane == 0) first = static_cast<int>(atomicAdd(&p.items[0], 1u));
    first = __shfl_sync(0xffffffffu, first, 0);
    if (lane == 0) item_slot[0] = first;
    if (first < n_items) build_list(first, 0);
  }
  __syncthreads();
  for (int item = item_slot[0]; item < n_items; item = item_slot[(item_n + 1) & 1], ++item_n) {
  const int rt = item % n_row_tiles, h = (item / n_row_tiles) % p.H, b = item / (n_row_tiles * p.H);
  const int r0 = rt * kRows;
  const uint16_t* tile_list = tile_lists + (item_n & 1) * kMaxTiles;
  const int T = n_tiles_slot[item_n & 1];

  if (warp == 2) {
    int nxt = 0;
    if (lane == 0) nxt = static_cast<int>(atomicAdd(&p.items[0], 1u));
    nxt = __shfl_sync(0xffffffffu, nxt, 0);
    if (lane == 0) item_slot[(item_n + 1) & 1] = nxt;
    if (nxt < n_items) build_list(nxt, (item_n + 1) & 1);
    __syncwarp();
    if (lane == 0) mbar_arrive(list_ready);
  }

  if (warp == 0) {
    // ================================ TMA producer ================================
    const int T_u = __shfl_sync(0xffffffffu, T, 0);
    auto load_resident = [&](int h_, int r0_, int b_, int buf) {
      if (elect_one()) {
        mbar_expect_tx(&res_full[buf], MODE == MODE_DQ ? 32768u + 4096u : 32768u);
        tma_load_4d(smem + TcSmem64::resA + buf * 16384, &tm_resA, &res_full[buf], 0, h_, r0_, b_);
        tma_load_4d(smem + TcSmem64::resB + buf * 16384, &tm_resB, &res_full[buf], 0, h_, r0_, b_);
        if (MODE == MODE_DQ) tma_load_4d(smem + TcSmem64::aug_res + buf * 4096, &tm_aug, &res_full[buf], 0, r0_, h_, b_);
      }
      __syncwarp();
    };
    auto load_tile = [&](int t, int h_, int b_) {
      uint8_t* st = smem + TcSmem64::stream + pstage * kStage64;
      mbar_wait(&st_empty[pstage], pphase ^ 1);
      if (elect_one()) {
        mbar_expect_tx(&st_full[pstage], MODE == MODE_DKV ? 16384u + 2048u : 16384u);
        tma_load_4d(st, &tm_stA, &st_full[pstage], 0, h_, t * kCols, b_);
        tma_load_4d(st + 8192, &tm_stB, &st_full[pstage], 0, h_, t * kCols, b_);
        if (MODE == MODE_DKV) tma_load_4d(st + 16384, &tm_aug, &st_full[pstage], 0, t * kCols, h_, b_);   // the queries' statistics rows
      }
      __syncwarp();
      if (++pstage == kNST64) { pstage = 0; pphase ^= 1; }
    };
    if (pre_cnt < 0) { load_resident(h, r0, b, item_n & 1); pre_cnt = 0; }
    for (int j = pre_cnt; j < T_u; ++j) load_tile(__shfl_sync(0xffffffffu, tile_list[j] & 0x7fff, 0), h, b);
    mbar_wait(list_ready, item_n & 1);
    const int nxt = __shfl_sync(0xffffffffu, item_slot[(item_n + 1) & 1], 0);
    pre_cnt = -1;
    if (nxt < n_items) {
      const int rt2 = nxt % n_row_tiles, h2 = (nxt / n_row_tiles) % p.H, b2 = nxt / (n_row_tiles * p.H);
      const uint16_t* list2 = tile_lists + ((item_n + 1) & 1) * kMaxTiles;
      const int T2 = __shfl_sync(0xffffffffu, n_tiles_slot[(item_n + 1) & 1], 0);
      load_resident(h2, rt2 * kRows, b2, (item_n + 1) & 1);
      pre_cnt = 0;
      const int ahead = T2 < kNST64 / 2 ? T2 : kNST64 / 2;
      for (int j = 0; j < ahead; ++j, ++pre_cnt) load_tile(__shfl_sync(0xffffffffu, list2[j] & 0x7fff, 0), h2, b2);
    }
  } else if (warp == 1) {
    // ================================ score-MMA issuer (SS mode) ================================
    constexpr uint32_t idesc_score = umma_idesc_bf16(kRows, kCols);
    const int T_u = __shfl_sync(0xffffffffu, T, 0);
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t stream = smem_u32(smem + TcSmem64::stream);
    const uint32_t buf = item_n & 1;
    const uint64_t dRA = umma_desc_sw128(smem_u32(smem + TcSmem64::resA) + buf * 16384);
    const uint64_t dRB = umma_desc_sw128(smem_u32(smem + TcSmem64::resB) + buf * 16384);
    const uint64_t dOnesS = umma_desc_sw32(smem_u32(smem + TcSmem64::ones));
    const uint64_t dOnesD = umma_desc_sw32(smem_u32(smem + TcSmem64::ones + 4096));
    const uint64_t dAugRes = umma_desc_sw32(smem_u32(smem + TcSmem64::aug_res) + buf * 4096);
    mbar_wait(&res_full[buf], (item_n >> 1) & 1);
    for (int js = 0; js < T_u; ++js) {
      const int gt = base + js;
      const int stage = gt % kNST64, g = gt % kNG, n = gt / kNG;
      uint64_t dS = umma_desc_sw128(stream + stage * kStage64), dD = umma_desc_sw128(stream + stage * kStage64 + 8192);
      uint32_t d_s = tmem_u + g * 128, d_dp = tmem_u + g * 128 + 64;
      // statistics K step: DKV  A = ones (keys), B = the tile's query statistics rows;  DQ  A = resident statistics rows,
      // B = ones (keys)
      uint64_t fA_s = dOnesS, fA_d = dOnesD, fB_s = umma_desc_sw32(stream + stage * kStage64 + 16384), fB_d = fB_s;
      if (MODE == MODE_DQ) { fA_s = fA_d = dAugRes; fB_s = dOnesS; fB_d = dOnesD; }
      asm volatile("" : "+l"(dS), "+l"(dD), "+r"(d_s), "+r"(d_dp), "+l"(fA_s), "+l"(fA_d), "+l"(fB_s), "+l"(fB_d));
      mbar_wait(&st_full[stage], (gt / kNST64) & 1);
      mbar_wait(&stage_free[g], (n & 1) ^ 1);
      tc_fence_after();
      if (elect_one()) {
        // a K step of 16 bf16 = 32 bytes = +2 in the descriptor's (address >> 4) field
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) umma_bf16(d_s, dRA + 2 * kk, dS + 2 * kk, idesc_score, kk > 0 ? 1u : 0u);
        umma_bf16(d_s, fA_s, fB_s, idesc_score, 1u);
        umma_commit(&sdp_full[g]);                     // S' complete: the warpgroup starts on the exponentials
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) umma_bf16(d_dp, dRB + 2 * kk, dD + 2 * kk, idesc_score, kk > 0 ? 1u : 0u);
        umma_bf16(d_dp, fA_d, fB_d, idesc_score, 1u);
        umma_commit(&dp_full[g]);
      }
      __syncwarp();
    }
  } else if (warp == 3) {
    // ================================ accumulate-MMA issuer (TS mode) ================================
    // B operand straight from the streamed stage: tile [64 tokens][64 dims], 128-byte rows, SWIZZLE_128B = the canonical
    // MN-major layout (N = 64 dims in one swizzle atom, 8-token groups 1024 B apart); a K step of 16 tokens = 2048 B.
    // DKV: dV += P^T dO (tile B), dK += dS^T Q (tile A).  DQ: dQ += dS K (tile A).
    constexpr uint32_t idesc_acc = umma_idesc_bf16(kRows, 64) | (1u << 16);
    const int T_u = __shfl_sync(0xffffffffu, T, 0);
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t stream = smem_u32(smem + TcSmem64::stream);
    for (int ia = 0; ia < T_u; ++ia) {
      const int gt = base + ia;
      const int stage = gt % kNST64, g = gt % kNG, n = gt / kNG;
      uint32_t ta = tmem_u + g * 128;                   // P pairs at +0..31, dS pairs at +64..95 (written in place)
      uint64_t dMA = umma_desc_sw128(stream + stage * kStage64 + 8192), dMB = umma_desc_sw128(stream + stage * kStage64);
      asm volatile("" : "+l"(dMA), "+l"(dMB), "+r"(ta));
      mbar_wait(&p_ready[g], n & 1);
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          if (MODE == MODE_DKV) umma_bf16_ts(tmem_u + kAcc64, ta + kk * 8, dMA + 128 * kk, idesc_acc, (ia > 0 || kk > 0) ? 1u : 0u);
          umma_bf16_ts(tmem_u + kAcc64 + 64, ta + 64 + kk * 8, dMB + 128 * kk, idesc_acc, (ia > 0 || kk > 0) ? 1u : 0u);
        }
        umma_commit(&stage_free[g]);
        umma_commit(&st_empty[stage]);
      }
      __syncwarp();
    }
    if (elect_one()) umma_commit(acc_full);
    __syncwarp();
  } else if (warp >= 4) {
    // ================================ compute warpgroups ================================
    // (the folded-statistics path of attn_bwd_tc_kernel: the score columns of a tile are the same 64 at either head_dim)
    const int g = (warp - 4) >> 2;
    const int q4 = warp & 3;
    const int r = q4 * 32 + lane;
    const int tid = r;
    const int row = r0 + r;
    const bool row_ok = row < p.S_row;
    int* ids_base = reinterpret_cast<int*>(smem + TcSmem64::ids) + g * 128;
    const int my_id = masked ? (row_ok ? p.row_id[static_cast<long long>(b) * p.S_row + row]
                                       : (MODE == MODE_DKV ? 0x7fffffff : -0x7fffffff))
                             : 0;
    int pre_i = 0;
    auto prefetch = [&](int j) {
      if (j >= T) return;
      const int c = (tile_list[j] & 0x7fff) * kCols + (tid & 63);
      const bool ok = c < p.S_col;
      if ((tile_list[j] & 0x8000) && tid < 64)
        pre_i = ok ? (masked ? p.col_id[static_cast<long long>(b) * p.S_col + c] : 0) : (MODE == MODE_DKV ? -0x7fffffff : 0x7fffffff);
    };
    const int j0 = (g + kNG - base % kNG) % kNG;
    prefetch(j0);
    for (int j = j0; j < T; j += kNG) {
      const int n = (base + j) / kNG;
      const bool need_mask = (tile_list[j] & 0x8000) != 0;
      int* s_id = ids_base + (n & 1) * 64;
      if (need_mask) {
        named_bar_sync(1 + g, 128);
        if (tid < 64) s_id[tid] = pre_i;
        named_bar_sync(1 + g, 128);
      }
      prefetch(j + kNG);
      mbar_wait(&sdp_full[g], n & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16) + g * 128;
      uint32_t sv[2][16], dv[2][16];
      float pf[16];
      auto expo = [&](uint32_t (&s16)[16], int i) {
        if (need_mask) {
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            const int cid = s_id[i * 16 + e];
            const bool hide = (MODE == MODE_DKV) ? (my_id > cid) : (cid > my_id);
            if (hide) s16[e] = 0xff800000u;
          }
        }
#pragma unroll
        for (int e = 0; e < 16; ++e) pf[e] = fast_ex2(__uint_as_float(s16[e]) * p.scale_log2);
      };
      tmem_ld16(taddr, sv[0]);
      tmem_wait1_16(sv[0]);
      tmem_ld16(taddr + 16, sv[1]);
      expo(sv[0], 0);
      mbar_wait(&dp_full[g], n & 1);
      tc_fence_after();
      tmem_ld16(taddr + 64, dv[0]);
#pragma unroll
      for (int i = 0; i < kSub; ++i) {
        const int cur = i & 1;
        if (i < kSub - 1) tmem_wait2_16(dv[cur], sv[cur ^ 1]); else tmem_wait1_16(dv[cur]);
        if (i < kSub - 1) tmem_ld16(taddr + 64 + (i + 1) * 16, dv[cur ^ 1]);
        if (i < kSub - 2) tmem_ld16(taddr + (i + 2) * 16, sv[cur]);
        uint32_t pw[8], dw[8];
#pragma unroll
        for (int e2 = 0; e2 < 8; ++e2) {
          const float s0 = pf[2 * e2] * __uint_as_float(dv[cur][2 * e2]);
          const float s1 = pf[2 * e2 + 1] * __uint_as_float(dv[cur][2 * e2 + 1]);
          if (MODE == MODE_DKV) pw[e2] = pack2(pf[2 * e2], pf[2 * e2 + 1]);
          dw[e2] = pack2(s0, s1);
        }
        if (MODE == MODE_DKV) tmem_st8(taddr + i * 8, pw);
        tmem_st8(taddr + 64 + i * 8, dw);
        if (i < kSub - 1) expo(sv[cur ^ 1], i + 1);
      }
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_ready[g]);
    }
    // ---- epilogue: accumulators (64 fp32 columns) -> bf16 -> global; wg0 -> dV, wg1 -> dK / dQ ----
    mbar_wait(acc_full, item_n & 1);
    tc_fence_after();
    const bool writes = (MODE == MODE_DKV) ? (g < 2) : (g == 1);
    if (writes) {
      const int which = (MODE == MODE_DKV) ? g : 1;
      const float sc = (which == 1) ? p.scale : 1.f;
      __nv_bfloat16* dst = nullptr;
      const float2* tb = nullptr;
      if (row_ok) {
        dst = (which == 0 ? p.out0 + b * p.o0_bs + static_cast<long long>(row) * p.o0_ts
                          : p.out1 + b * p.o1_bs + static_cast<long long>(row) * p.o1_ts) + h * 64;
        if (which == 1 && p.rope_table != nullptr) {
          int ps = p.rope_pos ? p.rope_pos[static_cast<long long>(b) * p.S_row + row] : row + p.rope_offset;
          ps = min(max(ps, 0), p.rope_len - 1);
          tb = p.rope_table + static_cast<long long>(ps) * 32;
        }
      }
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t acc[32];
        if (T > 0) {
          tmem_ld32(tmem_base + (static_cast<uint32_t>(q4 * 32) << 16) + kAcc64 + which * 64 + half * 32, acc);
          tmem_wait1_32(acc);
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) acc[i] = 0u;
        }
        if (row_ok) {
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            uint32_t w[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              float a0 = __uint_as_float(acc[c4 * 8 + e * 2]) * sc, a1 = __uint_as_float(acc[c4 * 8 + e * 2 + 1]) * sc;
              if (tb != nullptr) {         // gradient of a rotated operand: rotate back (conjugate)
                const float2 cs = tb[half * 16 + c4 * 4 + e];
                const float q0 = a0 * cs.x + a1 * cs.y, q1 = a1 * cs.x - a0 * cs.y;
                a0 = q0; a1 = q1;
              }
              w[e] = pack2(a0, a1);
            }
            *reinterpret_cast<uint4*>(dst + half * 32 + c4 * 8) = make_uint4(w[0], w[1], w[2], w[3]);
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  base += T;
  }   // item loop

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
  if (threadIdx.x == 0) {
    if (atomicAdd(&p.items[1], 1u) == gridDim.x - 1) {
      p.items[0] = 0u;
      p.items[1] = 0u;
      __threadfence();
    }
  }
}

// Merge of the key chunks of fk_attn_forward_kv_tc in chunk order (bit-reproducible): one thread per 4 columns of a
// (trial, head, query) row.  out = sum_c 2^(m_c - M) O_c / sum_c 2^(m_c - M) l_c with M = max_c m_c; a row that saw no
// key in any chunk gives zeros (lse = +inf, as in the unsplit kernels).
template <int HD>
__global__ void __launch_bounds__(256)
attn_kv_combine_kernel(const float* __restrict__ part_o, const float2* __restrict__ part_ml, __nv_bfloat16* __restrict__ out,
                       float* __restrict__ lse, int B, int H, int Sq, int n_chunks, long long o_bs, long long o_ts) {
  constexpr int kG = HD / 4;
  const long long t = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
  if (t >= static_cast<long long>(B) * H * Sq * kG) return;
  const int c4 = static_cast<int>(t % kG);
  const long long r = t / kG;                       // ((b * H + h) * Sq + row)
  const int row = static_cast<int>(r % Sq);
  const long long bh = r / Sq;
  const int h = static_cast<int>(bh % H), b = static_cast<int>(bh / H);
  const long long base = bh * n_chunks * Sq + row;  // partial row of chunk c: base + c * Sq
  float M = -INFINITY;
  for (int c = 0; c < n_chunks; ++c) M = fmaxf(M, part_ml[base + static_cast<long long>(c) * Sq].x);
  float L = 0.f, a[4] = {0.f, 0.f, 0.f, 0.f};
  if (M != -INFINITY) {
    for (int c = 0; c < n_chunks; ++c) {
      const long long pr = base + static_cast<long long>(c) * Sq;
      const float2 ml = part_ml[pr];
      if (!(ml.y > 0.f)) continue;
      const float w = exp2f(ml.x - M);
      const float4 o = *reinterpret_cast<const float4*>(part_o + pr * HD + c4 * 4);
      L += w * ml.y;
      a[0] += w * o.x; a[1] += w * o.y; a[2] += w * o.z; a[3] += w * o.w;
    }
  }
  const float inv = L > 0.f ? 1.f / L : 0.f;
  uint2 wv;
  wv.x = pack2(a[0] * inv, a[1] * inv);
  wv.y = pack2(a[2] * inv, a[3] * inv);
  *reinterpret_cast<uint2*>(out + b * o_bs + static_cast<long long>(row) * o_ts + h * HD + c4 * 4) = wv;
  if (lse != nullptr && c4 == 0) lse[bh * Sq + row] = L > 0.f ? M + log2f(L) : INFINITY;
}

}  // namespace fk

using namespace fk;

#define FK_API extern "C" __attribute__((visibility("default")))

FK_API int fk_attn_transpose(const void* x, long long bs, long long ts, int B, int S, int H, int head_dim, void* xt, int Sp,
                             void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(head_dim == 32, "fk_attn_transpose: only head_dim 32 is built");
  FK_REQUIRE(x && xt && B > 0 && S > 0 && H > 0 && Sp >= S && Sp % 8 == 0, "fk_attn_transpose: bad argument (Sp % 8 == 0)");
  FK_REQUIRE(ts % 8 == 0 && bs % 8 == 0, "fk_attn_transpose: strides must keep 16-byte alignment");
  attn_transpose_kernel<<<dim3((Sp + 63) / 64, H, B), 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(x), bs, ts, S, H, Sp,
                                                                        static_cast<__nv_bfloat16*>(xt));
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}

static int bwd_sm_count() { return fk_sm_count(); }

// head_dim 16 (attn_bwd_tc_kernel<.., 16>) and 64 (attn_bwd_tc64_kernel) backward: one path -- statistics folded (aug
// required), MN-major accumulate operands (no transposed copies), no stall-accounting build.  Arguments already checked by
// the caller as far as they are shared.
static int attn_backward_one_path(int head_dim, const void* q, const void* k, const void* v, const void* d_o, const void* qt, const void* kt,
                              const void* dot, const void* aug, void* dq, void* dk, void* dv, int B, int H, int S,
                              long long q_bs, long long q_ts, long long k_bs, long long k_ts, long long v_bs, long long v_ts,
                              long long do_bs, long long do_ts, long long dq_bs, long long dq_ts, long long dk_bs,
                              long long dk_ts, long long dv_bs, long long dv_ts, const int* qid, const int* kid,
                              const int* qmin, const int* qmax, const int* kmin, const int* kmax, float scale,
                              const float* lse, const float* delta, const float* rope_table, int rope_len,
                              const int* rope_pos, int rope_offset, int parts, unsigned int* counters,
                              const long long* g_attn_prof, cudaStream_t stream) {
  FK_REQUIRE(qt == nullptr && kt == nullptr && dot == nullptr, "fk_attn_backward_tc: head_dim 16 / 64 take no transposed operands");
  FK_REQUIRE(aug != nullptr && (reinterpret_cast<uintptr_t>(aug) & 31) == 0,
             "fk_attn_backward_tc: head_dim 16 / 64 need the statistics rows of fk_attn_aug (32-byte aligned)");
  FK_REQUIRE(g_attn_prof == nullptr, "fk_attn_backward_tc_profile: no stall-accounting build at head_dim 16 / 64");
  FK_REQUIRE(!(parts & 2) || (dk && dv), "fk_attn_backward_tc: dK/dV needs dk, dv");
  FK_REQUIRE(!(parts & 4) || dq, "fk_attn_backward_tc: dQ needs dq");
  FK_REQUIRE(dq_ts % 8 == 0 && dq_bs % 8 == 0 && dk_ts % 8 == 0 && dk_bs % 8 == 0 && dv_ts % 8 == 0 && dv_bs % 8 == 0,
             "fk_attn_backward_tc: gradient strides must keep 16-byte alignment");
  static bool attr_set_dev[FK_MAX_DEVICES];
  bool& attr_set = attr_set_dev[fk_device_ordinal()];
  if (!attr_set) {
    if (cudaFuncSetAttribute(attn_bwd_tc64_kernel<MODE_DKV>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem64::total) != cudaSuccess ||
        cudaFuncSetAttribute(attn_bwd_tc64_kernel<MODE_DQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem64::total) != cudaSuccess ||
        cudaFuncSetAttribute(attn_bwd_tc_kernel<MODE_DKV, 0, true, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem::total) != cudaSuccess ||
        cudaFuncSetAttribute(attn_bwd_tc_kernel<MODE_DQ, 0, true, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem::total) != cudaSuccess) {
      fk_set_last_error("cudaFuncSetAttribute(max dynamic smem) failed", __FILE__, __LINE__);
      return FK_ERR_CUDA;
    }
    attr_set = true;
  }
  CUtensorMap mQ128, mDO128, mK128, mV128, mQ64, mDO64, mK64, mV64, mAug64, mAug128;
  int rc = 0;
  auto make_map = head_dim == 64 ? make_tmap_heads_sw128 : make_tmap_heads_sw32;
  rc |= make_map(&mQ128, q, B, S, H, q_bs, q_ts, kRows);
  rc |= make_map(&mDO128, d_o, B, S, H, do_bs, do_ts, kRows);
  rc |= make_map(&mK128, k, B, S, H, k_bs, k_ts, kRows);
  rc |= make_map(&mV128, v, B, S, H, v_bs, v_ts, kRows);
  rc |= make_map(&mQ64, q, B, S, H, q_bs, q_ts, kCols);
  rc |= make_map(&mDO64, d_o, B, S, H, do_bs, do_ts, kCols);
  rc |= make_map(&mK64, k, B, S, H, k_bs, k_ts, kCols);
  rc |= make_map(&mV64, v, B, S, H, v_bs, v_ts, kCols);
  rc |= make_tmap_aug_sw32(&mAug64, aug, B, S, H, kCols);
  rc |= make_tmap_aug_sw32(&mAug128, aug, B, S, H, kRows);
  if (rc != 0) { fk_set_last_error("cuTensorMapEncodeTiled failed", __FILE__, __LINE__); return FK_ERR_DRIVER; }
  const long long n_items = static_cast<long long>((S + kRows - 1) / kRows) * H * B;
  FK_REQUIRE(n_items < (1ll << 31), "fk_attn_backward_tc: too many work items");
  const dim3 grid(static_cast<unsigned>(n_items < bwd_sm_count() ? n_items : bwd_sm_count()), 1, 1);
  TcParams p = {};
  p.lse = lse; p.delta = delta;
  p.B = B; p.H = H; p.S_row = S; p.S_col = S; p.Sq = S; p.scale = scale; p.scale_log2 = scale * 1.4426950408889634f;
  p.mn_major = 1;
  p.fold = 1;
  p.rope_table = reinterpret_cast<const float2*>(rope_table); p.rope_pos = rope_pos; p.rope_len = rope_len; p.rope_offset = rope_offset;
  int n = 0;
  if (parts & 2) {
    TcParams pk = p;
    pk.row_id = kid; pk.col_id = qid; pk.row_min = kmin; pk.row_max = kmax; pk.col_min = qmin; pk.col_max = qmax;
    pk.out0 = static_cast<__nv_bfloat16*>(dv); pk.o0_bs = dv_bs; pk.o0_ts = dv_ts;
    pk.out1 = static_cast<__nv_bfloat16*>(dk); pk.o1_bs = dk_bs; pk.o1_ts = dk_ts;
    pk.items = counters;
    if (head_dim == 64) attn_bwd_tc64_kernel<MODE_DKV><<<grid, kTcThreads, TcSmem64::total, stream>>>(mK128, mV128, mQ64, mDO64, mAug64, pk);
    else attn_bwd_tc_kernel<MODE_DKV, 0, true, 16><<<grid, kTcThreads, TcSmem::total, stream>>>(mK128, mV128, mQ64, mDO64, mDO64, mQ64, mAug64, pk);
    FK_CHECK_LAUNCH();
    ++n;
  }
  if (parts & 4) {
    TcParams pq = p;
    pq.row_id = qid; pq.col_id = kid; pq.row_min = qmin; pq.row_max = qmax; pq.col_min = kmin; pq.col_max = kmax;
    pq.out1 = static_cast<__nv_bfloat16*>(dq); pq.o1_bs = dq_bs; pq.o1_ts = dq_ts;
    pq.items = counters + 2;
    if (head_dim == 64) attn_bwd_tc64_kernel<MODE_DQ><<<grid, kTcThreads, TcSmem64::total, stream>>>(mQ128, mDO128, mK64, mV64, mAug128, pq);
    else attn_bwd_tc_kernel<MODE_DQ, 0, true, 16><<<grid, kTcThreads, TcSmem::total, stream>>>(mQ128, mDO128, mK64, mV64, mK64, mK64, mAug128, pq);
    FK_CHECK_LAUNCH();
    ++n;
  }
  fk_count_launch(n);
  return FK_OK;
}

// parts: 2 = dK/dV (needs qt, dot), 4 = dQ (needs kt).  delta must already hold rowsum(dO * O) (fk_attn_backward parts=1).
FK_API int fk_attn_backward_tc(const void* q, const void* k, const void* v, const void* d_o, const void* qt, const void* kt,
                               const void* dot, int Sp, const float* lse, const float* delta, const void* aug, void* dq, void* dk, void* dv,
                               int B, int H, int S, int head_dim, long long q_bs, long long q_ts, long long k_bs,
                               long long k_ts, long long v_bs, long long v_ts, long long do_bs, long long do_ts,
                               long long dq_bs, long long dq_ts, long long dk_bs, long long dk_ts, long long dv_bs,
                               long long dv_ts, const int* qid, const int* kid, const int* qmin, const int* qmax,
                               const int* kmin, const int* kmax, float scale, const float* rope_table, int rope_len,
                               const int* rope_pos, int rope_offset, int parts, unsigned int* counters, void* stream_) {
  return fk_attn_backward_tc_profile(q, k, v, d_o, qt, kt, dot, Sp, lse, delta, aug, dq, dk, dv, B, H, S, head_dim, q_bs, q_ts, k_bs,
                                     k_ts, v_bs, v_ts, do_bs, do_ts, dq_bs, dq_ts, dk_bs, dk_ts, dv_bs, dv_ts, qid, kid, qmin,
                                     qmax, kmin, kmax, scale, rope_table, rope_len, rope_pos, rope_offset, parts, counters,
                                     nullptr, 0, stream_);
}

// Same launch; prof != NULL selects the stall-accounting instantiation (diagnosis only, scripts/gpu_attn_stalls.py):
// prof_mode 1 = full stall accounting, 2 = light (lifetime + global timestamps + SM id).
FK_API int fk_attn_backward_tc_profile(const void* q, const void* k, const void* v, const void* d_o, const void* qt, const void* kt,
                               const void* dot, int Sp, const float* lse, const float* delta, const void* aug, void* dq, void* dk, void* dv,
                               int B, int H, int S, int head_dim, long long q_bs, long long q_ts, long long k_bs,
                               long long k_ts, long long v_bs, long long v_ts, long long do_bs, long long do_ts,
                               long long dq_bs, long long dq_ts, long long dk_bs, long long dk_ts, long long dv_bs,
                               long long dv_ts, const int* qid, const int* kid, const int* qmin, const int* qmax,
                               const int* kmin, const int* kmax, float scale, const float* rope_table, int rope_len,
                               const int* rope_pos, int rope_offset, int parts, unsigned int* counters, long long* g_attn_prof,
                               int g_attn_prof_mode, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(head_dim == 16 || head_dim == 32 || head_dim == 64, "fk_attn_backward_tc: head_dim must be 16, 32 or 64");
  FK_REQUIRE(counters != nullptr, "fk_attn_backward_tc: counters (4 zero-initialised uint32, one set per launch in flight) is null");
  FK_REQUIRE(rope_table == nullptr || rope_len > 0, "fk_attn_backward_tc: rope_len must be positive with a rope table");
  FK_REQUIRE(q && k && v && d_o && lse && delta && B > 0 && H > 0 && S > 0, "fk_attn_backward_tc: bad argument");
  FK_REQUIRE((parts & ~6) == 0 && parts != 0, "fk_attn_backward_tc: parts is a bitmask of 2 (dK/dV) and 4 (dQ)");
  FK_REQUIRE((qid == nullptr) == (kid == nullptr), "fk_attn_backward_tc: qid and kid go together");
  FK_REQUIRE(qid == nullptr || (qmin && qmax && kmin && kmax), "fk_attn_backward_tc: label ranges missing");
  FK_REQUIRE((S + kCols - 1) / kCols <= kMaxTiles, "fk_attn_backward_tc: sequence too long");
  FK_REQUIRE(Sp >= S && Sp % 8 == 0, "fk_attn_backward_tc: Sp must be >= S and a multiple of 8");
  if (head_dim != 32)
    return attn_backward_one_path(head_dim, q, k, v, d_o, qt, kt, dot, aug, dq, dk, dv, B, H, S, q_bs, q_ts, k_bs, k_ts, v_bs, v_ts, do_bs,
                              do_ts, dq_bs, dq_ts, dk_bs, dk_ts, dv_bs, dv_ts, qid, kid, qmin, qmax, kmin, kmax, scale, lse,
                              delta, rope_table, rope_len, rope_pos, rope_offset, parts, counters, g_attn_prof, stream);
  static bool attr_set_dev[FK_MAX_DEVICES];
  bool& attr_set = attr_set_dev[fk_device_ordinal()];
  if (!attr_set) {
    if (cudaFuncSetAttribute(attn_bwd_tc_kernel<MODE_DKV, 0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem::total) != cudaSuccess ||
        cudaFuncSetAttribute(attn_bwd_tc_kernel<MODE_DQ, 0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem::total) != cudaSuccess ||
        cudaFuncSetAttribute(attn_bwd_tc_kernel<MODE_DKV, 0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem::total) != cudaSuccess ||
        cudaFuncSetAttribute(attn_bwd_tc_kernel<MODE_DQ, 0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem::total) != cudaSuccess ||
        cudaFuncSetAttribute(attn_bwd_tc_kernel<MODE_DKV, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem::total) != cudaSuccess ||
        cudaFuncSetAttribute(attn_bwd_tc_kernel<MODE_DQ, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem::total) != cudaSuccess ||
        cudaFuncSetAttribute(attn_bwd_tc_kernel<MODE_DKV, 2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem::total) != cudaSuccess ||
        cudaFuncSetAttribute(attn_bwd_tc_kernel<MODE_DQ, 2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem::total) != cudaSuccess) {
      fk_set_last_error("cudaFuncSetAttribute(max dynamic smem) failed", __FILE__, __LINE__);
      return FK_ERR_CUDA;
    }
    attr_set = true;
  }
  CUtensorMap mQ128, mDO128, mK128, mV128, mQ64, mDO64, mK64, mV64, mQt, mKt, mDOt;
  int rc = 0;
  rc |= make_tmap_heads_sw64(&mQ128, q, B, S, H, q_bs, q_ts, kRows);
  rc |= make_tmap_heads_sw64(&mDO128, d_o, B, S, H, do_bs, do_ts, kRows);
  rc |= make_tmap_heads_sw64(&mK128, k, B, S, H, k_bs, k_ts, kRows);
  rc |= make_tmap_heads_sw64(&mV128, v, B, S, H, v_bs, v_ts, kRows);
  rc |= make_tmap_heads_sw64(&mQ64, q, B, S, H, q_bs, q_ts, kCols);
  rc |= make_tmap_heads_sw64(&mDO64, d_o, B, S, H, do_bs, do_ts, kCols);
  rc |= make_tmap_heads_sw64(&mK64, k, B, S, H, k_bs, k_ts, kCols);
  rc |= make_tmap_heads_sw64(&mV64, v, B, S, H, v_bs, v_ts, kCols);
  const uint64_t trows = static_cast<uint64_t>(B) * H * 32;
  // qt / kt / dot all null: the accumulate MMAs take their B operand MN-major from the [tokens][32] tiles (no copies)
  const int mn_major = (qt == nullptr && kt == nullptr && dot == nullptr) ? 1 : 0;
  mQt = mQ64; mDOt = mDO64; mKt = mK64;
  // aug (nullable): statistics rows from fk_attn_aug -> lse / delta folded into the score MMAs (needs the MN-major mode:
  // the statistics tile takes the place of the transposed operand in the streamed stage)
  const int fold = (aug != nullptr && mn_major && g_attn_prof == nullptr) ? 1 : 0;      // (the stall-accounting builds are staged)
  CUtensorMap mAug64 = mQ64, mAug128 = mQ64;
  if (fold) {
    FK_REQUIRE((reinterpret_cast<uintptr_t>(aug) & 31) == 0, "fk_attn_backward_tc: aug must be 32-byte aligned");
    rc |= make_tmap_aug_sw32(&mAug64, aug, B, S, H, kCols);
    rc |= make_tmap_aug_sw32(&mAug128, aug, B, S, H, kRows);
  }
  if ((parts & 2) && !mn_major) {
    FK_REQUIRE(qt && dot && dk && dv, "fk_attn_backward_tc: dK/dV needs qt, dot, dk, dv");
    rc |= make_tmap_bf16_sw128(&mQt, qt, trows, static_cast<uint64_t>(Sp), 32);
    rc |= make_tmap_bf16_sw128(&mDOt, dot, trows, static_cast<uint64_t>(Sp), 32);
  }
  if ((parts & 4) && !mn_major) {
    FK_REQUIRE(kt && dq, "fk_attn_backward_tc: dQ needs kt, dq");
    rc |= make_tmap_bf16_sw128(&mKt, kt, trows, static_cast<uint64_t>(Sp), 32);
  }
  FK_REQUIRE(!(parts & 2) || (dk && dv), "fk_attn_backward_tc: dK/dV needs dk, dv");
  FK_REQUIRE(!(parts & 4) || dq, "fk_attn_backward_tc: dQ needs dq");
  if (rc != 0) { fk_set_last_error("cuTensorMapEncodeTiled failed", __FILE__, __LINE__); return FK_ERR_DRIVER; }
  // persistent CTAs: one per SM (or per work item when there are fewer), looping over (row tile, head, batch) items
  const long long n_items = static_cast<long long>((S + kRows - 1) / kRows) * H * B;
  FK_REQUIRE(n_items < (1ll << 31), "fk_attn_backward_tc: too many work items");
  const dim3 grid(static_cast<unsigned>(n_items < bwd_sm_count() ? n_items : bwd_sm_count()), 1, 1);
  int n = 0;
  if (parts & 2) {
    TcParams p = {};
    p.row_id = kid; p.col_id = qid; p.row_min = kmin; p.row_max = kmax; p.col_min = qmin; p.col_max = qmax;
    p.lse = lse; p.delta = delta;
    p.out0 = static_cast<__nv_bfloat16*>(dv); p.o0_bs = dv_bs; p.o0_ts = dv_ts;
    p.out1 = static_cast<__nv_bfloat16*>(dk); p.o1_bs = dk_bs; p.o1_ts = dk_ts;
    p.B = B; p.H = H; p.S_row = S; p.S_col = S; p.Sq = S; p.scale = scale; p.scale_log2 = scale * 1.4426950408889634f;
    p.prof = g_attn_prof;
    p.items = counters;
    p.mn_major = mn_major;
    p.fold = fold;
    p.rope_table = reinterpret_cast<const float2*>(rope_table); p.rope_pos = rope_pos; p.rope_len = rope_len; p.rope_offset = rope_offset;
    if (g_attn_prof && g_attn_prof_mode == 2) attn_bwd_tc_kernel<MODE_DKV, 2, false><<<grid, kTcThreads, TcSmem::total, stream>>>(mK128, mV128, mQ64, mDO64, mDOt, mQt, mAug64, p);
    else if (g_attn_prof) attn_bwd_tc_kernel<MODE_DKV, 1, false><<<grid, kTcThreads, TcSmem::total, stream>>>(mK128, mV128, mQ64, mDO64, mDOt, mQt, mAug64, p);
    else if (fold) attn_bwd_tc_kernel<MODE_DKV, 0, true><<<grid, kTcThreads, TcSmem::total, stream>>>(mK128, mV128, mQ64, mDO64, mDOt, mQt, mAug64, p);
    else attn_bwd_tc_kernel<MODE_DKV, 0, false><<<grid, kTcThreads, TcSmem::total, stream>>>(mK128, mV128, mQ64, mDO64, mDOt, mQt, mAug64, p);
    FK_CHECK_LAUNCH();
    ++n;
  }
  if (parts & 4) {
    TcParams p = {};
    p.row_id = qid; p.col_id = kid; p.row_min = qmin; p.row_max = qmax; p.col_min = kmin; p.col_max = kmax;
    p.lse = lse; p.delta = delta;
    p.out0 = nullptr; p.out1 = static_cast<__nv_bfloat16*>(dq); p.o1_bs = dq_bs; p.o1_ts = dq_ts;
    p.B = B; p.H = H; p.S_row = S; p.S_col = S; p.Sq = S; p.scale = scale; p.scale_log2 = scale * 1.4426950408889634f;
    p.prof = g_attn_prof;
    p.items = counters + 2;
    p.mn_major = mn_major;
    p.fold = fold;
    p.rope_table = reinterpret_cast<const float2*>(rope_table); p.rope_pos = rope_pos; p.rope_len = rope_len; p.rope_offset = rope_offset;
    if (g_attn_prof && g_attn_prof_mode == 2) attn_bwd_tc_kernel<MODE_DQ, 2, false><<<grid, kTcThreads, TcSmem::total, stream>>>(mQ128, mDO128, mK64, mV64, mKt, mKt, mAug128, p);
    else if (g_attn_prof) attn_bwd_tc_kernel<MODE_DQ, 1, false><<<grid, kTcThreads, TcSmem::total, stream>>>(mQ128, mDO128, mK64, mV64, mKt, mKt, mAug128, p);
    else if (fold) attn_bwd_tc_kernel<MODE_DQ, 0, true><<<grid, kTcThreads, TcSmem::total, stream>>>(mQ128, mDO128, mK64, mV64, mKt, mKt, mAug128, p);
    else attn_bwd_tc_kernel<MODE_DQ, 0, false><<<grid, kTcThreads, TcSmem::total, stream>>>(mQ128, mDO128, mK64, mV64, mKt, mKt, mAug128, p);
    FK_CHECK_LAUNCH();
    ++n;
  }
  fk_count_launch(n);
  return FK_OK;
}

// delta = rowsum(dO * O) and the statistics rows the folded backward takes (see attn_aug_kernel): o / d_o bf16
// [B, S, H, head_dim] (16, 32 or 64) with strides in elements, lse fp32 [B, H, S] (log2 domain, from the forward), delta fp32
// [B, H, S], aug bf16 [B, H, S, 16].
FK_API int fk_attn_aug(const void* o, const void* d_o, const float* lse, float* delta, void* aug, int B, int H, int S,
                       int head_dim, long long o_bs, long long o_ts, long long do_bs, long long do_ts, float scale, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(head_dim == 16 || head_dim == 32 || head_dim == 64, "fk_attn_aug: head_dim must be 16, 32 or 64");
  FK_REQUIRE(o && d_o && lse && delta && aug && B > 0 && H > 0 && S > 0 && scale > 0.f, "fk_attn_aug: bad argument");
  FK_REQUIRE(o_ts % 8 == 0 && do_ts % 8 == 0 && o_bs % 8 == 0 && do_bs % 8 == 0, "fk_attn_aug: strides must keep 16-byte alignment");
  FK_REQUIRE((reinterpret_cast<uintptr_t>(aug) & 31) == 0, "fk_attn_aug: aug must be 32-byte aligned");
  const long long n = static_cast<long long>(B) * S * H;
  auto kern = head_dim == 64 ? attn_aug_kernel<64> : head_dim == 16 ? attn_aug_kernel<16> : attn_aug_kernel<32>;
  kern<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(
      static_cast<const __nv_bfloat16*>(o), static_cast<const __nv_bfloat16*>(d_o), lse, delta, static_cast<__nv_bfloat16*>(aug), B, H, S,
      o_bs, o_ts, do_bs, do_ts, 1.f / (scale * 1.4426950408889634f));
  FK_CHECK_LAUNCH();
  fk_count_launch();
  return FK_OK;
}

// The forward at head_dim 16, 32 or 64 on `grid` persistent CTAs: tensor maps of q / k / v with the swizzle of the head
// width, then that width's instantiation; the key-split one when `split` (the unsplit kernels take the parameter block
// without the chunk and band fields).
static int attn_fwd_launch(int head_dim, const void* q, const void* k, const void* v, long long q_bs, long long q_ts,
                           long long k_bs, long long k_ts, long long v_bs, long long v_ts, const FwdKvParams& p,
                           bool split, unsigned grid, cudaStream_t stream) {
  static bool attr_set_dev[FK_MAX_DEVICES];
  bool& attr_set = attr_set_dev[fk_device_ordinal()];
  if (!attr_set) {
    auto set_smem = [](auto kern, int bytes) {
      return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) == cudaSuccess;
    };
    if (!set_smem(attn_fwd_tc_kernel<16, false>, FwdSmem<16>::total) || !set_smem(attn_fwd_tc_kernel<16, true>, FwdSmem<16>::total) ||
        !set_smem(attn_fwd_tc_kernel<32, false>, FwdSmem<32>::total) || !set_smem(attn_fwd_tc_kernel<32, true>, FwdSmem<32>::total) ||
        !set_smem(attn_fwd_tc_kernel<64, false>, FwdSmem<64>::total) || !set_smem(attn_fwd_tc_kernel<64, true>, FwdSmem<64>::total)) {
      fk_set_last_error("cudaFuncSetAttribute(max dynamic smem) failed", __FILE__, __LINE__);
      return FK_ERR_CUDA;
    }
    attr_set = true;
  }
  CUtensorMap mQ, mK, mV;
  int rc = 0;
  auto make_map = head_dim == 64 ? make_tmap_heads_sw128 : head_dim == 16 ? make_tmap_heads_sw32 : make_tmap_heads_sw64;
  rc |= make_map(&mQ, q, p.B, p.Sq, p.H, q_bs, q_ts, 128);
  rc |= make_map(&mK, k, p.B, p.Sk, p.H, k_bs, k_ts, kFwdTileK);
  rc |= make_map(&mV, v, p.B, p.Sk, p.H, v_bs, v_ts, kFwdTileK);
  if (rc != 0) { fk_set_last_error("cuTensorMapEncodeTiled failed", __FILE__, __LINE__); return FK_ERR_DRIVER; }
  const FwdParams& p1 = p;
  if (split) {
    if (head_dim == 64) attn_fwd_tc_kernel<64, true><<<grid, kFwdThreads, FwdSmem<64>::total, stream>>>(mQ, mK, mV, p);
    else if (head_dim == 16) attn_fwd_tc_kernel<16, true><<<grid, kFwdThreads, FwdSmem<16>::total, stream>>>(mQ, mK, mV, p);
    else attn_fwd_tc_kernel<32, true><<<grid, kFwdThreads, FwdSmem<32>::total, stream>>>(mQ, mK, mV, p);
  } else {
    if (head_dim == 64) attn_fwd_tc_kernel<64><<<grid, kFwdThreads, FwdSmem<64>::total, stream>>>(mQ, mK, mV, p1);
    else if (head_dim == 16) attn_fwd_tc_kernel<16><<<grid, kFwdThreads, FwdSmem<16>::total, stream>>>(mQ, mK, mV, p1);
    else attn_fwd_tc_kernel<32><<<grid, kFwdThreads, FwdSmem<32>::total, stream>>>(mQ, mK, mV, p1);
  }
  FK_CHECK_LAUNCH();
  return FK_OK;
}

// Forward on tcgen05; q / k / v are strided views of the fused projection; same label / range conventions as fk_attn_forward.
FK_API int fk_attn_forward_tc(const void* q, const void* k, const void* v, void* out, float* lse, int B, int H, int S,
                              int head_dim, long long q_bs, long long q_ts, long long k_bs, long long k_ts, long long v_bs,
                              long long v_ts, long long o_bs, long long o_ts, const int* qid, const int* kid, const int* qmin,
                              const int* qmax, const int* kmin, const int* kmax, float scale, unsigned int* counters,
                              void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(head_dim == 16 || head_dim == 32 || head_dim == 64, "fk_attn_forward_tc: head_dim must be 16, 32 or 64");
  FK_REQUIRE(counters != nullptr, "fk_attn_forward_tc: counters (2 zero-initialised uint32, one pair per launch in flight) is null");
  FK_REQUIRE(q && k && v && out && B > 0 && H > 0 && S > 0, "fk_attn_forward_tc: bad argument");
  FK_REQUIRE((qid == nullptr) == (kid == nullptr), "fk_attn_forward_tc: qid and kid go together");
  FK_REQUIRE(qid == nullptr || (qmin && qmax && kmin && kmax), "fk_attn_forward_tc: label ranges missing");
  FK_REQUIRE((S + kFwdTileK - 1) / kFwdTileK <= kMaxTiles && S < (1 << 20), "fk_attn_forward_tc: sequence too long");
  FK_REQUIRE(o_ts % 8 == 0 && o_bs % 8 == 0, "fk_attn_forward_tc: output strides must keep 16-byte alignment");
  FwdKvParams p = {};
  p.qid = qid; p.kid = kid; p.qmin = qmin; p.qmax = qmax; p.kmin = kmin; p.kmax = kmax;
  p.out = static_cast<__nv_bfloat16*>(out); p.lse = lse; p.o_bs = o_bs; p.o_ts = o_ts;
  p.B = B; p.H = H; p.Sq = S; p.Sk = S; p.scale_log2 = scale * 1.4426950408889634f;
  p.items = counters;
  p.n_chunks = 1;
  // persistent CTAs: one per SM (or per work item when there are fewer), looping over (256-query block, head, trial) items
  const long long n_items = static_cast<long long>((S + 255) / 256) * H * B;
  FK_REQUIRE(n_items < (1ll << 31), "fk_attn_forward_tc: too many work items");
  const unsigned grid = static_cast<unsigned>(n_items < bwd_sm_count() ? n_items : bwd_sm_count());
  const int rc = attn_fwd_launch(head_dim, q, k, v, q_bs, q_ts, k_bs, k_ts, v_bs, v_ts, p, false, grid, stream);
  if (rc != FK_OK) return rc;
  fk_count_launch();
  return FK_OK;
}

// Split-key forward for queries and keys of different lengths (a streaming step against a key / value cache).
FK_API int fk_attn_kv_chunks(int B, int H, int Sq, int Sk, int max_ctas) {
  if (B < 1 || H < 1 || Sq < 1 || Sk < 1) return 1;
  const long long ctas = max_ctas > 0 ? max_ctas : fk_sm_count();
  const long long units = static_cast<long long>(B) * H * ((Sq + 255) / 256);
  const int n_k_tiles = (Sk + kFwdTileK - 1) / kFwdTileK;
  if (units >= ctas) return 1;
  const int want = static_cast<int>(std::min<long long>((ctas + units - 1) / units, n_k_tiles));
  const int per = (n_k_tiles + want - 1) / want;                 // key tiles per chunk; every chunk gets at least one
  return (n_k_tiles + per - 1) / per;
}

// fk_attn_forward_kv_tc with a label band.  A band below kNoBand runs the split kernel even with one chunk (merged by the
// combine kernel), so the unsplit kernels, which the training forward shares, never see a band.
FK_API int fk_attn_forward_kv_band_tc(const void* q, const void* k, const void* v, void* out, float* lse, int B, int H,
                                      int Sq, int Sk, int head_dim, long long q_bs, long long q_ts, long long k_bs,
                                      long long k_ts, long long v_bs, long long v_ts, long long o_bs, long long o_ts,
                                      const int* qid, const int* kid, const int* qmin, const int* qmax, const int* kmin,
                                      const int* kmax, float scale, float* part_o, float* part_ml, int n_chunks,
                                      long long band, unsigned int* counters, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  FK_REQUIRE(band >= 1, "fk_attn_forward_kv_band_tc: band must be >= 1");
  FK_REQUIRE(head_dim == 16 || head_dim == 32 || head_dim == 64, "fk_attn_forward_kv_tc: head_dim must be 16, 32 or 64");
  FK_REQUIRE(counters != nullptr, "fk_attn_forward_kv_tc: counters (2 zero-initialised uint32, one pair per launch in flight) is null");
  FK_REQUIRE(q && k && v && out && B > 0 && H > 0 && Sq > 0 && Sk > 0, "fk_attn_forward_kv_tc: bad argument");
  FK_REQUIRE((qid == nullptr) == (kid == nullptr), "fk_attn_forward_kv_tc: qid and kid go together");
  FK_REQUIRE(qid == nullptr || (qmin && qmax && kmin && kmax), "fk_attn_forward_kv_tc: label ranges missing");
  const bool banded = band < kNoBand;
  FK_REQUIRE(!banded || qid != nullptr, "fk_attn_forward_kv_band_tc: a band needs labels");
  FK_REQUIRE((Sk + kFwdTileK - 1) / kFwdTileK <= kMaxTiles && Sk < (1 << 20) && Sq < (1 << 20),
             "fk_attn_forward_kv_tc: sequence too long");
  FK_REQUIRE(q_bs % 8 == 0 && q_ts % 8 == 0 && k_bs % 8 == 0 && k_ts % 8 == 0 && v_bs % 8 == 0 && v_ts % 8 == 0 &&
             o_bs % 8 == 0 && o_ts % 8 == 0 && q_ts >= H * head_dim && k_ts >= H * head_dim && v_ts >= H * head_dim &&
             o_ts >= H * head_dim, "fk_attn_forward_kv_tc: strides must cover a token's heads and keep 16-byte alignment");
  const int n_k_tiles = (Sk + kFwdTileK - 1) / kFwdTileK;
  FK_REQUIRE(n_chunks >= 1 && n_chunks <= n_k_tiles, "fk_attn_forward_kv_tc: n_chunks must be in [1, key tiles of 128]");
  const bool split = n_chunks > 1 || banded;
  FK_REQUIRE(!split || (part_o && part_ml),
             "fk_attn_forward_kv_tc: part_o / part_ml are needed with more than one chunk or with a band");
  const long long n_units = static_cast<long long>((Sq + 255) / 256) * n_chunks;
  FK_REQUIRE(n_units * H * B < (1ll << 31), "fk_attn_forward_kv_tc: too many work items");
  FwdKvParams p = {};
  p.qid = qid; p.kid = kid; p.qmin = qmin; p.qmax = qmax; p.kmin = kmin; p.kmax = kmax;
  p.out = static_cast<__nv_bfloat16*>(out); p.lse = lse; p.o_bs = o_bs; p.o_ts = o_ts;
  p.B = B; p.H = H; p.Sq = Sq; p.Sk = Sk; p.scale_log2 = scale * 1.4426950408889634f;
  p.items = counters;
  p.part_o = part_o; p.part_ml = part_ml; p.n_chunks = n_chunks; p.chunk_tiles = (n_k_tiles + n_chunks - 1) / n_chunks;
  p.band = banded ? band : kNoBand;
  const long long n_items = n_units * H * B;
  const unsigned grid = static_cast<unsigned>(n_items < bwd_sm_count() ? n_items : bwd_sm_count());
  const int rc = attn_fwd_launch(head_dim, q, k, v, q_bs, q_ts, k_bs, k_ts, v_bs, v_ts, p, split, grid, stream);
  if (rc != FK_OK) return rc;
  if (!split) {
    // one chunk and no band: the unsplit kernels write O / l and lse themselves
    fk_count_launch();
    return FK_OK;
  }
  const long long n_threads = static_cast<long long>(B) * H * Sq * (head_dim / 4);
  auto combine = head_dim == 64 ? attn_kv_combine_kernel<64> : head_dim == 16 ? attn_kv_combine_kernel<16> : attn_kv_combine_kernel<32>;
  combine<<<static_cast<unsigned>((n_threads + 255) / 256), 256, 0, stream>>>(part_o, reinterpret_cast<const float2*>(part_ml),
                                                                                static_cast<__nv_bfloat16*>(out), lse, B, H, Sq,
                                                                                n_chunks, o_bs, o_ts);
  FK_CHECK_LAUNCH();
  fk_count_launch(2);
  return FK_OK;
}

FK_API int fk_attn_forward_kv_tc(const void* q, const void* k, const void* v, void* out, float* lse, int B, int H, int Sq,
                                 int Sk, int head_dim, long long q_bs, long long q_ts, long long k_bs, long long k_ts,
                                 long long v_bs, long long v_ts, long long o_bs, long long o_ts, const int* qid,
                                 const int* kid, const int* qmin, const int* qmax, const int* kmin, const int* kmax,
                                 float scale, float* part_o, float* part_ml, int n_chunks, unsigned int* counters,
                                 void* stream_) {
  return fk_attn_forward_kv_band_tc(q, k, v, out, lse, B, H, Sq, Sk, head_dim, q_bs, q_ts, k_bs, k_ts, v_bs, v_ts, o_bs, o_ts,
                                    qid, kid, qmin, qmax, kmin, kmax, scale, part_o, part_ml, n_chunks, kNoBand, counters,
                                    stream_);
}
