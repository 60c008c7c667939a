/* frankenstein-b200 C ABI  (libfk_b200.so, compiled for sm_100a only)
 *
 * Conventions (SURVEY.md section 8b):
 *  - plain pointers and sizes, no torch types; all pointers are DEVICE pointers unless stated;
 *  - the caller owns every buffer (kernels never allocate or free);
 *  - every call is asynchronous on `stream` (a cudaStream_t passed as void*), no implicit sync, and launches on the
 *    CURRENT device (the caller selects the device its pointers live on; host-side caches are per device ordinal);
 *  - no device-side global state: hand-out / last-block counters are caller-owned words (zero on entry, zero on exit),
 *    so calls are re-entrant per stream;
 *  - return value: 0 = ok, negative = error (fk_last_error() has the text);
 *    -1 bad argument, -2 CUDA launch error, -3 unsupported shape, -4 driver entry point missing;
 *  - no CPU path exists: without a Blackwell GPU every compute entry point fails.
 *
 * Each entry point names the reference interface it replaces.  "VQ" is the third-party
 * vector_quantize_pytorch.VectorQuantize constructed at models/vq_brain.py:184-193 and called at
 * models/vq_brain.py:209 / :233 (restated in oracle/vector_quantize_ref.py).
 */
#ifndef FK_B200_H
#define FK_B200_H

#ifdef __cplusplus
extern "C" {
#endif

/* ---- bookkeeping ---------------------------------------------------------------------------- */
const char* fk_last_error(void);
long long fk_launch_count(void);       /* kernels/memsets enqueued by this library since reset */
void fk_reset_launch_count(void);
int fk_abi_version(void);
int fk_target_sm(void);                 /* 100 */
int fk_device_ok(void);                 /* 1 if the current device is compute capability 10.x */

/* ---- VQ: operand preparation ---------------------------------------------------------------- */
/* VectorQuantize.forward `x = x.float()` + CosineSimCodebook `l2norm(x)` (F.normalize, eps 1e-12).
 * e: [N, D] dtype 0=f32 1=bf16 2=f16.  xn (nullable): fp32 [N, D] transformed rows;
 * x_bf16: [N, Dp] zero-padded tensor-core operand; inv_norm: [N] (cosine only). */
int fk_vq_prepare_input(const void* e, int dtype, long long N, int D, int Dp, int use_cosine, float* xn,
                        void* x_bf16, float* inv_norm, void* stream);
/* Codebook operand for the search: cb_bf16 [K, Dp], c2pad [Kpad] = |c|^2 (0 for cosine), +inf pad. */
int fk_vq_prepare_codebook(const float* embed, int K, int D, int Dp, int Kpad, int use_cosine, void* cb_bf16,
                           float* c2pad, void* stream);

/* ---- VQ: nearest-codeword search (tcgen05 / TMEM / TMA) -------------------------------------- */
/* Replaces `dist = -cdist(x, embed)` / `einsum('h n d, h c d -> h n c')` + `argmax` in
 * Euclidean/CosineSimCodebook.forward.  Writes per row S slots of 4 candidates (approximate key, code index; -1 = none): cand_val/cand_idx are [N, S, 4];
 * S = fk_vq_search_slots(N, K, max_ctas) (host helper, no GPU work).  max_ctas <= 0: all SMs. */
int fk_vq_search_slots(long long N, int K, int max_ctas);
int fk_vq_search(const void* x_bf16, const void* cb_bf16, const float* c2pad, long long N, int K, int Dp,
                 int use_cosine, float* cand_val, int* cand_idx, int S, int max_ctas, void* stream);

/* Same kernel; additionally dumps the raw fp32 accumulators x.c to dbg_scores [N, roundup(K,128)] (tests). */
int fk_vq_search_debug(const void* x_bf16, const void* cb_bf16, const float* c2pad, long long N, int K, int Dp,
                       int use_cosine, float* cand_val, int* cand_idx, int S, int max_ctas, float* dbg_scores,
                       void* stream);

/* Same kernel built with stall accounting (performance diagnosis only; scripts/gpu_search_stalls.py): prof is
 * int64 [n_ctas, 32] cycle counters (total, setup, producer / issuer / epilogue barrier waits; see vq_search.cu). */
int fk_vq_search_profile(const void* x_bf16, const void* cb_bf16, const float* c2pad, long long N, int K, int Dp,
                         int use_cosine, float* cand_val, int* cand_idx, int S, int max_ctas, long long* prof,
                         void* stream);

/* ---- VQ: exact re-score + gather + straight-through + commitment loss ------------------------ */
/* Replaces gumbel_sample(argmax), `quantize = onehot @ embed`, `x + (quantize - x).detach()` and
 * `F.mse_loss(quantize.detach(), x) * commitment_weight` (VectorQuantize.forward).
 * indices: int64 [N]; quantize: fp32 [N, D] (nullable when !training: indices only); loss: [1]; partials: [fk_vq_finish_partials(N)];
 * counter: one zero-initialised uint32 that the kernel leaves at zero. */
long long fk_vq_finish_partials(long long N);
int fk_vq_finish(const float* xn, const float* embed, const float* cand_val, const int* cand_idx, long long N,
                 int K, int D, int S, int use_cosine, int training, float commitment_weight, long long* indices,
                 float* quantize, float* loss, float* partials, unsigned int* counter, void* stream);

/* ---- VQ: EMA statistics, EMA finalize + dead-code reset -------------------------------------- */
/* Replaces `bins = onehot.sum()` and `embed_sum = einsum('h n d, h n c -> h c d')`.
 * stats: fp32 [K*D + K] = embed_sum || bins, one packed buffer so data-parallel ranks need ONE
 * all-reduce (every element is written by the call).  Segmented sum keyed by the code index: counting sort of the
 * rows, then one warp per code adds its rows in ascending row order (coalesced 16-byte loads, no atomics on data), so
 * the result is bit-reproducible.  ws: int32 [fk_vq_ema_stats_ws(N, K)] scratch.  D <= 256. */
long long fk_vq_ema_stats_ws(long long N, int K);
int fk_vq_ema_stats(const float* xn, const long long* indices, long long N, int K, int D, float* stats, int* ws,
                    void* stream);
/* Replaces ema_inplace x2, laplace_smoothing, `embed.copy_`, (cosine) l2norm and expire_codes_/
 * replace; also writes the next search's operand.  sample_rows (nullable): int64 [n_sample] rows of
 * xn; the i-th expired code (ascending code index) takes row sample_rows[i % n_sample].
 * Workspaces: total_ws [1] float, expire_rank_ws [K] int, n_expired [1] int (output). */
int fk_vq_ema_update(const float* stats, float* cluster_size, float* embed_avg, float* embed, int K, int D, int Dp,
                     int Kpad, int use_cosine, float decay, float eps, float threshold,
                     const long long* sample_rows, int n_sample, const float* xn, long long N, void* cb_bf16,
                     float* c2pad, float* total_ws, int* expire_rank_ws, int* n_expired, void* stream);

/* ---- VQ: backward ---------------------------------------------------------------------------- */
/* autograd of VectorQuantize.forward w.r.t. its input: g_out (nullable) [N, D], g_loss (nullable) [1]. */
int fk_vq_backward(const float* g_out, const float* g_loss, const float* xn, const float* quantize,
                   const float* inv_norm, long long N, int D, int use_cosine, float commitment_weight,
                   float* grad_in, void* stream);

/* ---- VQ: k-means init (upstream `kmeans`), one mean update from packed stats ----------------- */
int fk_vq_kmeans_update(const float* stats, float* means, int K, int D, int Dp, int Kpad, int use_cosine,
                        void* cb_bf16, float* c2pad, void* stream);

/* ---- SoundStream.calculate_perp (models/vq_brain.py:238-243) --------------------------------- */
int fk_vq_perplexity(const long long* indices, long long N, int K, float* bins_ws, float* out, void* stream);

/* ---- SoundStream.custom_l1_loss (models/vq_brain.py:220-227) --------------------------------- */
long long fk_masked_l1_partials(long long R);
int fk_masked_l1_forward(const void* pred, int dtype, const float* gt, long long R, int C, unsigned char* row_valid,
                         float* part_sum, float* part_cnt, unsigned int* counter, float* loss, float* denom,
                         void* stream);
int fk_masked_l1_backward(const void* pred, int dtype, const float* gt, const unsigned char* row_valid,
                          const float* g_loss, const float* denom, long long R, int C, void* grad_pred, void* stream);

/* ---- transformer blocks (models/brainformer.py, models/simple_mae) ---------------------------- */
/* nn.LayerNorm (brainformer.py:237-239,287) / RMSNorm (simple_mae:181-192).  dtype codes 0=f32 1=bf16.
 * Supported (x, y): (f32,bf16) (f32,f32) (bf16,bf16).  mean/rstd: [M] fp32 saved for backward (mean unused for rms).
 * D % 4 == 0 and D <= 1024 (forward and backward, also for fk_add_norm_*). */
int fk_norm_forward(const void* x, int x_dtype, const float* weight, const float* bias, void* y, int y_dtype,
                    float* mean, float* rstd, long long M, int D, float eps, int rms, void* stream);
/* dw_part/db_part: [fk_norm_backward_grid(), D] partial sums (caller reduces over dim 0).
 * Supported (x, g, dx): (f32,bf16,f32) (f32,f32,f32) (bf16,bf16,bf16). */
int fk_norm_backward_grid(void);
/* dw [D] (and db [D] when db_part != NULL) = column sums of the [nb, D] partials, one launch, fixed order. */
int fk_norm_reduce_partials(const float* dw_part, const float* db_part, int nb, int D, float* dw, float* db, void* stream);
int fk_norm_backward(const void* x, int x_dtype, const void* g, int g_dtype, const float* weight, const float* mean,
                     const float* rstd, void* dx, int dx_dtype, float* dw_part, float* db_part, long long M, int D,
                     int rms, void* stream);
/* ---- helpers of the implicit-GEMM convolutions (models/vq_brain.py:22-45: F.pad on the time axis; bias gradients) ---- */
/* out [(total_rows), C] bf16: trial b's T rows at out[b * rows_per_trial + left ...], zeros everywhere else (causal left
 * padding, right padding, slack rows), in one pass.  x [B, T, C]: f32 (0) or bf16 (1), channels contiguous, strides in
 * elements (multiples of 8). */
int fk_pad_rows(const void* x, int x_dtype, long long B, long long T, int C, long long stride_b, long long stride_t,
                void* out, long long rows_per_trial, long long left, long long total_rows, void* stream);
/* The GEMM input rows of one streamed causal convolution (SoundStream.stream; models/vq_brain.py:22-63), fk_pad_rows' layout:
 * out [(total_rows), C] bf16, trial b's rows at out[b * rows_per_trial ...] are hist_in[b] (h rows), then act(x[b] + r[b])
 * (n rows), then zeros up to the next trial and in the slack rows.  x [B, n, C]: f32 (0) or bf16 (1); r (nullable) bf16
 * [B, n, C], the ResidualUnit input added to its 1x1 convolution's output; x + r is rounded to bf16, then act: 0 = none,
 * 1 = ELU (alpha 1, fp32, torch's x > 0 ? x : expm1(x)), then bf16.  Strides in elements (multiples of 8, token strides
 * >= C), channels contiguous.  hist_in / hist_out: bf16 [B, h, C], distinct buffers (nullable when h == 0); hist_out[b]
 * = the last h rows of [hist_in[b] | act(x[b] + r[b])], also when n < h. */
int fk_conv_stream_rows(const void* x, int x_dtype, long long x_sb, long long x_st, const void* r, long long r_sb,
                        long long r_st, const void* hist_in, void* hist_out, long long B, long long n, int h, int C,
                        int act, void* out, long long rows_per_trial, long long total_rows, void* stream);
/* fk_conv_stream_rows with per-trial counts of new rows (a step in which the trials received different amounts of data):
 * counts (nullable) int32 [B] at this convolution's input rate; trial b's new rows are the first c = counts[b] rows of x
 * (clamped to [0, n]).  Rows h + c ... of its GEMM input are zeros, x[b] past c and r[b] past c are never read, and
 * hist_out[b] = the last h rows of [hist_in[b] | the c new rows], so c = 0 copies hist_in[b] bit for bit.  NULL: every
 * trial has n new rows, which is fk_conv_stream_rows. */
int fk_conv_stream_rows_counts(const void* x, int x_dtype, long long x_sb, long long x_st, const void* r, long long r_sb,
                               long long r_st, const void* hist_in, void* hist_out, const int* counts, long long B,
                               long long n, int h, int C, int act, void* out, long long rows_per_trial, long long total_rows,
                               void* stream);
/* column sums of a bf16 [M, N] matrix (row stride ld): part [fk_colsum_grid(), N] fp32 per-CTA partials in a fixed order;
 * reduce them with fk_norm_reduce_partials(part, NULL, fk_colsum_grid(), N, out, NULL).  Bias gradient of nn.Linear /
 * nn.Conv1d (sum of dY over tokens). */
int fk_colsum_grid(void);
int fk_colsum_partials(const void* g, long long M, int N, long long ld, float* part, void* stream);

/* MLP gate silu(w1 x) * (w3 x) (brainformer.py:123-124) on the fused bf16 projection h13 [M, 2H]. */
int fk_swiglu_forward(const void* h13, void* y, long long M, int H, void* stream);
int fk_swiglu_backward(const void* h13, const void* gy, void* dh13, long long M, int H, void* stream);
/* the same derivative on the block-interleaved h13 / dh13 of fk_gemm_nt's SwiGLU epilogue ([w1 block | w3 block] per
 * `block` hidden units); gy [M, H] in hidden-unit order. */
int fk_swiglu_backward_blocked(const void* h13, const void* gy, void* dh13, long long M, int H, int block, void* stream);
/* apply_rope (brainformer.py:70-91) in place on bf16 [B,S,H,head_dim] (head_dim 16, 32 or 64, strides in elements); table
 * [P,head_dim/2,2] fp32 (cos,sin) = view_as_real(build_complex_rope_cache); pos (nullable) [B,S] int32 else position =
 * s + pos_offset. */
int fk_rope(void* x, long long bs, long long ts, int B, int S, int H, int head_dim, const float* table, int P,
            const int* pos, int pos_offset, int inverse, void* stream);
/* F.scaled_dot_product_attention(q,k,v,attn_mask) (brainformer.py:168,215) with the mask given as integer labels:
 * key j visible to query i  <=>  kid[b][j] <= qid[b][i]  (null = no mask).  q/k/v/out: bf16 [B,S,H,32] with
 * batch/token strides in elements.  qmin..kmax: per-64-token-tile label ranges from fk_attn_label_ranges.
 * lse: [B,H,Sq] fp32 (log2 domain), nullable in inference. */
int fk_attn_label_ranges(const int* ids, int B, int S, int* tmin, int* tmax, void* stream);
/* Positions of one streaming step whose trials sit at different positions (brainformer.EncoderStream after a per-row reset):
 * trial b holds len_in[b] tokens (int32 [B]) and appends n_new at positions p = len_in[b] + i, i < n_new.  One launch
 * writes qid [B, n_new] = p / tokens_per_label (the block-causal label of p) with its per-64-token tile ranges qmin / qmax
 * [B, ceil(n_new / 64)] (as fk_attn_label_ranges), pos [B, n_new] = p (RoPE positions), rows int64 [B, n_new] =
 * b * cap + p (flat rows of a [B, cap, ...] cache) and len_out[b] = len_in[b] + n_new (len_out a buffer other than len_in).
 * The caller keeps len_in[b] + n_new <= cap.  B in [1, 65535], n_new in [1, cap], tokens_per_label >= 1; anything else is
 * rejected before the launch. */
int fk_stream_positions(const int* len_in, int* len_out, int B, int n_new, int tokens_per_label, int cap, int* qid,
                        int* qmin, int* qmax, int* pos, long long* rows, void* stream);
/* fk_stream_positions with per-trial counts of new tokens (trials that received different amounts of data in one step):
 * counts (nullable) int32 [B], clamped to [0, n_new].  Slot i < counts[b] is written as above.  A slot at or past it gets
 * qid = INT_MIN (no key label >= 0 satisfies it: the query sees no key, and its tile ranges skip every key tile),
 * pos = min(p, cap - 1) (inside the RoPE table) and rows = B * cap, a scratch row past every trial's window (the caller's
 * cache holds B * cap + 1 rows); len_out[b] = len_in[b] + counts[b], and the caller keeps that <= cap.  NULL: every
 * trial has n_new new tokens, which is fk_stream_positions. */
int fk_stream_positions_counts(const int* len_in, const int* counts, int* len_out, int B, int n_new, int tokens_per_label,
                               int cap, int* qid, int* qmin, int* qmax, int* pos, long long* rows, void* stream);
/* fk_stream_positions_counts for ring caches of cap tokens per trial (a sliding stream with no end): trial b holds len_in[b]
 * tokens (int64 [B], unbounded) and its new slot i < c = counts[b] (nullable, clamped to [0, n_new]; NULL: n_new) is the
 * token at p = len_in[b] + i.  One launch writes qid [B, n_new] = p / tokens_per_label with its per-64-token tile ranges
 * qmin / qmax, rows int64 [B, n_new] = b * cap + p mod cap, the key label kid[b][p mod cap] = p / tokens_per_label of the
 * ring kid int32 [B, cap], the key tile ranges kmin / kmax [B, ceil(cap / 64)] of every 64-slot tile it wrote (recomputed
 * from the ring), the RoPE rows rope fp32 [B * n_new, half, 2] = (cos, sin)(p * inv_freq[j]) computed in fp64 and rounded
 * (inv_freq fp32 [half]) and len_out[b] = len_in[b] + c.  A slot at or past c gets qid = INT_MIN (sees no key), the scratch
 * row B * cap (the caller's cache holds B * cap + 1 rows) and the RoPE row of position 0.  The caller keeps
 * p / tokens_per_label inside int32 and cap large enough that no slot a query still sees is overwritten.  B in [1, 65535],
 * n_new in [1, cap], tokens_per_label >= 1, half >= 1; anything else is rejected before the launch. */
int fk_stream_ring_positions(const long long* len_in, const int* counts, long long* len_out, int B, int n_new,
                             int tokens_per_label, int cap, int* qid, int* qmin, int* qmax, long long* rows, int* kid,
                             int* kmin, int* kmax, const float* inv_freq, int half, float* rope, void* stream);
int fk_attn_forward(const void* q, const void* k, const void* v, void* out, float* lse, int B, int H, int Sq, int Sk,
                    int head_dim, long long q_bs, long long q_ts, long long k_bs, long long k_ts, long long v_bs,
                    long long v_ts, long long o_bs, long long o_ts, const int* qid, const int* kid, const int* qmin,
                    const int* qmax, const int* kmin, const int* kmax, float scale, void* stream);
/* delta: [B,H,Sq] fp32 workspace.  dq/dk/dv: bf16, same addressing scheme as q/k/v.
 * parts: bitmask of the kernels to launch, in this order: 1 = delta = rowsum(dO*O), 2 = dK/dV, 4 = dQ (7 = all). */
int fk_attn_backward(const void* q, const void* k, const void* v, const void* o, const void* d_o, const float* lse,
                     float* delta, void* dq, void* dk, void* dv, int B, int H, int Sq, int Sk, int head_dim,
                     long long q_bs, long long q_ts, long long k_bs, long long k_ts, long long v_bs, long long v_ts,
                     long long o_bs, long long o_ts, long long do_bs, long long do_ts, long long dq_bs, long long dq_ts,
                     long long dk_bs, long long dk_ts, long long dv_bs, long long dv_ts, const int* qid, const int* kid,
                     const int* qmin, const int* qmax, const int* kmin, const int* kmax, float scale, int parts, void* stream);

/* tcgen05 / TMEM / TMA version of the attention backward (attention_tc.cu), head_dim 16, 32 or 64 (q/k/v/d_o/dq/dk/dv:
 * bf16 [B,S,H,head_dim], strides in elements; any other head_dim is rejected before anything is launched).  At head_dim 16
 * and 64 there is one path: aug from fk_attn_aug is required, qt = kt = dot = NULL, no stall accounting, gradient strides % 8 == 0.
 * qt = kt = dot = NULL (default): the
 * contractions over tokens read the Q / dO / K tiles MN-major straight from the strided inputs.  Cross-check mode:
 * fk_attn_transpose makes [B][H][32][Sp] copies (zero padded, Sp % 8 == 0) that serve as K-major operands instead:
 * qt, dot for dK/dV (parts & 2), kt for dQ (parts & 4).  delta must already hold rowsum(dO*O)
 * (fk_attn_backward with parts = 1).  Same labels / ranges / strides conventions as fk_attn_backward; Sq == Sk == S.
 * The kernels are persistent (one CTA per SM taking work items from a hand-out counter).  The counter words belong to
 * the CALLER: `counters` = 4 uint32 (2 per part), zero on entry; the last CTA of a launch puts them back to zero, so the
 * same words can serve every launch on one stream, and launches that may overlap (different streams / graph branches) must
 * be given different words.  The library itself holds no device-side state: every entry point is re-entrant per stream. */
int fk_attn_transpose(const void* x, long long bs, long long ts, int B, int S, int H, int head_dim, void* xt, int Sp,
                      void* stream);
/* fk_attn_aug: o / d_o bf16 [B,S,H,head_dim] (head_dim 16, 32 or 64);
 * delta [B,H,S] = rowsum(dO * O) and the statistics rows aug (bf16 [B,H,S,16], 32-byte aligned): -lse / c
 * and -delta as three bf16 terms each.  Passed to fk_attn_backward_tc as `aug` (nullable), they enter the score MMAs as one
 * more K step, so S - lse / c and dP - delta leave the tensor core and the compute warps neither stage nor subtract the
 * statistics (aug = NULL: the statistics are read from lse / delta as before). */
int fk_attn_aug(const void* o, const void* d_o, const float* lse, float* delta, void* aug, int B, int H, int S,
                int head_dim, long long o_bs, long long o_ts, long long do_bs, long long do_ts, float scale, void* stream);
int fk_attn_backward_tc(const void* q, const void* k, const void* v, const void* d_o, const void* qt, const void* kt,
                        const void* dot, int Sp, const float* lse, const float* delta, const void* aug, void* dq, void* dk, void* dv,
                        int B, int H, int S, int head_dim, long long q_bs, long long q_ts, long long k_bs,
                        long long k_ts, long long v_bs, long long v_ts, long long do_bs, long long do_ts,
                        long long dq_bs, long long dq_ts, long long dk_bs, long long dk_ts, long long dv_bs,
                        long long dv_ts, const int* qid, const int* kid, const int* qmin, const int* qmax,
                        const int* kmin, const int* kmax, float scale,
                        const float* rope_table /* [rope_len][head_dim/2][2] (cos, sin) or NULL: dq / dk are rotated back (the gradient of
                                                   apply_rope, brainformer.py:70-91) inside the kernel */,
                        int rope_len, const int* rope_pos /* [B][S] or NULL */, int rope_offset, int parts,
                        unsigned int* counters, void* stream);
/* Diagnosis only (scripts/gpu_attn_stalls.py): the same launch through a stall-accounting build of the kernel that writes
 * int64 [n_items, 24] cycle counters to prof (see attention_tc.cu); prof_mode 1 = full stall accounting, 2 = lifetime +
 * %globaltimer + %smid only.  prof == NULL behaves exactly like fk_attn_backward_tc. */
int fk_attn_backward_tc_profile(const void* q, const void* k, const void* v, const void* d_o, const void* qt,
                                const void* kt, const void* dot, int Sp, const float* lse, const float* delta, const void* aug,
                                void* dq, void* dk, void* dv, int B, int H, int S, int head_dim, long long q_bs, long long q_ts,
                                long long k_bs, long long k_ts, long long v_bs, long long v_ts, long long do_bs,
                                long long do_ts, long long dq_bs, long long dq_ts, long long dk_bs, long long dk_ts,
                                long long dv_bs, long long dv_ts, const int* qid, const int* kid, const int* qmin,
                                const int* qmax, const int* kmin, const int* kmax, float scale, const float* rope_table,
                                int rope_len, const int* rope_pos, int rope_offset, int parts, unsigned int* counters,
                                long long* prof, int prof_mode, void* stream);

/* tcgen05 / TMEM / TMA forward (attention_tc.cu): q / k / v are strided views ([B][S][H][head_dim], head_dim 16, 32 or 64,
 * strides in elements; any other head_dim is rejected before anything is launched);
 * the V tile is read MN-major by the P V MMAs, so no transposed copy is needed; Sq == Sk == S.
 * Labels: any int32 value is valid in qid and kid, INT32_MIN and INT32_MAX included (a query labelled INT32_MAX sees every
 * key); the key positions past S of the last tile are masked by position, not by a reserved label.
 * counters: 2 caller-owned uint32, zero on entry, zero again on exit (see fk_attn_backward_tc). */
int fk_attn_forward_tc(const void* q, const void* k, const void* v, void* out, float* lse, int B, int H, int S,
                       int head_dim, long long q_bs, long long q_ts, long long k_bs, long long k_ts, long long v_bs,
                       long long v_ts, long long o_bs, long long o_ts, const int* qid, const int* kid, const int* qmin,
                       const int* qmax, const int* kmin, const int* kmax, float scale, unsigned int* counters,
                       void* stream);
/* The same forward for queries and keys of different lengths (inference against a key / value cache, e.g. one streaming
 * step of brainformer.Encoder): q [B][Sq][H][head_dim], k / v [B][Sk][H][head_dim] bf16 strided views (all strides % 8 == 0,
 * token strides >= H * head_dim), head_dim 16, 32 or 64; labels qid [B, Sq], kid [B, Sk] with the ranges of
 * fk_attn_label_ranges for each side; any other head_dim, Sq < 1, Sk < 1 or bad strides are rejected before anything is
 * launched (counters untouched).  Work item = (256-query block, key chunk, head, trial): the key axis is cut into n_chunks
 * chunks of ceil(key tiles / n_chunks) 128-key tiles (1 <= n_chunks <= ceil(Sk / 128); fk_attn_kv_chunks picks enough to
 * fill max_ctas CTAs, <= 0: all SMs).  n_chunks == 1 runs the unsplit kernel (part_o / part_ml unused).  Otherwise each item
 * writes unnormalised partials, part_o fp32 [B, H, n_chunks, Sq, head_dim] and part_ml fp32 [B, H, n_chunks, Sq, 2] (running
 * maximum and sum, log2 domain), and a second launch merges them in chunk order (bit-reproducible).  out bf16; lse
 * [B, H, Sq] (log2 domain) nullable; a query that sees no key gives a zero row.  counters: as fk_attn_forward_tc.
 * Every k / v row below Sk must hold finite values, also rows no query sees: a tile that is only partly visible multiplies
 * P = 0 by every V row of the tile, and 0 * NaN or 0 * inf would reach the output.  (A cache of trials at different
 * lengths therefore starts zeroed; rows left by an earlier session are finite.) */
int fk_attn_kv_chunks(int B, int H, int Sq, int Sk, int max_ctas);
int fk_attn_forward_kv_tc(const void* q, const void* k, const void* v, void* out, float* lse, int B, int H, int Sq, int Sk,
                          int head_dim, long long q_bs, long long q_ts, long long k_bs, long long k_ts, long long v_bs,
                          long long v_ts, long long o_bs, long long o_ts, const int* qid, const int* kid, const int* qmin,
                          const int* qmax, const int* kmin, const int* kmax, float scale, float* part_o, float* part_ml,
                          int n_chunks, unsigned int* counters, void* stream);
/* fk_attn_forward_kv_tc with a label band (a sliding window over labels): key j is visible to query i iff
 * kid[b][j] <= qid[b][i] and qid[b][i] - kid[b][j] < band, the difference taken in 64 bits, so INT32_MIN and INT32_MAX stay
 * valid labels.  band >= 1; a band of 2^32 or more lets every difference of two int32 labels through and is no band, which
 * is fk_attn_forward_kv_tc bit for bit.  A narrower band needs labels and runs the split kernel even at n_chunks == 1, so
 * part_o / part_ml are then required at every chunk count; the unsplit kernels never see a band.  band < 1 is rejected
 * before anything is launched (counters untouched). */
int fk_attn_forward_kv_band_tc(const void* q, const void* k, const void* v, void* out, float* lse, int B, int H, int Sq,
                               int Sk, int head_dim, long long q_bs, long long q_ts, long long k_bs, long long k_ts,
                               long long v_bs, long long v_ts, long long o_bs, long long o_ts, const int* qid,
                               const int* kid, const int* qmin, const int* qmax, const int* kmin, const int* kmax,
                               float scale, float* part_o, float* part_ml, int n_chunks, long long band,
                               unsigned int* counters, void* stream);

/* Fused residual add + norm on the fp32 residual stream: x_out = x + delta (bf16), y = norm(x_out)
 * (the pair `x = x + branch(...)`; `ln(x)` of models/brainformer.py:243-244).  Backward: dx = norm_backward(g_y) + g_res
 * (g_res nullable = gradient reaching x_out through the residual path), written as fp32 and, if dx_bf16 != NULL, as a
 * bf16 copy for the delta branch.  y / g_y dtype codes as fk_norm_forward. */
int fk_add_norm_forward(const float* x, const void* delta_bf16, const float* weight, const float* bias, float* x_out,
                        void* y, int y_dtype, float* mean, float* rstd, long long M, int D, float eps, int rms,
                        long long x_period /* > 0: x has x_period rows, broadcast over the batch (brainformer.py:343) */,
                        void* stream);
int fk_add_norm_backward(const float* x_new, const void* g_y, int g_dtype, const float* g_res, const float* weight,
                         const float* mean, const float* rstd, float* dx, void* dx_bf16, float* dw_part, float* db_part,
                         long long M, int D, int rms, void* stream);

/* ---- dense bf16 GEMMs with fused epilogues (gemm.cu; tcgen05 / TMEM / TMA) ----------------------- */
/* C[M,N] (bf16) = A[M,K] (bf16, row-major, lda) x B[N,K]^T (bf16, row-major, ldb = an nn.Linear weight), fp32 accumulate.
 * Replaces the nn.Linear calls of models/brainformer.py:119-124 (MLP), :141-145,171 (qw/kw/vw fused, project), :285 (emb)
 * and, on transposed weight copies, their input gradients.  K % 8 == 0, N % 32 == 0.  K <= 512 runs the A-resident
 * kernel (all epilogues); longer K the streaming kernel (epilogue 0 only).  epilogue:
 *   0  C = A B^T (+ bias[N], nullable)
 *   1  apply_rope (brainformer.py:70-91) on columns [0, rope_cols) of C (heads of 32 columns; q | k of the fused
 *      projection): rope_table [rope_len][16][2] (cos, sin), position of row m = rope_pos ? rope_pos[m]
 *      : (m % rope_S) + rope_offset
 *   2  SwiGLU forward: B = w1 / w3 interleaved in blocks of 128 rows ([w1[0:128]; w3[0:128]; w1[128:256]; ...], N = 2 x
 *      hidden); writes the fused projection C = h13 [M, N] and C2 = gated [M, N/2] = silu(h1) * h3 (brainformer.py:123-124)
 *   3  removed (was the SwiGLU backward; rejected): d gated on epilogue 0, then fk_swiglu_backward_blocked
 *   4  as 1 for heads of 64 columns: rope_table [rope_len][32][2], rope_cols % 64 == 0
 *   5  as 1 for heads of 16 columns: rope_table [rope_len][8][2], rope_cols % 32 == 0 */
int fk_gemm_nt(const void* A, long long lda, const void* B, long long ldb, void* C, long long ldc, long long M, int N,
               int K, const float* bias, int epilogue, void* C2, long long ldc2, const float* rope_table, int rope_len,
               const int* rope_pos, int rope_offset, int rope_cols, int rope_S, void* stream);
/* out[Na,Nb] (fp32) = A[M,Na]^T x B[M,Nb] (bf16, row-major): the weight gradient dW = dY^T X of an nn.Linear.  The M rows
 * are cut into `splits` = fk_gemm_tn_splits(M, Na, Nb, 0) ranges whose partial sums go to ws (fp32 [splits, Na, Nb]) and
 * are added in a fixed order (bit-reproducible).  Na % 64 == 0, Nb % 64 == 0.  max_ctas <= 0: the SM count. */
int fk_gemm_tn_splits(long long M, int Na, int Nb, int max_ctas);
int fk_gemm_tn(const void* A, long long lda, const void* B, long long ldb, float* out, long long M, int Na, int Nb,
               float* ws, int splits, void* stream);

/* Patch embedding of brainformer.Encoder (brainformer.py:282 to_patches, :285 Linear(patch -> dim) + bias, :343 + electrode
 * embedding): x bf16 [n_rows = B * T, E] row-major (ldx), token (b, t, c) = x[b*T + t*patch .. + patch, c];
 * wt = W^T bf16 [patch, dim]; bias fp32 [dim] (nullable); emb fp32 [E, dim] (nullable) added per electrode;
 * out bf16 [n_rows / patch * E, dim] = token-major 'b (t c) d'.  The [B, S, patch] patch tensor is never materialised: TMA reads
 * x as the MN-major operand of a tcgen05 contraction over the patch's bins.  patch in {16, 32, 48, 64}, E % 64 == 0, dim % 64 == 0. */
int fk_patch_embed_forward(const void* x_bf16, long long ldx, const void* wt_bf16, const float* bias, const float* emb,
                           void* out_bf16, long long n_rows, int E, int patch, int dim, void* stream);

/* ---- input pipeline on the device (utils/data_utils.py; SURVEY 8f row N3) ------------------------------------------------
 * Ragged trials stored back to back: volt [sum_T, C1] fp32 (spike power), spk [sum_T, C2] fp32 (threshold crossings; C2 = 0
 * and spk = null for already concatenated data), offsets [n_trials + 1] int64 first row of each trial, block_id [n_trials]
 * int32 dense recording-block ids in [0, n_blocks).  C1 % 4 == 0, C2 % 4 == 0.
 *
 * fk_input_trial_moments: part [n_trials, C1 + C2] fp64 = per trial and channel sum of x (mean == null) or of
 *   (x - mean[block])^2 (mean = fp64 [n_blocks, C] from pass 0).
 * fk_input_block_reduce: adds the trials' partial sums per block in trial order.  pass 0 -> mean_d (fp64) and mean_f
 *   (fp32); pass 1 -> std_f (population std, as np.std / StandardScaler) with zero_policy 0: std == 0 -> 1
 *   (process_signal, data_utils.py:142) or 1: std < 10 eps -> 1 (StandardScaler, z_score_per_block_scaling :78-109).
 * fk_input_normalize: out [n_trials, T_out, C1 + C2] (out_dtype 0 = f32, 1 = bf16) = (x - mean) / std per block, smoothed
 *   over the trial's own bins with scipy's gaussian_filter1d(sigma = 1) when smooth != 0 (process_signal :115-156),
 *   zero padded / truncated to T_out bins (pad_truncate_brain_list :243-267). */
int fk_input_trial_moments(const float* volt, const float* spk, const long long* offsets, const int* block_id,
                           int n_trials, int C1, int C2, const double* mean, double* part, void* stream);
int fk_input_block_reduce(const double* part, const long long* offsets, const int* block_id, int n_trials, int n_blocks,
                          int C, int pass, int zero_policy, double* mean_d, float* mean_f, float* std_f, void* stream);
int fk_input_normalize(const float* volt, const float* spk, const long long* offsets, const int* block_id, const float* mean,
                       const float* stdv, int n_trials, int C1, int C2, int T_out, int smooth, void* out, int out_dtype,
                       void* stream);

/* ---- attention with few queries: the perceiver resampler (brainformer.py:175-219, :247-268; SURVEY 8f row N2) --------------
 * softmax(q k^T * scale) v for Tq <= 64 queries per (trial, head) against S keys, head_dim 16 / 32 / 64, no mask, bf16
 * [B, T, H, head_dim] operands with batch / token strides in elements (token strides % 8 == 0).  rope_table (nullable):
 * [rope_len, head_dim / 2, 2] fp32 (cos, sin); q row t is rotated by position rope_q0 + t, k row j by rope_k0 + j
 * (apply_rope, brainformer.py:70-91) and dq / dk are rotated back.  The key axis is split into
 * fk_small_attn_chunks(S) chunks of 256: part_o fp32 [B, H, chunks, Tq, head_dim], part_ml fp32 [B, H, chunks, Tq, 2],
 * part_dq like part_o; partials are merged in chunk order (deterministic).  lse [B, H, Tq] in the log2 domain.
 * k_len (forward only, nullable): int32 [B] per-trial key counts (a key / value cache whose trials hold different numbers
 * of tokens): key j of trial b takes part iff j < min(S, k_len[b]); a chunk past that writes the empty partial (m = -inf,
 * l = 0, O = 0), which the merge passes over exactly, and a trial with no key gets a zero row (lse = +inf).  Keys past
 * k_len[b] are never read.  NULL: every trial has S keys. */
int fk_small_attn_chunks(int S);
int fk_small_attn_forward(const void* q, long long q_bs, long long q_ts, const void* k, long long k_bs, long long k_ts,
                          const void* v, long long v_bs, long long v_ts, void* out, long long o_bs, long long o_ts,
                          float* lse, int B, int H, int Tq, int S, int head_dim, float scale, const float* rope_table,
                          int rope_len, int rope_q0, int rope_k0, float* part_o, float* part_ml, const int* k_len,
                          void* stream);
int fk_small_attn_backward(const void* q, long long q_bs, long long q_ts, const void* k, long long k_bs, long long k_ts,
                           const void* v, long long v_bs, long long v_ts, const void* out, long long o_bs, long long o_ts,
                           const void* dout, long long do_bs, long long do_ts, const float* lse, void* dq, void* dk,
                           void* dv, int B, int H, int Tq, int S, int head_dim, float scale, const float* rope_table,
                           int rope_len, int rope_q0, int rope_k0, float* part_dq, void* stream);

/* ---- encoder -> GPT-2 prefix hand-off (models/gpt2_model.py:178-196; SURVEY 8f row N2) -------------------------------------
 * out [B, Tc + T, D] = cat([prefix [B, Tc, D], wte[idx [B, T]]], dim 1) + wpe[0 .. Tc + T); wte [V, D], wpe [P, D] fp32;
 * prefix / out dtype 0 = f32, 1 = bf16; idx int64.  Backward: g [B, Tc + T, D] fp32 -> dwte [V, D] += scatter of the token
 * rows (fp32 atomics), dwpe [P, D] rows [0, Tc + T) += sum over the batch; d prefix is the view g[:, :Tc]. */
int fk_prefix_embed_forward(const void* prefix, int prefix_dtype, const long long* idx, const float* wte, const float* wpe,
                            void* out, int out_dtype, int B, int Tc, int T, int D, int V, int P, void* stream);
int fk_prefix_embed_backward(const float* g, const long long* idx, float* dwte, float* dwpe, int B, int Tc, int T, int D,
                             int V, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FK_B200_H */
