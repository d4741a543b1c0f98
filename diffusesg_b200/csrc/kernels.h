// Host-side launchers of every kernel in libdsg_b200.so (internal header).
//
// Conventions: all pointers are device pointers unless stated; "tokens" are the pixels of the
// N x N node-pair grid flattened row-major (token = i * res + j) and batched sample-major, so an
// activation is a row-major [B*L, C] matrix with the channel contiguous.  Launchers never allocate
// and never synchronise; they return 0 or a DSG_ERR_* code (see common.cuh).
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace dsg {

typedef __nv_bfloat16 bf16;

// ---------------------------------------------------------------------------------------------
// tcgen05 GEMM:  out[M, N] = epilogue(A[M, K] . W[N, K]^T)          (gemm.cu)
// ---------------------------------------------------------------------------------------------
enum GemmEpi : int {
  EPI_BF16 = 0,       // out bf16 = acc + bias
  EPI_GELU_BF16 = 1,  // out bf16 = gelu_erf(acc + bias)
  EPI_RES_F32 = 2,    // out f32 += acc + bias                  (in place: res == out)
  EPI_F32 = 3,        // out f32  = acc + bias
  EPI_ADJ_HEAD = 4,   // h = gelu(acc + bias) [N == 96]; y = W2 h + b2; masked (+ EDM precond) -> [B, Ce, n, n]
};

struct GemmParams {
  int M, N, K;
  const float* bias;   // [N] or nullptr
  const float* res;    // [M, ldo] fp32 (EPI_RES_F32)
  void* out;           // [M, ldo] bf16 / fp32; EPI_ADJ_HEAD: float [B, c_e, n, n]
  int ldo;
  int bn;              // tile width: 0 = gemm_block_n(N); 256 needs N % 256 == 0 and a W descriptor with that box
  int ksplit;          // launch_wgrad only, > 1: split the contraction into that many slices per output tile
  int scale_rows;      // weight-gradient GEMM: output rows < scale_rows are multiplied by row_scale (the q third of qkv)
  float row_scale;
  // EPI_ADJ_HEAD only
  const float* w2t;    // [96][8]: second layer of the adj read-out MLP, transposed and zero padded
  const float* b2;     // [8]
  int c_e;             // real output channels (<= 8)
  int n_img;           // N; a GEMM row m is pixel (b, i, j) = (m / N^2, (m / N) % N, m % N)
  const uint8_t* flags;  // [B, N] node validity
  const float* x_adj;    // preconditioning: D = c_skip * x + c_out * F; nullptr -> raw F
  const float* c_skip;   // [B]
  const float* c_out;    // [B]
  const int* perm;       // compact layout (padding skipping): the rows are a stack of side x side corners, image k =
  int side;              //   sample perm[k] (< 0: phantom, nothing is stored).  nullptr: dense rows
};

// Encode a TMA descriptor for a row-major bf16 matrix [rows, cols] (cols contiguous), box = 64 cols x
// box_rows rows, 128-byte swizzle.  Pure host work (driver entry point), no stream interaction.
int make_tmap_bf16(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int box_rows);
// Output descriptor of a GEMM with epilogue `epi`: [rows, cols] bf16 / fp32, box = 32 cols x 128 rows
// (64-byte swizzle for bf16, 128-byte for fp32).  Not used by EPI_ADJ_HEAD.
int make_tmap_out(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int epi);

// Weight gradient dW [n_out, out_cols] += dY^T . X with dY [tokens, n_out], X [tokens, x_cols] read as MN-major operands
// straight from their row-major tensors (no transposes), contraction over the tokens split into `ksplit` slices.
int launch_wgrad(const void* dy, const void* x, float* dw, long long tokens, int n_out, int x_cols, int out_cols, int ksplit,
                 int scale_rows, float row_scale, cudaStream_t st);

// N must be a multiple of 96; K a multiple of 32; rows beyond M are neither read as valid nor written.
// box_rows of the W descriptor must equal gemm_block_n(N).
int gemm_block_n(int N);
// Tile width the schedule uses for a [rows x N x K] GEMM: 256-wide tiles (16 % fewer operand bytes per flop through the
// SM's shared memory than 192-wide ones) where N divides, the K loop is long enough and the waves stay full.
int gemm_choose_bn(long long rows, int N, int K, int epi, bool pair);
// Whether a GEMM of `rows` rows, contraction K and epilogue `epi` runs on CTA pairs (cta_group::2, 256-row tiles).
bool gemm_use_pair(long long rows, int K, int epi);
// EPI_RES_F32 accumulates in place with a TMA reduce-add: p.res must alias p.out.
// pair = true runs CTA pairs (cta_group::2, 256-row tiles): tmW must then have box_rows = gemm_block_n(N) / 2.
int launch_gemm(const CUtensorMap* tmA, const CUtensorMap* tmW, const CUtensorMap* tmO, int epi, const GemmParams& p,
                cudaStream_t st, bool pair = false);

// ---------------------------------------------------------------------------------------------
// fused MLP:  x += fc2(gelu(fc1(y))), y = LN(x) in bf16                 (mlp.cu)
// ---------------------------------------------------------------------------------------------
// Built for C = 96 and 192 (hidden 4C).  tmY: y [rows, C] bf16, box 64 x 128 (make_tmap_bf16); tmW1: fc1.weight
// [4C, C] bf16, box 64 x fused_mlp_w1_box_rows(C); tmW2: fc2.weight [C, 4C] bf16, box 64 x C; tmX: x [rows, C] fp32
// output descriptor (make_tmap_out, EPI_RES_F32).
bool fused_mlp_supported(int C);
int fused_mlp_w1_box_rows(int C);
int launch_fused_mlp(const CUtensorMap* tmY, const CUtensorMap* tmW1, const CUtensorMap* tmW2, const CUtensorMap* tmX,
                     const float* b1, const float* b2, long long rows, int C, cudaStream_t st);

// ---------------------------------------------------------------------------------------------
// fused block tail:  x += proj(att) + b_p;  x += fc2(gelu(fc1(LN2(x)) + b1)) + b2     (blocktail.cu)
// ---------------------------------------------------------------------------------------------
// Built for C = 96.  tmAtt: att [rows, C] bf16, box 32 x 128 (64-byte swizzle); tmWp: proj.weight [C, C] bf16, box
// 32 x C; tmW1: fc1.weight [4C, C] bf16, box 32 x 128; tmW2: fc2.weight [C, 4C] bf16, box 64 x C (128-byte swizzle);
// tmX: x [rows, C] fp32, box 32 x 128 (make_tmap_out, EPI_RES_F32); x: the same buffer, written in place.
int make_tmap_2d(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int elem_bytes, int box_cols,
                 int box_rows);
bool block_tail_supported(int C);
int launch_block_tail(const CUtensorMap* tmAtt, const CUtensorMap* tmWp, const CUtensorMap* tmW1,
                      const CUtensorMap* tmW2, const CUtensorMap* tmX, const float* bp, const float* gamma,
                      const float* beta, const float* b1, const float* b2, float* x, long long rows, int C,
                      cudaStream_t st, const CUtensorMap* tmY = nullptr,
                      const float* gamma_f = nullptr, const float* beta_f = nullptr);
// tmY / gamma_f / beta_f (all or none): the LAST block of the network - the kernel applies the final LayerNorm
// (:758) to the block output and stores only y = LN(x) as bf16 through tmY ([M, C] bf16, 32-column boxes); x is not
// written back.

// ---------------------------------------------------------------------------------------------
// fused attention projection + residual + LayerNorm2 for C = 192 / 384 (projln.cu):
//   x += att W_proj^T + b_proj (in place, fp32);  y = LN(x) gamma + beta (bf16).  tmA: [rows, C] bf16, box 64 x 128;
//   tmW: the proj weight [C, C] bf16, box 64 x 192 (= gemm_block_n(C)).
// ---------------------------------------------------------------------------------------------
bool proj_ln_supported(int C);
int launch_proj_ln(const CUtensorMap* tmA, const CUtensorMap* tmW, const float* bias, const float* gamma, const float* beta,
                   float* x, bf16* y, long long rows, int C, cudaStream_t st);

// ---------------------------------------------------------------------------------------------
// fused block head:  x = silu(FiLM(x));  qkv = LN1(x) W_qkv^T + b_qkv                     (blockhead.cu)
// ---------------------------------------------------------------------------------------------
// Built for C = 96.  tmXin / tmXout: x [rows, C] fp32 in / out (make_tmap_out, EPI_F32; may be the same buffer);
// tmW: qkv.weight [3C, C] bf16, box 32 x C (64-byte swizzle); tmQ: qkv [rows, 3C] bf16 (make_tmap_out, EPI_BF16).
bool block_head_supported(int C);
int launch_block_head(const CUtensorMap* tmXin, const CUtensorMap* tmXout, const CUtensorMap* tmW, const CUtensorMap* tmQ,
                      const float* film, int film_ld, int cond_uniform, int tokens_per_sample, const float* gamma,
                      const float* beta, const float* bqkv, long long rows, int C, cudaStream_t st);

// ---------------------------------------------------------------------------------------------
// shifted-window attention                                             (attention.cu)
// ---------------------------------------------------------------------------------------------
// qkv [B*res*res, 3*C] bf16 (q pre-scaled through the packed weights), layout per token [3][heads][32];
// bias [heads, T, T] fp32 = gathered relative-position bias; mask [nW, T, T] fp32 (0 / -100) for shifted blocks,
// nullptr otherwise; out [B*res*res, C] bf16 at the un-shifted token positions.
int make_tmap_3d_bf16(CUtensorMap* map, const void* base, int64_t d0, int64_t d1, int64_t d2, int64_t s1, int64_t s2, int b0,
                      int b1, int b2);
// tcgen05 version for un-shifted 8 x 8 windows (attention_tc.cu): two windows per 128-row MMA tile, scores and
// probabilities in tensor memory.  Returns DSG_ERR_INVALID for shapes it does not take.
bool window_attention_tc_supported(int batch, int res, int window, int shift, int heads);
int launch_window_attention_tc(const bf16* qkv, const float* bias, bf16* out, int batch, int res, int shift, int heads,
                               cudaStream_t st);
// several stacks of square grids in one launch (the buckets of the padding skipping): group g = counts[g] grids of
// res[g] x res[g] tokens starting at token tok_off[g]; un-shifted windows, an even number of windows per group, <= 4 groups
int launch_window_attention_tc_groups(const bf16* qkv, const float* bias, bf16* out, int n_groups, const int* counts,
                                      const int* res, const long long* tok_off, int heads, cudaStream_t st);
// quad-box tcgen05 version (one window per tile): even windows up to 10 x 10, shift 0 or window / 2; the SW-MSA mask
// is generated in the kernel, so a shifted block may only take it when check_mask_canonical() found the model's
// attn_mask buffer equal to the reference's construction (synchronous; called at model finalisation).
bool window_attention_quad_supported(int batch, int res, int window, int shift, int heads);
int launch_window_attention_quad(const bf16* qkv, const float* bias, bf16* out, int batch, int res, int window, int shift,
                                 int heads, cudaStream_t st);
int check_mask_canonical(const float* mask, int res, int window, int shift, cudaStream_t st, int* canonical);
// 16 x 16 windows (T = 256): query halves of 128 rows against 256 keys, bias looked up from the head's offset table;
// needs check_bias_toeplitz() (bias[h][q][k] depends on the token offset only; synchronous, at finalisation).
bool window_attention_w16_supported(int batch, int res, int window, int shift, int heads);
int launch_window_attention_w16(const bf16* qkv, const float* bias, bf16* out, int batch, int res, int shift, int heads,
                                cudaStream_t st);
int check_bias_toeplitz(const float* bias, int heads, int window, cudaStream_t st, int* toeplitz);
// canonical: bit 0 = `mask` is known to hold the reference's SW-MSA values (ignored for un-shifted blocks),
//            bit 1 = `bias` is known to be a function of the token offset
enum { ATTN_MASK_CANONICAL = 1, ATTN_BIAS_TOEPLITZ = 2 };
int launch_window_attention(const bf16* qkv, const float* bias, const float* mask, bf16* out, int batch, int res,
                            int window, int shift, int heads, cudaStream_t st, int canonical = 0);

// ---------------------------------------------------------------------------------------------
// row kernels: LayerNorm / FiLM / merge / breakup / embed / heads       (rowops.cu)
// ---------------------------------------------------------------------------------------------
// x_out = silu(shift_b + x_in * (1 + scale_b)); y = LN(x_out) * g + b  (bf16).  film [n_cond, film_ld]
// holds (scale[C], shift[C]) at column film_off; sample s uses row (cond_uniform ? 0 : s).
int launch_film_ln(const float* x_in, float* x_out, bf16* y, const float* film, int film_ld, int film_off,
                   int cond_uniform, const float* gamma, const float* beta, int batch, int tokens_per_sample,
                   int C, cudaStream_t st, const int* src_rows = nullptr);
// src_rows [rows]: output row r reads input row src_rows[r] (layout changes of the padding skipping; not in place)
int launch_ln(const float* x, bf16* y, const float* gamma, const float* beta, int64_t rows, int C, cudaStream_t st);
// PatchMerging front half: gather the 2x2 neighbourhood (order (0,0),(1,0),(0,1),(1,1)), LN(4C) -> bf16; C = 96, 192, 384
int launch_merge_ln(const float* x, bf16* y, const float* gamma, const float* beta, int batch, int res, int C,
                    cudaStream_t st);
// PatchBreakup input: y[m, 0:C] = bf16(x[m]), y[m, C:2C] = bf16(skip[m])
int launch_concat_bf16(const float* x, const float* skip, bf16* y, int64_t rows, int C, cudaStream_t st,
                       const int* skip_rows = nullptr);   // skip_rows: row r reads skip row skip_rows[r]
// PatchBreakup middle: LN(D) over each row of t [B*res*res, D], split into 4 chunks of D/4, chunk k goes to
// pixel (2y + k%2, 2x + k/2) of the 2res x 2res grid, LN(D/4) -> bf16 [B*4*res*res, D/4]; D = 384, 768, 1536
int launch_breakup_ln(const float* t, bf16* y, const float* g1, const float* b1, const float* g2, const float* b2,
                      int batch, int res, int D, cudaStream_t st, const int* tok0 = nullptr, const int* width = nullptr,
                      int sh = 0, const int* src_perm = nullptr);
// tok0 / width (both or neither): y is a compact layout of the padding skipping (model.cu) in which sample b is a
// (width[b] >> sh)^2 image starting at token tok0[b] >> 2 sh; only the children inside it are written.  src_perm: t is
// itself a compact stack whose image b shows sample src_perm[b] (< 0: the phantom, no children); nullptr: sample b

// sigma conditioning: noise_labels [n_cond] -> emb [n_cond, 512] -> film [n_cond, film_total]
// scratch: emb0 [n_cond, embed], emb1 [n_cond, 512], emb [n_cond, 512]
int launch_cond(const float* noise_labels, long long label_stride, int n_cond, const float* w0, const float* b0, const float* w1,
                const float* b1, const float* w_film, const float* b_film, int film_total, float* emb0, float* emb1,
                float* emb, float* film, int embed, cudaStream_t st);

// per-sample EDM coefficients from sigma: coef[0..3][B] = c_in, c_skip, c_out, c_noise
int launch_precond_coef(const float* sigmas, int sigma_stride, float* coef, int batch, cudaStream_t st);

// node row/col projections of the patch embedding: rc[b, i, 0:E] = W_row . nodecat[b, i], rc[b, i, E:2E] = W_col . nodecat
int launch_node_proj(const float* node, const float* sc_node, const float* in_scale, const float* w_rc,
                     float* rc, int batch, int n, int c_n, int self_cond, int embed, cudaStream_t st);
// patch embed + LN + FiLM-SiLU -> x0 [B*n*n, E] fp32
int launch_patch_embed(const float* adj, const float* sc_adj, const float* in_scale, const uint8_t* flags,
                       const float* rc, const float* w_adj, const float* bias, const float* gamma,
                       const float* beta, const float* film, int film_ld, int film_off, int cond_uniform,
                       float* x0, int batch, int n, int c_e, int self_cond, int embed, cudaStream_t st,
                       const int* perm = nullptr, int side = 0);
// perm / side: compact layout of the padding skipping (model.cu): x0 is a stack of `batch` corners of side x side
// pixels, image k showing the top-left corner of sample perm[k] (-1 = the all-padding phantom)
// node head: masked row mean of y = LN(x) [B*n*n, E] bf16 -> folded read_out -> MLP -> (precond) -> out_node [B, n, c_n]
// fold_t [E][E], w1t [E][E] and w2t [E][c_n] are transposed (input-channel major)
int launch_node_head(const bf16* rep, const uint8_t* flags, const float* fold_t, const float* fold_b, const float* w1t,
                     const float* b1, const float* w2t, const float* b2, const float* x_node, const float* c_skip, const float* c_out,
                     float* out_node, int batch, int n, int c_n, int embed, cudaStream_t st, const int* tok0 = nullptr,
                     const int* width = nullptr, float* scratch = nullptr);
// scratch [B n, 128] fp32: with it (embed 96, c_n <= 32) the head runs as two kernels - masked row sums, then the MLP
// for 32 rows per CTA with the weights in shared memory; without it, the single-kernel version
// tok0 / width: compact layout - `rep` holds sample b as a width[b]^2 corner starting at token tok0[b]


// ---------------------------------------------------------------------------------------------
// fused EDM step kernels                                               (edm.cu)
// ---------------------------------------------------------------------------------------------
int launch_edm_pre_step(const float* adj, const float* node, const float* eps_adj, const float* eps_node,
                        const uint8_t* flags, float noise_coef, float* adj_hat, float* node_hat, int batch,
                        int c_e, int n, int c_n, cudaStream_t st);
// same, eps drawn in the kernel exactly as torch.randn_like would from generator state (seed, offset_*); grid_* =
// ATen's launch grid for a tensor of that size (see edm.cu)
int launch_edm_pre_step_philox(const float* adj, const float* node, const uint8_t* flags, float noise_coef,
                               unsigned long long seed, unsigned long long offset_adj, int grid_adj,
                               unsigned long long offset_node, int grid_node, const void* dev_params, float* adj_hat,
                               float* node_hat, int batch, int c_e, int n, int c_n, cudaStream_t st);
// dev_params: device dsg_edm_step_params the scalars are read from (CUDA-graph replay), or nullptr
int launch_edm_post_step(const float* adj_hat, const float* node_hat, const float* d1_adj, const float* d1_node,
                         const float* d2_adj, const float* d2_node, const uint8_t* flags, float inv_t_hat,
                         float h, float inv_t_prime, const void* dev_params, float* adj_next, float* node_next, int batch,
                         int c_e, int n, int c_n, cudaStream_t st);
int launch_edm_step_advance(const void* table, void* cur, int* counter, cudaStream_t st);
// completion (known entries held; NaN = free): the two pre-steps with the known state, and x = mask(isnan(k) ? x : k)
// in place after the last post-step
int launch_edm_pre_step_known(const float* adj, const float* node, const float* eps_adj, const float* eps_node,
                              const float* known_adj, const float* known_node, const uint8_t* flags, float noise_coef,
                              float t_hat, float* adj_hat, float* node_hat, int batch, int c_e, int n, int c_n,
                              cudaStream_t st);
int launch_edm_pre_step_philox_known(const float* adj, const float* node, const float* known_adj, const float* known_node,
                                     const uint8_t* flags, float noise_coef, float t_hat, unsigned long long seed,
                                     unsigned long long offset_adj, int grid_adj, unsigned long long offset_node,
                                     int grid_node, const void* dev_params, float* adj_hat, float* node_hat, int batch,
                                     int c_e, int n, int c_n, cudaStream_t st);
int launch_edm_apply_known(float* adj, float* node, const float* known_adj, const float* known_node, const uint8_t* flags,
                           int batch, int c_e, int n, int c_n, cudaStream_t st);
// guided completion: update == 0: out = mask(isnan(o) ? 0 : d - o) (o = known state); else out = mask(d - w o) (o = G)
int launch_edm_guidance(const float* d_adj, const float* d_node, const float* o_adj, const float* o_node,
                        const uint8_t* flags, float w, int update, float* out_adj, float* out_node, int batch, int c_e,
                        int n, int c_n, cudaStream_t st);
// class ids (-1 = free) and boxes (NaN row = free) -> NaN-coded known state; any input may be nullptr
int launch_encode_known(const int32_t* node_cls, const float* bbox, const int32_t* adj_cls, float* known_adj,
                        float* known_node, int batch, int c_e, int n, int c_n, cudaStream_t st);
// last (Euler) step + decode of the final sample in one pass; adj_next / node_next may be nullptr
int launch_edm_final_decode(const float* adj_hat, const float* node_hat, const float* d1_adj, const float* d1_node,
                            const uint8_t* flags, float inv_t_hat, float h, const void* dev_params, float* adj_next,
                            float* node_next, int32_t* adj_cls, int32_t* node_cls, float* bbox, int num_adj_type,
                            int num_node_type, int batch, int c_e, int n, int c_n, cudaStream_t st);
int launch_mask_scale(const float* adj, const float* node, const uint8_t* flags, float scale, float* adj_out,
                      float* node_out, int batch, int c_e, int n, int c_n, cudaStream_t st);

// bits -> class ids (+ boxes) of the final sample; adj_cls [B, n, n], node_cls [B, n] int32, bbox [B, n, 4]
int launch_decode(const float* adj, const float* node, const uint8_t* flags, int32_t* adj_cls, int32_t* node_cls,
                  float* bbox, int num_adj_type, int num_node_type, int batch, int c_e, int n, int c_n, cudaStream_t st);

// ---------------------------------------------------------------------------------------------
// EDM training objective: noising and masked weighted squared-error sums            (train.cu)
// ---------------------------------------------------------------------------------------------
// x_adj = mask(y_adj + sigma_b e_adj), n_adj = mask(sigma_b e_adj); n_node = mask(sigma_b e_node), x_node = y_node + n_node
int launch_train_noise(const float* y_adj, const float* y_node, const float* e_adj, const float* e_node,
                       const float* sigmas, const uint8_t* flags, float* x_adj, float* n_adj, float* x_node,
                       float* n_node, int batch, int c_e, int n, int c_n, cudaStream_t st);
// s_adj[b] = sum mask w_b (d_adj - y_adj)^2, s_node[b] likewise; weights == nullptr means 1
int launch_loss_sums(const float* d_adj, const float* y_adj, const float* d_node, const float* y_node,
                     const float* weights, const uint8_t* flags, float* s_adj, float* s_node, int batch, int c_e, int n,
                     int c_n, cudaStream_t st);
// gradient of the two sums w.r.t. the predictions, scaled by the upstream gradients g_adj / g_node [B]
int launch_loss_sums_backward(const float* d_adj, const float* y_adj, const float* d_node, const float* y_node,
                              const float* weights, const uint8_t* flags, const float* g_adj, const float* g_node,
                              float* gd_adj, float* gd_node, int batch, int c_e, int n, int c_n, cudaStream_t st);


// ---------------------------------------------------------------------------------------------
// weight packing helpers (run once per weight update)                  (pack.cu)
// ---------------------------------------------------------------------------------------------
// dst bf16 = src * (i < n_scaled ? scale : 1)
int launch_pack_bf16(const float* src, bf16* dst, int64_t numel, int64_t n_scaled, float scale, cudaStream_t st);
int launch_scale_copy(const float* src, float* dst, int64_t numel, int64_t n_scaled, float scale, cudaStream_t st);
// *flag |= 1 when the two buffers differ in any 32-bit word (weight staleness probe)
int launch_compare_words(const void* a, const void* b, int64_t words, int* flag, cudaStream_t st);
// dst[c * dst_pitch + r] = src[r * ld + col0 + c], r < R, c < ncols   (dst is NOT cleared)
int launch_transpose(const float* src, float* dst, int R, int ld, int col0, int ncols, int dst_pitch, cudaStream_t st);
// out[h, p, q] = table[index[p, q], h]                              (diffusesg.py:121-124)
int launch_bias_expand(const float* table, const int64_t* index, float* out, int T, int heads, int table_rows,
                       cudaStream_t st);
// C[o][i] = sum_k A[o][k] * (trans_b ? B[i][k] : B[k][i]), n x n fp32
int launch_small_mm(const float* A, const float* B, float* C, int n, int trans_b, cudaStream_t st);
// y = A x + b
int launch_small_mv(const float* A, const float* x, const float* b, float* y, int n, cudaStream_t st);

}  // namespace dsg
