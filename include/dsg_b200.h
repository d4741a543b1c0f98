/* libdsg_b200 — C ABI of the B200-native DiffuseSG denoising hot path.
 *
 * The reference (ubc-vision/DiffuseSG) is pure Python/PyTorch and has no FFI of its own; its seam for this
 * path is the pair of Python objects built by utils/learning_utils.py:33 get_network() and
 * utils/sampling_utils.py:8 get_mc_sampler().  This header is what the drop-in Python classes in
 * diffusesg_b200/ bind through ctypes (see INTEGRATION.md).  Each entry point cites the reference code it
 * replaces; paths are relative to DiffuseSG/ in the reference repository.
 *
 * Conventions
 *   - plain C, no exceptions: every function returns 0 (DSG_OK) or a DSG_ERR_* code; dsg_last_error() gives
 *     the message of the last failure on the calling thread.
 *   - all tensor pointers are DEVICE pointers (fp32 unless stated) owned by the caller; nothing is allocated
 *     behind the caller's back: weights live in a caller-provided arena, activations in a caller-provided
 *     workspace.  Calls are asynchronous on the given CUDA stream and never synchronise it.
 *   - one host thread per dsg_model; different models may be used from different threads.
 *   - there is no CPU path: without an sm_100 device every compute call fails with DSG_ERR_CUDA.
 */
#ifndef DSG_B200_H_
#define DSG_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSG_ABI_VERSION 4

#if defined(__GNUC__)
#define DSG_API __attribute__((visibility("default")))
#else
#define DSG_API
#endif

enum {
  DSG_OK = 0,
  DSG_ERR_INVALID = 1,     /* bad argument / shape */
  DSG_ERR_CUDA = 2,        /* a CUDA runtime / driver call failed (includes: no device) */
  DSG_ERR_STATE = 3,       /* call order violated (e.g. forward before finalize) */
  DSG_ERR_UNKNOWN_KEY = 4, /* set_tensor with a key the configuration does not define */
  DSG_ERR_WORKSPACE = 5    /* arena / workspace too small or not bound */
};

typedef void* dsg_stream_t;          /* cudaStream_t */
typedef struct dsg_model dsg_model;  /* opaque: configuration + packed weights + TMA descriptors */

/* Constructor arguments of the reference denoiser, DiffuseSG.__init__ (model/diffusesg/diffusesg.py:587-720) as
 * called from utils/learning_utils.py:47-64.  patch_size is 1, mlp_ratio 4, head_dim 32 and all drop rates 0 there. */
typedef struct dsg_config {
  int32_t img_size;       /* N: dataset.max_node_num */
  int32_t embed_dim;      /* model.feature_dims[-1]; 96 */
  int32_t num_stages;     /* len(model.depths), <= 4 */
  int32_t depths[4];
  int32_t num_heads[4];   /* [3, 6, 12, 24]; dim / heads must be 32 */
  int32_t window_size;
  int32_t c_e;            /* out_chans_adj: edge channels (<= 8) */
  int32_t c_n;            /* out_chans_node: node channels */
  int32_t self_condition; /* train.self_cond */
} dsg_config;

DSG_API int dsg_abi_version(void);
DSG_API const char* dsg_last_error(void);
/* Number of CUDA kernels this library has launched in the calling process (all models). */
DSG_API uint64_t dsg_launch_count(void);
/* Kernels launched by replaying a CUDA graph captured from this library's launches are not seen by the counter
 * above; the caller that replays the graph adds the number recorded at capture time. */
DSG_API void dsg_launch_count_add(uint64_t n);

/* ---- model life cycle -------------------------------------------------------------------------------------- */
DSG_API int dsg_model_create(const dsg_config* cfg, dsg_model** out);
DSG_API void dsg_model_destroy(dsg_model* m);

/* The arena holds the fp32 master copy of every state_dict tensor plus the packed bf16 / transposed / folded
 * forms the kernels read.  Bind once; rebinding invalidates loaded tensors. */
DSG_API size_t dsg_model_arena_bytes(const dsg_model* m);
DSG_API int dsg_model_bind_arena(dsg_model* m, void* arena, size_t bytes);

/* Enumerate the state_dict of the reference module (same keys, shapes and dtypes as
 * DiffuseSG(...).state_dict(); strict checkpoint loading at utils/sampling_utils.py:34-60 relies on it).
 * dtype: 0 = float32, 1 = int64 (the relative_position_index buffers). */
DSG_API int dsg_model_num_tensors(const dsg_model* m);
DSG_API int dsg_model_tensor_info(const dsg_model* m, int index, const char** key, int64_t* numel, int32_t* dtype);

/* Copy one state_dict tensor (contiguous, dtype as reported above) into the arena.  src may be a device or a
 * host pointer (src_is_host != 0). */
DSG_API int dsg_model_set_tensor(dsg_model* m, const char* key, const void* src, int64_t bytes, int src_is_host,
                         dsg_stream_t stream);
/* Staleness probe: *flag |= 1 (device int32, caller-zeroed) when `src` (device, same dtype / size as the tensor
 * `key`) differs from the fp32 / int64 master the arena holds.  The Python module uses it to notice parameter
 * updates that bypass autograd's version counters (`p.data.copy_()`, ema_pytorch's `.data.lerp_()`:
 * utils/learning_utils.py:145-166 wraps the model in EMA and the reference samples from `ema_model`). */
DSG_API int dsg_model_tensor_differs(const dsg_model* m, const char* key, const void* src, int64_t bytes, int32_t* flag,
                                     dsg_stream_t stream);
/* Build the packed forms (bf16 weights with the q scale folded in, gathered relative-position bias, folded
 * read_out chain, transposed head weights) and the weight TMA descriptors.  Call after all tensors are set and
 * again whenever any of them changed.  For shifted blocks / 16 x 16 windows it also compares the attn_mask buffer
 * with the reference's SW-MSA construction (diffusesg.py:207-222) and checks that the gathered bias depends on the
 * token offset only; the tcgen05 attention kernels, which generate the mask and look the bias up themselves, are
 * only selected when that holds.  These checks SYNCHRONISE the stream (one small readback per such block); the
 * denoiser passes themselves never do. */
DSG_API int dsg_model_finalize(dsg_model* m, dsg_stream_t stream);

/* ---- denoiser forward --------------------------------------------------------------------------------------- */
/* n_cond = 1 when every sample shares one noise level (sampling: runner/mcmc_sampler/edm.py:371 expands a
 * scalar), = batch otherwise (training). */
DSG_API size_t dsg_workspace_bytes(const dsg_model* m, int batch, int n_cond);

/* ---- padding skipping (SURVEY 8f-4; model/diffusesg/diffusesg.py:796-802, :812-825) ------------------------------
 * A graph with n_b < N nodes occupies the top-left n_b x n_b corner of the N x N pair grid; every other pixel is
 * padding: its inputs are zeroed by mask_adjs (:800) and its outputs are masked (:822-825).  The reference still
 * computes on it.  For the leading resolution stages whose blocks are all UN-shifted window attention, nothing moves
 * between aligned windows, so every window outside the corner of side R_b = ceil(n_b / granule) * granule (i) holds,
 * in the encoder, one and the same token value for every sample - computed once on an all-padding "phantom" image
 * and filled in where the first dense stage needs it - and (ii) cannot influence any unmasked output in the decoder.
 * Those stages run on a compact layout: the samples are grouped into buckets by R_b, bucket k is a stack of count[k]
 * images of side[k] x side[k] pixels, the buckets follow each other in memory.  In exact arithmetic the result equals
 * the dense computation; tests/test_gpu_denoiser.py::test_padding_skipping_* hold it to the dense path (bit-identical
 * on every tested input) and to the reference's golden outputs at the tolerances of DESIGN.md section 1.
 * dsg_model_skip_info: stages = number of compactable leading stages (0: none for this geometry), granule in pixels.
 * The caller builds, from the node counts, one int32 table on the device (dsg_forward_args.skip_tables):
 *     perm[skip_table_images] | tok0[B] | width[B]
 * perm[k]: the sample shown by compact image k, bucket by bucket (-1: an all-padding image - the phantom, or the
 * dummy that keeps a bucket's image count even); tok0[b]: stage-0 token offset of sample b's image in the compact
 * layout; width[b] = R_b.  skip_phantom_tok0: token offset of the phantom image (it lives in the bucket of side
 * `granule`).  Needs n_cond == 1 (one shared noise level, as in sampling). */
DSG_API int dsg_model_skip_info(const dsg_model* m, int32_t* stages, int32_t* granule);
/* Second level (0: not available): when the first block of the first DENSE stage and that stage's last block on the way
 * up are un-shifted as well (Visual Genome: the C = 384 stage, blocks [un-shifted, shifted, un-shifted]), those two
 * blocks, the encoder skip of that stage and the PatchBreakup input run on a second compact layout with the coarser
 * granule2 (that stage's window in pixels), described by dsg_forward_args.skip2_* exactly like the first
 * (perm2 | tok2 | width2 with its own phantom image); the shifted blocks in between stay dense. */
DSG_API int dsg_model_skip_info2(const dsg_model* m, int32_t* granule2);

typedef struct dsg_forward_args {
  uint32_t struct_size;     /* sizeof(dsg_forward_args) */
  int32_t batch;
  int32_t n_cond;           /* 1 or batch */
  /* mode 0: raw network, DiffuseSG.forward(adj, node, node_flags, noise_labels, self_cond_x, self_cond_feat)
   *         (model/diffusesg/diffusesg.py:765); `noise` holds noise_labels (c_noise = ln(sigma) / 4).
   * mode 1: EDM-preconditioned denoiser, the non-coin-flip body of NodeAdjPrecond.forward
   *         (model/precond/precond.py:100-105): `noise` holds sigmas; inputs are scaled by c_in inside the
   *         patch embedding, outputs are c_skip * x + c_out * F, masked. */
  int32_t mode;
  const float* adj;         /* [B, c_e, N, N] */
  const float* node;        /* [B, N, c_n] */
  const uint8_t* flags;     /* [B, N] bool (node_flags), 4-byte aligned */
  const float* noise;       /* n_cond values, element stride noise_stride */
  int64_t noise_stride;
  const float* sc_adj;      /* self-conditioning inputs or NULL (zeros), same shapes as adj / node */
  const float* sc_node;
  float* out_adj;           /* [B, c_e, N, N] */
  float* out_node;          /* [B, N, c_n] */
  void* workspace;
  size_t workspace_bytes;
  const int32_t* skip_tables; /* NULL: dense.  Device table described at dsg_model_skip_info */
  int32_t skip_table_images;  /* length of the perm section (>= sum of skip_count) */
  int32_t skip_buckets;       /* K <= 8 (0: dense) */
  int32_t skip_count[8];      /* images per bucket, even */
  int32_t skip_side[8];       /* corner side of the bucket's images in pixels: a multiple of the granule */
  int64_t skip_phantom_tok0;  /* stage-0 token offset of the phantom image */
  /* Row maps of the layout changes (int32 token indices at the first dense stage; a reader in layout Y of a tensor stored
   * in layout X reads row map[r] - tokens outside X's kept corner point at X's phantom token):
   *   skip_map_dense_from_c1 [B res^2]   without a second level: the dense grid reads the merge output of the last compact
   *                                      stage (first dense block on the way down, skip concat on the way up)
   *   skip2_map_c2_from_c1   [tokens of the second layout]   the same readers when there is a second level
   *   skip2_map_dense_from_c2 [B res^2]  the shifted block after the level-2 block reads its output
   *   skip2_map_c2_from_dense [tokens of the second layout]   the level-2 block on the way up reads the dense grid */
  const int32_t* skip_map_dense_from_c1;
  const int32_t* skip2_map_c2_from_c1;
  const int32_t* skip2_map_dense_from_c2;
  const int32_t* skip2_map_c2_from_dense;
  const int32_t* skip2_tables; /* second level (dsg_model_skip_info2), same layout; NULL: none */
  int32_t skip2_table_images;
  int32_t skip2_buckets;
  int32_t skip2_count[8];
  int32_t skip2_side[8];
  int64_t skip2_phantom_tok0;
} dsg_forward_args;

DSG_API int dsg_denoiser_forward(dsg_model* m, const dsg_forward_args* args, dsg_stream_t stream);

/* ---- EDM stochastic-Heun sampler steps (runner/mcmc_sampler/edm.py:350-434) ------------------------------- */
/* x_hat = mask(x + noise_coef * eps), noise_coef = sqrt(t_hat^2 - t_cur^2) * S_noise          (:361-366) */
DSG_API int dsg_edm_pre_step(const float* adj, const float* node, const float* eps_adj, const float* eps_node,
                     const uint8_t* flags, float noise_coef, float* adj_hat, float* node_hat, int batch, int c_e,
                     int n, int c_n, dsg_stream_t stream);
/* The same step with eps drawn inside the kernel, bit-identical to `eps_adj = randn_like(adjs); eps_node =
 * randn_like(nodes)` of the reference (:358-364) on this device: Philox4x32-10 keyed by the torch CUDA generator's
 * seed, counter offsets offset_adj / offset_node, and ATen's launch grids for tensors of those sizes
 * (grid = min(SMs * (max threads per SM / 256), ceil(numel / 256)); ATen/native/cuda/DistributionTemplates.h).
 * The caller advances the generator by ((numel - 1) / (256 * grid * 4) + 1) * 4 per tensor.  No eps tensor is
 * materialised (SURVEY 8f-3). */
DSG_API int dsg_edm_pre_step_philox(const float* adj, const float* node, const uint8_t* flags, float noise_coef,
                            uint64_t seed, uint64_t offset_adj, int grid_adj, uint64_t offset_node, int grid_node,
                            float* adj_hat, float* node_hat, int batch, int c_e, int n, int c_n, dsg_stream_t stream);
/* Heun update from (x_hat, D1, D2); pass d2_* = NULL for the Euler update of the last step     (:384-422).
 * inv_t_hat = 1 / t_hat, h = t_next - t_hat, inv_t_prime = 1 / (t_hat + h), all evaluated in fp32 by the caller
 * exactly as the reference does. */
DSG_API int dsg_edm_post_step(const float* adj_hat, const float* node_hat, const float* d1_adj, const float* d1_node,
                      const float* d2_adj, const float* d2_node, const uint8_t* flags, float inv_t_hat, float h,
                      float inv_t_prime, float* adj_next, float* node_next, int batch, int c_e, int n, int c_n,
                      dsg_stream_t stream);
/* ---- the same steps for CUDA-graph replay: per-step scalars read from device memory -------------------------------
 * A captured Heun step cannot carry per-step host scalars, so the sampler uploads ONE row per step (the values the
 * reference derives at :355-356, :361, :369, :384-391, :414, evaluated on the host exactly as before, plus the Philox
 * counter offsets of that step's two randn_like draws) and every captured launch reads the current row:
 *   dsg_edm_step_advance: cur = table[*counter]; ++*counter   (first node of each captured step)
 *   *_dev entry points:   as above with the scalars taken from `cur`; `cur->t_hat` is also what the captured
 *                         dsg_denoiser_forward(mode 1, n_cond 1) is given as its sigma pointer. */
typedef struct dsg_edm_step_params {
  float noise_coef;    /* sqrt(t_hat^2 - t_cur^2) * S_noise                      (:361) */
  float inv_t_hat;     /* sigma'(t_hat) / sigma(t_hat) = 1 / t_hat               (:384) */
  float h;             /* t_next - t_hat                                         (:389) */
  float inv_t_prime;   /* 1 / (t_hat + h); 0 on the last step                    (:414) */
  float t_hat;         /* the noise level both denoiser calls of the step see    (:371) */
  float reserved;
  uint64_t seed;        /* torch CUDA generator seed */
  uint64_t offset_adj;  /* Philox counter offset of randn_like(adjs) of this step */
  uint64_t offset_node; /* ... of randn_like(nodes) */
} dsg_edm_step_params;
DSG_API int dsg_edm_step_advance(const dsg_edm_step_params* table, dsg_edm_step_params* cur, int32_t* counter,
                                 dsg_stream_t stream);
DSG_API int dsg_edm_pre_step_philox_dev(const float* adj, const float* node, const uint8_t* flags,
                                        const dsg_edm_step_params* cur, int grid_adj, int grid_node, float* adj_hat,
                                        float* node_hat, int batch, int c_e, int n, int c_n, dsg_stream_t stream);
DSG_API int dsg_edm_post_step_dev(const float* adj_hat, const float* node_hat, const float* d1_adj, const float* d1_node,
                                  const float* d2_adj, const float* d2_node, const uint8_t* flags,
                                  const dsg_edm_step_params* cur, float* adj_next, float* node_next, int batch, int c_e,
                                  int n, int c_n, dsg_stream_t stream);
/* x_out = mask(x * scale): masking of the initial noise and its scaling by sigma(t_0)         (:276-289, :346-347) */
DSG_API int dsg_edm_mask_scale(const float* adj, const float* node, const uint8_t* flags, float scale, float* adj_out,
                       float* node_out, int batch, int c_e, int n, int c_n, dsg_stream_t stream);

/* ---- decode of the final sample ("next" row f-1: runner/sampler/sampler_node_adj.py:199-285, 'bits' encodings) -- */
/* adj_cls[b,i,j] = clamp(bin2dec(adj[b,:,i,j] > 0), 0, num_adj_type-1) for valid i != j else 0 (self-loops
 * removed, :283); node_cls[b,i] = clamp(bin2dec(node[b,i,:c_n-4] > 0), 0, num_node_type-1) for valid i else 0;
 * bbox[b,i,:] = node[b,i,c_n-4:] * 0.5 + 0.5 for valid i else 0 (:202-209).  Bits are MSB first
 * (utils/attribute_code.py:319-328).  Only the int32 classes and 4 floats per node need to leave the GPU. */
DSG_API int dsg_decode_samples(const float* adj, const float* node, const uint8_t* flags, int32_t* adj_cls,
                               int32_t* node_cls, float* bbox, int num_adj_type, int num_node_type, int batch,
                               int c_e, int n, int c_n, dsg_stream_t stream);

/* The LAST sampler step (Euler, :389-396) fused with that decode: one pass over (x_hat, D1) writes the classes and
 * boxes; the fp32 state is written only when adj_next / node_next are non-NULL.  Scalars from `cur` when it is
 * non-NULL (graph replay), else from inv_t_hat / h. */
DSG_API int dsg_edm_final_step_decode(const float* adj_hat, const float* node_hat, const float* d1_adj,
                                      const float* d1_node, const uint8_t* flags, float inv_t_hat, float h,
                                      const dsg_edm_step_params* cur, float* adj_next, float* node_next,
                                      int32_t* adj_cls, int32_t* node_cls, float* bbox, int num_adj_type,
                                      int num_node_type, int batch, int c_e, int n, int c_n, dsg_stream_t stream);

/* ---- EDM training objective (BASELINE config 4; forward only) ---------------------------------------------------
 * dsg_train_noise replaces NodeAdjEDMObjectiveGenerator.get_network_input (runner/objectives/edm.py:233-254) over
 * add_sym_normal_noise(non_symmetric=True) (utils/graph_utils.py:122-152): eps_* are the caller's N(0,1) draws
 * (torch.randn_like, in the reference's order: adjacency first, nodes second), sigmas is [batch]; the four outputs are
 * bit-identical to the reference's fp32 expressions.
 * dsg_edm_loss_sums replaces the elementwise part of NodeAdjRainbowLoss.get_regression_loss (loss/rainbow_loss.py:60-99):
 * sum_adj[b] = sum mask w_b (pred - target)^2 over [C_e, N, N], sum_node[b] over [N, C_n]; weights may be NULL (= 1).
 * The [batch]-sized normalisations (n_b^2 C_e, n_b C_n, loss weights, 'mean' / 'none') stay on the host. */
DSG_API int dsg_train_noise(const float* clean_adj, const float* clean_node, const float* eps_adj, const float* eps_node,
                            const float* sigmas, const uint8_t* flags, float* noisy_adj, float* noise_adj,
                            float* noisy_node, float* noise_node, int batch, int c_e, int n, int c_n, dsg_stream_t stream);
DSG_API int dsg_edm_loss_sums(const float* pred_adj, const float* target_adj, const float* pred_node,
                              const float* target_node, const float* weights, const uint8_t* flags, float* sum_adj,
                              float* sum_node, int batch, int c_e, int n, int c_n, dsg_stream_t stream);
/* Backward of dsg_edm_loss_sums for loss.backward() (runner/trainer/trainer_node_adj.py:173): grad_pred = grad_sum[b] *
 * 2 w_b (pred - target) on valid entries, 0 on masked ones; the targets, weights and flags carry no gradient. */
DSG_API int dsg_edm_loss_sums_backward(const float* pred_adj, const float* target_adj, const float* pred_node,
                                       const float* target_node, const float* weights, const uint8_t* flags,
                                       const float* grad_sum_adj, const float* grad_sum_node, float* grad_pred_adj,
                                       float* grad_pred_node, int batch, int c_e, int n, int c_n, dsg_stream_t stream);


/* ---- building blocks, exported for the kernel-level parity tests ------------------------------------------- */
/* out[M, N] = epilogue(A[M, K] . W[N, K]^T + bias); A, W bf16 row-major.  epi: 0 bf16, 1 gelu->bf16,
 * 2 fp32 + residual (res may alias out), 3 fp32.  tcgen05/TMEM/TMA kernel (nn.Linear of the reference). */
DSG_API int dsg_gemm_bf16(const void* a, const void* w, const float* bias, const float* res, void* out, int M, int N, int K,
                  int epi, dsg_stream_t stream);
/* x[M, C] += att[M, C] . w[C, C]^T + bias (fp32, in place);  y[M, C] = LayerNorm(x) * gamma + beta (bf16): the fused
 * attention projection + residual + norm2 of the C = 192 / 384 Swin blocks (diffusesg.py:137, :272, :275). */
DSG_API int dsg_proj_ln(const void* att, const void* w, const float* bias, const float* gamma, const float* beta, float* x,
                void* y, int M, int C, dsg_stream_t stream);
/* qkv [B*res*res, 3*heads*32] bf16 -> out [B*res*res, heads*32] bf16 (WindowAttention.forward, :108-139, q
 * pre-scaled); bias [heads, T, T] fp32, mask [nW, T, T] fp32 or NULL (shift == 0).  Runs the same mask / bias
 * checks as dsg_model_finalize on every call (synchronous) and then the kernel the denoiser would pick. */
DSG_API int dsg_window_attention(const void* qkv, const float* bias, const float* mask, void* out, int batch, int res,
                         int window, int shift, int heads, dsg_stream_t stream);
/* The two halves of dsg_window_attention: the (stream-synchronising) checks of the mask / bias buffers, once, and the
 * launch with their result - what a CUDA-graph capture of a training step needs (no synchronisation inside a capture). */
DSG_API int dsg_window_attention_check(const float* bias, const float* mask, int batch, int res, int window, int shift,
                                       int heads, dsg_stream_t stream, int* flags_out);
DSG_API int dsg_window_attention_flags(const void* qkv, const float* bias, const float* mask, void* out, int batch, int res,
                                       int window, int shift, int heads, int flags, dsg_stream_t stream);

/* ---- training step (SURVEY 8 f-2): loss.backward() and optimizer.step() of runner/trainer/trainer_node_adj.py:171-178 ---
 * Row-wise forward kernels in the form the backward pass needs (out of place, pre-activations kept) and every backward
 * kernel that is not a GEMM.  fp32 unless a pointer is `void*` (bf16).  The host-side tape that strings them together is
 * diffusesg_b200/model/diffusesg/train_graph.py. */
/* nn.LayerNorm (diffusesg.py:243, :275, :333, :386, :400, :571, :758), eps 1e-5: y as bf16 and / or fp32 (either may be
 * NULL).  Backward: dx = LN'(dy) (+ dx_add, may alias dx), dgamma / dbeta ACCUMULATED (atomicAdd). */
DSG_API int dsg_tr_ln_fwd(const float* x, const float* gamma, const float* beta, void* y_bf16, float* y_f32, long long M, int C,
                          dsg_stream_t stream);
DSG_API int dsg_tr_ln_bwd(const float* dy, const float* x, const float* gamma, const float* dx_add, float* dx, float* dgamma,
                          float* dbeta, long long M, int C, dsg_stream_t stream);
/* Noise conditioning out = silu(shift_b + v (1 + scale_b)) (diffusesg.py:238-240, :574-576); (scale, shift) of sample b =
 * film[b * ldf + off + (0..C)], [.. + C + (0..C)].  Backward: dv written, dfilm[b, off .. off + 2C) ACCUMULATED. */
DSG_API int dsg_tr_film_silu_fwd(const float* v, const float* film, int ldf, int off, float* out, int B, int L, int C,
                                 dsg_stream_t stream);
DSG_API int dsg_tr_film_silu_bwd(const float* dout, const float* v, const float* film, int ldf, int off, float* dv, float* dfilm,
                                 int B, int L, int C, dsg_stream_t stream);
/* nn.GELU (erf form, diffusesg.py:15) on bf16, evaluated with the inference kernels' tanh-form fit (|error| <= 2.6e-5) and its
 * analytic derivative (<= 1.1e-4): dh == NULL: out = gelu(pre); else out = dh * gelu'(pre).  n % 8 == 0. */
DSG_API int dsg_tr_gelu(const void* pre, const void* dh, void* out, long long n, dsg_stream_t stream);
/* the same on fp32 (the node read-out MLP, :818): dout == NULL: forward */
DSG_API int dsg_tr_gelu_f32(const float* pre, const float* dout, float* out, long long n, dsg_stream_t stream);
/* out[c] += sum_r src[r, c] (bias gradients of the small fp32 layers) */
DSG_API int dsg_tr_colsum(const float* src, float* out, long long M, int C, dsg_stream_t stream);
/* out [4, B] = c_skip | c_out | c_in | c_noise of runner/objectives/edm.py:122-126 ('edm', sigma_data 0.5) */
DSG_API int dsg_tr_precond_coef(const float* sigmas, float* out, int B, dsg_stream_t stream);
/* silu on fp32 (:769-771): dout == NULL: out = silu(pre); else out = dout * silu'(pre). */
DSG_API int dsg_tr_silu(const float* pre, const float* dout, float* out, long long n, dsg_stream_t stream);
DSG_API int dsg_tr_add_inplace(float* y, const float* x, long long n, dsg_stream_t stream);
/* The weight gradient of an nn.Linear without transposes: dw [n_out, out_cols] += dy^T . x with dy [tokens, n_out] and
 * x [tokens, x_cols] bf16 row-major, read by TMA as they lie and fed to tcgen05.mma as MN-major operands (the
 * non-contracted index is the contiguous one); contraction over the tokens in `ksplit` slices combined by the reduce-add
 * epilogue; rows < scale_rows of dw are multiplied by row_scale (the q third of qkv, :118); out_cols <= x_cols (a zero
 * padded input).  tokens % 16 == 0, widths % 8 == 0.  dsg_tr_cast_colsum prepares its operand: colsum [C] += column sums
 * of dy (the bias gradient; columns < scale_cols scaled) and, for an fp32 dy, the bf16 copy. */
DSG_API int dsg_tr_wgrad(const void* dy, const void* x, float* dw, long long tokens, int n_out, int x_cols, int out_cols,
                         int ksplit, int scale_rows, float row_scale, dsg_stream_t stream);
DSG_API int dsg_tr_cast_colsum(const void* src, int src_is_bf16, void* cast, float* colsum, long long M, int C,
                               int scale_cols, float scale, dsg_stream_t stream);
/* fine [B, 2H, 2W, C] <-> coarse [B, H, W, 4, C], chunk k = dy + 2 dx: the gather of PatchMerging (:325-329) and the
 * scatter of PatchBreakup (:394-397); to_coarse selects the direction (each is the other's backward). */
DSG_API int dsg_tr_shuffle2x2(const float* src, float* dst, int B, int H, int W, int C, int to_coarse, dsg_stream_t stream);
/* dst[:, dcol : dcol + ncols] (=, +=) src[:, scol : scol + ncols], dst fp32 or bf16: torch.cat of :753 and its split */
DSG_API int dsg_tr_copy_cols(const float* src, int lds, int scol, void* dst, int ldd, int dcol, int ncols, long long M,
                             int dst_bf16, int accumulate, dsg_stream_t stream);
/* the input grid of :791-802 (self-conditioning first, node planes masked) as a bf16 GEMM operand [B N N, ld], inputs
 * scaled by c_in[b] when given (model/precond/precond.py:100) */
DSG_API int dsg_tr_embed_input(const float* adj, const float* node, const float* sc_adj, const float* sc_node,
                               const uint8_t* flags, const float* c_in, void* out, int B, int n, int c_e, int c_n,
                               int self_cond, int ld, dsg_stream_t stream);
/* head outputs, token-major -> the reference's tensors with masks (:822-825) and D = c_skip x + c_out F
 * (precond.py:102-105; x == NULL: raw F); backward != 0: `in` is the output gradient, `out` the token-major gradient */
DSG_API int dsg_tr_adj_out(const float* in, const uint8_t* flags, const float* x_adj, const float* c_skip, const float* c_out,
                           float* out, int B, int n, int c_e, int backward, dsg_stream_t stream);
DSG_API int dsg_tr_node_out(const float* in, const uint8_t* flags, const float* x_node, const float* c_skip, const float* c_out,
                            float* out, int B, int n, int c_n, int backward, dsg_stream_t stream);
/* second layer of the adjacency read-out MLP (:806-809), c_e <= 8 outputs from embed <= 128 hidden channels (h bf16):
 * dtok == NULL: tok [M, c_e] = h w^T + b; else dw [c_e, embed] += dtok^T h (the bias gradient is dsg_tr_colsum of dtok) */
DSG_API int dsg_tr_adj_fc2(const void* h, const float* w, const float* b, float* tok, const float* dtok, float* dw, long long M,
                           int E, int ce, dsg_stream_t stream);
/* masked mean of :812-813: dpooled == NULL: pooled [B n, C] from rep [B n n, C]; else drep += its backward */
DSG_API int dsg_tr_node_pool(const float* rep, const uint8_t* flags, float* pooled, const float* dpooled, float* drep, int B,
                             int n, int C, dsg_stream_t stream);
/* PositionalEmbedding (:507-513) */
DSG_API int dsg_tr_posemb(const float* labels, float* out, int B, int embed, dsg_stream_t stream);
/* bias[h, t, u] = table[index[t, u], h] (:121-124); backward != 0: dtable[index[t, u], h] += bias[h, t, u] */
DSG_API int dsg_tr_bias_gather(const float* table, const int64_t* index, float* bias, int heads, int T, int backward,
                               float* dtable, dsg_stream_t stream);
/* C[m, n] (=, +=) sum_k A[m sam + k sak] B[k sbk + n sbn] (+ bias[n]); fp32 CUDA-core GEMM for the small matrices (noise
 * embedding MLP, FiLM generators, node read-out, c_e / c_n wide output layers) and their gradients; ksplit > 1 or
 * accumulate: atomicAdd onto C. */
DSG_API int dsg_tr_sgemm(const void* A, int a_is_bf16, long long sam, long long sak, const void* B, int b_is_bf16,
                         long long sbk, long long sbn, const float* bias, float* C, long long ldc, int M, int N, int K,
                         int ksplit, int accumulate, dsg_stream_t stream);
/* backward of dsg_window_attention (:108-139 with the roll / partition index arithmetic of :28-57, :248-267): qkv
 * [B res res, 3 heads 32] bf16 (q pre-scaled), datt [B res res, heads 32] bf16 -> dqkv (same layout as qkv; dq w.r.t. the
 * scaled q), dbias [heads, T, T] ACCUMULATED.  mask [nW, T, T] is required when shift > 0.  T = window^2 <= 100. */
DSG_API int dsg_tr_window_attention_bwd(const void* qkv, const void* datt, const float* bias, const float* mask, void* dqkv,
                                        float* dbias, int batch, int res, int window, int shift, int heads,
                                        dsg_stream_t stream);
/* optimizer.step(): out[0] = sum g^2 (for clip_grad_norm_, trainer_node_adj.py:174); then Adam with torch.optim.Adam
 * semantics (utils/learning_utils.py:126-145) and n_ema <= 8 exponential moving averages (ema_pytorch.EMA.update, :148-166:
 * ema += (1 - decay) (p - ema)) over one flat parameter buffer in one launch; gsumsq (device) and max_norm > 0 apply the
 * gradient clipping coefficient min(1, max_norm / (sqrt(gsumsq) + 1e-6)).  m == v == NULL: only the moving averages move
 * (ema.update() without a fused optimiser); decay 0 copies the parameters (ema_pytorch's first updates). */
DSG_API int dsg_tr_sumsq(const float* g, long long n, float* out, dsg_stream_t stream);
DSG_API int dsg_tr_adam_ema(float* p, const float* g, float* m, float* v, long long n, const float* gsumsq, float lr,
                            float beta1, float beta2, float eps, float weight_decay, int step, float max_norm, int n_ema,
                            float* const* ema, const float* ema_decay, dsg_stream_t stream);
/* bf16 shadows of the fp32 master weights for the tcgen05 GEMMs of a training step, one launch: jobs_device is an array
 * of { const float* src; void* dst; void* dst_t; int32 rows, cols, ldd, rows_t; int64 scale_elems; float scale; int32
 * dst_f32 } (dsg_tr_prep_job_bytes() each): dst [rows, ldd] = src [rows, cols] zero padded (bf16, or fp32 when dst_f32),
 * dst_t [rows_t, rows] its transpose (the dgrad operand) or NULL, the first scale_elems source elements scaled. */
DSG_API int dsg_tr_prep_weights(const void* jobs_device, int n_jobs, dsg_stream_t stream);
DSG_API int dsg_tr_prep_job_bytes(void);

/* ---- per-kernel-class timing (bench.py roofline numbers) ------------------------------------------------------- */
/* While enabled, every pass_stride-th dsg_denoiser_forward and every dsg_edm_* call brackets each of its kernel
 * launches with a pair of CUDA events on the launching stream.  dsg_profile_read waits for the recorded events
 * and returns per-class totals since dsg_profile_begin: launches, device milliseconds, ALGORITHMIC flops and
 * bytes (2MNK per GEMM; each distinct tensor touched once per elementwise kernel).  Process-global, one thread. */
typedef struct dsg_profile_class {
  char name[24];
  uint64_t launches;
  double ms;
  double flops;
  double bytes;
} dsg_profile_class;
DSG_API int dsg_profile_begin(int pass_stride);
DSG_API int dsg_profile_read(dsg_profile_class* out, int max_classes, int* n_classes);
/* Write the records gathered since the last dsg_profile_read, one line per launch in launch order
 * (index,class,label,rows,k,ms,flops,bytes), to a CSV file.  Call before dsg_profile_read (which consumes them). */
DSG_API int dsg_profile_dump(const char* path);
DSG_API void dsg_profile_stop(void);

/* ---- test hooks (used by tests/ to localise a parity failure; not part of the product path) ------------------- */
/* Leave dsg_denoiser_forward after n_stages schedule stages (0: patch embedding, then one per Swin block /
 * PatchMerging / PatchBreakup in execution order); -1 restores the full schedule.  Process-global. */
DSG_API void dsg_debug_set_stop_after(int n_stages);
/* While enabled, every kernel launch of the library is followed by a kernel (legacy default stream: use it with torch's
 * default stream only) that fills the shared memory of every SM with `pattern` (e.g. 0x7fc00000, a NaN): what a foreign
 * kernel - NCCL, another library - may leave behind.  A kernel that reads shared memory it never wrote, e.g. a
 * zero-weighted padding slot, then produces NaN (tests/test_gpu_denoiser.py::test_kernels_ignore_shared_memory_leftovers).
 * Process-global. */
DSG_API void dsg_debug_set_smem_poison(unsigned pattern, int enable);
/* Byte offset and size of a named activation buffer ("X", "Y", "QKV", "ATT", "H", "T", "REP", "skip0".."skip2",
 * "film", "rc", "emb", "coef") inside a workspace laid out for (batch, n_cond). */
DSG_API int dsg_debug_buffer(const dsg_model* m, int batch, int n_cond, const char* name, size_t* offset, size_t* bytes);

#ifdef __cplusplus
}
#endif
#endif /* DSG_B200_H_ */
