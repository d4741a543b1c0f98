// dsg_model: configuration, weight arena, packing and the kernel schedule of one denoiser forward.
//
// The schedule restates DiffuseSG.forward / forward_features (model/diffusesg/diffusesg.py:739-830 of the
// reference) as ~110 launches of the kernels in gemm.cu / attention.cu / rowops.cu on one stream.  All shapes
// are static per (model, batch), so the whole forward is CUDA-graph capturable (no host sync, no allocation).
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/dsg_b200.h"
#include "common.cuh"
#include "kernels.h"

namespace dsg {

// ------------------------------------------------------------------------------------------------
// error / launch bookkeeping
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";
static unsigned long long g_launches = 0;
static int g_stop_after = -1;  // test hook: leave the forward schedule after this many stages (-1: run all)

void set_last_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
// test hook (dsg_debug_set_smem_poison): after every counted launch, a kernel on the legacy default stream overwrites the
// shared memory of every SM with a bit pattern - a kernel that reads shared memory it never wrote then shows it
static unsigned g_smem_poison = 0;
static bool g_smem_poison_on = false;
__global__ void poison_smem_kernel(unsigned pattern, int words) {
  extern __shared__ unsigned psm[];
  for (int i = threadIdx.x; i < words; i += blockDim.x) psm[i] = pattern;
  __syncthreads();
  if (psm[(threadIdx.x * 7) % words] != pattern) __trap();   // keeps the stores alive
}
static void poison_smem_now() {
  constexpr int bytes = 200 * 1024;
  static PerDeviceOnce configured;
  if (configured.first()) cudaFuncSetAttribute(poison_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  poison_smem_kernel<<<device_sm_count() * 2, 256, bytes, 0>>>(g_smem_poison, bytes / 4);
}
void count_launch(int n) {
  __atomic_fetch_add(&g_launches, static_cast<unsigned long long>(n), __ATOMIC_RELAXED);
  if (g_smem_poison_on) poison_smem_now();
}

// ------------------------------------------------------------------------------------------------
// optional per-kernel-class timing with CUDA events on the launching stream (bench.py roofline numbers)
// ------------------------------------------------------------------------------------------------
enum ProfClass { PC_GEMM = 0, PC_ATTN, PC_ROW, PC_EMBED_HEAD, PC_EDM, PC_MLP, PC_EDM_NOISE, PC_COUNT };
static const char* kProfNames[PC_COUNT] = {"gemm_tcgen05", "window_attention", "row_ln_film", "embed_heads_cond", "edm_step",
                                           "fused_mlp_tcgen05", "edm_pre_step_philox"};
struct ProfRec { int cls; double flops, bytes; cudaEvent_t e0, e1; char label[56]; long long rows; int c; };
static bool g_prof_on = false;        // between dsg_profile_begin and dsg_profile_stop
static bool g_prof_pass = false;      // the current denoiser pass is being bracketed
static int g_prof_stride = 1, g_prof_counter = 0;
static std::vector<ProfRec> g_prof_recs;
static std::vector<cudaEvent_t> g_prof_pool;
static dsg_profile_class g_prof_tot[PC_COUNT];

static cudaEvent_t prof_event() {
  cudaEvent_t e = nullptr;
  if (!g_prof_pool.empty()) { e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
  if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
  return e;
}

// event brackets are not recorded while the stream is being captured into a CUDA graph
static bool stream_capturing(cudaStream_t st) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) { cudaGetLastError(); return false; }
  return cs != cudaStreamCaptureStatusNone;
}
static bool prof_every_launch(cudaStream_t st) { return g_prof_on && !stream_capturing(st); }

struct ProfScope {
  bool active = false;
  ProfRec rec;
  cudaStream_t st;
  ProfScope(bool enabled, int cls, double flops, double bytes, cudaStream_t s, const char* label = "", long long rows = 0,
            int c = 0) : st(s) {
    if (!enabled) return;
    rec.cls = cls; rec.flops = flops; rec.bytes = bytes; rec.rows = rows; rec.c = c;
    size_t n = 0;  // label = the launcher's name: the text up to the first '(' of the bracketed expression
    while (label[n] != 0 && label[n] != '(' && n + 1 < sizeof(rec.label)) { rec.label[n] = label[n]; ++n; }
    rec.label[n] = 0;
    rec.e0 = prof_event(); rec.e1 = prof_event();
    if (rec.e0 == nullptr || rec.e1 == nullptr) return;
    active = cudaEventRecord(rec.e0, st) == cudaSuccess;
  }
  ~ProfScope() {
    if (!active) return;
    if (cudaEventRecord(rec.e1, st) == cudaSuccess) g_prof_recs.push_back(rec);
  }
};

namespace {

constexpr size_t kAlign = 256;
inline size_t align_up(size_t v) { return (v + kAlign - 1) / kAlign * kAlign; }

struct TensorSpec {
  std::string key;
  int64_t numel = 0;
  int dtype = 0;  // 0 fp32, 1 int64
  size_t offset = 0;
  bool loaded = false;
  size_t bytes() const { return static_cast<size_t>(numel) * (dtype == 1 ? 8 : 4); }
};

struct Weight {       // packed bf16 [N, K] + its TMA descriptor
  size_t offset = 0;  // into the arena
  int N = 0, K = 0;
  CUtensorMap tmap;       // box 64 x gemm_block_n(N)
  CUtensorMap tmap_half;  // box 64 x gemm_block_n(N) / 2: the B half each CTA of a pair loads
  CUtensorMap tmap256, tmap256_half;  // N % 256 == 0: boxes of 256 / 128 rows for the 256-wide tiles
};

struct Block {
  std::string prefix;
  int dim, res, heads, window, shift, stage;
  int film_off;        // column of (scale, shift) in the film row
  Weight qkv, proj, fc1, fc2;
  CUtensorMap mlp_w1, mlp_w2;  // descriptors of fc1 / fc2 with the fused-MLP box shapes (C = 96, 192)
  CUtensorMap tail_wp, tail_w1;  // proj / fc1 with the fused block-tail box shapes (32-column k-blocks)
  CUtensorMap head_w;            // qkv with the fused block-head box shape (32 x C)
  size_t qkv_bias_off;  // fp32 [3C], q part pre-scaled
  size_t attn_bias_off; // fp32 [heads, T, T]
  int mask_canonical = 0;  // ATTN_MASK_CANONICAL / ATTN_BIAS_TOEPLITZ bits, checked at finalisation
};

struct Merge { std::string prefix; int C, res; Weight reduction; };
struct Breakup { std::string prefix; int D, res; Weight pre, post; };

}  // namespace
}  // namespace dsg

using namespace dsg;

struct dsg_model {
  dsg_config cfg;
  int nl, N, E;
  int planes_adj, planes_node, cin;
  std::vector<TensorSpec> tensors;           // state_dict order
  std::map<std::string, int> index;          // key -> tensors[]
  std::vector<Block> blocks;                 // execution order
  std::vector<int> down_first, up_first;     // index of the first block of each down / up layer
  std::vector<Merge> merges;                 // after down layer s (s < nl - 1)
  std::vector<Breakup> breakups;             // before up layer u (u >= 1), index u - 1
  int film_total = 0;
  size_t film_w_off = 0, film_b_off = 0;     // contiguous [film_total, 512] and [film_total]
  // packed extras
  size_t w_adj_off = 0, w_rc_off = 0, fold_t1_off = 0, fold_f_off = 0, fold_b_off = 0, fold_tv_off = 0;
  size_t adj_w2t_off = 0, adj_b2_off = 0, adj_b1_off = 0, node_w1t_off = 0, node_w2t_off = 0, fold_ft_off = 0;
  Weight adj_fc1;  // readout_adj_mlp.fc1 composed with the folded read_out chain
  size_t arena_bytes = 0;
  uint8_t* arena = nullptr;
  bool finalized = false;
  // the unfused schedules these three switches select are what the fusion tests compare the fused kernels against
  bool use_fused_mlp = true;  // DSG_NO_FUSED_MLP=1 keeps the LayerNorm + two-GEMM schedule
  bool use_tail = true;       // DSG_NO_TAIL=1 keeps proj GEMM + LayerNorm + fused MLP as separate launches
  bool use_head = true;       // DSG_NO_HEAD=1 keeps the FiLM + LayerNorm row kernel and the qkv GEMM as two launches
  // Padded-row skipping (SURVEY 8f-4; dsg_forward_args.skip_*): the leading `skip_stages` resolution stages are
  // computed on a compact layout holding, per sample, only the first R_b image rows (R_b = n_b rounded up to
  // `skip_granule` pixels).  0 = the geometry does not allow it (see skip_geometry below).
  int skip_stages = 0, skip_granule = 0;
  // Second level: the first block of the first DENSE stage (encoder) and that stage's last block (decoder) are
  // un-shifted too; they run on a second, coarser compact layout (corner side rounded up to skip2_granule pixels =
  // that stage's window).  0 = not available.
  int skip2_granule = 0;
  std::map<std::tuple<const void*, long long, int>, CUtensorMap> a_maps;

  const float* f32(const std::string& key) const {
    return reinterpret_cast<const float*>(arena + tensors[index.at(key)].offset);
  }
  template <typename T> T* at(size_t off) const { return reinterpret_cast<T*>(arena + off); }
};

namespace {

void skip_geometry(dsg_model* m);

void add_tensor(dsg_model* m, const std::string& key, int64_t numel, int dtype = 0) {
  TensorSpec t;
  t.key = key;
  t.numel = numel;
  t.dtype = dtype;
  m->index[key] = static_cast<int>(m->tensors.size());
  m->tensors.push_back(t);
}
void add_linear(dsg_model* m, const std::string& p, int out, int in, bool bias = true) {
  add_tensor(m, p + ".weight", static_cast<int64_t>(out) * in);
  if (bias) add_tensor(m, p + ".bias", out);
}
void add_ln(dsg_model* m, const std::string& p, int c) {
  add_tensor(m, p + ".weight", c);
  add_tensor(m, p + ".bias", c);
}

// Registration order of the reference module tree (model/diffusesg/diffusesg.py:611-720; blocks :158-230).
void add_block(dsg_model* m, const std::string& p, int dim, int res, int heads, int j, int stage) {
  const int window = m->cfg.window_size;
  Block b;
  b.prefix = p;
  b.dim = dim; b.res = res; b.heads = heads; b.stage = stage;
  if (res <= window) { b.window = res; b.shift = 0; }              // :189-192
  else { b.window = window; b.shift = (j % 2 == 0) ? 0 : window / 2; }  // :459
  const int T = b.window * b.window;
  if (b.shift > 0) {
    const int nw = (res / b.window) * (res / b.window);
    add_tensor(m, p + ".attn_mask", static_cast<int64_t>(nw) * T * T);
  }
  add_linear(m, p + ".affine", 2 * dim, 512);
  add_ln(m, p + ".norm1", dim);
  add_tensor(m, p + ".attn.relative_position_bias_table",
             static_cast<int64_t>(2 * b.window - 1) * (2 * b.window - 1) * heads);
  add_tensor(m, p + ".attn.relative_position_index", static_cast<int64_t>(T) * T, 1);
  add_linear(m, p + ".attn.qkv", 3 * dim, dim);
  add_linear(m, p + ".attn.proj", dim, dim);
  add_ln(m, p + ".norm2", dim);
  add_linear(m, p + ".mlp.fc1", 4 * dim, dim);
  add_linear(m, p + ".mlp.fc2", dim, 4 * dim);
  m->blocks.push_back(b);
}

size_t reserve(size_t& cursor, size_t bytes) {
  const size_t off = cursor;
  cursor = align_up(cursor + bytes);
  return off;
}

void reserve_weight(size_t& cursor, Weight& w, int N, int K) {
  w.N = N; w.K = K;
  w.offset = reserve(cursor, static_cast<size_t>(N) * K * 2);
}

int build(dsg_model* m) {
  const dsg_config& c = m->cfg;
  DSG_REQUIRE(c.num_stages >= 1 && c.num_stages <= 4, "config: num_stages %d", c.num_stages);
  DSG_REQUIRE(c.embed_dim == 96, "config: embed_dim %d (this build supports 96)", c.embed_dim);
  DSG_REQUIRE(c.c_e >= 1 && c.c_e <= 8 && c.c_n >= 1 && c.c_n <= 64, "config: c_e %d c_n %d", c.c_e, c.c_n);
  DSG_REQUIRE(c.img_size > 0 && c.img_size % (1 << (c.num_stages - 1)) == 0 && c.img_size % 4 == 0,
              "config: img_size %d is not divisible by the %d-stage pyramid (and by 4)", c.img_size, c.num_stages);
  m->nl = c.num_stages; m->N = c.img_size; m->E = c.embed_dim;
  const int sc = c.self_condition ? 2 : 1;
  m->planes_adj = c.c_e * sc;
  m->planes_node = c.c_n * sc;
  m->cin = m->planes_adj + 2 * m->planes_node;
  for (int s = 0; s < m->nl; ++s) {
    const int dim = m->E << s, res = m->N >> s;
    DSG_REQUIRE(c.depths[s] >= 1, "config: depth of stage %d", s);
    DSG_REQUIRE(c.num_heads[s] * 32 == dim, "config: stage %d needs %d heads of 32 channels", s, dim / 32);
    const int w = res <= c.window_size ? res : c.window_size;
    DSG_REQUIRE(res % w == 0 && (w * w) % 2 == 0 && w * w <= 256, "config: window %d on a %d-grid", w, res);
  }
  // ---- state_dict enumeration ------------------------------------------------------------------
  add_linear(m, "patch_embed.affine", 2 * m->E, 512);
  add_tensor(m, "patch_embed.proj.weight", static_cast<int64_t>(m->E) * m->cin);
  add_tensor(m, "patch_embed.proj.bias", m->E);
  add_ln(m, "patch_embed.norm", m->E);
  char buf[128];
  for (int s = 0; s < m->nl; ++s) {
    const int dim = m->E << s, res = m->N >> s;
    m->down_first.push_back(static_cast<int>(m->blocks.size()));
    for (int j = 0; j < c.depths[s]; ++j) {
      snprintf(buf, sizeof(buf), "down_layers.%d.blocks.%d", s, j);
      add_block(m, buf, dim, res, c.num_heads[s], j, s);
    }
    if (s < m->nl - 1) {
      snprintf(buf, sizeof(buf), "down_layers.%d.downsample", s);
      Merge mg; mg.prefix = buf; mg.C = dim; mg.res = res;
      add_linear(m, mg.prefix + ".reduction", 2 * dim, 4 * dim, false);
      add_ln(m, mg.prefix + ".norm", 4 * dim);
      m->merges.push_back(mg);
    }
  }
  for (int u = 0; u < m->nl; ++u) {
    const int s = m->nl - 1 - u;
    const int dim = m->E << s, res = m->N >> s;
    if (u > 0) {
      snprintf(buf, sizeof(buf), "up_layers.%d.upsample", u);
      Breakup bu; bu.prefix = buf; bu.D = 4 * dim; bu.res = res / 2;
      add_linear(m, bu.prefix + ".pre_linear", bu.D, bu.D, false);
      add_ln(m, bu.prefix + ".norm", bu.D);
      add_linear(m, bu.prefix + ".post_linear", bu.D / 4, bu.D / 4, false);
      add_ln(m, bu.prefix + ".post_norm", bu.D / 4);
      m->breakups.push_back(bu);
    }
    m->up_first.push_back(static_cast<int>(m->blocks.size()));
    for (int j = 0; j < c.depths[s]; ++j) {
      snprintf(buf, sizeof(buf), "up_layers.%d.blocks.%d", u, j);
      add_block(m, buf, dim, res, c.num_heads[s], j, s);
    }
  }
  skip_geometry(m);
  for (int k = 0; k < 3; ++k) {
    snprintf(buf, sizeof(buf), "read_out.%d", k);
    add_linear(m, buf, m->E, m->E);
  }
  add_linear(m, "map_layer0", 512, m->E);
  add_linear(m, "map_layer1", 512, 512);
  add_ln(m, "norm", m->E);
  add_linear(m, "readout_adj_mlp.fc1", m->E, m->E);
  add_linear(m, "readout_adj_mlp.fc2", c.c_e, m->E);
  add_linear(m, "readout_node_mlp.fc1", m->E, m->E);
  add_linear(m, "readout_node_mlp.fc2", c.c_n, m->E);

  // ---- arena layout ------------------------------------------------------------------------------
  size_t cur = 0;
  // all FiLM generators back to back: one [film_total, 512] matrix, one [film_total] bias
  std::vector<std::string> film_keys;
  film_keys.push_back("patch_embed.affine");
  for (const Block& b : m->blocks) film_keys.push_back(b.prefix + ".affine");
  m->film_w_off = cur;
  int off = 0;
  for (size_t i = 0; i < film_keys.size(); ++i) {
    TensorSpec& t = m->tensors[m->index[film_keys[i] + ".weight"]];
    t.offset = cur;
    cur += t.bytes();
    if (i > 0) m->blocks[i - 1].film_off = off;
    off += static_cast<int>(t.numel / 512);
  }
  m->film_total = off;
  cur = align_up(cur);
  m->film_b_off = cur;
  for (const std::string& k : film_keys) {
    TensorSpec& t = m->tensors[m->index[k + ".bias"]];
    t.offset = cur;
    cur += t.bytes();
  }
  cur = align_up(cur);
  for (TensorSpec& t : m->tensors) {
    if (t.key.size() > 7 && t.key.find(".affine.") != std::string::npos) continue;
    t.offset = reserve(cur, t.bytes());
  }
  // packed forms
  for (Block& b : m->blocks) {
    const int C = b.dim, T = b.window * b.window;
    reserve_weight(cur, b.qkv, 3 * C, C);
    reserve_weight(cur, b.proj, C, C);
    reserve_weight(cur, b.fc1, 4 * C, C);
    reserve_weight(cur, b.fc2, C, 4 * C);
    b.qkv_bias_off = reserve(cur, static_cast<size_t>(3 * C) * 4);
    b.attn_bias_off = reserve(cur, static_cast<size_t>(b.heads) * T * T * 4);
  }
  for (Merge& g : m->merges) reserve_weight(cur, g.reduction, 2 * g.C, 4 * g.C);
  for (Breakup& u : m->breakups) {
    reserve_weight(cur, u.pre, u.D, u.D);
    reserve_weight(cur, u.post, u.D / 4, u.D / 4);
  }
  const int E = m->E;
  m->w_adj_off = reserve(cur, static_cast<size_t>(m->planes_adj) * E * 4);
  m->w_rc_off = reserve(cur, static_cast<size_t>(2) * m->planes_node * E * 4);
  m->fold_t1_off = reserve(cur, static_cast<size_t>(E) * E * 4);
  m->fold_f_off = reserve(cur, static_cast<size_t>(E) * E * 4);
  m->fold_b_off = reserve(cur, static_cast<size_t>(E) * 4);
  m->fold_tv_off = reserve(cur, static_cast<size_t>(E) * 4);
  m->fold_ft_off = reserve(cur, static_cast<size_t>(E) * E * 4);
  m->adj_b1_off = reserve(cur, static_cast<size_t>(E) * 4);
  reserve_weight(cur, m->adj_fc1, E, E);
  m->adj_w2t_off = reserve(cur, static_cast<size_t>(E) * 8 * 4);
  m->adj_b2_off = reserve(cur, 8 * 4);
  m->node_w1t_off = reserve(cur, static_cast<size_t>(E) * E * 4);
  m->node_w2t_off = reserve(cur, static_cast<size_t>(E) * c.c_n * 4);
  m->arena_bytes = cur;
  return DSG_OK;
}

// Leading stages whose blocks are all un-shifted window attention on the tcgen05 kernels.  Why un-shifted only: inside
// such a stage information moves only within aligned windows, so (a) in the encoder a window that lies entirely in the
// padding of its sample (rows >= n_b: every input of mask_adjs'ed pixels is zero, diffusesg.py:796-802) holds ONE token
// value, the same for every such window of every sample at a given sigma - it is computed once, on an all-padding
// "phantom" sample; (b) in the decoder nothing computed in such a window can reach a valid output pixel (the heads mask
// padded pixels, diffusesg.py:812-825).  The first shifted block / merged-down dense stage mixes everything, so from
// there on the grid is dense (the skipped rows are filled with the phantom's token first).
void skip_geometry(dsg_model* m) {
  m->skip_stages = 0;
  m->skip_granule = 0;
  int S = 0;
  for (int s = 0; s + 1 < m->nl; ++s) {
    bool ok = true;
    for (int j = 0; j < m->cfg.depths[s]; ++j) {
      const Block& b = m->blocks[m->down_first[s] + j];
      const Block& u = m->blocks[m->up_first[m->nl - 1 - s] + j];
      // 8 x 8 windows: two windows per tile (the plan keeps every bucket's image count even); others: quad kernel
      ok = ok && b.shift == 0 && u.shift == 0 && b.window < b.res &&
           (b.window == 8 || window_attention_quad_supported(1, b.res, b.window, 0, b.heads));
    }
    if (!ok) break;
    S = s + 1;
  }
  while (S > 0) {
    const int g = m->blocks[m->down_first[S - 1]].window << (S - 1);  // window of the coarsest compact stage, in pixels
    if (g < m->N && m->N % g == 0) { m->skip_stages = S; m->skip_granule = g; break; }
    --S;  // a single window spans the whole grid there: nothing to skip at that stage
  }
  m->skip2_granule = 0;
  if (S == 0 || S > m->nl - 1) return;
  // level 2 at stage S: its first encoder block and its last decoder block must be un-shifted window attention over more
  // than one window, with at least one (shifted) block between them and the rest of the network
  const int d = m->cfg.depths[S];
  if (d < 2) return;
  const Block& e0 = m->blocks[m->down_first[S]];
  const Block& dl = m->blocks[m->up_first[m->nl - 1 - S] + d - 1];
  const bool ok = e0.shift == 0 && dl.shift == 0 && e0.window < e0.res && dl.window == e0.window &&
                  (e0.window == 8 || window_attention_quad_supported(1, e0.res, e0.window, 0, e0.heads));
  const int g2 = e0.window << S;
  if (ok && g2 < m->N && m->N % g2 == 0 && g2 % m->skip_granule == 0) m->skip2_granule = g2;
}

int pack_weight(dsg_model* m, Weight& w, const std::string& key, cudaStream_t st, int64_t n_scaled = 0,
                float scale = 1.f) {
  int rc = launch_pack_bf16(m->f32(key), m->at<bf16>(w.offset), static_cast<int64_t>(w.N) * w.K, n_scaled, scale, st);
  if (rc) return rc;
  if (int rc2 = make_tmap_bf16(&w.tmap_half, m->arena + w.offset, w.N, w.K, gemm_block_n(w.N) / 2)) return rc2;
  if (w.N % 256 == 0) {
    if (int rc2 = make_tmap_bf16(&w.tmap256, m->arena + w.offset, w.N, w.K, 256)) return rc2;
    if (int rc2 = make_tmap_bf16(&w.tmap256_half, m->arena + w.offset, w.N, w.K, 128)) return rc2;
  }
  return make_tmap_bf16(&w.tmap, m->arena + w.offset, w.N, w.K, gemm_block_n(w.N));
}

struct Workspace {
  float *X, *T, *coef, *emb0, *emb1, *emb, *film, *rc;
  std::vector<float*> skip;
  bf16 *Y, *QKV, *ATT, *H;
  size_t bytes;
};

// Token layout of an activation.  The compact layouts of the padding skipping (see skip_geometry) group the samples into
// K buckets by the side of their kept corner: bucket k is a stack of count[k] images of side[k] x side[k] pixels (>> s
// tokens at stage s), image i showing sample perm[img0[k] + i]; the buckets follow each other in memory.  The dense grid is
// the special case of one bucket of B images of side N and no tables.  Every geometry-aware kernel runs once per bucket on
// an ordinary (batch, res) = (count[k], side[k] >> s) tensor; every row-wise kernel runs once over all tokens.
struct Layout {
  int level = 0;                    // 0: the dense grid; 1, 2: the compaction level of the padding skipping
  int K = 0;
  int count[8], side[8], img0[8];   // images, side in pixels, index of the first image in `perm`
  long long tok[9];                 // stage-0 token offset of each bucket; tok[K] = all tokens
  const int *perm = nullptr, *tok0 = nullptr, *width = nullptr;   // device tables (include/dsg_b200.h); null: dense
  bool dense() const { return perm == nullptr; }
  const int* bucket_perm(int k) const { return perm != nullptr ? perm + img0[k] : nullptr; }
  long long tokens(int s) const { return tok[K] >> (2 * s); }
  long long at(int k, int s) const { return tok[k] >> (2 * s); }
};

Layout dense_layout(int B, int N) {
  Layout l;
  l.K = 1;
  l.count[0] = B; l.side[0] = N; l.img0[0] = 0;
  l.tok[0] = 0; l.tok[1] = static_cast<long long>(B) * N * N;
  return l;
}

// The compact layout of compaction level `level` from the plan of dsg_forward_args (skip_* / skip2_* fields): a batch of
// B samples of side N, corner sides a multiple of the granule G.
int parse_plan(Layout& c, int level, const int32_t* tables, int table_images, int buckets, const int32_t* counts,
               const int32_t* sides, long long phantom_tok0, int G, int B, int N) {
  DSG_REQUIRE(buckets > 0 && buckets <= 8 && table_images > 0, "forward: %d buckets", buckets);
  c.level = level;
  c.K = buckets;
  long long tok = 0;
  int img = 0;
  for (int k = 0; k < c.K; ++k) {
    c.count[k] = counts[k];
    c.side[k] = sides[k];
    DSG_REQUIRE(c.count[k] > 0 && c.count[k] % 2 == 0 && c.side[k] >= G && c.side[k] <= N && c.side[k] % G == 0,
                "forward: bucket %d holds %d images of side %d (granule %d)", k, c.count[k], c.side[k], G);
    c.img0[k] = img;
    c.tok[k] = tok;
    img += c.count[k];
    tok += static_cast<long long>(c.count[k]) * c.side[k] * c.side[k];
  }
  c.tok[c.K] = tok;
  DSG_REQUIRE(img <= table_images && tok <= static_cast<long long>(B + 1) * N * N,
              "forward: the compact plan holds %d images / %lld pixels (table %d, capacity %lld)", img, tok, table_images,
              static_cast<long long>(B + 1) * N * N);
  DSG_REQUIRE(phantom_tok0 >= 0 && phantom_tok0 + static_cast<long long>(G) * G <= tok, "forward: phantom offset");
  c.perm = tables;
  c.tok0 = c.perm + table_images;
  c.width = c.tok0 + B;
  return DSG_OK;
}

// The dsg_forward_args row map through which a kernel running in layout `to` reads a tensor stored in layout `from`;
// nullptr when both are the same.  Level 1 is entered only by the breakup, which writes it directly, so no map leads there.
const int* row_map(const dsg_forward_args* a, const Layout& from, const Layout& to) {
  if (from.level == to.level) return nullptr;
  if (from.level == 1) return to.level == 2 ? a->skip2_map_c2_from_c1 : a->skip_map_dense_from_c1;
  return to.level == 2 ? a->skip2_map_c2_from_dense : a->skip2_map_dense_from_c2;
}

Workspace carve(const dsg_model* m, int batch, int n_cond, void* base) {
  Workspace w;
  uint8_t* p = static_cast<uint8_t*>(base);
  size_t cur = 0;
  // one extra sample of capacity: the compact layout of the padding skipping adds the phantom and up to one dummy
  // image per bucket (a plan that would not fit is refused by the caller and the dense schedule runs)
  const size_t tok0 = static_cast<size_t>(batch + (m->skip_stages > 0 ? 1 : 0)) * m->N * m->N;
  const size_t full = tok0 * m->E;  // elements of a stage-0 activation; later stages hold full / 2^s
  auto take = [&](size_t bytes) { void* r = p ? p + cur : nullptr; cur = align_up(cur + bytes); return r; };
  w.X = static_cast<float*>(take(full * 4));
  w.T = static_cast<float*>(take(full * 4));
  w.Y = static_cast<bf16*>(take(full * 2));
  w.QKV = static_cast<bf16*>(take(full * 3 * 2));
  w.ATT = static_cast<bf16*>(take(full * 2));
  w.H = static_cast<bf16*>(take(full * 4 * 2));
  for (int s = 0; s + 1 < m->nl; ++s) w.skip.push_back(static_cast<float*>(take((full >> (s + 1)) * 4)));
  w.coef = static_cast<float*>(take(static_cast<size_t>(4) * batch * 4));
  w.emb0 = static_cast<float*>(take(static_cast<size_t>(n_cond) * m->E * 4));
  w.emb1 = static_cast<float*>(take(static_cast<size_t>(n_cond) * 512 * 4));
  w.emb = static_cast<float*>(take(static_cast<size_t>(n_cond) * 512 * 4));
  w.film = static_cast<float*>(take(static_cast<size_t>(n_cond) * m->film_total * 4));
  w.rc = static_cast<float*>(take(static_cast<size_t>(batch) * m->N * 2 * m->E * 4));
  w.bytes = cur;
  return w;
}

int gemm(dsg_model* m, const bf16* A, long long rows, const Weight& W, int epi, const float* bias, const float* res,
         void* out, cudaStream_t st, const GemmParams* extra = nullptr) {
  DSG_REQUIRE(rows > 0 && rows < 2147483647LL, "gemm: %lld rows", rows);
  auto key = std::make_tuple(static_cast<const void*>(A), rows, W.K);
  auto it = m->a_maps.find(key);
  if (it == m->a_maps.end()) {
    CUtensorMap tm;
    int rc = make_tmap_bf16(&tm, A, rows, W.K, 128);
    if (rc) return rc;
    if (m->a_maps.size() > 4096) m->a_maps.clear();
    it = m->a_maps.emplace(key, tm).first;
  }
  const CUtensorMap* tmo = &it->second;  // placeholder for the adj-head epilogue, which stores directly
  if (epi != EPI_ADJ_HEAD) {
    auto okey = std::make_tuple(static_cast<const void*>(out), rows, -(W.N * 8 + epi));
    auto ot = m->a_maps.find(okey);
    if (ot == m->a_maps.end()) {
      CUtensorMap tm;
      int rc = make_tmap_out(&tm, out, rows, W.N, epi);
      if (rc) return rc;
      ot = m->a_maps.emplace(okey, tm).first;
    }
    tmo = &ot->second;
  }
  GemmParams p;
  if (extra) p = *extra; else memset(&p, 0, sizeof(p));
  p.M = static_cast<int>(rows); p.N = W.N; p.K = W.K;
  p.bias = bias; p.res = res; p.out = out; p.ldo = W.N;
  const double mn = static_cast<double>(rows) * W.N;
  const double out_bytes = epi == EPI_ADJ_HEAD ? static_cast<double>(rows) * (extra ? extra->c_e : 0) * 4
                                               : mn * ((epi == EPI_BF16 || epi == EPI_GELU_BF16) ? 2 : 4);
  char label[56];
  snprintf(label, sizeof(label), "gemm_n%d_k%d_epi%d", W.N, W.K, epi);
  ProfScope ps(g_prof_pass, PC_GEMM, 2.0 * mn * W.K,
               static_cast<double>(rows) * W.K * 2 + static_cast<double>(W.N) * W.K * 2 + out_bytes +
                   (epi == EPI_RES_F32 ? mn * 4 : 0), st, label, rows, W.K);
  const bool pair = gemm_use_pair(rows, W.K, epi);
  p.bn = gemm_choose_bn(rows, W.N, W.K, epi, pair);
  if (p.bn == 256) return launch_gemm(&it->second, pair ? &W.tmap256_half : &W.tmap256, tmo, epi, p, st, pair);
  return launch_gemm(&it->second, pair ? &W.tmap_half : &W.tmap, tmo, epi, p, st, pair);
}

#define DSG_TRY(expr)        \
  do {                       \
    int _rc = (expr);        \
    if (_rc) return _rc;     \
  } while (0)

// same, bracketed by a pair of CUDA events when this pass is being profiled (algorithmic flops / bytes attached)
#define DSG_TRY_P(cls, flops, bytes, expr)                                    \
  do {                                                                        \
    ProfScope _ps(g_prof_pass, cls, flops, bytes, st, #expr);                 \
    int _rc = (expr);                                                         \
    if (_rc) return _rc;                                                      \
  } while (0)

// lay: the layout the block runs in - the activation holds lay.tokens(stage) tokens, bucket by bucket (see Layout)
// x_in_rows: x_in is in another layout; row r of this block reads x_in row x_in_rows[r] (x_in must not be w.X)
// fuse_final_ln: this is the last block of the network; if it runs the fused tail, the tail also applies the final
// LayerNorm and writes only Y (*fused_final_ln = true), and the caller skips the separate LayerNorm launch.
int run_block(dsg_model* m, const Block& b, const Workspace& w, const float* x_in, const Layout& lay, const int* x_in_rows,
              int cond_uniform, cudaStream_t st, bool fuse_final_ln, bool* fused_final_ln) {
  const int C = b.dim;
  const int L = b.res * b.res;
  const long long rows = lay.tokens(b.stage);
  const std::string& p = b.prefix;
  const double rc = static_cast<double>(rows) * C;
  auto tmap = [&](const void* ptr, int key, auto make) -> const CUtensorMap* {
    auto k = std::make_tuple(ptr, rows, key);
    auto it = m->a_maps.find(k);
    if (it == m->a_maps.end()) {
      CUtensorMap tm;
      if (make(&tm)) return nullptr;
      it = m->a_maps.emplace(k, tm).first;
    }
    return &it->second;
  };
  DSG_REQUIRE(x_in_rows == nullptr || (x_in != w.X && !block_head_supported(C)), "run_block: layout-changing input at C = %d", C);
  if (m->use_head && block_head_supported(C)) {
    // x = silu(FiLM(x)); qkv = LN1(x) W^T + b in one launch                (:238-243, :115)
    const CUtensorMap* ti = tmap(x_in, -(C * 8 + EPI_RES_F32), [&](CUtensorMap* t) { return make_tmap_out(t, x_in, rows, C, EPI_RES_F32); });
    const CUtensorMap* to = tmap(w.X, -(C * 8 + EPI_RES_F32), [&](CUtensorMap* t) { return make_tmap_out(t, w.X, rows, C, EPI_RES_F32); });
    const CUtensorMap* tq = tmap(w.QKV, -(3 * C * 8 + EPI_BF16), [&](CUtensorMap* t) { return make_tmap_out(t, w.QKV, rows, 3 * C, EPI_BF16); });
    if (ti == nullptr || to == nullptr || tq == nullptr) return DSG_ERR_CUDA;
    DSG_TRY_P(PC_MLP, 6.0 * rc * C, rc * 14,
              launch_block_head(ti, to, &b.head_w, tq, w.film + b.film_off, m->film_total, cond_uniform, L,
                                m->f32(p + ".norm1.weight"), m->f32(p + ".norm1.bias"), m->at<float>(b.qkv_bias_off), rows,
                                C, st));
  } else {
    // x = silu(FiLM(x)); y = LN1(x)                                        (:238-243)
    // per-sample FiLM rows exist only on the dense grid: a compact layout needs one shared condition
    const int per_sample = cond_uniform ? static_cast<int>(rows) : L;
    DSG_TRY_P(PC_ROW, 0, rc * 10, launch_film_ln(x_in, w.X, w.Y, w.film, m->film_total, b.film_off, cond_uniform,
                                                 m->f32(p + ".norm1.weight"), m->f32(p + ".norm1.bias"),
                                                 static_cast<int>(rows / per_sample), per_sample, C, st, x_in_rows));
    DSG_TRY(gemm(m, w.Y, rows, b.qkv, EPI_BF16, m->at<float>(b.qkv_bias_off), nullptr, w.QKV, st));
  }
  const float* mask = b.shift > 0 ? m->f32(p + ".attn_mask") : nullptr;
  if (!lay.dense() && b.window == 8 && lay.K <= 4) {
    // 8 x 8 windows: all buckets in ONE launch (a tensor-map pair per bucket); per-bucket launches of the persistent
    // kernel each paid its prologue and pipeline ramp for a handful of windows per CTA
    int res_k[4];
    long long tok_k[4];
    for (int k = 0; k < lay.K; ++k) { res_k[k] = lay.side[k] >> b.stage; tok_k[k] = lay.at(k, b.stage); }
    DSG_TRY_P(PC_ATTN, 4.0 * rc * b.window * b.window, rc * 8,
              launch_window_attention_tc_groups(w.QKV, m->at<float>(b.attn_bias_off), w.ATT, lay.K, lay.count, res_k, tok_k, b.heads, st));
  } else {
    for (int k = 0; k < lay.K; ++k) {   // one (count, side) tensor per bucket
      const long long t0 = lay.at(k, b.stage), tk = lay.at(k + 1, b.stage) - t0;
      DSG_TRY_P(PC_ATTN, 4.0 * tk * C * b.window * b.window, static_cast<double>(tk) * C * 8,
                launch_window_attention(w.QKV + t0 * 3 * C, m->at<float>(b.attn_bias_off), mask, w.ATT + t0 * C, lay.count[k],
                                        lay.side[k] >> b.stage, b.window, b.shift, b.heads, st, b.mask_canonical));
    }
  }
  if (m->use_tail && block_tail_supported(C)) {
    // x += proj(attn); x += fc2(gelu(fc1(LN2(x))))  in one launch        (:137, :272, :275)
    const CUtensorMap* ta = tmap(w.ATT, 100000 + C, [&](CUtensorMap* t) { return make_tmap_2d(t, w.ATT, rows, C, 2, 32, 128); });
    const CUtensorMap* tx = tmap(w.X, -(C * 8 + EPI_RES_F32), [&](CUtensorMap* t) { return make_tmap_out(t, w.X, rows, C, EPI_RES_F32); });
    if (ta == nullptr || tx == nullptr) return DSG_ERR_CUDA;
    const CUtensorMap* ty = nullptr;
    if (fuse_final_ln) {
      ty = tmap(w.Y, -(C * 8 + EPI_BF16), [&](CUtensorMap* t) { return make_tmap_out(t, w.Y, rows, C, EPI_BF16); });
      if (ty == nullptr) return DSG_ERR_CUDA;
      if (fused_final_ln) *fused_final_ln = true;
    }
    DSG_TRY_P(PC_MLP, 18.0 * rc * C, rc * (fuse_final_ln ? 8 : 10),
              launch_block_tail(ta, &b.tail_wp, &b.tail_w1, &b.mlp_w2, tx, m->f32(p + ".attn.proj.bias"),
                                m->f32(p + ".norm2.weight"), m->f32(p + ".norm2.bias"), m->f32(p + ".mlp.fc1.bias"),
                                m->f32(p + ".mlp.fc2.bias"), w.X, rows, C, st, ty,
                                fuse_final_ln ? m->f32("norm.weight") : nullptr,
                                fuse_final_ln ? m->f32("norm.bias") : nullptr));
    return DSG_OK;
  }
  if (C == 384) {  // the fused kernel: 126 vs 146 us at C = 384, only break-even at C = 192 (projln.cu)
    // x = x + proj(attn);  y = LN2(x)  in one launch                     (:137, :272, :275)
    const CUtensorMap* ta = tmap(w.ATT, C, [&](CUtensorMap* t) { return make_tmap_bf16(t, w.ATT, rows, C, 128); });
    if (ta == nullptr) return DSG_ERR_CUDA;
    DSG_TRY_P(PC_MLP, 2.0 * rc * C, rc * 12,
              launch_proj_ln(ta, &b.proj.tmap, m->f32(p + ".attn.proj.bias"), m->f32(p + ".norm2.weight"),
                             m->f32(p + ".norm2.bias"), w.X, w.Y, rows, C, st));
  } else {
    // x = x + proj(attn)                                                   (:137, :272)
    DSG_TRY(gemm(m, w.ATT, rows, b.proj, EPI_RES_F32, m->f32(p + ".attn.proj.bias"), w.X, w.X, st));
    // y = LN2(x)                                                           (:275)
    DSG_TRY_P(PC_ROW, 0, rc * 6, launch_ln(w.X, w.Y, m->f32(p + ".norm2.weight"), m->f32(p + ".norm2.bias"), rows, C, st));
  }
  // x = x + fc2(gelu(fc1(y)))                                            (:275)
  if (m->use_fused_mlp && fused_mlp_supported(C)) {
    const CUtensorMap* ty = tmap(w.Y, C, [&](CUtensorMap* t) { return make_tmap_bf16(t, w.Y, rows, C, 128); });
    const CUtensorMap* tx = tmap(w.X, -(C * 8 + EPI_RES_F32), [&](CUtensorMap* t) { return make_tmap_out(t, w.X, rows, C, EPI_RES_F32); });
    if (ty == nullptr || tx == nullptr) return DSG_ERR_CUDA;
    DSG_TRY_P(PC_MLP, 16.0 * rc * C, rc * 10,
              launch_fused_mlp(ty, &b.mlp_w1, &b.mlp_w2, tx, m->f32(p + ".mlp.fc1.bias"), m->f32(p + ".mlp.fc2.bias"), rows,
                               C, st));
    return DSG_OK;
  }
  DSG_TRY(gemm(m, w.Y, rows, b.fc1, EPI_GELU_BF16, m->f32(p + ".mlp.fc1.bias"), nullptr, w.H, st));
  DSG_TRY(gemm(m, w.H, rows, b.fc2, EPI_RES_F32, m->f32(p + ".mlp.fc2.bias"), w.X, w.X, st));
  return DSG_OK;
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int dsg_abi_version(void) { return DSG_ABI_VERSION; }
void dsg_debug_set_smem_poison(unsigned pattern, int enable) {
  g_smem_poison = pattern;
  g_smem_poison_on = enable != 0;
}
const char* dsg_last_error(void) { return g_err; }
uint64_t dsg_launch_count(void) { return __atomic_load_n(&g_launches, __ATOMIC_RELAXED); }

int dsg_model_create(const dsg_config* cfg, dsg_model** out) {
  DSG_REQUIRE(cfg != nullptr && out != nullptr, "dsg_model_create: null argument");
  dsg_model* m = new dsg_model();
  m->cfg = *cfg;
  const char* no_fuse = getenv("DSG_NO_FUSED_MLP");
  m->use_fused_mlp = !(no_fuse != nullptr && no_fuse[0] == '1');
  const char* no_tail = getenv("DSG_NO_TAIL");
  m->use_tail = !(no_tail != nullptr && no_tail[0] == '1');
  const char* no_head = getenv("DSG_NO_HEAD");
  m->use_head = !(no_head != nullptr && no_head[0] == '1');
  const int rc = build(m);
  if (rc) { delete m; return rc; }
  *out = m;
  return DSG_OK;
}

void dsg_model_destroy(dsg_model* m) { delete m; }

size_t dsg_model_arena_bytes(const dsg_model* m) { return m ? m->arena_bytes : 0; }

int dsg_model_bind_arena(dsg_model* m, void* arena, size_t bytes) {
  DSG_REQUIRE(m != nullptr && arena != nullptr, "bind_arena: null argument");
  if (bytes < m->arena_bytes || (reinterpret_cast<uintptr_t>(arena) & (kAlign - 1)) != 0) {
    set_last_error("bind_arena: need %zu bytes aligned to %zu, got %zu at %p", m->arena_bytes, kAlign, bytes, arena);
    return DSG_ERR_WORKSPACE;
  }
  m->arena = static_cast<uint8_t*>(arena);
  m->finalized = false;
  for (TensorSpec& t : m->tensors) t.loaded = false;
  return DSG_OK;
}

int dsg_model_num_tensors(const dsg_model* m) { return m ? static_cast<int>(m->tensors.size()) : 0; }

int dsg_model_tensor_info(const dsg_model* m, int i, const char** key, int64_t* numel, int32_t* dtype) {
  DSG_REQUIRE(m != nullptr && i >= 0 && i < static_cast<int>(m->tensors.size()), "tensor_info: index %d", i);
  if (key) *key = m->tensors[i].key.c_str();
  if (numel) *numel = m->tensors[i].numel;
  if (dtype) *dtype = m->tensors[i].dtype;
  return DSG_OK;
}

int dsg_model_set_tensor(dsg_model* m, const char* key, const void* src, int64_t bytes, int src_is_host,
                         dsg_stream_t stream) {
  DSG_REQUIRE(m != nullptr && key != nullptr && src != nullptr, "set_tensor: null argument");
  if (m->arena == nullptr) { set_last_error("set_tensor: no arena bound"); return DSG_ERR_STATE; }
  auto it = m->index.find(key);
  if (it == m->index.end()) { set_last_error("set_tensor: unknown key '%s'", key); return DSG_ERR_UNKNOWN_KEY; }
  TensorSpec& t = m->tensors[it->second];
  DSG_REQUIRE(static_cast<size_t>(bytes) == t.bytes(), "set_tensor: '%s' expects %zu bytes, got %lld", key, t.bytes(),
              static_cast<long long>(bytes));
  DSG_CUDA_CHECK(cudaMemcpyAsync(m->arena + t.offset, src, t.bytes(),
                                 src_is_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice,
                                 static_cast<cudaStream_t>(stream)));
  t.loaded = true;
  m->finalized = false;
  return DSG_OK;
}

int dsg_model_tensor_differs(const dsg_model* m, const char* key, const void* src, int64_t bytes, int32_t* flag,
                             dsg_stream_t stream) {
  DSG_REQUIRE(m != nullptr && key != nullptr && src != nullptr && flag != nullptr, "tensor_differs: null argument");
  if (m->arena == nullptr) { set_last_error("tensor_differs: no arena bound"); return DSG_ERR_STATE; }
  auto it = m->index.find(key);
  if (it == m->index.end()) { set_last_error("tensor_differs: unknown key '%s'", key); return DSG_ERR_UNKNOWN_KEY; }
  const TensorSpec& t = m->tensors[it->second];
  DSG_REQUIRE(static_cast<size_t>(bytes) == t.bytes() && (reinterpret_cast<uintptr_t>(src) & 3) == 0,
              "tensor_differs: '%s' expects %zu bytes (4-byte aligned), got %lld", key, t.bytes(), static_cast<long long>(bytes));
  return launch_compare_words(m->arena + t.offset, src, static_cast<int64_t>(t.bytes() / 4), flag,
                              static_cast<cudaStream_t>(stream));
}

int dsg_model_finalize(dsg_model* m, dsg_stream_t stream) {
  DSG_REQUIRE(m != nullptr, "finalize: null model");
  if (m->arena == nullptr) { set_last_error("finalize: no arena bound"); return DSG_ERR_STATE; }
  for (const TensorSpec& t : m->tensors)
    if (!t.loaded) { set_last_error("finalize: tensor '%s' was never set", t.key.c_str()); return DSG_ERR_STATE; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float qscale = 0.17677669529663687f;  // head_dim ** -0.5 with head_dim = 32 (diffusesg.py:76, :118)
  for (Block& b : m->blocks) {
    const int C = b.dim, T = b.window * b.window;
    const std::string& p = b.prefix;
    DSG_TRY(pack_weight(m, b.qkv, p + ".attn.qkv.weight", st, static_cast<int64_t>(C) * C, qscale));
    DSG_TRY(launch_scale_copy(m->f32(p + ".attn.qkv.bias"), m->at<float>(b.qkv_bias_off), 3 * C, C, qscale, st));
    DSG_TRY(pack_weight(m, b.proj, p + ".attn.proj.weight", st));
    DSG_TRY(pack_weight(m, b.fc1, p + ".mlp.fc1.weight", st));
    DSG_TRY(pack_weight(m, b.fc2, p + ".mlp.fc2.weight", st));
    if (fused_mlp_supported(C)) {
      DSG_TRY(make_tmap_bf16(&b.mlp_w1, m->arena + b.fc1.offset, 4 * C, C, fused_mlp_w1_box_rows(C)));
      DSG_TRY(make_tmap_bf16(&b.mlp_w2, m->arena + b.fc2.offset, C, 4 * C, C));
    }
    if (block_head_supported(C)) DSG_TRY(make_tmap_2d(&b.head_w, m->arena + b.qkv.offset, 3 * C, C, 2, 32, C));
    if (block_tail_supported(C)) {
      DSG_TRY(make_tmap_2d(&b.tail_wp, m->arena + b.proj.offset, C, C, 2, 32, C));
      DSG_TRY(make_tmap_2d(&b.tail_w1, m->arena + b.fc1.offset, 4 * C, C, 2, 32, 128));
    }
    const TensorSpec& idx = m->tensors[m->index[p + ".attn.relative_position_index"]];
    DSG_TRY(launch_bias_expand(m->f32(p + ".attn.relative_position_bias_table"),
                               reinterpret_cast<const int64_t*>(m->arena + idx.offset), m->at<float>(b.attn_bias_off), T,
                               b.heads, (2 * b.window - 1) * (2 * b.window - 1), st));
    // the tcgen05 attention kernels generate the SW-MSA mask in registers: only for the reference's own values
    b.mask_canonical = 0;
    const bool w16 = window_attention_w16_supported(1, b.res, b.window, b.shift, b.heads);
    if (b.shift > 0 && (w16 || window_attention_quad_supported(1, b.res, b.window, b.shift, b.heads))) {
      int ok = 0;
      DSG_TRY(check_mask_canonical(m->f32(p + ".attn_mask"), b.res, b.window, b.shift, st, &ok));
      if (ok) b.mask_canonical |= ATTN_MASK_CANONICAL;
    }
    if (w16) {  // the 16 x 16 kernel looks the bias up by token offset
      int ok = 0;
      DSG_TRY(check_bias_toeplitz(m->at<float>(b.attn_bias_off), b.heads, b.window, st, &ok));
      if (ok) b.mask_canonical |= ATTN_BIAS_TOEPLITZ;
    }
  }
  for (Merge& g : m->merges) DSG_TRY(pack_weight(m, g.reduction, g.prefix + ".reduction.weight", st));
  for (Breakup& u : m->breakups) {
    DSG_TRY(pack_weight(m, u.pre, u.prefix + ".pre_linear.weight", st));
    DSG_TRY(pack_weight(m, u.post, u.prefix + ".post_linear.weight", st));
  }
  const int E = m->E;
  // patch embedding: split the 1x1 conv into its adjacency and node row / column parts, input-channel major
  const float* wp = m->f32("patch_embed.proj.weight");  // [E, cin]
  DSG_TRY(launch_transpose(wp, m->at<float>(m->w_adj_off), E, m->cin, 0, m->planes_adj, E, st));
  DSG_TRY(launch_transpose(wp, m->at<float>(m->w_rc_off), E, m->cin, m->planes_adj, m->planes_node, E, st));
  DSG_TRY(launch_transpose(wp, m->at<float>(m->w_rc_off) + static_cast<size_t>(m->planes_node) * E, E, m->cin,
                           m->planes_adj + m->planes_node, m->planes_node, E, st));
  // read_out = ConvTranspose2d(1x1) -> Conv2d(1x1) -> Conv2d(1x1) with no activation between (:705-709): one
  // 96x96 map.  ConvTranspose2d stores its weight as [in, out].
  float* t1 = m->at<float>(m->fold_t1_off);
  float* ff = m->at<float>(m->fold_f_off);
  float* tv = m->at<float>(m->fold_tv_off);
  DSG_TRY(launch_small_mm(m->f32("read_out.1.weight"), m->f32("read_out.0.weight"), t1, E, 1, st));
  DSG_TRY(launch_small_mm(m->f32("read_out.2.weight"), t1, ff, E, 0, st));
  DSG_TRY(launch_small_mv(m->f32("read_out.1.weight"), m->f32("read_out.0.bias"), m->f32("read_out.1.bias"), tv, E, st));
  DSG_TRY(launch_small_mv(m->f32("read_out.2.weight"), tv, m->f32("read_out.2.bias"), m->at<float>(m->fold_b_off), E, st));
  // adj head: fc1 composed with the folded read_out (fp32 composition, one bf16 rounding of the product), so the
  // shared representation [B, 96, N, N] of :761 is never written; the node head pools LN(x) and applies the
  // fold after the (linear) masked row mean
  DSG_TRY(launch_small_mm(m->f32("readout_adj_mlp.fc1.weight"), ff, t1, E, 0, st));
  DSG_TRY(launch_pack_bf16(t1, m->at<bf16>(m->adj_fc1.offset), static_cast<int64_t>(E) * E, 0, 1.f, st));
  DSG_TRY(make_tmap_bf16(&m->adj_fc1.tmap, m->arena + m->adj_fc1.offset, E, E, gemm_block_n(E)));
  DSG_TRY(launch_small_mv(m->f32("readout_adj_mlp.fc1.weight"), m->at<float>(m->fold_b_off),
                          m->f32("readout_adj_mlp.fc1.bias"), m->at<float>(m->adj_b1_off), E, st));
  DSG_TRY(launch_transpose(ff, m->at<float>(m->fold_ft_off), E, E, 0, E, E, st));
  DSG_CUDA_CHECK(cudaMemsetAsync(m->at<float>(m->adj_w2t_off), 0, static_cast<size_t>(E) * 8 * 4, st));
  DSG_CUDA_CHECK(cudaMemsetAsync(m->at<float>(m->adj_b2_off), 0, 8 * 4, st));
  DSG_TRY(launch_transpose(m->f32("readout_adj_mlp.fc2.weight"), m->at<float>(m->adj_w2t_off), m->cfg.c_e, E, 0, E, 8, st));
  DSG_CUDA_CHECK(cudaMemcpyAsync(m->at<float>(m->adj_b2_off), m->f32("readout_adj_mlp.fc2.bias"), m->cfg.c_e * 4,
                                 cudaMemcpyDeviceToDevice, st));
  DSG_TRY(launch_transpose(m->f32("readout_node_mlp.fc1.weight"), m->at<float>(m->node_w1t_off), E, E, 0, E, E, st));
  DSG_TRY(launch_transpose(m->f32("readout_node_mlp.fc2.weight"), m->at<float>(m->node_w2t_off), m->cfg.c_n, E, 0, E,
                           m->cfg.c_n, st));
  m->finalized = true;
  return DSG_OK;
}

int dsg_model_skip_info(const dsg_model* m, int32_t* stages, int32_t* granule) {
  DSG_REQUIRE(m != nullptr && stages != nullptr && granule != nullptr, "skip_info: null argument");
  *stages = m->skip_stages;
  *granule = m->skip_granule;
  return DSG_OK;
}

int dsg_model_skip_info2(const dsg_model* m, int32_t* granule2) {
  DSG_REQUIRE(m != nullptr && granule2 != nullptr, "skip_info2: null argument");
  *granule2 = m->skip2_granule;
  return DSG_OK;
}

size_t dsg_workspace_bytes(const dsg_model* m, int batch, int n_cond) {
  if (m == nullptr || batch <= 0 || n_cond <= 0) return 0;
  return carve(m, batch, n_cond, nullptr).bytes;
}

int dsg_denoiser_forward(dsg_model* m, const dsg_forward_args* a, dsg_stream_t stream) {
  DSG_REQUIRE(m != nullptr && a != nullptr, "forward: null argument");
  DSG_REQUIRE(a->struct_size == sizeof(dsg_forward_args), "forward: dsg_forward_args size %u, library expects %zu",
              a->struct_size, sizeof(dsg_forward_args));
  if (!m->finalized) { set_last_error("forward: dsg_model_finalize has not been called since the last weight update"); return DSG_ERR_STATE; }
  DSG_REQUIRE(a->batch > 0 && (a->n_cond == 1 || a->n_cond == a->batch), "forward: batch %d n_cond %d", a->batch, a->n_cond);
  DSG_REQUIRE(a->mode == 0 || a->mode == 1, "forward: mode %d", a->mode);
  DSG_REQUIRE(a->adj && a->node && a->flags && a->noise && a->out_adj && a->out_node, "forward: null tensor");
  DSG_REQUIRE((reinterpret_cast<uintptr_t>(a->flags) & 3) == 0, "forward: node_flags must be 4-byte aligned");
  DSG_REQUIRE(static_cast<long long>(a->batch) * m->N * m->N < 2147483647LL, "forward: batch %d too large", a->batch);
  const int B = a->batch, N = m->N, E = m->E;
  Workspace w = carve(m, B, a->n_cond, a->workspace);   // X and T trade places at the layout changes of the padding skipping
  if (a->workspace == nullptr || a->workspace_bytes < w.bytes ||
      (reinterpret_cast<uintptr_t>(a->workspace) & (kAlign - 1)) != 0) {
    set_last_error("forward: workspace needs %zu bytes aligned to %zu (got %zu at %p)", w.bytes, kAlign,
                   a->workspace_bytes, a->workspace);
    return DSG_ERR_WORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int uniform = a->n_cond == 1 ? 1 : 0;
  const float *c_in = nullptr, *c_skip = nullptr, *c_out = nullptr;
  const float* labels = a->noise;
  long long label_stride = a->noise_stride;
  if (a->mode == 1) {
    // coefficients for every sample (a shared sigma is broadcast), c_noise doubles as the noise labels
    DSG_TRY(launch_precond_coef(a->noise, uniform ? 0 : static_cast<int>(a->noise_stride), w.coef, B, st));
    c_in = w.coef; c_skip = w.coef + B; c_out = w.coef + 2 * B;
    labels = w.coef + 3 * B;
    label_stride = 1;
  }
  // ---- layouts: the dense grid and the compact layouts of the padding skipping (see skip_geometry, Layout) ----------
  const Layout dense = dense_layout(B, N);
  Layout l1, l2;
  int S = 0;            // stages 0 .. S - 1 run in l1
  bool level2 = false;  // the first encoder block and the last decoder block of stage S run in l2
  if (a->skip_tables != nullptr && a->skip_buckets > 0) {
    DSG_REQUIRE(m->skip_stages > 0, "forward: this geometry has no compactable stage (skip_tables given)");
    DSG_REQUIRE(uniform, "forward: padding skipping needs one shared noise level (n_cond == 1)");
    DSG_REQUIRE(g_stop_after < 0, "forward: the stage-walk test hook runs on the dense schedule");
    DSG_TRY(parse_plan(l1, 1, a->skip_tables, a->skip_table_images, a->skip_buckets, a->skip_count, a->skip_side,
                       a->skip_phantom_tok0, m->skip_granule, B, N));
    S = m->skip_stages;
    DSG_REQUIRE((a->skip2_tables != nullptr && a->skip2_buckets > 0) || a->skip_map_dense_from_c1 != nullptr,
                "forward: the row map dense <- compact is missing");
    if (a->skip2_tables != nullptr && a->skip2_buckets > 0) {
      DSG_REQUIRE(a->skip2_map_c2_from_c1 && a->skip2_map_dense_from_c2 && a->skip2_map_c2_from_dense,
                  "forward: the level-2 row maps are missing");
      DSG_REQUIRE(m->skip2_granule > 0, "forward: this geometry has no second compaction level (skip2_tables given)");
      DSG_TRY(parse_plan(l2, 2, a->skip2_tables, a->skip2_table_images, a->skip2_buckets, a->skip2_count, a->skip2_side,
                         a->skip2_phantom_tok0, m->skip2_granule, B, N));
      level2 = true;
    }
  }
  // the layout of stage s: patch embedding, merges, encoder skips and breakup outputs
  auto stage_layout = [&](int s) -> const Layout& { return s < S ? l1 : dense; };
  // block j of stage s; j2 is the level-2 block of stage S (encoder: the first, decoder: the last)
  auto block_layout = [&](int s, int j, int j2) -> const Layout& {
    return s < S ? l1 : (level2 && s == S && j == j2) ? l2 : dense;
  };
  bool final_ln_done = false;
  // a block reads an input stored in another layout through a row map; a mapped read cannot be in place, so X and T
  // trade places when the input is X
  auto block = [&](const Block& b, const float* x_in, const Layout& from, const Layout& lay, bool last) -> int {
    const int* rows_map = row_map(a, from, lay);
    if (rows_map != nullptr && x_in == w.X) std::swap(w.X, w.T);
    return run_block(m, b, w, x_in, lay, rows_map, uniform, st, last, &final_ln_done);
  };
  g_prof_pass = g_prof_on && !stream_capturing(st) && (g_prof_counter++ % g_prof_stride == 0);
  struct ProfPassGuard { ~ProfPassGuard() { g_prof_pass = false; } } prof_pass_guard;
  DSG_TRY_P(PC_EMBED_HEAD, 0, 0, launch_cond(labels, label_stride, a->n_cond, m->f32("map_layer0.weight"),
                      m->f32("map_layer0.bias"), m->f32("map_layer1.weight"), m->f32("map_layer1.bias"),
                      m->at<float>(m->film_w_off), m->at<float>(m->film_b_off), m->film_total, w.emb0, w.emb1, w.emb,
                      w.film, E, st));
  // patch embedding straight from (adj, node): the [B, cin, N, N] grid of :784-802 is never built
  DSG_TRY_P(PC_EMBED_HEAD, 0, 0, launch_node_proj(a->node, a->sc_node, c_in, m->at<float>(m->w_rc_off), w.rc, B, N, m->cfg.c_n,
                           m->cfg.self_condition, E, st));
  const Layout& l0 = stage_layout(0);
  for (int k = 0; k < l0.K; ++k) {
    const double pxk = static_cast<double>(l0.count[k]) * l0.side[k] * l0.side[k];
    DSG_TRY_P(PC_EMBED_HEAD, 0, pxk * (m->planes_adj * 4 + E * 4),
              launch_patch_embed(a->adj, a->sc_adj, c_in, a->flags, w.rc, m->at<float>(m->w_adj_off),
                                 m->f32("patch_embed.proj.bias"), m->f32("patch_embed.norm.weight"),
                                 m->f32("patch_embed.norm.bias"), w.film, m->film_total, 0, uniform, w.X + l0.tok[k] * E,
                                 l0.count[k], N, m->cfg.c_e, m->cfg.self_condition, E, st, l0.bucket_perm(k), l0.side[k]));
  }
  const Layout* xl = &l0;   // the layout of the activation in X
  int stage_no = 0;
#define DSG_STAGE_DONE() do { if (g_stop_after >= 0 && stage_no++ == g_stop_after) return DSG_OK; } while (0)
  DSG_STAGE_DONE();
  // encoder                                                                  (:746-748)
  for (int s = 0; s < m->nl; ++s) {
    // the first block of a stage after the first reads the merge output, stored in the previous stage's layout
    const float* x_in = s == 0 ? w.X : w.skip[s - 1];
    const Layout* in = s == 0 ? xl : &stage_layout(s - 1);
    for (int j = 0; j < m->cfg.depths[s]; ++j) {
      const Layout& lay = block_layout(s, j, 0);
      DSG_TRY(block(m->blocks[m->down_first[s] + j], x_in, *in, lay, false));
      x_in = w.X;
      in = xl = &lay;
      DSG_STAGE_DONE();
    }
    if (s < m->nl - 1) {
      const Merge& g = m->merges[s];
      const Layout& lay = stage_layout(s);
      for (int k = 0; k < lay.K; ++k) {
        const double rk = static_cast<double>(lay.at(k + 1, s + 1) - lay.at(k, s + 1));
        DSG_TRY_P(PC_ROW, 0, rk * 4 * g.C * 6,
                  launch_merge_ln(w.X + lay.at(k, s) * g.C, w.Y + lay.at(k, s + 1) * 4 * g.C, m->f32(g.prefix + ".norm.weight"),
                                  m->f32(g.prefix + ".norm.bias"), lay.count[k], lay.side[k] >> s, g.C, st));
      }
      DSG_TRY(gemm(m, w.Y, lay.tokens(s + 1), g.reduction, EPI_F32, nullptr, nullptr, w.skip[s], st));
      DSG_STAGE_DONE();
    }
  }
  // decoder                                                                  (:751-756)
  for (int u = 0; u < m->nl; ++u) {
    const int s = m->nl - 1 - u;
    if (u > 0) {
      // the low-resolution stream is in X (every stage has a block); the skip (the merge output of the way down) is
      // stored in the stage's layout `up`.  Entering another layout, the breakup writes only the children inside each
      // sample's kept corner of `up`.
      const Breakup& bu = m->breakups[u - 1];
      const Layout &low = *xl, &up = stage_layout(s);
      const bool change = low.level != up.level;
      const long long rows_low = low.tokens(s + 1);
      DSG_TRY_P(PC_ROW, 0, static_cast<double>(rows_low) * bu.D * 6,
                launch_concat_bf16(w.X, w.skip[s], w.Y, rows_low, bu.D / 2, st, row_map(a, up, low)));
      DSG_TRY(gemm(m, w.Y, rows_low, bu.pre, EPI_F32, nullptr, nullptr, w.T, st));
      for (int k = 0; k < low.K; ++k) {
        const double rk = static_cast<double>(low.at(k + 1, s + 1) - low.at(k, s + 1));
        DSG_TRY_P(PC_ROW, 0, rk * bu.D * 6,
                  launch_breakup_ln(w.T + low.at(k, s + 1) * bu.D, change ? w.Y : w.Y + up.at(k, s) * (bu.D / 4),
                                    m->f32(bu.prefix + ".norm.weight"), m->f32(bu.prefix + ".norm.bias"),
                                    m->f32(bu.prefix + ".post_norm.weight"), m->f32(bu.prefix + ".post_norm.bias"),
                                    low.count[k], low.side[k] >> (s + 1), bu.D, st, change ? up.tok0 : nullptr,
                                    change ? up.width : nullptr, s, change ? low.bucket_perm(k) : nullptr));
      }
      DSG_TRY(gemm(m, w.Y, up.tokens(s), bu.post, EPI_F32, nullptr, nullptr, w.X, st));
      xl = &up;
      DSG_STAGE_DONE();
    }
    for (int j = 0; j < m->cfg.depths[s]; ++j) {
      // the last block: the final LayerNorm rides on its fused tail (not while a test walks the stages: those read X)
      const bool last = u == m->nl - 1 && j == m->cfg.depths[s] - 1 && g_stop_after < 0;
      const Layout& lay = block_layout(s, j, m->cfg.depths[s] - 1);
      DSG_TRY(block(m->blocks[m->up_first[u] + j], w.X, *xl, lay, last));
      xl = &lay;
      DSG_STAGE_DONE();
    }
  }
  // read-out                                                                 (:758-761, :806-825)
  const long long pixels = l0.tokens(0);
  if (!l0.dense())  // pixels that are not computed are padding: their outputs are the masked zeros
    DSG_CUDA_CHECK(cudaMemsetAsync(a->out_adj, 0, static_cast<size_t>(B) * m->cfg.c_e * N * N * 4, st));
  if (!final_ln_done)
    DSG_TRY_P(PC_ROW, 0, static_cast<double>(pixels) * E * 6, launch_ln(w.X, w.Y, m->f32("norm.weight"), m->f32("norm.bias"), pixels, E, st));
  GemmParams hp;
  memset(&hp, 0, sizeof(hp));
  hp.w2t = m->at<float>(m->adj_w2t_off);
  hp.b2 = m->at<float>(m->adj_b2_off);
  hp.c_e = m->cfg.c_e;
  hp.n_img = N;
  hp.flags = a->flags;
  hp.x_adj = a->mode == 1 ? a->adj : nullptr;
  hp.c_skip = c_skip;
  hp.c_out = c_out;
  for (int k = 0; k < l0.K; ++k) {   // the epilogue maps a GEMM row to its pixel through the bucket's geometry
    hp.perm = l0.bucket_perm(k);
    hp.side = l0.side[k];
    DSG_TRY(gemm(m, w.Y + l0.tok[k] * E, l0.tok[k + 1] - l0.tok[k], m->adj_fc1, EPI_ADJ_HEAD, m->at<float>(m->adj_b1_off),
                 nullptr, a->out_adj, st, &hp));
  }
  DSG_TRY_P(PC_EMBED_HEAD, 0, static_cast<double>(pixels) * E * 2, launch_node_head(w.Y, a->flags, m->at<float>(m->fold_ft_off), m->at<float>(m->fold_b_off),
                           m->at<float>(m->node_w1t_off), m->f32("readout_node_mlp.fc1.bias"),
                           m->at<float>(m->node_w2t_off), m->f32("readout_node_mlp.fc2.bias"),
                           a->mode == 1 ? a->node : nullptr, c_skip, c_out, a->out_node, B, N, m->cfg.c_n, E, st,
                           l0.tok0, l0.width, 2 * E >= 128 ? w.rc : nullptr));   // rc (row / column planes of the embedding) is dead by now
  return DSG_OK;
}

void dsg_launch_count_add(uint64_t n) { __atomic_fetch_add(&g_launches, static_cast<unsigned long long>(n), __ATOMIC_RELAXED); }
void dsg_debug_set_stop_after(int n_stages) { g_stop_after = n_stages; }

int dsg_profile_begin(int pass_stride) {
  DSG_REQUIRE(pass_stride >= 1, "profile_begin: stride %d", pass_stride);
  for (int c = 0; c < PC_COUNT; ++c) {
    memset(&g_prof_tot[c], 0, sizeof(g_prof_tot[c]));
    strncpy(g_prof_tot[c].name, kProfNames[c], sizeof(g_prof_tot[c].name) - 1);
  }
  g_prof_stride = pass_stride;
  g_prof_counter = 0;
  g_prof_on = true;
  return DSG_OK;
}

int dsg_profile_dump(const char* path) {
  DSG_REQUIRE(path != nullptr, "profile_dump: null path");
  FILE* f = fopen(path, "w");
  DSG_REQUIRE(f != nullptr, "profile_dump: cannot open %s", path);
  fprintf(f, "index,class,label,rows,k,ms,flops,bytes\n");
  int i = 0;
  for (ProfRec& r : g_prof_recs) {
    float ms = 0.f;
    if (cudaEventSynchronize(r.e1) != cudaSuccess || cudaEventElapsedTime(&ms, r.e0, r.e1) != cudaSuccess) ms = -1.f;
    fprintf(f, "%d,%s,%s,%lld,%d,%.6f,%.0f,%.0f\n", i++, kProfNames[r.cls], r.label, r.rows, r.c, ms, r.flops, r.bytes);
  }
  fclose(f);
  return DSG_OK;
}

int dsg_profile_read(dsg_profile_class* out, int max_classes, int* n_classes) {
  for (ProfRec& r : g_prof_recs) {
    float ms = 0.f;
    DSG_CUDA_CHECK(cudaEventSynchronize(r.e1));
    DSG_CUDA_CHECK(cudaEventElapsedTime(&ms, r.e0, r.e1));
    dsg_profile_class& t = g_prof_tot[r.cls];
    t.launches += 1; t.ms += ms; t.flops += r.flops; t.bytes += r.bytes;
    g_prof_pool.push_back(r.e0);
    g_prof_pool.push_back(r.e1);
  }
  g_prof_recs.clear();
  if (out != nullptr)
    for (int c = 0; c < PC_COUNT && c < max_classes; ++c) out[c] = g_prof_tot[c];
  if (n_classes) *n_classes = PC_COUNT;
  return DSG_OK;
}

void dsg_profile_stop(void) { g_prof_on = false; g_prof_pass = false; }

int dsg_debug_buffer(const dsg_model* m, int batch, int n_cond, const char* name, size_t* offset, size_t* bytes) {
  DSG_REQUIRE(m && name && offset && bytes && batch > 0 && n_cond > 0, "debug_buffer: bad argument");
  uint8_t* base = reinterpret_cast<uint8_t*>(kAlign);  // fake non-null base: only offsets are wanted
  Workspace w = carve(m, batch, n_cond, base);
  const size_t full = static_cast<size_t>(batch) * m->N * m->N * m->E;
  struct { const char* n; const void* p; size_t b; } tab[] = {
      {"X", w.X, full * 4}, {"T", w.T, full * 4}, {"Y", w.Y, full * 2}, {"QKV", w.QKV, full * 6},
      {"ATT", w.ATT, full * 2}, {"H", w.H, full * 8},
      {"skip0", w.skip.size() > 0 ? w.skip[0] : nullptr, full * 2}, {"skip1", w.skip.size() > 1 ? w.skip[1] : nullptr, full},
      {"skip2", w.skip.size() > 2 ? w.skip[2] : nullptr, full / 2}, {"coef", w.coef, static_cast<size_t>(16) * batch},
      {"emb", w.emb, static_cast<size_t>(n_cond) * 2048}, {"film", w.film, static_cast<size_t>(n_cond) * m->film_total * 4},
      {"rc", w.rc, static_cast<size_t>(batch) * m->N * 2 * m->E * 4}};
  for (auto& t : tab)
    if (strcmp(t.n, name) == 0 && t.p != nullptr) {
      *offset = static_cast<size_t>(static_cast<const uint8_t*>(t.p) - base);
      *bytes = t.b;
      return DSG_OK;
    }
  set_last_error("debug_buffer: no buffer named '%s'", name);
  return DSG_ERR_INVALID;
}

int dsg_edm_pre_step(const float* adj, const float* node, const float* eps_adj, const float* eps_node,
                     const uint8_t* flags, float noise_coef, float* adj_hat, float* node_hat, int batch, int c_e, int n,
                     int c_n, dsg_stream_t stream) {
  DSG_REQUIRE(adj && node && eps_adj && eps_node && flags && adj_hat && node_hat, "edm_pre_step: null tensor");
  const double el = static_cast<double>(batch) * (static_cast<double>(c_e) * n * n + static_cast<double>(n) * c_n);
  ProfScope ps(prof_every_launch(static_cast<cudaStream_t>(stream)), PC_EDM, 2 * el, 12 * el, static_cast<cudaStream_t>(stream));
  return launch_edm_pre_step(adj, node, eps_adj, eps_node, flags, noise_coef, adj_hat, node_hat, batch, c_e, n, c_n,
                             static_cast<cudaStream_t>(stream));
}

int dsg_edm_pre_step_philox(const float* adj, const float* node, const uint8_t* flags, float noise_coef, uint64_t seed,
                            uint64_t offset_adj, int grid_adj, uint64_t offset_node, int grid_node, float* adj_hat,
                            float* node_hat, int batch, int c_e, int n, int c_n, dsg_stream_t stream) {
  DSG_REQUIRE(adj && node && flags && adj_hat && node_hat, "edm_pre_step_philox: null tensor");
  const double el = static_cast<double>(batch) * (static_cast<double>(c_e) * n * n + static_cast<double>(n) * c_n);
  ProfScope ps(prof_every_launch(static_cast<cudaStream_t>(stream)), PC_EDM_NOISE, 2 * el, 8 * el, static_cast<cudaStream_t>(stream));  // Philox / Box-Muller bound
  return launch_edm_pre_step_philox(adj, node, flags, noise_coef, seed, offset_adj, grid_adj, offset_node, grid_node,
                                    nullptr, adj_hat, node_hat, batch, c_e, n, c_n, static_cast<cudaStream_t>(stream));
}

int dsg_edm_step_advance(const dsg_edm_step_params* table, dsg_edm_step_params* cur, int32_t* counter, dsg_stream_t stream) {
  DSG_REQUIRE(table && cur && counter, "edm_step_advance: null pointer");
  return launch_edm_step_advance(table, cur, counter, static_cast<cudaStream_t>(stream));
}

int dsg_edm_pre_step_philox_dev(const float* adj, const float* node, const uint8_t* flags, const dsg_edm_step_params* cur,
                                int grid_adj, int grid_node, float* adj_hat, float* node_hat, int batch, int c_e, int n,
                                int c_n, dsg_stream_t stream) {
  DSG_REQUIRE(adj && node && flags && cur && adj_hat && node_hat, "edm_pre_step_philox_dev: null tensor");
  const double el = static_cast<double>(batch) * (static_cast<double>(c_e) * n * n + static_cast<double>(n) * c_n);
  ProfScope ps(prof_every_launch(static_cast<cudaStream_t>(stream)), PC_EDM_NOISE, 2 * el, 8 * el, static_cast<cudaStream_t>(stream));
  return launch_edm_pre_step_philox(adj, node, flags, 0.f, 0, 0, grid_adj, 0, grid_node, cur, adj_hat, node_hat, batch,
                                    c_e, n, c_n, static_cast<cudaStream_t>(stream));
}

int dsg_edm_post_step_dev(const float* adj_hat, const float* node_hat, const float* d1_adj, const float* d1_node,
                          const float* d2_adj, const float* d2_node, const uint8_t* flags, const dsg_edm_step_params* cur,
                          float* adj_next, float* node_next, int batch, int c_e, int n, int c_n, dsg_stream_t stream) {
  DSG_REQUIRE(adj_hat && node_hat && d1_adj && d1_node && flags && cur && adj_next && node_next, "edm_post_step_dev: null tensor");
  DSG_REQUIRE((d2_adj == nullptr) == (d2_node == nullptr), "edm_post_step_dev: d2_adj / d2_node must both be given or both NULL");
  const double el = static_cast<double>(batch) * (static_cast<double>(c_e) * n * n + static_cast<double>(n) * c_n);
  ProfScope ps(prof_every_launch(static_cast<cudaStream_t>(stream)), PC_EDM, (d2_adj ? 11 : 4) * el, (d2_adj ? 16 : 12) * el,
               static_cast<cudaStream_t>(stream));
  return launch_edm_post_step(adj_hat, node_hat, d1_adj, d1_node, d2_adj, d2_node, flags, 0.f, 0.f, 0.f, cur, adj_next,
                              node_next, batch, c_e, n, c_n, static_cast<cudaStream_t>(stream));
}

int dsg_edm_final_step_decode(const float* adj_hat, const float* node_hat, const float* d1_adj, const float* d1_node,
                              const uint8_t* flags, float inv_t_hat, float h, const dsg_edm_step_params* cur, float* adj_next,
                              float* node_next, int32_t* adj_cls, int32_t* node_cls, float* bbox, int num_adj_type,
                              int num_node_type, int batch, int c_e, int n, int c_n, dsg_stream_t stream) {
  DSG_REQUIRE(adj_hat && node_hat && d1_adj && d1_node && flags && adj_cls && node_cls && bbox, "edm_final_step_decode: null tensor");
  DSG_REQUIRE((adj_next == nullptr) == (node_next == nullptr), "edm_final_step_decode: adj_next / node_next both or neither");
  return launch_edm_final_decode(adj_hat, node_hat, d1_adj, d1_node, flags, inv_t_hat, h, cur, adj_next, node_next, adj_cls,
                                 node_cls, bbox, num_adj_type, num_node_type, batch, c_e, n, c_n,
                                 static_cast<cudaStream_t>(stream));
}

int dsg_edm_post_step(const float* adj_hat, const float* node_hat, const float* d1_adj, const float* d1_node,
                      const float* d2_adj, const float* d2_node, const uint8_t* flags, float inv_t_hat, float h,
                      float inv_t_prime, float* adj_next, float* node_next, int batch, int c_e, int n, int c_n,
                      dsg_stream_t stream) {
  DSG_REQUIRE(adj_hat && node_hat && d1_adj && d1_node && flags && adj_next && node_next, "edm_post_step: null tensor");
  DSG_REQUIRE((d2_adj == nullptr) == (d2_node == nullptr), "edm_post_step: d2_adj / d2_node must both be given or both NULL");
  const double el = static_cast<double>(batch) * (static_cast<double>(c_e) * n * n + static_cast<double>(n) * c_n);
  ProfScope ps(prof_every_launch(static_cast<cudaStream_t>(stream)), PC_EDM, (d2_adj ? 11 : 4) * el, (d2_adj ? 16 : 12) * el, static_cast<cudaStream_t>(stream));
  return launch_edm_post_step(adj_hat, node_hat, d1_adj, d1_node, d2_adj, d2_node, flags, inv_t_hat, h, inv_t_prime,
                              nullptr, adj_next, node_next, batch, c_e, n, c_n, static_cast<cudaStream_t>(stream));
}

int dsg_edm_mask_scale(const float* adj, const float* node, const uint8_t* flags, float scale, float* adj_out,
                       float* node_out, int batch, int c_e, int n, int c_n, dsg_stream_t stream) {
  DSG_REQUIRE(adj && node && flags && adj_out && node_out, "edm_mask_scale: null tensor");
  return launch_mask_scale(adj, node, flags, scale, adj_out, node_out, batch, c_e, n, c_n,
                           static_cast<cudaStream_t>(stream));
}

int dsg_decode_samples(const float* adj, const float* node, const uint8_t* flags, int32_t* adj_cls, int32_t* node_cls,
                       float* bbox, int num_adj_type, int num_node_type, int batch, int c_e, int n, int c_n,
                       dsg_stream_t stream) {
  DSG_REQUIRE(adj && node && flags && adj_cls && node_cls && bbox, "decode_samples: null tensor");
  return launch_decode(adj, node, flags, adj_cls, node_cls, bbox, num_adj_type, num_node_type, batch, c_e, n, c_n,
                       static_cast<cudaStream_t>(stream));
}

int dsg_train_noise(const float* clean_adj, const float* clean_node, const float* eps_adj, const float* eps_node,
                    const float* sigmas, const uint8_t* flags, float* noisy_adj, float* noise_adj, float* noisy_node,
                    float* noise_node, int batch, int c_e, int n, int c_n, dsg_stream_t stream) {
  DSG_REQUIRE(clean_adj && clean_node && eps_adj && eps_node && sigmas && flags && noisy_adj && noise_adj && noisy_node &&
                  noise_node,
              "train_noise: null tensor");
  return launch_train_noise(clean_adj, clean_node, eps_adj, eps_node, sigmas, flags, noisy_adj, noise_adj, noisy_node,
                            noise_node, batch, c_e, n, c_n, static_cast<cudaStream_t>(stream));
}

int dsg_edm_loss_sums(const float* pred_adj, const float* target_adj, const float* pred_node, const float* target_node,
                      const float* weights, const uint8_t* flags, float* sum_adj, float* sum_node, int batch, int c_e,
                      int n, int c_n, dsg_stream_t stream) {
  DSG_REQUIRE(pred_adj && target_adj && pred_node && target_node && flags && sum_adj && sum_node,
              "edm_loss_sums: null tensor");
  return launch_loss_sums(pred_adj, target_adj, pred_node, target_node, weights, flags, sum_adj, sum_node, batch, c_e, n,
                          c_n, static_cast<cudaStream_t>(stream));
}

int dsg_edm_loss_sums_backward(const float* pred_adj, const float* target_adj, const float* pred_node,
                               const float* target_node, const float* weights, const uint8_t* flags, const float* grad_sum_adj,
                               const float* grad_sum_node, float* grad_pred_adj, float* grad_pred_node, int batch, int c_e,
                               int n, int c_n, dsg_stream_t stream) {
  DSG_REQUIRE(pred_adj && target_adj && pred_node && target_node && flags && grad_sum_adj && grad_sum_node && grad_pred_adj &&
                  grad_pred_node, "edm_loss_sums_backward: null tensor");
  return launch_loss_sums_backward(pred_adj, target_adj, pred_node, target_node, weights, flags, grad_sum_adj, grad_sum_node,
                                   grad_pred_adj, grad_pred_node, batch, c_e, n, c_n, static_cast<cudaStream_t>(stream));
}

int dsg_gemm_bf16(const void* a, const void* w, const float* bias, const float* res, void* out, int M, int N, int K,
                  int epi, dsg_stream_t stream) {
  DSG_REQUIRE(a && w && out && epi >= 0 && epi <= 3, "gemm_bf16: bad argument");
  CUtensorMap ta, tw, to;
  DSG_TRY(make_tmap_bf16(&ta, a, M, K, 128));
  const bool pair = gemm_use_pair(M, K, epi);
  const int bn = gemm_choose_bn(M, N, K, epi, pair);
  DSG_TRY(make_tmap_bf16(&tw, w, N, K, pair ? bn / 2 : bn));
  DSG_TRY(make_tmap_out(&to, out, M, N, epi));
  if (epi == EPI_RES_F32) {
    DSG_REQUIRE(res != nullptr, "gemm_bf16: residual epilogue without residual");
    if (res != out)  // the kernel accumulates in place: seed the output with the residual
      DSG_CUDA_CHECK(cudaMemcpyAsync(out, res, static_cast<size_t>(M) * N * 4, cudaMemcpyDeviceToDevice,
                                     static_cast<cudaStream_t>(stream)));
    res = static_cast<const float*>(out);
  }
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.M = M; p.N = N; p.K = K; p.bias = bias; p.res = res; p.out = out; p.ldo = N; p.bn = bn;
  return launch_gemm(&ta, &tw, &to, epi, p, static_cast<cudaStream_t>(stream), pair);
}

int dsg_proj_ln(const void* att, const void* w, const float* bias, const float* gamma, const float* beta, float* x, void* y,
                int M, int C, dsg_stream_t stream) {
  DSG_REQUIRE(att && w && bias && gamma && beta && x && y, "proj_ln: null tensor");
  DSG_REQUIRE(proj_ln_supported(C), "proj_ln: C = %d (192 / 384)", C);
  CUtensorMap ta, tw;
  DSG_TRY(make_tmap_bf16(&ta, att, M, C, 128));
  DSG_TRY(make_tmap_bf16(&tw, w, C, C, gemm_block_n(C)));
  return launch_proj_ln(&ta, &tw, bias, gamma, beta, x, static_cast<bf16*>(y), M, C, static_cast<cudaStream_t>(stream));
}

int dsg_window_attention_check(const float* bias, const float* mask, int batch, int res, int window, int shift, int heads,
                               dsg_stream_t stream, int* flags_out) {
  DSG_REQUIRE(bias && flags_out, "window_attention_check: null argument");
  int canonical = 0;
  const bool w16 = window_attention_w16_supported(batch, res, window, shift, heads);
  if (mask != nullptr && shift > 0 && (w16 || window_attention_quad_supported(batch, res, window, shift, heads))) {
    int ok = 0;
    DSG_TRY(check_mask_canonical(mask, res, window, shift, static_cast<cudaStream_t>(stream), &ok));
    if (ok) canonical |= ATTN_MASK_CANONICAL;
  }
  if (w16) {
    int ok = 0;
    DSG_TRY(check_bias_toeplitz(bias, heads, window, static_cast<cudaStream_t>(stream), &ok));
    if (ok) canonical |= ATTN_BIAS_TOEPLITZ;
  }
  *flags_out = canonical;
  return DSG_OK;
}

int dsg_window_attention_flags(const void* qkv, const float* bias, const float* mask, void* out, int batch, int res, int window,
                               int shift, int heads, int flags, dsg_stream_t stream) {
  DSG_REQUIRE(qkv && bias && out, "window_attention: null tensor");
  return launch_window_attention(static_cast<const bf16*>(qkv), bias, mask, static_cast<bf16*>(out), batch, res, window,
                                 shift, heads, static_cast<cudaStream_t>(stream), flags);
}

int dsg_window_attention(const void* qkv, const float* bias, const float* mask, void* out, int batch, int res, int window,
                         int shift, int heads, dsg_stream_t stream) {
  int flags = 0;
  DSG_TRY(dsg_window_attention_check(bias, mask, batch, res, window, shift, heads, stream, &flags));
  return dsg_window_attention_flags(qkv, bias, mask, out, batch, res, window, shift, heads, flags, stream);
}

}  // extern "C"
