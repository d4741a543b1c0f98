// Fused elementwise kernels of the EDM stochastic-Heun sampler (runner/mcmc_sampler/edm.py:350-434 of the
// reference; ~113 ATen launches per step there, two here).
//
// State layout: adj [B, C_e, N, N] and node [B, N, C_n], fp32, exactly the reference's tensors.  Pure
// HBM-bound streaming: 128-bit loads/stores over the adjacency tensor (N % 4 == 0), grid-stride with a grid
// that is a multiple of the SM count.  Arithmetic is written with explicit round-to-nearest intrinsics in
// the reference's operation order (no FMA contraction) so that, given the same inputs, the results are
// bit-identical to the fp32 torch expressions:
//
//   pre :  x_hat  = mask(x + c * eps)                      c = sqrt(t_hat^2 - t_cur^2) * S_noise     (:361-366)
//   post:  k      = mask(inv_t * x_hat - inv_t * D1)                                                  (:384-387)
//          x'     = x_hat + h * k                                                                    (:389-390)
//          x_next = mask(x_hat + h * (0.5 k + 0.5 (inv_tp * x' - inv_tp * D2)))     (Heun, :414-422)
//          x_next = mask(x')                                                        (last step, :395-396)
//
// Completion (sampling with known entries held; DESIGN.md §3.6): k = known state, NaN = free entry
//   pre :  x_hat  = mask(isnan(k) ? x + c * eps : k + t_hat * eps)     same eps, same element as the plain pre-step
//   last:  x      = mask(isnan(k) ? x : k)                             once, after the last post-step
//
// Guided completion (reconstruction guidance, DESIGN.md §3.7): G = grad_x_hat 1/2 sum_known (D(x_hat) - k)^2
//   residual: r      = mask(isnan(k) ? 0 : D - k)                      the output gradient the denoiser backward takes
//   update:   D~     = mask(D - w * G)                                 replaces D in the post-step and self-conditioning
#include <curand_kernel.h>

#include "common.cuh"
#include "kernels.h"

namespace dsg {
namespace {

struct EdmShape {
  int batch, c_e, n, c_n;
};

DSG_DEVICE float pre_one(float x, float e, float c) { return __fadd_rn(x, __fmul_rn(c, e)); }
// replacement at noise level t_hat for a known entry k (finite), the plain pre-step for a free one (k = NaN)
DSG_DEVICE float pre_known_one(float x, float e, float k, float c, float t_hat) {
  return isnan(k) ? pre_one(x, e, c) : pre_one(k, e, t_hat);
}

DSG_DEVICE float post_one(float xh, float d1, float d2, float inv_t, float h, float inv_tp, bool heun) {
  const float k = __fsub_rn(__fmul_rn(inv_t, xh), __fmul_rn(inv_t, d1));
  const float xp = __fadd_rn(xh, __fmul_rn(h, k));
  if (!heun) return xp;
  const float kp = __fsub_rn(__fmul_rn(inv_tp, xp), __fmul_rn(inv_tp, d2));
  return __fadd_rn(xh, __fmul_rn(h, __fadd_rn(__fmul_rn(0.5f, k), __fmul_rn(0.5f, kp))));
}

// Per-step scalars in device memory (CUDA-graph replays: the captured launches read the row the step-advance kernel
// copied into `cur`; include/dsg_b200.h: dsg_edm_step_params)
struct StepParams {
  float noise_coef, inv_t_hat, h, inv_t_prime, t_hat, pad;
  unsigned long long seed, offset_adj, offset_node;
};
static_assert(sizeof(StepParams) == sizeof(dsg_edm_step_params), "StepParams mirrors dsg_edm_step_params");

__global__ void step_advance_kernel(const StepParams* __restrict__ table, StepParams* __restrict__ cur, int* counter) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    const int i = *counter;
    *cur = table[i];
    *counter = i + 1;
  }
}

// MODE 0: pre-step, 1: post-step (heun), 2: post-step (euler / last), 3: x = mask(x * scale),
// 4: pre-step with known entries (a2 / n2 = known, s1 = t_hat)
// Streaming layout: the adjacency tensor is walked as float4 vectors, U = 4 vectors per thread per trip, all loads of a
// trip issued before the first store (12 x 16 B in flight per thread in the Heun post-step); 32-bit index arithmetic
// (the launcher checks the vector count), streaming (evict-first) loads: every operand is read exactly once.
constexpr int EDM_U = 4;
template <int MODE>
__global__ void __launch_bounds__(256)
edm_kernel(const float* __restrict__ a0, const float* __restrict__ a1, const float* __restrict__ a2,
           float* __restrict__ a_out, const float* __restrict__ n0, const float* __restrict__ n1,
           const float* __restrict__ n2, float* __restrict__ n_out, const uint8_t* __restrict__ flags, float s0,
           float s1, float s2, const StepParams* __restrict__ P, EdmShape sh) {
  if (P != nullptr) {
    if (MODE == 0) { s0 = P->noise_coef; }
    else if (MODE == 4) { s0 = P->noise_coef; s1 = P->t_hat; }
    else { s0 = P->inv_t_hat; s1 = P->h; s2 = P->inv_t_prime; }
  }
  const unsigned n = sh.n, n4 = sh.n >> 2, nce = n * sh.c_e;
  const unsigned adj_vec = static_cast<unsigned>(sh.batch) * sh.c_e * n * n4;
  const unsigned trip = gridDim.x * blockDim.x * EDM_U;
  const float4* A0 = reinterpret_cast<const float4*>(a0);
  const float4* A1 = reinterpret_cast<const float4*>(a1);
  const float4* A2 = reinterpret_cast<const float4*>(a2);
  float4* AO = reinterpret_cast<float4*>(a_out);
  for (unsigned base = blockIdx.x * blockDim.x * EDM_U + threadIdx.x; base < adj_vec; base += trip) {
    float4 x[EDM_U], p[EDM_U], q[EDM_U];
#pragma unroll
    for (int u = 0; u < EDM_U; ++u) {
      const unsigned v = base + u * blockDim.x;
      if (v < adj_vec) {
        x[u] = __ldcs(A0 + v);
        if (MODE == 0 || MODE == 1 || MODE == 2 || MODE == 4) p[u] = __ldcs(A1 + v);
        if (MODE == 1 || MODE == 4) q[u] = __ldcs(A2 + v);
      }
    }
#pragma unroll
    for (int u = 0; u < EDM_U; ++u) {
      const unsigned v = base + u * blockDim.x;
      if (v >= adj_vec) continue;
      const unsigned r = v / n4, j4 = v - r * n4;
      const unsigned b = r / nce, i = r % n;
      const uint8_t* f = flags + b * n;
      const bool fi = f[i] != 0;
      const uchar4 fj = *reinterpret_cast<const uchar4*>(f + 4 * j4);
      float4 o;
      if (MODE == 0) {
        o = make_float4(pre_one(x[u].x, p[u].x, s0), pre_one(x[u].y, p[u].y, s0), pre_one(x[u].z, p[u].z, s0),
                        pre_one(x[u].w, p[u].w, s0));
      } else if (MODE == 1 || MODE == 2) {
        const float4 d1 = p[u];
        const float4 d2 = MODE == 1 ? q[u] : p[u];
        o = make_float4(post_one(x[u].x, d1.x, d2.x, s0, s1, s2, MODE == 1), post_one(x[u].y, d1.y, d2.y, s0, s1, s2, MODE == 1),
                        post_one(x[u].z, d1.z, d2.z, s0, s1, s2, MODE == 1), post_one(x[u].w, d1.w, d2.w, s0, s1, s2, MODE == 1));
      } else if (MODE == 4) {
        o = make_float4(pre_known_one(x[u].x, p[u].x, q[u].x, s0, s1), pre_known_one(x[u].y, p[u].y, q[u].y, s0, s1),
                        pre_known_one(x[u].z, p[u].z, q[u].z, s0, s1), pre_known_one(x[u].w, p[u].w, q[u].w, s0, s1));
      } else {
        o = make_float4(__fmul_rn(x[u].x, s0), __fmul_rn(x[u].y, s0), __fmul_rn(x[u].z, s0), __fmul_rn(x[u].w, s0));
      }
      o.x = (fi && fj.x) ? o.x : 0.f;
      o.y = (fi && fj.y) ? o.y : 0.f;
      o.z = (fi && fj.z) ? o.z : 0.f;
      o.w = (fi && fj.w) ? o.w : 0.f;
      AO[v] = o;
    }
  }
  const unsigned node_el = static_cast<unsigned>(sh.batch) * n * sh.c_n;
  const unsigned stride = gridDim.x * blockDim.x;
  for (unsigned v = blockIdx.x * blockDim.x + threadIdx.x; v < node_el; v += stride) {
    const bool ok = flags[v / static_cast<unsigned>(sh.c_n)] != 0;
    const float x = n0[v];
    float o;
    if (MODE == 0) {
      o = pre_one(x, n1[v], s0);
    } else if (MODE == 1) {
      o = post_one(x, n1[v], n2[v], s0, s1, s2, true);
    } else if (MODE == 2) {
      o = post_one(x, n1[v], 0.f, s0, s1, s2, false);
    } else if (MODE == 4) {
      o = pre_known_one(x, n1[v], n2[v], s0, s1);
    } else {
      o = __fmul_rn(x, s0);
    }
    n_out[v] = ok ? o : 0.f;
  }
}

// Last sampler step fused with the decode of the final sample (SURVEY 8f-1): Euler update (edm.py:389-396), mask, and
// the reference's bits -> class rule (runner/sampler/sampler_node_adj.py:222-285) in one pass over (x_hat, D1); the
// fp32 state is written only if the caller wants it (adj_next / node_next may be NULL), so that only int32 classes and
// four box floats per node have to leave the GPU.  One thread per 4 neighbouring pixels, channels walked in the loop.
__global__ void __launch_bounds__(256)
edm_final_decode_kernel(const float* __restrict__ adj_hat, const float* __restrict__ node_hat, const float* __restrict__ d1_adj,
                        const float* __restrict__ d1_node, const uint8_t* __restrict__ flags, float inv_t, float h,
                        const StepParams* __restrict__ P, float* __restrict__ adj_next, float* __restrict__ node_next,
                        int32_t* __restrict__ adj_cls, int32_t* __restrict__ node_cls, float* __restrict__ bbox,
                        int num_adj_type, int num_node_type, EdmShape sh) {
  if (P != nullptr) { inv_t = P->inv_t_hat; h = P->h; }
  const unsigned n = sh.n, n4 = sh.n >> 2, plane4 = n * n4;
  const unsigned groups = static_cast<unsigned>(sh.batch) * plane4;
  const unsigned stride = gridDim.x * blockDim.x;
  const unsigned tid = blockIdx.x * blockDim.x + threadIdx.x;
  for (unsigned g = tid; g < groups; g += stride) {
    const unsigned b = g / plane4, ij4 = g - b * plane4;
    const unsigned i = ij4 / n4, j4 = ij4 - i * n4;
    const uint8_t* f = flags + b * n;
    const bool fi = f[i] != 0;
    const uchar4 fj = *reinterpret_cast<const uchar4*>(f + 4 * j4);
    const bool ok[4] = {fi && fj.x, fi && fj.y, fi && fj.z, fi && fj.w};
    int v[4] = {0, 0, 0, 0};
    for (int c = 0; c < sh.c_e; ++c) {
      const size_t at = (static_cast<size_t>(b) * sh.c_e + c) * plane4 + ij4;
      const float4 xh = __ldcs(reinterpret_cast<const float4*>(adj_hat) + at);
      const float4 d1 = __ldcs(reinterpret_cast<const float4*>(d1_adj) + at);
      float o[4] = {post_one(xh.x, d1.x, 0.f, inv_t, h, 0.f, false), post_one(xh.y, d1.y, 0.f, inv_t, h, 0.f, false),
                    post_one(xh.z, d1.z, 0.f, inv_t, h, 0.f, false), post_one(xh.w, d1.w, 0.f, inv_t, h, 0.f, false)};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        o[k] = ok[k] ? o[k] : 0.f;
        v[k] = (v[k] << 1) | (o[k] > 0.0f ? 1 : 0);
      }
      if (adj_next != nullptr) reinterpret_cast<float4*>(adj_next)[at] = make_float4(o[0], o[1], o[2], o[3]);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      v[k] = v[k] > num_adj_type - 1 ? num_adj_type - 1 : v[k];
      if (!ok[k] || i == 4 * j4 + k) v[k] = 0;  // invalid pairs and self-loops (sampler_node_adj.py:283)
    }
    reinterpret_cast<int4*>(adj_cls)[g] = make_int4(v[0], v[1], v[2], v[3]);
  }
  const int nb = sh.c_n - 4;
  const unsigned nodes = static_cast<unsigned>(sh.batch) * n;
  for (unsigned bi = tid; bi < nodes; bi += stride) {
    const bool ok = flags[bi] != 0;
    int v = 0;
    for (int c = 0; c < sh.c_n; ++c) {
      const size_t at = static_cast<size_t>(bi) * sh.c_n + c;
      float o = post_one(node_hat[at], d1_node[at], 0.f, inv_t, h, 0.f, false);
      o = ok ? o : 0.f;
      if (node_next != nullptr) node_next[at] = o;
      if (c < nb) v = (v << 1) | (o > 0.0f ? 1 : 0);
      else bbox[static_cast<size_t>(bi) * 4 + (c - nb)] = ok ? __fadd_rn(__fmul_rn(o, 0.5f), 0.5f) : 0.f;
    }
    v = v > num_node_type - 1 ? num_node_type - 1 : v;
    node_cls[bi] = ok ? v : 0;
  }
}

// Decode of the final sample (runner/sampler/sampler_node_adj.py:199-285 of the reference, 'bits' encodings):
//   class = clamp(bin2dec(x > 0, MSB first), 0, num_types - 1), masked; self-loops removed; box = x * 0.5 + 0.5, masked.
// (clamp(x, -1, 1) > 0 == x > 0, so the reference's clamp -> sign -> gt(0) chain collapses to one comparison.)
__global__ void __launch_bounds__(256)
decode_kernel(const float* __restrict__ adj, const float* __restrict__ node, const uint8_t* __restrict__ flags,
              int32_t* __restrict__ adj_cls, int32_t* __restrict__ node_cls, float* __restrict__ bbox, int num_adj_type,
              int num_node_type, EdmShape sh) {
  const int n = sh.n, nn = sh.n * sh.n;
  const long long pixels = static_cast<long long>(sh.batch) * nn;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  const long long tid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  for (long long px = tid; px < pixels; px += stride) {
    const int b = static_cast<int>(px / nn);
    const int ij = static_cast<int>(px - static_cast<long long>(b) * nn);
    const int i = ij / n, j = ij - i * n;
    int v = 0;
    if (i != j && flags[b * n + i] != 0 && flags[b * n + j] != 0) {
      for (int c = 0; c < sh.c_e; ++c) v = (v << 1) | (adj[(static_cast<size_t>(b) * sh.c_e + c) * nn + ij] > 0.0f ? 1 : 0);
      v = v < 0 ? 0 : (v > num_adj_type - 1 ? num_adj_type - 1 : v);
    }
    adj_cls[px] = v;
  }
  const int nb = sh.c_n - 4;  // class bits; the last four node channels are the box
  const long long nodes = static_cast<long long>(sh.batch) * n;
  for (long long bi = tid; bi < nodes; bi += stride) {
    const bool ok = flags[bi] != 0;
    const float* x = node + bi * sh.c_n;
    int v = 0;
    if (ok) {
      for (int c = 0; c < nb; ++c) v = (v << 1) | (x[c] > 0.0f ? 1 : 0);
      v = v < 0 ? 0 : (v > num_node_type - 1 ? num_node_type - 1 : v);
    }
    node_cls[bi] = v;
#pragma unroll
    for (int c = 0; c < 4; ++c) bbox[bi * 4 + c] = ok ? __fadd_rn(__fmul_rn(x[nb + c], 0.5f), 0.5f) : 0.f;
  }
}

// Pre-step with the noise drawn IN the kernel, bit-compatible with the two `torch.randn_like` calls of the reference
// (runner/mcmc_sampler/edm.py:358-364): ATen's normal_ on CUDA is a grid-stride kernel over Philox4x32-10,
//   curand_init(seed, thread, offset); per iteration  float4 r = curand_normal4()  ->  elements  li + k T, k < 4,
//   T = 256 * grid threads, grid = min(SMs * (max threads per SM / 256), ceil(numel / 256))
// (ATen/native/cuda/DistributionTemplates.h: calc_execution_policy, distribution_elementwise_grid_stride_kernel).
// Launching the same virtual grid with the generator's (seed, offset) reproduces eps element for element; the caller
// advances the generator by the same counter offset.  One launch per tensor (each has its own offset and grid).
template <bool ADJ>
__global__ void __launch_bounds__(256)
edm_pre_philox_kernel(const float* __restrict__ x, float* __restrict__ out, const uint8_t* __restrict__ flags, float c,
                      unsigned long long seed, unsigned long long offset, long long numel, const StepParams* __restrict__ P,
                      EdmShape sh) {
  if (P != nullptr) { c = P->noise_coef; seed = P->seed; offset = ADJ ? P->offset_adj : P->offset_node; }
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  curandStatePhilox4_32_10_t state;
  curand_init(seed, idx, offset, &state);
  const long long T = static_cast<long long>(blockDim.x) * gridDim.x;
  const long long rounded = ((numel - 1) / (T * 4) + 1) * T * 4;
  const int n = sh.n;
  for (long long li = idx; li < rounded; li += T * 4) {
    const float4 r = curand_normal4(&state);
#pragma unroll
    for (int ii = 0; ii < 4; ++ii) {
      const long long e = li + T * ii;
      if (e < numel) {
        const float eps = ii == 0 ? r.x : (ii == 1 ? r.y : (ii == 2 ? r.z : r.w));
        bool ok;
        const unsigned eu = static_cast<unsigned>(e);  // numel < 2^31 (checked by the launcher): 32-bit divisions
        if (ADJ) {
          const unsigned un = static_cast<unsigned>(n);
          const unsigned rr = eu / un, j = eu - rr * un;
          const unsigned q2 = rr / un, i = rr - q2 * un;       // q2 = b * c_e + c
          const unsigned b = q2 / static_cast<unsigned>(sh.c_e);
          ok = flags[b * un + i] != 0 && flags[b * un + j] != 0;
        } else {
          ok = flags[eu / static_cast<unsigned>(sh.c_n)] != 0;
        }
        out[e] = ok ? pre_one(x[e], eps, c) : 0.f;
      }
    }
  }
}

// The same draw for the completion pre-step (pre_known_one): `known` has the shape of x.  A kernel of its own so that
// the plain pre-step above stays exactly as it is.
template <bool ADJ>
__global__ void __launch_bounds__(256)
edm_pre_philox_known_kernel(const float* __restrict__ x, const float* __restrict__ known, float* __restrict__ out,
                            const uint8_t* __restrict__ flags, float c, float t_hat, unsigned long long seed,
                            unsigned long long offset, long long numel, const StepParams* __restrict__ P, EdmShape sh) {
  if (P != nullptr) { c = P->noise_coef; t_hat = P->t_hat; seed = P->seed; offset = ADJ ? P->offset_adj : P->offset_node; }
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  curandStatePhilox4_32_10_t state;
  curand_init(seed, idx, offset, &state);
  const long long T = static_cast<long long>(blockDim.x) * gridDim.x;
  const long long rounded = ((numel - 1) / (T * 4) + 1) * T * 4;
  const unsigned un = static_cast<unsigned>(sh.n);
  for (long long li = idx; li < rounded; li += T * 4) {
    const float4 r = curand_normal4(&state);
#pragma unroll
    for (int ii = 0; ii < 4; ++ii) {
      const long long e = li + T * ii;
      if (e < numel) {
        const float eps = ii == 0 ? r.x : (ii == 1 ? r.y : (ii == 2 ? r.z : r.w));
        bool ok;
        const unsigned eu = static_cast<unsigned>(e);
        if (ADJ) {
          const unsigned rr = eu / un, j = eu - rr * un;
          const unsigned q2 = rr / un, i = rr - q2 * un;
          const unsigned b = q2 / static_cast<unsigned>(sh.c_e);
          ok = flags[b * un + i] != 0 && flags[b * un + j] != 0;
        } else {
          ok = flags[eu / static_cast<unsigned>(sh.c_n)] != 0;
        }
        out[e] = ok ? pre_known_one(x[e], eps, known[e], c, t_hat) : 0.f;
      }
    }
  }
}

// Completion, after the last post-step: x = mask(isnan(k) ? x : k), in place.  Same streaming layout as edm_kernel
// (one float4 per thread per trip over the adjacency tensor, scalars over the nodes); runs once per sampling run.
__global__ void __launch_bounds__(256)
apply_known_kernel(float* adj, float* node, const float* __restrict__ k_adj, const float* __restrict__ k_node,
                   const uint8_t* __restrict__ flags, EdmShape sh) {
  const unsigned n = sh.n, n4 = sh.n >> 2, nce = n * sh.c_e;
  const unsigned adj_vec = static_cast<unsigned>(sh.batch) * sh.c_e * n * n4;
  const unsigned stride = gridDim.x * blockDim.x;
  const unsigned tid = blockIdx.x * blockDim.x + threadIdx.x;
  for (unsigned v = tid; v < adj_vec; v += stride) {
    const unsigned r = v / n4, j4 = v - r * n4;
    const unsigned b = r / nce, i = r % n;
    const uint8_t* f = flags + b * n;
    const bool fi = f[i] != 0;
    const uchar4 fj = *reinterpret_cast<const uchar4*>(f + 4 * j4);
    const float4 x = reinterpret_cast<const float4*>(adj)[v];
    const float4 k = __ldcs(reinterpret_cast<const float4*>(k_adj) + v);
    float4 o;
    o.x = (fi && fj.x) ? (isnan(k.x) ? x.x : k.x) : 0.f;
    o.y = (fi && fj.y) ? (isnan(k.y) ? x.y : k.y) : 0.f;
    o.z = (fi && fj.z) ? (isnan(k.z) ? x.z : k.z) : 0.f;
    o.w = (fi && fj.w) ? (isnan(k.w) ? x.w : k.w) : 0.f;
    reinterpret_cast<float4*>(adj)[v] = o;
  }
  const unsigned node_el = static_cast<unsigned>(sh.batch) * n * sh.c_n;
  for (unsigned v = tid; v < node_el; v += stride) {
    const bool ok = flags[v / static_cast<unsigned>(sh.c_n)] != 0;
    const float k = k_node[v];
    node[v] = ok ? (isnan(k) ? node[v] : k) : 0.f;
  }
}

// Reconstruction guidance (DESIGN.md §3.7), elementwise over both tensors, same streaming layout as apply_known_kernel:
//   kUpdate = false: out = mask(isnan(o) ? 0 : d - o)   o = known state: the residual, the output gradient of
//                                                      1/2 sum_known (D - k)^2
//   kUpdate = true:  out = mask(d - w * o)              o = the input gradient G of that loss: the guided D
// `out` may alias `d` (each element is read before it is written, by the same thread).
DSG_DEVICE float guide_one(float d, float o, float w, bool ok, bool update) {
  if (!ok) return 0.f;
  if (update) return __fsub_rn(d, __fmul_rn(w, o));
  return isnan(o) ? 0.f : __fsub_rn(d, o);
}

template <bool kUpdate>
__global__ void __launch_bounds__(256)
guidance_kernel(const float* d_adj, const float* d_node, const float* __restrict__ o_adj, const float* __restrict__ o_node,
                const uint8_t* __restrict__ flags, float w, float* out_adj, float* out_node, EdmShape sh) {
  const unsigned n = sh.n, n4 = sh.n >> 2, nce = n * sh.c_e;
  const unsigned adj_vec = static_cast<unsigned>(sh.batch) * sh.c_e * n * n4;
  const unsigned stride = gridDim.x * blockDim.x;
  const unsigned tid = blockIdx.x * blockDim.x + threadIdx.x;
  for (unsigned v = tid; v < adj_vec; v += stride) {
    const unsigned r = v / n4, j4 = v - r * n4;
    const unsigned b = r / nce, i = r % n;
    const uint8_t* f = flags + b * n;
    const bool fi = f[i] != 0;
    const uchar4 fj = *reinterpret_cast<const uchar4*>(f + 4 * j4);
    const float4 d = reinterpret_cast<const float4*>(d_adj)[v];
    const float4 o = reinterpret_cast<const float4*>(o_adj)[v];
    float4 y;
    y.x = guide_one(d.x, o.x, w, fi && fj.x, kUpdate);
    y.y = guide_one(d.y, o.y, w, fi && fj.y, kUpdate);
    y.z = guide_one(d.z, o.z, w, fi && fj.z, kUpdate);
    y.w = guide_one(d.w, o.w, w, fi && fj.w, kUpdate);
    reinterpret_cast<float4*>(out_adj)[v] = y;
  }
  const unsigned node_el = static_cast<unsigned>(sh.batch) * n * sh.c_n;
  for (unsigned v = tid; v < node_el; v += stride)
    out_node[v] = guide_one(d_node[v], o_node[v], w, flags[v / static_cast<unsigned>(sh.c_n)] != 0, kUpdate);
}

// User-level conditions -> the NaN-coded known state (the inverse of decode_kernel for the 'bits' encodings):
// a known class (>= 0) is written as its bits, MSB first, +1 for a set bit and -1 for a clear one, a known box
// coordinate b as 2 b - 1; everything else is NaN (free).  adj_cls [B,N,N] fills all c_e channels of its pair,
// node_cls [B,N] the first c_n - 4 node channels, bbox [B,N,4] the last four.  Any input may be NULL (all free).
__global__ void __launch_bounds__(256)
encode_known_kernel(const int32_t* __restrict__ node_cls, const float* __restrict__ bbox, const int32_t* __restrict__ adj_cls,
                    float* __restrict__ k_adj, float* __restrict__ k_node, EdmShape sh) {
  const unsigned n = sh.n, nn = n * n;
  const unsigned pixels = static_cast<unsigned>(sh.batch) * nn;
  const unsigned stride = gridDim.x * blockDim.x;
  const unsigned tid = blockIdx.x * blockDim.x + threadIdx.x;
  const float nan = __int_as_float(0x7fc00000);
  for (unsigned px = tid; px < pixels; px += stride) {
    const unsigned b = px / nn, ij = px - b * nn;
    const int v = adj_cls != nullptr ? adj_cls[px] : -1;
    for (int c = 0; c < sh.c_e; ++c)
      k_adj[(static_cast<size_t>(b) * sh.c_e + c) * nn + ij] = v < 0 ? nan : (((v >> (sh.c_e - 1 - c)) & 1) ? 1.f : -1.f);
  }
  const int nb = sh.c_n - 4;
  const unsigned nodes = static_cast<unsigned>(sh.batch) * n;
  for (unsigned bi = tid; bi < nodes; bi += stride) {
    const int v = node_cls != nullptr ? node_cls[bi] : -1;
    float* out = k_node + static_cast<size_t>(bi) * sh.c_n;
    for (int c = 0; c < nb; ++c) out[c] = v < 0 ? nan : (((v >> (nb - 1 - c)) & 1) ? 1.f : -1.f);
#pragma unroll
    for (int c = 0; c < 4; ++c) out[nb + c] = bbox != nullptr ? __fsub_rn(__fmul_rn(2.f, bbox[bi * 4 + c]), 1.f) : nan;
  }
}

template <int MODE>
int launch_mode(const float* a0, const float* a1, const float* a2, float* a_out, const float* n0, const float* n1,
                const float* n2, float* n_out, const uint8_t* flags, float s0, float s1, float s2, const void* dev_params,
                int batch, int c_e, int n, int c_n, cudaStream_t st) {
  DSG_REQUIRE(batch > 0 && c_e > 0 && n > 0 && c_n > 0 && n % 4 == 0, "edm step: bad shape B=%d C_e=%d N=%d C_n=%d",
              batch, c_e, n, c_n);
  DSG_REQUIRE(((reinterpret_cast<uintptr_t>(a0) | reinterpret_cast<uintptr_t>(a_out) | reinterpret_cast<uintptr_t>(a1) |
                reinterpret_cast<uintptr_t>(a2)) & 15) == 0 && (reinterpret_cast<uintptr_t>(flags) & 3) == 0,
              "edm step: adjacency tensors must be 16-byte aligned (flags 4-byte)");
  const long long vec = static_cast<long long>(batch) * c_e * n * (n / 4);
  DSG_REQUIRE(vec < 2147483647LL - 148LL * 8 * 256 * EDM_U && static_cast<long long>(batch) * n * c_n < 2147483647LL,
              "edm step: %lld vectors (32-bit indexing)", vec);
  long long blocks = (vec + 256 * EDM_U - 1) / (256 * EDM_U);
  const long long cap = 148LL * 8;  // 8 resident CTAs of 256 threads per SM
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  EdmShape sh{batch, c_e, n, c_n};
  edm_kernel<MODE><<<static_cast<unsigned>(blocks), 256, 0, st>>>(a0, a1, a2, a_out, n0, n1, n2, n_out, flags, s0, s1,
                                                                  s2, static_cast<const StepParams*>(dev_params), sh);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

}  // namespace

int launch_edm_pre_step(const float* adj, const float* node, const float* eps_adj, const float* eps_node,
                        const uint8_t* flags, float noise_coef, float* adj_hat, float* node_hat, int batch, int c_e,
                        int n, int c_n, cudaStream_t st) {
  return launch_mode<0>(adj, eps_adj, nullptr, adj_hat, node, eps_node, nullptr, node_hat, flags, noise_coef, 0.f, 0.f,
                        nullptr, batch, c_e, n, c_n, st);
}

int launch_edm_pre_step_philox(const float* adj, const float* node, const uint8_t* flags, float noise_coef,
                               unsigned long long seed, unsigned long long offset_adj, int grid_adj,
                               unsigned long long offset_node, int grid_node, const void* dev_params, float* adj_hat,
                               float* node_hat, int batch, int c_e, int n, int c_n, cudaStream_t st) {
  DSG_REQUIRE(batch > 0 && c_e > 0 && n > 0 && c_n > 0 && grid_adj > 0 && grid_node > 0,
              "edm philox pre-step: bad shape / grid B=%d C_e=%d N=%d C_n=%d grids %d %d", batch, c_e, n, c_n, grid_adj,
              grid_node);
  EdmShape sh{batch, c_e, n, c_n};
  const long long na = static_cast<long long>(batch) * c_e * n * n, nn = static_cast<long long>(batch) * n * c_n;
  DSG_REQUIRE(na < 2147483647LL && nn < 2147483647LL, "edm philox pre-step: %lld / %lld elements (32-bit indexing)", na, nn);
  const StepParams* P = static_cast<const StepParams*>(dev_params);
  edm_pre_philox_kernel<true><<<static_cast<unsigned>(grid_adj), 256, 0, st>>>(adj, adj_hat, flags, noise_coef, seed,
                                                                               offset_adj, na, P, sh);
  DSG_LAUNCH_CHECK();
  edm_pre_philox_kernel<false><<<static_cast<unsigned>(grid_node), 256, 0, st>>>(node, node_hat, flags, noise_coef, seed,
                                                                                 offset_node, nn, P, sh);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_edm_pre_step_known(const float* adj, const float* node, const float* eps_adj, const float* eps_node,
                              const float* known_adj, const float* known_node, const uint8_t* flags, float noise_coef,
                              float t_hat, float* adj_hat, float* node_hat, int batch, int c_e, int n, int c_n,
                              cudaStream_t st) {
  return launch_mode<4>(adj, eps_adj, known_adj, adj_hat, node, eps_node, known_node, node_hat, flags, noise_coef, t_hat,
                        0.f, nullptr, batch, c_e, n, c_n, st);
}

int launch_edm_pre_step_philox_known(const float* adj, const float* node, const float* known_adj, const float* known_node,
                                     const uint8_t* flags, float noise_coef, float t_hat, unsigned long long seed,
                                     unsigned long long offset_adj, int grid_adj, unsigned long long offset_node,
                                     int grid_node, const void* dev_params, float* adj_hat, float* node_hat, int batch,
                                     int c_e, int n, int c_n, cudaStream_t st) {
  DSG_REQUIRE(batch > 0 && c_e > 0 && n > 0 && c_n > 0 && grid_adj > 0 && grid_node > 0,
              "edm philox pre-step (known): bad shape / grid B=%d C_e=%d N=%d C_n=%d grids %d %d", batch, c_e, n, c_n,
              grid_adj, grid_node);
  DSG_REQUIRE(((reinterpret_cast<uintptr_t>(adj) | reinterpret_cast<uintptr_t>(known_adj) |
                reinterpret_cast<uintptr_t>(adj_hat)) & 15) == 0 && (reinterpret_cast<uintptr_t>(flags) & 3) == 0,
              "edm philox pre-step (known): adjacency tensors must be 16-byte aligned (flags 4-byte)");
  EdmShape sh{batch, c_e, n, c_n};
  const long long na = static_cast<long long>(batch) * c_e * n * n, nn = static_cast<long long>(batch) * n * c_n;
  DSG_REQUIRE(na < 2147483647LL && nn < 2147483647LL, "edm philox pre-step (known): %lld / %lld elements (32-bit indexing)",
              na, nn);
  const StepParams* P = static_cast<const StepParams*>(dev_params);
  edm_pre_philox_known_kernel<true><<<static_cast<unsigned>(grid_adj), 256, 0, st>>>(
      adj, known_adj, adj_hat, flags, noise_coef, t_hat, seed, offset_adj, na, P, sh);
  DSG_LAUNCH_CHECK();
  edm_pre_philox_known_kernel<false><<<static_cast<unsigned>(grid_node), 256, 0, st>>>(
      node, known_node, node_hat, flags, noise_coef, t_hat, seed, offset_node, nn, P, sh);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_edm_apply_known(float* adj, float* node, const float* known_adj, const float* known_node, const uint8_t* flags,
                           int batch, int c_e, int n, int c_n, cudaStream_t st) {
  DSG_REQUIRE(batch > 0 && c_e > 0 && n > 0 && c_n > 0 && n % 4 == 0, "apply_known: bad shape B=%d C_e=%d N=%d C_n=%d",
              batch, c_e, n, c_n);
  DSG_REQUIRE(((reinterpret_cast<uintptr_t>(adj) | reinterpret_cast<uintptr_t>(known_adj)) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(flags) & 3) == 0,
              "apply_known: adjacency tensors must be 16-byte aligned (flags 4-byte)");
  const long long vec = static_cast<long long>(batch) * c_e * n * (n / 4);
  DSG_REQUIRE(vec < 2147483647LL - 148LL * 8 * 256 && static_cast<long long>(batch) * n * c_n < 2147483647LL,
              "apply_known: %lld vectors (32-bit indexing)", vec);
  long long blocks = (vec + 255) / 256;
  if (blocks > 148LL * 8) blocks = 148LL * 8;
  EdmShape sh{batch, c_e, n, c_n};
  apply_known_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(adj, node, known_adj, known_node, flags, sh);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_edm_guidance(const float* d_adj, const float* d_node, const float* o_adj, const float* o_node,
                        const uint8_t* flags, float w, int update, float* out_adj, float* out_node, int batch, int c_e,
                        int n, int c_n, cudaStream_t st) {
  DSG_REQUIRE(batch > 0 && c_e > 0 && n > 0 && c_n > 0 && n % 4 == 0, "edm guidance: bad shape B=%d C_e=%d N=%d C_n=%d",
              batch, c_e, n, c_n);
  DSG_REQUIRE(((reinterpret_cast<uintptr_t>(d_adj) | reinterpret_cast<uintptr_t>(o_adj) |
                reinterpret_cast<uintptr_t>(out_adj)) & 15) == 0 && (reinterpret_cast<uintptr_t>(flags) & 3) == 0,
              "edm guidance: adjacency tensors must be 16-byte aligned (flags 4-byte)");
  const long long vec = static_cast<long long>(batch) * c_e * n * (n / 4);
  DSG_REQUIRE(vec < 2147483647LL - 148LL * 8 * 256 && static_cast<long long>(batch) * n * c_n < 2147483647LL,
              "edm guidance: %lld vectors (32-bit indexing)", vec);
  long long blocks = (vec + 255) / 256;
  if (blocks > 148LL * 8) blocks = 148LL * 8;
  EdmShape sh{batch, c_e, n, c_n};
  if (update)
    guidance_kernel<true><<<static_cast<unsigned>(blocks), 256, 0, st>>>(d_adj, d_node, o_adj, o_node, flags, w, out_adj,
                                                                         out_node, sh);
  else
    guidance_kernel<false><<<static_cast<unsigned>(blocks), 256, 0, st>>>(d_adj, d_node, o_adj, o_node, flags, 0.f, out_adj,
                                                                          out_node, sh);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_encode_known(const int32_t* node_cls, const float* bbox, const int32_t* adj_cls, float* known_adj,
                        float* known_node, int batch, int c_e, int n, int c_n, cudaStream_t st) {
  DSG_REQUIRE(batch > 0 && c_e > 0 && c_e <= 30 && n > 0 && c_n > 4 && c_n - 4 <= 30,
              "encode_known: bad shape B=%d C_e=%d N=%d C_n=%d", batch, c_e, n, c_n);
  const long long pixels = static_cast<long long>(batch) * n * n;
  DSG_REQUIRE(pixels < 2147483647LL - 148LL * 8 * 256, "encode_known: %lld pixels (32-bit indexing)", pixels);
  long long blocks = (pixels + 255) / 256;
  if (blocks > 148LL * 8) blocks = 148LL * 8;
  EdmShape sh{batch, c_e, n, c_n};
  encode_known_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(node_cls, bbox, adj_cls, known_adj, known_node, sh);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_edm_post_step(const float* adj_hat, const float* node_hat, const float* d1_adj, const float* d1_node,
                         const float* d2_adj, const float* d2_node, const uint8_t* flags, float inv_t_hat, float h,
                         float inv_t_prime, const void* dev_params, float* adj_next, float* node_next, int batch, int c_e,
                         int n, int c_n, cudaStream_t st) {
  if (d2_adj != nullptr)
    return launch_mode<1>(adj_hat, d1_adj, d2_adj, adj_next, node_hat, d1_node, d2_node, node_next, flags, inv_t_hat, h,
                          inv_t_prime, dev_params, batch, c_e, n, c_n, st);
  return launch_mode<2>(adj_hat, d1_adj, nullptr, adj_next, node_hat, d1_node, nullptr, node_next, flags, inv_t_hat, h,
                        0.f, dev_params, batch, c_e, n, c_n, st);
}

int launch_edm_step_advance(const void* table, void* cur, int* counter, cudaStream_t st) {
  step_advance_kernel<<<1, 32, 0, st>>>(static_cast<const StepParams*>(table), static_cast<StepParams*>(cur), counter);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_edm_final_decode(const float* adj_hat, const float* node_hat, const float* d1_adj, const float* d1_node,
                            const uint8_t* flags, float inv_t_hat, float h, const void* dev_params, float* adj_next,
                            float* node_next, int32_t* adj_cls, int32_t* node_cls, float* bbox, int num_adj_type,
                            int num_node_type, int batch, int c_e, int n, int c_n, cudaStream_t st) {
  DSG_REQUIRE(batch > 0 && c_e > 0 && c_e <= 30 && n > 0 && n % 4 == 0 && c_n > 4 && c_n - 4 <= 30 && num_adj_type > 0 &&
                  num_node_type > 0, "final step + decode: bad shape B=%d C_e=%d N=%d C_n=%d", batch, c_e, n, c_n);
  DSG_REQUIRE(((reinterpret_cast<uintptr_t>(adj_hat) | reinterpret_cast<uintptr_t>(d1_adj) |
                reinterpret_cast<uintptr_t>(adj_next) | reinterpret_cast<uintptr_t>(adj_cls)) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(flags) & 3) == 0, "final step + decode: tensors must be 16-byte aligned");
  const long long groups = static_cast<long long>(batch) * n * (n / 4);
  DSG_REQUIRE(groups < 2147483647LL, "final step + decode: %lld pixel groups (32-bit indexing)", groups);
  long long blocks = (groups + 255) / 256;
  if (blocks > 148LL * 8) blocks = 148LL * 8;
  EdmShape sh{batch, c_e, n, c_n};
  edm_final_decode_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(
      adj_hat, node_hat, d1_adj, d1_node, flags, inv_t_hat, h, static_cast<const StepParams*>(dev_params), adj_next,
      node_next, adj_cls, node_cls, bbox, num_adj_type, num_node_type, sh);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_decode(const float* adj, const float* node, const uint8_t* flags, int32_t* adj_cls, int32_t* node_cls,
                  float* bbox, int num_adj_type, int num_node_type, int batch, int c_e, int n, int c_n, cudaStream_t st) {
  DSG_REQUIRE(batch > 0 && c_e > 0 && c_e <= 30 && n > 0 && c_n > 4 && c_n - 4 <= 30 && num_adj_type > 0 && num_node_type > 0,
              "decode: bad shape B=%d C_e=%d N=%d C_n=%d", batch, c_e, n, c_n);
  const long long pixels = static_cast<long long>(batch) * n * n;
  long long blocks = (pixels + 255) / 256;
  if (blocks > 148LL * 8) blocks = 148LL * 8;
  EdmShape sh{batch, c_e, n, c_n};
  decode_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(adj, node, flags, adj_cls, node_cls, bbox, num_adj_type,
                                                              num_node_type, sh);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_mask_scale(const float* adj, const float* node, const uint8_t* flags, float scale, float* adj_out,
                      float* node_out, int batch, int c_e, int n, int c_n, cudaStream_t st) {
  return launch_mode<3>(adj, nullptr, nullptr, adj_out, node, nullptr, nullptr, node_out, flags, scale, 0.f, 0.f, nullptr,
                        batch, c_e, n, c_n, st);
}

}  // namespace dsg
