// Row kernels of the denoiser: everything that is not a GEMM or attention.
//
// HBM-bound by construction: each kernel reads its fp32 rows once with 128-bit loads (one warp per row, the
// whole row in registers), does LayerNorm / FiLM / gather / scatter in registers and writes once.  The
// window / merge / breakup reshuffles of the reference (model/diffusesg/diffusesg.py:28-57, :314-335, :374-403)
// are index arithmetic on the row addresses of these kernels; the 60-channel input grid (:784-802) is never
// materialised.
#include "common.cuh"
#include "kernels.h"

namespace dsg {
namespace {

constexpr int kRowThreads = 256;  // 8 rows per CTA
constexpr float kLnEps = 1e-5f;   // nn.LayerNorm default (diffusesg.py:175 etc.)

DSG_DEVICE uint2 pack4_bf16(float a, float b, float c, float d) { return make_uint2(pack_bf16x2(a, b), pack_bf16x2(c, d)); }

// Sum over the LPR consecutive lanes that share a row.
template <int LPR>
DSG_DEVICE float group_sum(float v) {
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// A row of C fp32 values spread over LPR lanes (32 = a whole warp): float4 number (sub + LPR i) lives in v[i],
// sub = lane % LPR.  Narrow rows (C = 96, 192) use 8 / 16 lanes per row so that no lane idles.
template <int NV, int LPR = 32>
struct Row {
  float4 v[NV];
  DSG_DEVICE void load(const float* p, int C, int lane) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int e = (lane + LPR * i) * 4;
      v[i] = (e < C) ? *reinterpret_cast<const float4*>(p + e) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  DSG_DEVICE void store(float* p, int C, int lane) const {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int e = (lane + LPR * i) * 4;
      if (e < C) *reinterpret_cast<float4*>(p + e) = v[i];
    }
  }
  // (x - mean) * rstd over the C valid entries, in place
  DSG_DEVICE void normalize(int C, int lane) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    const float mean = group_sum<LPR>(s) / C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int e = (lane + LPR * i) * 4;
      if (e < C) {
        v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
        q += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
      }
    }
    const float rstd = rsqrtf(group_sum<LPR>(q) / C + kLnEps);
#pragma unroll
    for (int i = 0; i < NV; ++i) { v[i].x *= rstd; v[i].y *= rstd; v[i].z *= rstd; v[i].w *= rstd; }
  }
  DSG_DEVICE void affine(const float* g, const float* b, int C, int lane) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int e = (lane + LPR * i) * 4;
      if (e < C) {
        const float4 gg = __ldg(reinterpret_cast<const float4*>(g + e));
        const float4 bb = __ldg(reinterpret_cast<const float4*>(b + e));
        v[i].x = fmaf(v[i].x, gg.x, bb.x); v[i].y = fmaf(v[i].y, gg.y, bb.y);
        v[i].z = fmaf(v[i].z, gg.z, bb.z); v[i].w = fmaf(v[i].w, gg.w, bb.w);
      }
    }
  }
  DSG_DEVICE void store_bf16(bf16* p, int C, int lane) const {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int e = (lane + LPR * i) * 4;
      if (e < C) *reinterpret_cast<uint2*>(p + e) = pack4_bf16(v[i].x, v[i].y, v[i].z, v[i].w);
    }
  }
};

// ---------------------------------------------------------------------------------------------------------
// FiLM + SiLU (+ shortcut write) + LayerNorm            (SwinTransformerBlock.forward :238-243)
// ---------------------------------------------------------------------------------------------------------
template <int NV, int LPR>
__global__ void __launch_bounds__(kRowThreads)
film_ln_kernel(const float* __restrict__ x_in, float* __restrict__ x_out, bf16* __restrict__ y,
               const float* __restrict__ film, int film_ld, int cond_uniform, const float* __restrict__ gamma,
               const float* __restrict__ beta, long long rows, int tokens_per_sample, int C,
               const int* __restrict__ src_rows) {
  const int lane = threadIdx.x % LPR;
  long long row = static_cast<long long>(blockIdx.x) * (kRowThreads / LPR) + threadIdx.x / LPR;
  const bool valid = row < rows;  // surplus lane groups stay for the shuffles but never store
  if (!valid) row = rows - 1;
  const int b = cond_uniform ? 0 : static_cast<int>(row / tokens_per_sample);
  const float* sc = film + static_cast<size_t>(b) * film_ld;  // scale[C] then shift[C]
  Row<NV, LPR> r;
  // src_rows: the input lives in another layout of the padding skipping (model.cu); output row `row` reads input row
  // src_rows[row] - the layout change costs nothing beyond the 4-byte index (x_in must not alias x_out then)
  r.load(x_in + (src_rows != nullptr ? static_cast<long long>(src_rows[row]) : row) * C, C, lane);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int e = (lane + LPR * i) * 4;
    if (e < C) {
      const float4 s = __ldg(reinterpret_cast<const float4*>(sc + e));
      const float4 t = __ldg(reinterpret_cast<const float4*>(sc + C + e));
      r.v[i].x = silu_f(fmaf(r.v[i].x, s.x + 1.f, t.x));
      r.v[i].y = silu_f(fmaf(r.v[i].y, s.y + 1.f, t.y));
      r.v[i].z = silu_f(fmaf(r.v[i].z, s.z + 1.f, t.z));
      r.v[i].w = silu_f(fmaf(r.v[i].w, s.w + 1.f, t.w));
    }
  }
  if (valid) r.store(x_out + row * C, C, lane);
  r.normalize(C, lane);
  r.affine(gamma, beta, C, lane);
  if (valid) r.store_bf16(y + row * C, C, lane);
}

template <int NV, int LPR>
__global__ void __launch_bounds__(kRowThreads)
ln_kernel(const float* __restrict__ x, bf16* __restrict__ y, const float* __restrict__ gamma,
          const float* __restrict__ beta, long long rows, int C) {
  const int lane = threadIdx.x % LPR;
  long long row = static_cast<long long>(blockIdx.x) * (kRowThreads / LPR) + threadIdx.x / LPR;
  const bool valid = row < rows;
  if (!valid) row = rows - 1;
  Row<NV, LPR> r;
  r.load(x + row * C, C, lane);
  r.normalize(C, lane);
  r.affine(gamma, beta, C, lane);
  if (valid) r.store_bf16(y + row * C, C, lane);
}

// ---------------------------------------------------------------------------------------------------------
// PatchMerging front half (2x2 gather + LN(4C), :314-333) and PatchBreakup middle (LN(D) -> depth-to-space -> LN(D/4),
// :386-400) for the widths the geometries use, C and Dq = D / 4 of 96, 192 or 384: lanes [8k, 8k + 8) own source pixel /
// chunk k, so
// the 2x2 gather (scatter) is plain address arithmetic per lane group, the per-chunk LayerNorm is an 8-lane shuffle
// reduction, and no lane divides by a run-time width.  Generic one-warp-per-row versions spent ~1.4 k instructions per
// row on that index arithmetic and were issue-bound at 2 TB/s.
// ---------------------------------------------------------------------------------------------------------
template <int NV>  // NV = C / 32 float4 per lane
__global__ void __launch_bounds__(kRowThreads)
merge_ln_q_kernel(const float* __restrict__ x, bf16* __restrict__ y, const float* __restrict__ gamma,
                  const float* __restrict__ beta, long long rows_out, int res) {
  constexpr int C = NV * 32, C4 = 4 * C;
  const int lane = threadIdx.x & 31, q = lane >> 3, sub = lane & 7;
  const long long row = static_cast<long long>(blockIdx.x) * (kRowThreads / 32) + (threadIdx.x >> 5);
  if (row >= rows_out) return;
  const int half = res >> 1;
  const int ox = static_cast<int>(row % half);
  const int oy = static_cast<int>((row / half) % half);
  const long long b = row / (static_cast<long long>(half) * half);
  // channel block q holds pixel (2y + q % 2, 2x + q / 2)                         (:325-329)
  const float* src = x + ((b * res + (2 * oy + (q & 1))) * res + (2 * ox + (q >> 1))) * C;
  float4 v[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = *reinterpret_cast<const float4*>(src + (sub + 8 * i) * 4);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  const float mean = warp_sum(s) * (1.0f / C4);
  float qq = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
    qq += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
  }
  const float rstd = rsqrtf(warp_sum(qq) * (1.0f / C4) + kLnEps);
  bf16* dst = y + row * C4 + q * C;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int e = (sub + 8 * i) * 4;
    const float4 gg = __ldg(reinterpret_cast<const float4*>(gamma + q * C + e));
    const float4 bb = __ldg(reinterpret_cast<const float4*>(beta + q * C + e));
    *reinterpret_cast<uint2*>(dst + e) = pack4_bf16(fmaf(v[i].x * rstd, gg.x, bb.x), fmaf(v[i].y * rstd, gg.y, bb.y),
                                                    fmaf(v[i].z * rstd, gg.z, bb.z), fmaf(v[i].w * rstd, gg.w, bb.w));
  }
}

template <int NV>  // NV = Dq / 32 float4 per lane, Dq = D / 4
__global__ void __launch_bounds__(kRowThreads)
breakup_ln_q_kernel(const float* __restrict__ t, bf16* __restrict__ y, const float* __restrict__ g1,
                    const float* __restrict__ b1, const float* __restrict__ g2, const float* __restrict__ b2,
                    long long rows_in, int res, const int* __restrict__ tok0, const int* __restrict__ width, int sh,
                    const int* __restrict__ src_perm) {
  constexpr int Dq = NV * 32, D = 4 * Dq;
  const int lane = threadIdx.x & 31, k = lane >> 3, sub = lane & 7;
  const long long row = static_cast<long long>(blockIdx.x) * (kRowThreads / 32) + (threadIdx.x >> 5);
  if (row >= rows_in) return;
  const int ix = static_cast<int>(row % res);
  const int iy = static_cast<int>((row / res) % res);
  const long long b = row / (static_cast<long long>(res) * res);
  // compacting variant (padding skipping, model.cu): the input is the dense [B, res, res] grid, the output the compact
  // layout in which sample b is a (width[b] >> sh)^2 image starting at token tok0[b] >> 2 sh
  const int res2 = 2 * res;
  long long out_tok0 = ((b * res2 + 2 * iy) * res2) + 2 * ix;   // token of the (dy, dx) = (0, 0) child, dense
  int out_pitch = res2;
  if (tok0 != nullptr) {
    // the input image shows sample src_perm[b] when the input itself is a compact stack (nullptr: dense, sample b)
    const long long sb = src_perm != nullptr ? src_perm[b] : b;
    if (sb < 0) return;                          // an all-padding image has no children anyone reads
    const int wc = width[sb] >> sh;
    if (2 * iy >= wc || 2 * ix >= wc) return;   // children outside the kept corner: dead, never read
    out_pitch = wc;
    out_tok0 = (static_cast<long long>(tok0[sb]) >> (2 * sh)) + static_cast<long long>(2 * iy) * wc + 2 * ix;
  }
  const float* src = t + row * D + k * Dq;  // lanes [8k, 8k + 8) own chunk k = elements [k Dq, (k + 1) Dq)
  float4 v[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = *reinterpret_cast<const float4*>(src + (sub + 8 * i) * 4);
  // LayerNorm(D) over the whole row                                              (:386)
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  const float mean = warp_sum(s) * (1.0f / D);
  float qq = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
    qq += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
  }
  const float rstd = rsqrtf(warp_sum(qq) * (1.0f / D) + kLnEps);
  float s2 = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int e = k * Dq + (sub + 8 * i) * 4;
    const float4 gg = __ldg(reinterpret_cast<const float4*>(g1 + e));
    const float4 bb = __ldg(reinterpret_cast<const float4*>(b1 + e));
    v[i].x = fmaf(v[i].x * rstd, gg.x, bb.x); v[i].y = fmaf(v[i].y * rstd, gg.y, bb.y);
    v[i].z = fmaf(v[i].z * rstd, gg.z, bb.z); v[i].w = fmaf(v[i].w * rstd, gg.w, bb.w);
    s2 += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  // LayerNorm(D / 4) of this lane group's chunk                                   (:399)
  const float mean2 = group_sum<8>(s2) * (1.0f / Dq);
  float q2 = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i].x -= mean2; v[i].y -= mean2; v[i].z -= mean2; v[i].w -= mean2;
    q2 += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
  }
  const float rstd2 = rsqrtf(group_sum<8>(q2) * (1.0f / Dq) + kLnEps);
  // chunk k lands on pixel (2y + k % 2, 2x + k / 2) of the up-sampled grid        (:394-397)
  bf16* dst = y + (out_tok0 + static_cast<long long>(k & 1) * out_pitch + (k >> 1)) * Dq;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (sub + 8 * i) * 4;
    const float4 gg = __ldg(reinterpret_cast<const float4*>(g2 + c));
    const float4 bb = __ldg(reinterpret_cast<const float4*>(b2 + c));
    *reinterpret_cast<uint2*>(dst + c) = pack4_bf16(fmaf(v[i].x * rstd2, gg.x, bb.x), fmaf(v[i].y * rstd2, gg.y, bb.y),
                                                    fmaf(v[i].z * rstd2, gg.z, bb.z), fmaf(v[i].w * rstd2, gg.w, bb.w));
  }
}

// y[m] = bf16([x[m], skip[m]])                                                    (:753 torch.cat)
__global__ void __launch_bounds__(256)
concat_bf16_kernel(const float* __restrict__ x, const float* __restrict__ skip, bf16* __restrict__ y, long long rows,
                   int C, const int* __restrict__ skip_rows) {
  const int c4 = C >> 2;
  const long long total = rows * 2 * c4;
  for (long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long row = idx / (2 * c4);
    const int e = static_cast<int>(idx - row * (2 * c4));
    // skip_rows: the skip tensor lives in another layout of the padding skipping (see film_ln_kernel)
    const long long srow = skip_rows != nullptr ? static_cast<long long>(skip_rows[row]) : row;
    const float* src = (e < c4) ? x + row * C + e * 4 : skip + srow * C + (e - c4) * 4;
    const float4 v = *reinterpret_cast<const float4*>(src);
    *reinterpret_cast<uint2*>(y + row * (2 * C) + e * 4) = pack4_bf16(v.x, v.y, v.z, v.w);
  }
}

// ---------------------------------------------------------------------------------------------------------
// sigma conditioning                                                   (:507-513, :768-771, affine layers)
// ---------------------------------------------------------------------------------------------------------
__global__ void sinusoid_kernel(const float* __restrict__ labels, long long label_stride, float* __restrict__ e0,
                                int n_cond, int embed) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int half = embed >> 1;
  if (idx >= n_cond * half) return;
  const int r = idx / half, k = idx - r * half;
  const float f = powf(1.0f / 10000.0f, static_cast<float>(k) / static_cast<float>(half));
  const float a = labels[r * label_stride] * f;
  e0[r * embed + k] = cosf(a);
  e0[r * embed + half + k] = sinf(a);
}

// y[r, o] = act(W[o, :] . x[r, :] + b[o]); one warp per output
__global__ void __launch_bounds__(256)
small_linear_kernel(const float* __restrict__ x, const float* __restrict__ W, const float* __restrict__ bias,
                    float* __restrict__ y, int n, int K, int O, int act_silu) {
  const long long wid = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (wid >= static_cast<long long>(n) * O) return;
  const int r = static_cast<int>(wid / O), o = static_cast<int>(wid - static_cast<long long>(r) * O);
  const float* xr = x + static_cast<size_t>(r) * K;
  const float* wr = W + static_cast<size_t>(o) * K;
  float s = 0.f;
  for (int k = lane; k < K; k += 32) s = fmaf(__ldg(wr + k), xr[k], s);
  s = warp_sum(s);
  if (lane == 0) {
    s += bias ? bias[o] : 0.f;
    y[static_cast<size_t>(r) * O + o] = act_silu ? silu_f(s) : s;
  }
}

// coef[0..3][n] = c_in, c_skip, c_out, c_noise                    (runner/objectives/edm.py:122-126, sigma_data 0.5)
__global__ void precond_coef_kernel(const float* __restrict__ sigmas, int sigma_stride, float* __restrict__ coef,
                                    int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float s = sigmas[static_cast<size_t>(i) * sigma_stride];
  const float s2 = __fadd_rn(__fmul_rn(s, s), 0.25f);
  coef[i] = __fdiv_rn(1.0f, __fsqrt_rn(s2));
  coef[n + i] = __fdiv_rn(0.25f, s2);
  coef[2 * n + i] = __fdiv_rn(__fmul_rn(s, 0.5f), __fsqrt_rn(s2));
  coef[3 * n + i] = __fdiv_rn(logf(s), 4.0f);
}

// ---------------------------------------------------------------------------------------------------------
// patch embedding without the 60-channel grid                                   (:784-802, :569-577)
// ---------------------------------------------------------------------------------------------------------
// rc[b, i, 0:E]  = sum_c W[:, row-plane c] * nodecat[b, i, c]      nodecat = [self-cond node, c_in * node]
// rc[b, i, E:2E] = sum_c W[:, col-plane c] * nodecat[b, i, c]
// w_rc is [2, 2 c_n(self_cond) or c_n, E] (input-channel major so that lanes read consecutive e).
// One thread per output column e2 keeps its <= 32 weights in registers and walks kNodeRows rows (b, i); the rows' node
// vectors are staged in shared memory.  (One CTA per row re-read the 18 KB weight table 32768 times: 87 us.)
constexpr int kNodeRows = 16;
__global__ void node_proj_kernel(const float* __restrict__ node, const float* __restrict__ sc_node,
                                 const float* __restrict__ in_scale, const float* __restrict__ w_rc,
                                 float* __restrict__ rc, int batch, int n, int c_n, int self_cond, int embed) {
  __shared__ float sv[kNodeRows][32];
  const int cin = self_cond ? 2 * c_n : c_n;  // <= 32 (checked by the launcher)
  const long long rows = static_cast<long long>(batch) * n;
  const long long row0 = static_cast<long long>(blockIdx.x) * kNodeRows;
  // all 32 channel slots are written: the product loop below runs over 32 channels with zero weights beyond cin, and
  // 0 x (whatever an earlier kernel left in this SM's shared memory) is NaN whenever the leftover is a NaN / Inf pattern
  for (int idx = threadIdx.x; idx < kNodeRows * 32; idx += blockDim.x) {
    const int r = idx >> 5, ch = idx & 31;
    const long long bi = row0 + r;
    float v = 0.f;
    if (bi < rows && ch < cin) {
      if (self_cond && ch < c_n) {
        v = sc_node ? sc_node[bi * c_n + ch] : 0.f;
      } else {
        const float sc = in_scale ? in_scale[bi / n] : 1.f;
        v = __fmul_rn(sc, node[bi * c_n + (self_cond ? ch - c_n : ch)]);
      }
    }
    sv[r][ch] = v;
  }
  __syncthreads();
  const int e2 = threadIdx.x;  // 0 .. 2E-1
  if (e2 >= 2 * embed) return;
  const int which = e2 / embed, e = e2 - which * embed;
  const float* w = w_rc + static_cast<size_t>(which) * cin * embed + e;
  float wr[32];
#pragma unroll
  for (int ch = 0; ch < 32; ++ch) wr[ch] = ch < cin ? w[ch * embed] : 0.f;
  for (int r = 0; r < kNodeRows && row0 + r < rows; ++r) {
    float acc = 0.f;
#pragma unroll
    for (int ch = 0; ch < 32; ++ch) acc = fmaf(wr[ch], sv[r][ch], acc);  // same order as the reference's channel cat
    rc[(row0 + r) * 2 * embed + e2] = acc;
  }
}

// Sixteen consecutive pixels (b, i, j) per warp step, on the legacy warp MMA (m16n8k16 bf16 -> fp32):
//   conv1x1:  [16 pixels x 16 planes] . [16 planes x 96 channels], planes = c_e (x2 with self-conditioning), K padded
//             with zeros.  Inputs and weights stay fp32-accurate: both are split into bf16 hi + lo parts and three
//             products are accumulated (hi hi + hi lo + lo hi; the dropped lo lo term is 2^-16 relative).
//   epilogue: on the accumulator fragments (thread (g, t) owns channel pairs 8 nt + 2t, +1 of pixels g and g + 8):
//             + row / column node planes, LayerNorm over the 96 channels (quad shuffles), FiLM, SiLU, 8-byte stores
//             (four lanes write one 32-byte sector).
// The scalar versions of this kernel (one thread per pixel, then eight lanes per pixel) spent ~130 warp instructions
// per pixel on the 1152 FMAs + weight loads of the conv and ran at 1.3 TB/s; this one needs ~35.
// x0 = silu(shift + LN(conv1x1(input)) * (1 + scale))
constexpr int kPE = 96;
__global__ void __launch_bounds__(kRowThreads, 3)
patch_embed_kernel(const float* __restrict__ adj, const float* __restrict__ sc_adj, const float* __restrict__ in_scale,
                   const uint8_t* __restrict__ flags, const float* __restrict__ rc, const float* __restrict__ w_adj,
                   const float* __restrict__ bias, const float* __restrict__ gamma, const float* __restrict__ beta,
                   const float* __restrict__ film, int film_ld, int cond_uniform, float* __restrict__ x0,
                   long long pixels, int n, int c_e, int self_cond, const int* __restrict__ perm, int side) {
  constexpr int E = kPE, NT = E / 8;
  __shared__ uint4 sBf[NT][32];                 // B fragments of n-tile nt for lane: {hi k0-7, hi k8-15, lo k0-7, lo k8-15}
  __shared__ __align__(16) float sBias[E], sGam[E], sBet[E];
  const int planes = self_cond ? 2 * c_e : c_e;
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  auto split2 = [](float a, float b, uint32_t& hi, uint32_t& lo) {
    const __nv_bfloat16 ah = __float2bfloat16_rn(a), bh = __float2bfloat16_rn(b);
    hi = pack_bf16x2(__bfloat162float(ah), __bfloat162float(bh));
    lo = pack_bf16x2(a - __bfloat162float(ah), b - __bfloat162float(bh));
  };
  for (int idx = threadIdx.x; idx < NT * 32; idx += kRowThreads) {
    const int nt = idx >> 5, l = idx & 31, ch = nt * 8 + (l >> 2), k0 = 2 * (l & 3);
    auto w = [&](int k) { return k < planes ? w_adj[k * E + ch] : 0.f; };  // B[k][n] = W[plane k][channel]
    uint4 f;
    split2(w(k0), w(k0 + 1), f.x, f.z);
    split2(w(k0 + 8), w(k0 + 9), f.y, f.w);
    sBf[nt][l] = f;
  }
  for (int i = threadIdx.x; i < E; i += kRowThreads) { sBias[i] = bias[i]; sGam[i] = gamma[i]; sBet[i] = beta[i]; }
  __syncthreads();
  const int nn = n * n;
  const long long groups = (pixels + 15) / 16;
  const long long warps_total = static_cast<long long>(gridDim.x) * (kRowThreads / 32);
  // A-fragment inputs of a step: planes [self-cond adj (c_e), c_in * adj (c_e)] at k = 2t, 2t + 1, 2t + 8, 2t + 9 of
  // fragment rows g and g + 8.  They are the only HBM reads of the kernel and are fetched ONE STEP AHEAD (the warp
  // otherwise sits on this round trip with nothing else to do: 46 % long-scoreboard stalls in the ncu profile).
  // (raw values only: the first USE of a loaded register stalls the in-order warp, so c_in is applied a step later)
  auto load_planes = [&](long long grp, float (&pv)[8], float (&scl)[2]) {
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const long long px = grp * 16 + g + 8 * r;
      const long long pc = px < pixels ? px : pixels - 1;
      int b_ = static_cast<int>(pc / nn);
      int ij_ = static_cast<int>(pc - static_cast<long long>(b_) * nn);
      if (perm != nullptr) {  // compact layout: a stack of side x side corners; image k is sample perm[k] (-1: all padding)
        const int img = static_cast<int>(pc / (side * side));
        const int rem = static_cast<int>(pc - static_cast<long long>(img) * side * side);
        const int i_ = rem / side;
        b_ = perm[img];
        ij_ = i_ * n + (rem - i_ * side);
      }
      scl[r] = (in_scale && b_ >= 0) ? in_scale[b_] : 1.f;
      if (b_ < 0) {
#pragma unroll
        for (int h = 0; h < 4; ++h) pv[r * 4 + h] = 0.f;
        continue;
      }
#pragma unroll
      for (int h = 0; h < 4; ++h) {
        const int k = 2 * t + (h & 1) + 8 * (h >> 1);
        float a = 0.f;
        if (k < planes) {
          if (self_cond && k < c_e) {
            if (sc_adj) a = sc_adj[(static_cast<size_t>(b_) * c_e + k) * nn + ij_];
          } else {
            a = adj[(static_cast<size_t>(b_) * c_e + (self_cond ? k - c_e : k)) * nn + ij_];
          }
        }
        pv[r * 4 + h] = a;
      }
    }
  };
  const long long grp0 = static_cast<long long>(blockIdx.x) * (kRowThreads / 32) + (threadIdx.x >> 5);
  float pv_next[8], sc_next[2];
  if (grp0 < groups) load_planes(grp0, pv_next, sc_next);
  for (long long grp = grp0; grp < groups; grp += warps_total) {
    float pv[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {  // c_in * adj for the adjacency planes (self-conditioning planes are not scaled)
      const int kk = 2 * t + (k & 1) + 8 * ((k >> 1) & 1);
      pv[k] = (self_cond && kk < c_e) ? pv_next[k] : __fmul_rn(sc_next[k >> 2], pv_next[k]);
    }
    if (grp + warps_total < groups) load_planes(grp + warps_total, pv_next, sc_next);
    // the two pixels (fragment rows g and g + 8) of this thread
    long long pix[2];
    int bb[2], ij[2];
    bool valid[2], pair_ok[2];
    const float *rrow[2], *rcol[2], *fs[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      pix[r] = grp * 16 + g + 8 * r;
      valid[r] = pix[r] < pixels;
      const long long pc = valid[r] ? pix[r] : pixels - 1;
      bb[r] = static_cast<int>(pc / nn);
      ij[r] = static_cast<int>(pc - static_cast<long long>(bb[r]) * nn);
      if (perm != nullptr) {
        const int img = static_cast<int>(pc / (side * side));
        const int rem = static_cast<int>(pc - static_cast<long long>(img) * side * side);
        const int ii = rem / side;
        bb[r] = perm[img];
        ij[r] = ii * n + (rem - ii * side);
      }
      const int i_ = ij[r] / n, j_ = ij[r] - i_ * n;
      const int bs = bb[r] < 0 ? 0 : bb[r];
      pair_ok[r] = bb[r] >= 0 && flags[bs * n + i_] != 0 && flags[bs * n + j_] != 0;
      rrow[r] = rc + (static_cast<size_t>(bs) * n + i_) * 2 * E;
      rcol[r] = rc + (static_cast<size_t>(bs) * n + j_) * 2 * E + E;
      fs[r] = film + static_cast<size_t>(cond_uniform ? 0 : bs) * film_ld;  // scale[E] then shift[E]
    }
    uint32_t a_hi[4], a_lo[4];   // A fragment registers: (row g, k lo) (row g + 8, k lo) (row g, k hi) (row g + 8, k hi)
    split2(pv[0], pv[1], a_hi[0], a_lo[0]);
    split2(pv[4], pv[5], a_hi[1], a_lo[1]);
    split2(pv[2], pv[3], a_hi[2], a_lo[2]);
    split2(pv[6], pv[7], a_hi[3], a_lo[3]);
    float acc[NT][4];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const float2 bv = *reinterpret_cast<const float2*>(&sBias[nt * 8 + 2 * t]);
      acc[nt][0] = bv.x; acc[nt][1] = bv.y; acc[nt][2] = bv.x; acc[nt][3] = bv.y;
      const uint4 f = sBf[nt][lane];
      const uint32_t b_hi[2] = {f.x, f.y}, b_lo[2] = {f.z, f.w};
      mma_m16n8k16_bf16(acc[nt], a_lo, b_hi);
      mma_m16n8k16_bf16(acc[nt], a_hi, b_lo);
      mma_m16n8k16_bf16(acc[nt], a_hi, b_hi);
    }
    // ---- epilogue on packed fp32 pairs: pr[nt][r] = channels (8 nt + 2t, + 1) of fragment row r
    f32x2 pr[NT][2];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      pr[nt][0] = f2_pack(acc[nt][0], acc[nt][1]);
      pr[nt][1] = f2_pack(acc[nt][2], acc[nt][3]);
    }
    // node planes (zeroed on padded rows / columns, mask_adjs at :800) and the LayerNorm statistics
    float mean[2], rstd[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      if (pair_ok[r]) {
        const float2* p1 = reinterpret_cast<const float2*>(rrow[r] + 2 * t);
        const float2* p2 = reinterpret_cast<const float2*>(rcol[r] + 2 * t);
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
          const float2 r1 = __ldg(p1 + 4 * nt), r2 = __ldg(p2 + 4 * nt);
          pr[nt][r] = f2_add(pr[nt][r], f2_add(f2_pack(r1.x, r1.y), f2_pack(r2.x, r2.y)));
        }
      }
      f32x2 s2 = pr[0][r];
#pragma unroll
      for (int nt = 1; nt < NT; ++nt) s2 = f2_add(s2, pr[nt][r]);
      float sa, sb;
      f2_unpack(s2, sa, sb);
      float sm = sa + sb;
      sm += __shfl_xor_sync(0xffffffffu, sm, 1);
      sm += __shfl_xor_sync(0xffffffffu, sm, 2);
      mean[r] = sm * (1.0f / E);
      const f32x2 nm = f2_splat(-mean[r]);
      f32x2 q2 = f2_splat(0.f);
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        pr[nt][r] = f2_add(pr[nt][r], nm);
        q2 = f2_fma(pr[nt][r], pr[nt][r], q2);
      }
      f2_unpack(q2, sa, sb);
      float qq = sa + sb;
      qq += __shfl_xor_sync(0xffffffffu, qq, 1);
      qq += __shfl_xor_sync(0xffffffffu, qq, 2);
      rstd[r] = rsqrtf(qq * (1.0f / E) + kLnEps);
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const f32x2 rs = f2_splat(rstd[r]);
      const float2* psc = reinterpret_cast<const float2*>(fs[r] + 2 * t);
      const float2* psh = reinterpret_cast<const float2*>(fs[r] + E + 2 * t);
      float2* orow = reinterpret_cast<float2*>(x0 + pix[r] * E + 2 * t);
      if (valid[r]) {
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
          const float2 gg = *reinterpret_cast<const float2*>(&sGam[nt * 8 + 2 * t]);
          const float2 be = *reinterpret_cast<const float2*>(&sBet[nt * 8 + 2 * t]);
          const float2 fsc = __ldg(psc + 4 * nt), fsh = __ldg(psh + 4 * nt);
          // silu(LN(v) (1 + scale) + shift),  silu(x) = x / (1 + 2^(-x log2 e))
          const f32x2 y = f2_fma(f2_mul(pr[nt][r], rs), f2_pack(gg.x, gg.y), f2_pack(be.x, be.y));
          const f32x2 z = f2_fma(y, f2_add(f2_pack(fsc.x, fsc.y), f2_splat(1.f)), f2_pack(fsh.x, fsh.y));
          float z0, z1, u0, u1;
          f2_unpack(z, z0, z1);
          f2_unpack(f2_mul(z, f2_splat(-1.4426950408889634f)), u0, u1);
          const f32x2 den = f2_add(f2_pack(ex2_approx(u0), ex2_approx(u1)), f2_splat(1.f));
          float d0, d1;
          f2_unpack(den, d0, d1);
          orow[4 * nt] = make_float2(z0 * rcp_approx(d0), z1 * rcp_approx(d1));
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// node read-out: masked row mean -> MLP -> mask (-> EDM output preconditioning)   (:812-822, precond.py:103-105)
// ---------------------------------------------------------------------------------------------------------
// One CTA (256 threads) per kHeadRows consecutive rows (b, i): the three weight matrices (77 KB from L2) are read
// once per CTA instead of once per row, and the phases of the eight rows overlap each other's latencies.  y is LN(x)
// of the last stage [B n n, E] (bf16); the folded read_out map (fold_t [E][E] input-major, fold_b) is applied after
// pooling: mean_j m_ij (F y_ij + f) = F mean_j(m_ij y_ij) + f cnt/n.
constexpr int kHeadRows = 8;
__global__ void __launch_bounds__(256)
node_head_kernel(const bf16* __restrict__ rep, const uint8_t* __restrict__ flags, const float* __restrict__ fold_t,
                 const float* __restrict__ fold_b, const float* __restrict__ w1t,
                 const float* __restrict__ b1, const float* __restrict__ w2t, const float* __restrict__ b2,
                 const float* __restrict__ x_node, const float* __restrict__ c_skip, const float* __restrict__ c_out,
                 float* __restrict__ out_node, long long rows, int n, int c_n, int embed, const int* __restrict__ tok0,
                 const int* __restrict__ width) {
  __shared__ float va[kHeadRows][128];  // masked row means, then the hidden layer
  __shared__ float vb[kHeadRows][128];  // pooled read-out
  __shared__ float frac[kHeadRows];     // valid columns / n
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row0 = static_cast<long long>(blockIdx.x) * kHeadRows;
  // ---- masked mean over j of row (b, i) = row0 + warp: lanes 0 .. embed / 4 - 1 own four channels each
  {
    const long long bi = row0 + warp;
    const bool live = bi < rows && flags[bi] != 0;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    int cnt = 0;
    if (live) {
      const int b = static_cast<int>(bi / n);
      const uint8_t* fj = flags + static_cast<size_t>(b) * n;
      // compact layout: sample b is a width[b]^2 corner starting at token tok0[b]; valid nodes always lie inside it
      const int nj = tok0 != nullptr ? width[b] : n;
      const size_t row_tok = tok0 != nullptr ? static_cast<size_t>(tok0[b]) + static_cast<size_t>(bi - static_cast<long long>(b) * n) * nj
                                             : static_cast<size_t>(bi) * n;
      const bf16* p = rep + row_tok * embed + 4 * lane;
      const bool mine = 4 * lane < embed;
      // unconditional, unrolled loads (masked columns are multiplied by zero): eight 8-byte loads in flight per lane
#pragma unroll 8
      for (int j = 0; j < nj; ++j) {
        const float m = fj[j] != 0 ? 1.f : 0.f;
        cnt += fj[j] != 0;
        if (mine) {
          const uint2 v = *reinterpret_cast<const uint2*>(p + static_cast<size_t>(j) * embed);
          const __nv_bfloat162 lo = *reinterpret_cast<const __nv_bfloat162*>(&v.x);
          const __nv_bfloat162 hi = *reinterpret_cast<const __nv_bfloat162*>(&v.y);
          s.x = fmaf(m, __low2float(lo), s.x); s.y = fmaf(m, __high2float(lo), s.y);
          s.z = fmaf(m, __low2float(hi), s.z); s.w = fmaf(m, __high2float(hi), s.w);
        }
      }
    }
    if (4 * lane < embed) {  // mean over the full row length N, not over the valid count (:813)
      va[warp][4 * lane] = s.x / n; va[warp][4 * lane + 1] = s.y / n;
      va[warp][4 * lane + 2] = s.z / n; va[warp][4 * lane + 3] = s.w / n;
    }
    if (lane == 0) frac[warp] = static_cast<float>(cnt) / n;
  }
  __syncthreads();
  // ---- three small matrix products, thread (e, rh): output column e of rows 4 rh .. 4 rh + 3
  const int e = threadIdx.x % 128, rh = threadIdx.x / 128;
  if (e < embed) {
    float acc[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) acc[r] = fold_b[e] * frac[4 * rh + r];
#pragma unroll 16
    for (int k = 0; k < embed; ++k) {  // sixteen independent L2 loads in flight
      const float w = fold_t[k * embed + e];
#pragma unroll
      for (int r = 0; r < 4; ++r) acc[r] = fmaf(w, va[4 * rh + r][k], acc[r]);
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) vb[4 * rh + r][e] = acc[r];
  }
  __syncthreads();
  if (e < embed) {
    float acc[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) acc[r] = b1[e];
#pragma unroll 16
    for (int k = 0; k < embed; ++k) {
      const float w = w1t[k * embed + e];
#pragma unroll
      for (int r = 0; r < 4; ++r) acc[r] = fmaf(w, vb[4 * rh + r][k], acc[r]);
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) va[4 * rh + r][e] = gelu_erf(acc[r]);
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < kHeadRows * c_n; idx += blockDim.x) {
    const int r = idx / c_n, c = idx - r * c_n;
    const long long bi = row0 + r;
    if (bi >= rows) continue;
    const size_t o = static_cast<size_t>(bi) * c_n + c;
    if (flags[bi] == 0) {  // masked node: output row is zero regardless of the features
      out_node[o] = 0.f;
      continue;
    }
    float sum = b2[c];
#pragma unroll 16
    for (int k = 0; k < embed; ++k) sum = fmaf(w2t[k * c_n + c], va[r][k], sum);
    const int b = static_cast<int>(bi / n);
    if (x_node != nullptr) sum = __fadd_rn(__fmul_rn(c_skip[b], x_node[o]), __fmul_rn(c_out[b], sum));
    out_node[o] = sum;
  }
}

// ---------------------------------------------------------------------------------------------------------
// node read-out in two kernels (embed = 96): (1) masked row sums, one warp per row (b, i), 16-byte loads, masked
// columns never loaded; (2) the three small matrix products for 32 rows per CTA with the weights staged in shared
// memory once per CTA (the single-kernel version above read 77 KB of weights from L2 per 8 rows and ran at 1.1 TB/s).
// pooled [B n, 128]: columns 0..95 = mean over j of the masked features (divided by n, :813), column 96 = valid / n.
// ---------------------------------------------------------------------------------------------------------
constexpr int kPoolPitch = 128;
__global__ void __launch_bounds__(256)
node_pool_kernel(const bf16* __restrict__ rep, const uint8_t* __restrict__ flags, float* __restrict__ pooled, long long rows,
                 int n, const int* __restrict__ tok0, const int* __restrict__ width) {
  constexpr int E = 96;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long bi = static_cast<long long>(blockIdx.x) * 8 + warp;
  if (bi >= rows) return;
  float* out = pooled + bi * kPoolPitch;
  if (flags[bi] == 0) {   // masked node: its output row is zero whatever the features are
    for (int c = lane; c <= E; c += 32) out[c] = 0.f;
    return;
  }
  const int b = static_cast<int>(bi / n);
  const uint8_t* fj = flags + static_cast<size_t>(b) * n;
  const int nj = tok0 != nullptr ? width[b] : n;
  const size_t row_tok = tok0 != nullptr ? static_cast<size_t>(tok0[b]) + static_cast<size_t>(bi - static_cast<long long>(b) * n) * nj
                                         : static_cast<size_t>(bi) * n;
  const int tsub = lane / 12, c8 = lane - 12 * tsub;   // lanes 0..23: token parity, 8-channel chunk
  // the row's column mask as two 32-bit words (n <= 64): the data loads below depend on registers only, not on a flag
  // load per token, so the compiler keeps eight of them in flight
  const unsigned m_lo = __ballot_sync(0xffffffffu, lane < nj && fj[lane] != 0);
  const unsigned m_hi = __ballot_sync(0xffffffffu, lane + 32 < nj && fj[lane + 32] != 0);
  const unsigned long long mask = (static_cast<unsigned long long>(m_hi) << 32) | m_lo;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (lane < 24) {
    const bf16* p = rep + row_tok * E + 8 * c8;
#pragma unroll 8
    for (int j = tsub; j < nj; j += 2) {
      if (((mask >> j) & 1ull) == 0) continue;
      const uint4 v = *reinterpret_cast<const uint4*>(p + static_cast<size_t>(j) * E);
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
      for (int k = 0; k < 4; ++k) { acc[2 * k] += __low2float(h[k]); acc[2 * k + 1] += __high2float(h[k]); }
    }
  }
  const int cnt = __popcll(mask);
#pragma unroll
  for (int k = 0; k < 8; ++k) acc[k] += __shfl_down_sync(0xffffffffu, acc[k], 12);
  if (lane < 12) {
    const float inv = 1.0f / n;
#pragma unroll
    for (int k = 0; k < 8; ++k) out[8 * c8 + k] = acc[k] * inv;
  }
  if (lane == 0) out[E] = static_cast<float>(cnt) / n;
}

constexpr int kMlpRows = 32;
// activations are kept k-major in shared memory (vT[k][row]): for one k the 16 rows of a thread are four broadcast
// 16-byte loads, so a k step costs 5 shared-memory loads per 16 FMAs (row-major: 17)
__global__ void __launch_bounds__(192)
node_mlp_kernel(const float* __restrict__ pooled, const uint8_t* __restrict__ flags, const float* __restrict__ fold_t,
                const float* __restrict__ fold_b, const float* __restrict__ w1t, const float* __restrict__ b1,
                const float* __restrict__ w2t, const float* __restrict__ b2, const float* __restrict__ x_node,
                const float* __restrict__ c_skip, const float* __restrict__ c_out, float* __restrict__ out_node, long long rows,
                int n, int c_n) {
  constexpr int E = 96, R = kMlpRows, RH = R / 2;
  extern __shared__ __align__(16) float sm[];
  float* sW2 = sm;                    // [E][c_n]; the two E x E matrices are read through L1 (one coalesced load per 16 FMAs)
  float* vaT = sW2 + E * 32;          // [E + 1][R]: pooled features (row E: valid fraction), later the hidden layer
  float* vbT = vaT + (E + 1) * R;     // [E][R]
  __shared__ int any_live;
  const long long row0 = static_cast<long long>(blockIdx.x) * R;
  if (threadIdx.x == 0) any_live = 0;
  __syncthreads();
  if (threadIdx.x < R && row0 + threadIdx.x < rows && flags[row0 + threadIdx.x] != 0) any_live = 1;
  __syncthreads();
  if (!any_live) {   // a block of masked nodes: zeros, no weights needed
    for (int idx = threadIdx.x; idx < R * c_n; idx += blockDim.x) {
      const long long bi = row0 + idx / c_n;
      if (bi < rows) out_node[bi * c_n + idx % c_n] = 0.f;
    }
    return;
  }
  {
    // pooled features: thread = (row, 16-float segment), six segments per row + the valid fraction
    const int pr = threadIdx.x / 6, ps = threadIdx.x - 6 * pr;
    float4 pv[4];
    const bool prow = row0 + pr < rows;
#pragma unroll
    for (int q = 0; q < 4; ++q)
      pv[q] = prow ? *reinterpret_cast<const float4*>(pooled + (row0 + pr) * kPoolPitch + 16 * ps + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      vaT[(16 * ps + 4 * q) * R + pr] = pv[q].x; vaT[(16 * ps + 4 * q + 1) * R + pr] = pv[q].y;
      vaT[(16 * ps + 4 * q + 2) * R + pr] = pv[q].z; vaT[(16 * ps + 4 * q + 3) * R + pr] = pv[q].w;
    }
    if (threadIdx.x < R) vaT[E * R + threadIdx.x] = row0 + threadIdx.x < rows ? pooled[(row0 + threadIdx.x) * kPoolPitch + E] : 0.f;
  }
  for (int i = threadIdx.x; i < E * c_n; i += blockDim.x) sW2[i] = w2t[i];
  __syncthreads();
  const int e = threadIdx.x % E, rg = threadIdx.x / E;   // output column, half of the rows
  auto matvec = [&](const float* W, const float* vT, float (&acc)[RH]) {
#pragma unroll 8
    for (int k = 0; k < E; ++k) {
      const float w = __ldg(W + k * E + e);
      const float4* v4 = reinterpret_cast<const float4*>(vT + k * R + rg * RH);
#pragma unroll
      for (int q = 0; q < RH / 4; ++q) {
        const float4 v = v4[q];
        acc[4 * q] = fmaf(w, v.x, acc[4 * q]);
        acc[4 * q + 1] = fmaf(w, v.y, acc[4 * q + 1]);
        acc[4 * q + 2] = fmaf(w, v.z, acc[4 * q + 2]);
        acc[4 * q + 3] = fmaf(w, v.w, acc[4 * q + 3]);
      }
    }
  };
  {
    float acc[RH];
    const float fb = fold_b[e];
#pragma unroll
    for (int r = 0; r < RH; ++r) acc[r] = fb * vaT[E * R + rg * RH + r];
    matvec(fold_t, vaT, acc);
#pragma unroll
    for (int r = 0; r < RH; ++r) vbT[e * R + rg * RH + r] = acc[r];
  }
  __syncthreads();
  {
    float acc[RH];
    const float bb = b1[e];
#pragma unroll
    for (int r = 0; r < RH; ++r) acc[r] = bb;
    matvec(w1t, vbT, acc);
#pragma unroll
    for (int r = 0; r < RH; ++r) vaT[e * R + rg * RH + r] = gelu_erf(acc[r]);   // vaT's features were consumed before the barrier above
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < R * c_n; idx += blockDim.x) {
    const int r = idx / c_n, c = idx - r * c_n;
    const long long bi = row0 + r;
    if (bi >= rows) continue;
    const size_t o = static_cast<size_t>(bi) * c_n + c;
    if (flags[bi] == 0) { out_node[o] = 0.f; continue; }
    float sum = b2[c];
#pragma unroll 16
    for (int k = 0; k < E; ++k) sum = fmaf(sW2[k * c_n + c], vaT[k * R + r], sum);
    const int b = static_cast<int>(bi / n);
    if (x_node != nullptr) sum = __fadd_rn(__fmul_rn(c_skip[b], x_node[o]), __fmul_rn(c_out[b], sum));
    out_node[o] = sum;
  }
}

inline unsigned row_grid(long long rows, int lpr = 32) {
  const int per_cta = kRowThreads / lpr;
  return static_cast<unsigned>((rows + per_cta - 1) / per_cta);
}

}  // namespace

// (float4 per lane, lanes per row): 96 -> (3, 8), 192 -> (3, 16), 384 -> (3, 32), 768 -> (6, 32)
#define DSG_DISPATCH_ROW(C, CALL)                                                         \
  switch (C) {                                                                            \
    case 96: { constexpr int NV = 3, LPR = 8; CALL; break; }                              \
    case 192: { constexpr int NV = 3, LPR = 16; CALL; break; }                            \
    case 384: { constexpr int NV = 3, LPR = 32; CALL; break; }                            \
    case 768: { constexpr int NV = 6, LPR = 32; CALL; break; }                            \
    default:                                                                              \
      set_last_error("row kernel: unsupported width %d (96/192/384/768)", C);             \
      return DSG_ERR_INVALID;                                                             \
  }

int launch_film_ln(const float* x_in, float* x_out, bf16* y, const float* film, int film_ld, int film_off,
                   int cond_uniform, const float* gamma, const float* beta, int batch, int tokens_per_sample, int C,
                   cudaStream_t st, const int* src_rows) {
  const long long rows = static_cast<long long>(batch) * tokens_per_sample;
  DSG_REQUIRE(src_rows == nullptr || x_in != x_out, "film_ln: a gathering launch cannot run in place");
  DSG_DISPATCH_ROW(C, (film_ln_kernel<NV, LPR><<<row_grid(rows, LPR), kRowThreads, 0, st>>>(
                          x_in, x_out, y, film + film_off, film_ld, cond_uniform, gamma, beta, rows, tokens_per_sample, C,
                          src_rows)));
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_ln(const float* x, bf16* y, const float* gamma, const float* beta, int64_t rows, int C, cudaStream_t st) {
  DSG_DISPATCH_ROW(C, (ln_kernel<NV, LPR><<<row_grid(rows, LPR), kRowThreads, 0, st>>>(x, y, gamma, beta, rows, C)));
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_merge_ln(const float* x, bf16* y, const float* gamma, const float* beta, int batch, int res, int C,
                    cudaStream_t st) {
  DSG_REQUIRE(res % 2 == 0, "merge: odd resolution %d", res);
  const long long rows = static_cast<long long>(batch) * (res / 2) * (res / 2);
  const unsigned grid = row_grid(rows);
  if (C == 96) merge_ln_q_kernel<3><<<grid, kRowThreads, 0, st>>>(x, y, gamma, beta, rows, res);
  else if (C == 192) merge_ln_q_kernel<6><<<grid, kRowThreads, 0, st>>>(x, y, gamma, beta, rows, res);
  else if (C == 384) merge_ln_q_kernel<12><<<grid, kRowThreads, 0, st>>>(x, y, gamma, beta, rows, res);
  else { set_last_error("merge: unsupported width %d (96/192/384)", C); return DSG_ERR_INVALID; }
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_concat_bf16(const float* x, const float* skip, bf16* y, int64_t rows, int C, cudaStream_t st, const int* skip_rows) {
  DSG_REQUIRE(C % 4 == 0, "concat: width %d", C);
  const long long total = rows * 2 * (C / 4);
  const unsigned grid = static_cast<unsigned>(total / 256 + 1 < 148LL * 16 ? total / 256 + 1 : 148LL * 16);
  concat_bf16_kernel<<<grid, 256, 0, st>>>(x, skip, y, rows, C, skip_rows);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_breakup_ln(const float* t, bf16* y, const float* g1, const float* b1, const float* g2, const float* b2,
                      int batch, int res, int D, cudaStream_t st, const int* tok0, const int* width, int sh,
                      const int* src_perm) {
  DSG_REQUIRE((tok0 == nullptr) == (width == nullptr), "breakup: tok0 / width must both be given or both NULL");
  const long long rows = static_cast<long long>(batch) * res * res;
  const unsigned grid = row_grid(rows);
  if (D == 384) breakup_ln_q_kernel<3><<<grid, kRowThreads, 0, st>>>(t, y, g1, b1, g2, b2, rows, res, tok0, width, sh, src_perm);
  else if (D == 768) breakup_ln_q_kernel<6><<<grid, kRowThreads, 0, st>>>(t, y, g1, b1, g2, b2, rows, res, tok0, width, sh, src_perm);
  else if (D == 1536) breakup_ln_q_kernel<12><<<grid, kRowThreads, 0, st>>>(t, y, g1, b1, g2, b2, rows, res, tok0, width, sh, src_perm);
  else { set_last_error("breakup: unsupported width %d (384/768/1536)", D); return DSG_ERR_INVALID; }
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_cond(const float* noise_labels, long long label_stride, int n_cond, const float* w0, const float* b0, const float* w1,
                const float* b1, const float* w_film, const float* b_film, int film_total, float* emb0, float* emb1,
                float* emb, float* film, int embed, cudaStream_t st) {
  const int half = embed / 2;
  sinusoid_kernel<<<(n_cond * half + 127) / 128, 128, 0, st>>>(noise_labels, label_stride, emb0, n_cond, embed);
  DSG_LAUNCH_CHECK();
  auto lin = [&](const float* x, const float* W, const float* b, float* y, int K, int O, int act) {
    const long long warps = static_cast<long long>(n_cond) * O;
    small_linear_kernel<<<static_cast<unsigned>((warps + 7) / 8), 256, 0, st>>>(x, W, b, y, n_cond, K, O, act);
  };
  lin(emb0, w0, b0, emb1, embed, 512, 1);
  DSG_LAUNCH_CHECK();
  lin(emb1, w1, b1, emb, 512, 512, 1);
  DSG_LAUNCH_CHECK();
  lin(emb, w_film, b_film, film, 512, film_total, 0);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_precond_coef(const float* sigmas, int sigma_stride, float* coef, int n, cudaStream_t st) {
  precond_coef_kernel<<<(n + 127) / 128, 128, 0, st>>>(sigmas, sigma_stride, coef, n);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_node_proj(const float* node, const float* sc_node, const float* in_scale, const float* w_rc, float* rc,
                     int batch, int n, int c_n, int self_cond, int embed, cudaStream_t st) {
  DSG_REQUIRE(2 * embed <= 1024 && (self_cond ? 2 : 1) * c_n <= 32, "node_proj: embed %d, c_n %d", embed, c_n);
  const long long rows = static_cast<long long>(batch) * n;
  node_proj_kernel<<<static_cast<unsigned>((rows + kNodeRows - 1) / kNodeRows), 2 * embed, 0, st>>>(
      node, sc_node, in_scale, w_rc, rc, batch, n, c_n, self_cond, embed);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_patch_embed(const float* adj, const float* sc_adj, const float* in_scale, const uint8_t* flags,
                       const float* rc, const float* w_adj, const float* bias, const float* gamma, const float* beta,
                       const float* film, int film_ld, int film_off, int cond_uniform, float* x0, int batch, int n,
                       int c_e, int self_cond, int embed, cudaStream_t st, const int* perm, int side) {
  DSG_REQUIRE(embed == 96, "patch_embed: embed_dim %d (only 96 is built)", embed);
  // perm: `batch` counts the images of a compact stack of side x side corners (see patch_embed_kernel)
  const long long pixels = perm != nullptr ? static_cast<long long>(batch) * side * side : static_cast<long long>(batch) * n * n;
  DSG_REQUIRE((self_cond ? 2 : 1) * c_e <= 16, "patch_embed: %d adjacency planes (max 16)", (self_cond ? 2 : 1) * c_e);
  long long blocks = (pixels / 16 + 7) / 8;  // one warp per 16 pixels per step
  if (blocks > 148 * 3) blocks = 148 * 3;  // persistent: three resident CTAs per SM, the weight-fragment prologue is paid once each
  patch_embed_kernel<<<static_cast<unsigned>(blocks), kRowThreads, 0, st>>>(adj, sc_adj, in_scale, flags, rc, w_adj,
                                                                           bias, gamma, beta, film + film_off, film_ld,
                                                                           cond_uniform, x0, pixels, n, c_e, self_cond,
                                                                           perm, side);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int launch_node_head(const bf16* rep, const uint8_t* flags, const float* fold_t, const float* fold_b, const float* w1t,
                     const float* b1, const float* w2t, const float* b2, const float* x_node, const float* c_skip,
                     const float* c_out, float* out_node, int batch, int n, int c_n, int embed, cudaStream_t st,
                     const int* tok0, const int* width, float* scratch) {
  DSG_REQUIRE(embed <= 128 && embed % 4 == 0 && c_n <= 128, "node_head: embed %d c_n %d", embed, c_n);
  const long long rows = static_cast<long long>(batch) * n;
  if (embed == 96 && c_n <= 32 && n <= 64 && scratch != nullptr) {
    // two kernels: masked row sums, then the MLP for 32 rows per CTA with the weights in shared memory
    node_pool_kernel<<<static_cast<unsigned>((rows + 7) / 8), 256, 0, st>>>(rep, flags, scratch, rows, n, tok0, width);
    DSG_LAUNCH_CHECK();
    constexpr int smem = (96 * 32 + (2 * 96 + 1) * kMlpRows) * 4;
    static PerDeviceOnce configured;
    if (configured.first())
      DSG_CUDA_CHECK(cudaFuncSetAttribute(node_mlp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    node_mlp_kernel<<<static_cast<unsigned>((rows + kMlpRows - 1) / kMlpRows), 192, smem, st>>>(
        scratch, flags, fold_t, fold_b, w1t, b1, w2t, b2, x_node, c_skip, c_out, out_node, rows, n, c_n);
    DSG_LAUNCH_CHECK();
    return DSG_OK;
  }
  node_head_kernel<<<static_cast<unsigned>((rows + kHeadRows - 1) / kHeadRows), 256, 0, st>>>(
      rep, flags, fold_t, fold_b, w1t, b1, w2t, b2, x_node, c_skip, c_out, out_node, rows, n, c_n, embed, tok0, width);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

}  // namespace dsg
