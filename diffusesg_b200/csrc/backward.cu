// Training step of the denoiser (SURVEY 8 f-2): the row-wise forward kernels that keep what the backward pass needs,
// and every backward kernel that is not a GEMM.  The GEMMs of the backward pass (dgrad: dX = dY . W, wgrad:
// dW = dY^T . X contracted over the tokens with split-K) run on gemm_kernel (gemm.cu) - the wgrad operands are read
// MN-major straight from the row-major dY and X.
//
// Reference: loss.backward() of runner/trainer/trainer_node_adj.py:171-178 through model/diffusesg/diffusesg.py
// (LayerNorm :243/:275, FiLM + SiLU :238-240/:574-576, nn.GELU :15, PatchMerging :314-335, PatchBreakup :374-403,
// WindowAttention :108-139, the read-out heads :806-825) and model/precond/precond.py:100-105.
//
// All kernels are HBM-bound row kernels (one warp per token row, 16-byte accesses) except the window-attention backward
// (window_attention_bwd_tc_kernel: warp-level tensor cores, five T x T x 32 products per window-head from shared memory)
// and the small strided fp32 GEMM for the batch-sized layers.
#include <math.h>
#include <mma.h>

#include "common.cuh"
#include "kernels.h"

namespace dsg {
namespace {

typedef __nv_bfloat16 bf16_t;

DSG_DEVICE float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
DSG_DEVICE void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
DSG_DEVICE void st4_bf16(bf16_t* p, float4 v) {
  uint2 w;
  w.x = pack_bf16x2(v.x, v.y);
  w.y = pack_bf16x2(v.z, v.w);
  *reinterpret_cast<uint2*>(p) = w;
}
DSG_DEVICE float4 ld4_bf16(const bf16_t* p) {
  const uint2 w = *reinterpret_cast<const uint2*>(p);
  const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&w.x);
  const __nv_bfloat162 b = *reinterpret_cast<const __nv_bfloat162*>(&w.y);
  return make_float4(__low2float(a), __high2float(a), __low2float(b), __high2float(b));
}
DSG_DEVICE void unpack8(const uint4& w, float (&f)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&w);
#pragma unroll
  for (int j = 0; j < 4; ++j) { f[2 * j] = __low2float(h[j]); f[2 * j + 1] = __high2float(h[j]); }
}
DSG_DEVICE uint4 pack8(const float (&f)[8]) {
  uint4 w;
  w.x = pack_bf16x2(f[0], f[1]); w.y = pack_bf16x2(f[2], f[3]); w.z = pack_bf16x2(f[4], f[5]); w.w = pack_bf16x2(f[6], f[7]);
  return w;
}
DSG_DEVICE float sigmoid_f(float x) { return 1.0f / (1.0f + __expf(-x)); }

constexpr float kLnEps = 1e-5f;  // nn.LayerNorm default

// ---------------------------------------------------------------------------------------------------------
// LayerNorm forward (training form): y = (x - mean) * rstd * gamma + beta, one warp per row held in registers, mean and
// centred variance as two exact reductions.  Writes bf16 (GEMM operand) and / or fp32.
// ---------------------------------------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(256)
ln_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
              bf16_t* __restrict__ y16, float* __restrict__ y32, long long M, int C) {
  // a lane owns the float4 groups lane + 32 k (k < NV) of every row: the row is read once and stays in registers
  const int lane = threadIdx.x & 31;
  const long long warps = static_cast<long long>(gridDim.x) * 8;
  const int nv = C >> 2;
  const float invC = 1.0f / C;
  for (long long row = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5); row < M; row += warps) {
    const float* xr = x + row * C;
    float4 a[NV];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int v = lane + 32 * k;
      a[k] = v < nv ? ld4(xr + 4 * v) : make_float4(0.f, 0.f, 0.f, 0.f);
      s += (a[k].x + a[k].y) + (a[k].z + a[k].w);
    }
    const float mean = warp_sum(s) * invC;
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      if (lane + 32 * k < nv) {
        a[k].x -= mean; a[k].y -= mean; a[k].z -= mean; a[k].w -= mean;
        q += (a[k].x * a[k].x + a[k].y * a[k].y) + (a[k].z * a[k].z + a[k].w * a[k].w);
      }
    }
    const float rstd = rsqrtf(warp_sum(q) * invC + kLnEps);
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int v = lane + 32 * k;
      if (v < nv) {
        const float4 g = ld4(gamma + 4 * v), b = ld4(beta + 4 * v);
        const float4 o = make_float4(a[k].x * rstd * g.x + b.x, a[k].y * rstd * g.y + b.y, a[k].z * rstd * g.z + b.z,
                                     a[k].w * rstd * g.w + b.w);
        if (y16 != nullptr) st4_bf16(y16 + row * C + 4 * v, o);
        if (y32 != nullptr) st4(y32 + row * C + 4 * v, o);
      }
    }
  }
}

// LayerNorm backward: dx = rstd (g - mean(g) - xhat mean(g xhat)) with g = dy gamma, statistics recomputed from x;
// dx (+= dx_add when given: the gradient arriving over the residual connection).  dgamma / dbeta: a lane owns the same
// NV float4 column groups in every row, so the parameter gradients accumulate in registers over the rows of the warp and
// are combined once per CTA (shared memory, then one atomicAdd per channel per CTA).  The row is held in registers.
template <int NV>
__global__ void __launch_bounds__(256)
ln_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ gamma,
              const float* dx_add, float* dx, float* __restrict__ dgamma, float* __restrict__ dbeta, long long M, int C) {
  extern __shared__ float sacc[];  // [2][C]
  for (int i = threadIdx.x; i < 2 * C; i += 256) sacc[i] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long warps = static_cast<long long>(gridDim.x) * 8;
  const int nv = C >> 2;
  constexpr bool kGammaInRegs = NV <= 3;   // wide rows re-read gamma (L1) instead of holding it: register budget
  float4 gm[kGammaInRegs ? NV : 1], ag[NV], ab[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int v = lane + 32 * k;
    if (kGammaInRegs) gm[k] = v < nv ? ld4(gamma + 4 * v) : make_float4(0.f, 0.f, 0.f, 0.f);
    ag[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    ab[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const float invC = 1.0f / C;
  for (long long row = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5); row < M; row += warps) {
    const float* xr = x + row * C;
    const float* dr = dy + row * C;
    float4 a[NV], d[NV];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int v = lane + 32 * k;
      a[k] = v < nv ? ld4(xr + 4 * v) : make_float4(0.f, 0.f, 0.f, 0.f);
      d[k] = v < nv ? ld4(dr + 4 * v) : make_float4(0.f, 0.f, 0.f, 0.f);
      s += (a[k].x + a[k].y) + (a[k].z + a[k].w);
    }
    const float mean = warp_sum(s) * invC;
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      if (lane + 32 * k < nv) {
        a[k].x -= mean; a[k].y -= mean; a[k].z -= mean; a[k].w -= mean;
        q += (a[k].x * a[k].x + a[k].y * a[k].y) + (a[k].z * a[k].z + a[k].w * a[k].w);
      }
    }
    const float rstd = rsqrtf(warp_sum(q) * invC + kLnEps);
    float m1 = 0.f, m2 = 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      a[k].x *= rstd; a[k].y *= rstd; a[k].z *= rstd; a[k].w *= rstd;      // xhat (zero in the unused groups)
      ag[k].x += d[k].x * a[k].x; ag[k].y += d[k].y * a[k].y; ag[k].z += d[k].z * a[k].z; ag[k].w += d[k].w * a[k].w;
      ab[k].x += d[k].x; ab[k].y += d[k].y; ab[k].z += d[k].z; ab[k].w += d[k].w;
      const float4 gk = kGammaInRegs ? gm[kGammaInRegs ? k : 0]
                                     : (lane + 32 * k < nv ? ld4(gamma + 4 * (lane + 32 * k)) : make_float4(0.f, 0.f, 0.f, 0.f));
      d[k].x *= gk.x; d[k].y *= gk.y; d[k].z *= gk.z; d[k].w *= gk.w;   // g = dy gamma
      m1 += (d[k].x + d[k].y) + (d[k].z + d[k].w);
      m2 += (d[k].x * a[k].x + d[k].y * a[k].y) + (d[k].z * a[k].z + d[k].w * a[k].w);
    }
    m1 = warp_sum(m1) * invC;
    m2 = warp_sum(m2) * invC;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int v = lane + 32 * k;
      if (v < nv) {
        float4 o = make_float4(rstd * (d[k].x - m1 - a[k].x * m2), rstd * (d[k].y - m1 - a[k].y * m2),
                               rstd * (d[k].z - m1 - a[k].z * m2), rstd * (d[k].w - m1 - a[k].w * m2));
        if (dx_add != nullptr) {
          const float4 e = ld4(dx_add + row * C + 4 * v);
          o.x += e.x; o.y += e.y; o.z += e.z; o.w += e.w;
        }
        st4(dx + row * C + 4 * v, o);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int v = lane + 32 * k;
    if (v < nv) {
      atomicAdd(&sacc[4 * v], ag[k].x); atomicAdd(&sacc[4 * v + 1], ag[k].y);
      atomicAdd(&sacc[4 * v + 2], ag[k].z); atomicAdd(&sacc[4 * v + 3], ag[k].w);
      atomicAdd(&sacc[C + 4 * v], ab[k].x); atomicAdd(&sacc[C + 4 * v + 1], ab[k].y);
      atomicAdd(&sacc[C + 4 * v + 2], ab[k].z); atomicAdd(&sacc[C + 4 * v + 3], ab[k].w);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += 256) {
    atomicAdd(&dgamma[i], sacc[i]);
    atomicAdd(&dbeta[i], sacc[C + i]);
  }
}

// ---------------------------------------------------------------------------------------------------------
// FiLM + SiLU: out = silu(shift_b + v (1 + scale_b)), (scale, shift) = film[b, off : off + C], [off + C : off + 2C]
// (diffusesg.py:238-240, :574-576).  One CTA per (sample, chunk of 32 tokens).
// ---------------------------------------------------------------------------------------------------------
constexpr int kFilmTokens = 32;
__global__ void __launch_bounds__(256)
film_silu_fwd_kernel(const float* __restrict__ v, const float* __restrict__ film, int ldf, int off,
                     float* __restrict__ out, int L, int C) {
  const int chunks = (L + kFilmTokens - 1) / kFilmTokens;
  const int b = blockIdx.x / chunks, t0 = (blockIdx.x - b * chunks) * kFilmTokens;
  const int nt = min(kFilmTokens, L - t0);
  const float* fs = film + static_cast<size_t>(b) * ldf + off;
  const size_t base = (static_cast<size_t>(b) * L + t0) * C;
  const int nv = C >> 2;
  for (int i = threadIdx.x; i < nt * nv; i += 256) {
    const int c = (i % nv) * 4;
    const size_t o = base + static_cast<size_t>(i / nv) * C + c;
    const float4 a = ld4(v + o), sc = ld4(fs + c), sh = ld4(fs + C + c);
    const float u0 = fmaf(a.x, sc.x + 1.f, sh.x), u1 = fmaf(a.y, sc.y + 1.f, sh.y), u2 = fmaf(a.z, sc.z + 1.f, sh.z),
                u3 = fmaf(a.w, sc.w + 1.f, sh.w);
    st4(out + o, make_float4(u0 * sigmoid_f(u0), u1 * sigmoid_f(u1), u2 * sigmoid_f(u2), u3 * sigmoid_f(u3)));
  }
}

// du = dout silu'(u); dv = du (1 + scale); dscale[b, c] += sum_tokens du v; dshift[b, c] += sum_tokens du.
// A thread keeps one float4 channel group for a strided run of the chunk's tokens, so the two parameter gradients
// accumulate in registers; threads of the same group meet in shared memory once per CTA (one atomic per channel per CTA).
constexpr int kFilmBwdTokens = 128;
__global__ void __launch_bounds__(256)
film_silu_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ v, const float* __restrict__ film, int ldf,
                     int off, float* __restrict__ dv, float* __restrict__ dfilm, int L, int C) {
  extern __shared__ float sacc[];  // [2][C]
  for (int i = threadIdx.x; i < 2 * C; i += 256) sacc[i] = 0.f;
  __syncthreads();
  const int chunks = (L + kFilmBwdTokens - 1) / kFilmBwdTokens;
  const int b = blockIdx.x / chunks, t0 = (blockIdx.x - b * chunks) * kFilmBwdTokens;
  const int nt = min(kFilmBwdTokens, L - t0);
  const float* fs = film + static_cast<size_t>(b) * ldf + off;
  const size_t base = (static_cast<size_t>(b) * L + t0) * C;
  const int nv = C >> 2;
  // groups are walked in passes of 256 threads: thread -> (group g = (pass * 256 + tid) % nv is NOT fixed), so fix it:
  // rows-per-pass R = 256 / nvp threads share a group, nvp = groups handled per pass
  const int nvp = nv < 256 ? nv : 256;          // groups per pass
  const int R = 256 / nvp;                      // token rows in flight per pass
  const int gl = threadIdx.x % nvp, rl = threadIdx.x / nvp;
  for (int g0 = 0; g0 < nv; g0 += nvp) {
    const int g = g0 + gl;
    if (g >= nv || rl >= R) continue;
    const int c = 4 * g;
    const float4 sc = ld4(fs + c), sh = ld4(fs + C + c);
    const float scv[4] = {sc.x, sc.y, sc.z, sc.w}, shv[4] = {sh.x, sh.y, sh.z, sh.w};
    float as[4] = {0.f, 0.f, 0.f, 0.f}, ah[4] = {0.f, 0.f, 0.f, 0.f};
    for (int t = rl; t < nt; t += R) {
      const size_t o = base + static_cast<size_t>(t) * C + c;
      const float4 a = ld4(v + o), gd = ld4(dout + o);
      const float av[4] = {a.x, a.y, a.z, a.w}, gv[4] = {gd.x, gd.y, gd.z, gd.w};
      float r[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float u = fmaf(av[k], scv[k] + 1.f, shv[k]);
        const float sg = sigmoid_f(u);
        const float du = gv[k] * sg * (1.f + u * (1.f - sg));
        r[k] = du * (scv[k] + 1.f);
        as[k] = fmaf(du, av[k], as[k]);
        ah[k] += du;
      }
      st4(dv + o, make_float4(r[0], r[1], r[2], r[3]));
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) { atomicAdd(&sacc[c + k], as[k]); atomicAdd(&sacc[C + c + k], ah[k]); }
  }
  __syncthreads();
  float* df = dfilm + static_cast<size_t>(b) * ldf + off;
  for (int i = threadIdx.x; i < 2 * C; i += 256) atomicAdd(&df[i], sacc[i]);
}

// ---------------------------------------------------------------------------------------------------------
// erf GELU (nn.GELU default), exact form for the training path: forward on the pre-activation kept for backward
// ---------------------------------------------------------------------------------------------------------
DSG_DEVICE float gelu_exact(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752f)); }
DSG_DEVICE float gelu_grad(float x) {
  return 0.5f * (1.f + erff(x * 0.70710678118654752f)) + x * 0.3989422804014327f * __expf(-0.5f * x * x);
}
// The bf16 MLP activations use the inference path's form of erf GELU (common.cuh: x/2 (1 + tanh(x q(x^2))), q a minimax
// fit, |error| <= 2.6e-5) and its analytic derivative (|error| <= 1.1e-4, rms 6.5e-5 under N(0,1) - both far below the bf16
// rounding of the stored value): ~3x fewer issue slots than erff + expf, which bound these kernels, and the training
// forward then computes exactly what the inference kernels compute.  The polynomial is evaluated on x clamped to +-10
// (tanh is saturated long before; beyond |x| = 11 the unclamped quartic would change sign).
DSG_DEVICE float gelu_fast(float x) {
  const float xc = fminf(fmaxf(x, -10.f), 10.f), x2 = xc * xc;
  const float q = fmaf(x2, fmaf(x2, -3.51516789e-04f, 3.70056460e-02f), 7.97507884e-01f);
  const float h = 0.5f * x;
  return fmaf(h, tanh_approx(xc * q), h);
}
DSG_DEVICE float gelu_fast_grad(float x) {
  const float xc = fminf(fmaxf(x, -10.f), 10.f), x2 = xc * xc;
  const float q = fmaf(x2, fmaf(x2, -3.51516789e-04f, 3.70056460e-02f), 7.97507884e-01f);
  const float dq = fmaf(x2, fmaf(x2, 5.f * -3.51516789e-04f, 3.f * 3.70056460e-02f), 7.97507884e-01f);   // d(x q)/dx
  const float t = tanh_approx(xc * q);
  return fmaf(0.5f * x * dq, fmaf(-t, t, 1.f), fmaf(0.5f, t, 0.5f));
}
// n8 = element count / 8; pointers 16-byte aligned
__global__ void __launch_bounds__(256)
gelu_fwd_kernel(const bf16_t* __restrict__ pre, bf16_t* __restrict__ out, long long n8) {
  const uint4* in = reinterpret_cast<const uint4*>(pre);
  uint4* o = reinterpret_cast<uint4*>(out);
  const long long stride = static_cast<long long>(gridDim.x) * 256;
  for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < n8; i += 2 * stride) {
    const bool two = i + stride < n8;
    const uint4 w0 = in[i], w1 = two ? in[i + stride] : w0;
    float f[8];
    unpack8(w0, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = gelu_fast(f[j]);
    o[i] = pack8(f);
    if (two) {
      unpack8(w1, f);
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = gelu_fast(f[j]);
      o[i + stride] = pack8(f);
    }
  }
}
__global__ void __launch_bounds__(256)
gelu_bwd_kernel(const bf16_t* __restrict__ dh, const bf16_t* __restrict__ pre, bf16_t* __restrict__ dpre, long long n8) {
  const uint4* in = reinterpret_cast<const uint4*>(pre);
  const uint4* gin = reinterpret_cast<const uint4*>(dh);
  uint4* o = reinterpret_cast<uint4*>(dpre);
  const long long stride = static_cast<long long>(gridDim.x) * 256;
  for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < n8; i += 2 * stride) {
    const bool two = i + stride < n8;
    const uint4 a0 = in[i], g0 = gin[i], a1 = two ? in[i + stride] : a0, g1 = two ? gin[i + stride] : g0;
    float f[8], g[8];
    unpack8(a0, f); unpack8(g0, g);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = g[j] * gelu_fast_grad(f[j]);
    o[i] = pack8(f);
    if (two) {
      unpack8(a1, f); unpack8(g1, g);
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = g[j] * gelu_fast_grad(f[j]);
      o[i + stride] = pack8(f);
    }
  }
}
__global__ void __launch_bounds__(256)
gelu_f32_kernel(const float* __restrict__ pre, const float* __restrict__ dout, float* __restrict__ out, long long n) {
  for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * 256)
    out[i] = dout == nullptr ? gelu_exact(pre[i]) : dout[i] * gelu_grad(pre[i]);
}
// out[c] += sum over rows of src[r, c] (bias gradients of the small fp32 layers): a thread per column for wide matrices;
// for narrow ones (the c_e = 6 / c_n = 12 wide outputs: a thread per column would leave most of the CTA idle) a flat
// mapping - thread t walks elements t, t + 256, ... of the CTA's row chunk, coalesced whatever C is - with a private
// shared-memory accumulator row per thread (no atomics, no contention), reduced once per CTA.
__global__ void __launch_bounds__(256)
colsum_f32_kernel(const float* __restrict__ src, float* __restrict__ out, long long M, int C, int rows_per_cta) {
  const long long r0 = static_cast<long long>(blockIdx.x) * rows_per_cta, r1 = min(M, r0 + rows_per_cta);
  const int c = blockIdx.y * 256 + threadIdx.x;      // grid.y = column blocks: a [128, 9792] matrix still fills the GPU
  if (c >= C) return;
  float s = 0.f;
  for (long long r = r0; r < r1; ++r) s += src[r * C + c];
  atomicAdd(&out[c], s);
}
__global__ void __launch_bounds__(256)
colsum_narrow_kernel(const float* __restrict__ src, float* __restrict__ out, long long M, int C, int rows_per_cta) {
  extern __shared__ float priv[];  // [256][C]
  float* mine = priv + threadIdx.x * C;
  for (int c = 0; c < C; ++c) mine[c] = 0.f;
  const long long r0 = static_cast<long long>(blockIdx.x) * rows_per_cta, r1 = min(M, r0 + rows_per_cta);
  const long long n = (r1 - r0) * C;
  const float* p = src + r0 * C;
  int c = threadIdx.x % C;
  const int step = 256 % C;
  for (long long i = threadIdx.x; i < n; i += 256) {
    mine[c] += p[i];
    c += step;
    if (c >= C) c -= C;
  }
  __syncthreads();
  for (int cc = threadIdx.x; cc < C; cc += 256) {
    float s = 0.f;
    for (int t = 0; t < 256; ++t) s += priv[t * C + cc];
    atomicAdd(&out[cc], s);
  }
}
// EDM preconditioning coefficients (runner/objectives/edm.py:122-126), sigma_data = 0.5: out = [c_skip | c_out | c_in | c_noise]
__global__ void precond_coef_kernel(const float* __restrict__ sigmas, float* __restrict__ out, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const float s = sigmas[b], sd = 0.5f;
  const float q = s * s + sd * sd;
  out[b] = sd * sd / q;
  out[B + b] = s * sd / sqrtf(q);
  out[2 * B + b] = 1.0f / sqrtf(q);
  out[3 * B + b] = logf(s) / 4.0f;
}
__global__ void __launch_bounds__(256)
silu_fwd_kernel(const float* __restrict__ pre, float* __restrict__ out, long long n) {
  for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * 256) {
    const float u = pre[i];
    out[i] = u * sigmoid_f(u);
  }
}
__global__ void __launch_bounds__(256)
silu_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ pre, float* __restrict__ dpre, long long n) {
  for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * 256) {
    const float u = pre[i], sg = sigmoid_f(u);
    dpre[i] = dout[i] * sg * (1.f + u * (1.f - sg));
  }
}
// y += x (gradient accumulation where a tensor has two consumers)
__global__ void __launch_bounds__(256)
add_inplace_kernel(float* __restrict__ y, const float* __restrict__ x, long long n4) {
  for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < n4; i += static_cast<long long>(gridDim.x) * 256) {
    const float4 a = ld4(y + 4 * i), b = ld4(x + 4 * i);
    st4(y + 4 * i, make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w));
  }
}

// Bias gradient and bf16 operand of a weight-gradient GEMM in one pass over dY [M, C] (C % 8 == 0): colsum[c] += sum over
// rows (columns < scale_cols scaled), cast [M, C] = bf16(dY) when dY is fp32.  A thread owns one 8-column group for a
// strided run of rows (a warp reads 32 consecutive groups of one row), four rows in flight.
constexpr int kCsRows = 512;
template <typename T>
__global__ void __launch_bounds__(256)
cast_colsum_kernel(const T* __restrict__ src, bf16_t* __restrict__ cast, float* __restrict__ colsum, long long M, int C,
                   int scale_cols, float scale) {
  __shared__ float part[8][256];
  const int g = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c = (blockIdx.x * 32 + g) * 8;
  const bool col_ok = c < C;
  const long long r_begin = static_cast<long long>(blockIdx.y) * kCsRows, r_end = min(M, r_begin + kCsRows);
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (long long r0 = r_begin + rl; r0 < r_end; r0 += 32) {
    float v[4][8];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long r = r0 + 8 * u;
      const bool ok = col_ok && r < r_end;
      const T* p = src + (ok ? r * C + c : 0);
      if (sizeof(T) == 2) {
        uint4 w = *reinterpret_cast<const uint4*>(p);
        if (!ok) w = make_uint4(0u, 0u, 0u, 0u);
        unpack8(w, v[u]);
      } else {
        float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
        if (!ok) { a = make_float4(0.f, 0.f, 0.f, 0.f); b = a; }
        v[u][0] = a.x; v[u][1] = a.y; v[u][2] = a.z; v[u][3] = a.w; v[u][4] = b.x; v[u][5] = b.y; v[u][6] = b.z; v[u][7] = b.w;
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long r = r0 + 8 * u;
      if (cast != nullptr && col_ok && r < r_end) *reinterpret_cast<uint4*>(cast + r * C + c) = pack8(v[u]);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += v[u][j];
    }
  }
  if (colsum != nullptr) {
#pragma unroll
    for (int j = 0; j < 8; ++j) part[rl][8 * g + j] = acc[j];
    __syncthreads();
    const int cc = blockIdx.x * 256 + threadIdx.x;
    if (cc < C) {
      float t = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) t += part[k][threadIdx.x];
      atomicAdd(&colsum[cc], cc < scale_cols ? t * scale : t);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// 2 x 2 space <-> depth: fine [B, 2H, 2W, C] <-> coarse [B, H, W, 4, C], chunk k = dy + 2 dx (PatchMerging's
// x0..x3 order, diffusesg.py:325-329, and PatchBreakup's scatter, :394-397: the same map).  fp32, pure permutation.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
shuffle2x2_kernel(const float* __restrict__ src, float* __restrict__ dst, int B, int H, int W, int C, int to_coarse) {
  const int nv = C >> 2;
  const long long total = static_cast<long long>(B) * H * W * 4 * nv;
  for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * 256) {
    const int v = static_cast<int>(i % nv);
    long long t = i / nv;
    const int k = static_cast<int>(t & 3);
    t >>= 2;
    const int xw = static_cast<int>(t % W);
    t /= W;
    const int yh = static_cast<int>(t % H);
    const int b = static_cast<int>(t / H);
    const long long coarse = i * 4;  // ((((b H + y) W + x) 4 + k) C + 4 v
    const long long fine = ((static_cast<long long>(b) * 2 * H + 2 * yh + (k & 1)) * 2 * W + 2 * xw + (k >> 1)) * C + 4 * v;
    if (to_coarse) st4(dst + coarse, ld4(src + fine));
    else st4(dst + fine, ld4(src + coarse));
  }
}

// dst[:, dcol : dcol + n] (=, +=) src[:, scol : scol + n]; src fp32, dst fp32 or bf16 (skip concat and its split).
// VEC: 16-byte accesses (every column count / pitch / offset a multiple of 4); otherwise element-wise.
template <bool VEC>
__global__ void __launch_bounds__(256)
copy_cols_kernel(const float* __restrict__ src, int lds, int scol, void* __restrict__ dst, int ldd, int dcol, int ncols,
                 long long M, int dst_bf16, int accumulate) {
  constexpr int W = VEC ? 4 : 1;
  const int nv = ncols / W;
  const long long total = M * nv;
  for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * 256) {
    const long long r = i / nv;
    const int c = static_cast<int>(i - r * nv) * W;
    if (VEC) {
      float4 a = ld4(src + r * lds + scol + c);
      if (dst_bf16) {
        st4_bf16(static_cast<bf16_t*>(dst) + r * ldd + dcol + c, a);
      } else {
        float* d = static_cast<float*>(dst) + r * ldd + dcol + c;
        if (accumulate) { const float4 e = ld4(d); a.x += e.x; a.y += e.y; a.z += e.z; a.w += e.w; }
        st4(d, a);
      }
    } else {
      const float a = src[r * lds + scol + c];
      if (dst_bf16) {
        static_cast<bf16_t*>(dst)[r * ldd + dcol + c] = __float2bfloat16_rn(a);
      } else {
        float* d = static_cast<float*>(dst) + r * ldd + dcol + c;
        *d = accumulate ? *d + a : a;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// Input grid of the patch embedding as a GEMM operand: row (b, i, j) = [sc_adj(Ce) | c_in adj(Ce) | node planes of i:
// sc_node, c_in node (2 Cn) | node planes of j (2 Cn) | zero pad to `ld`], node planes masked by flag_i & flag_j
// (diffusesg.py:791-802; c_in of model/precond/precond.py:100).  Without self-conditioning the sc blocks are absent.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
embed_input_kernel(const float* __restrict__ adj, const float* __restrict__ node, const float* __restrict__ sc_adj,
                   const float* __restrict__ sc_node, const uint8_t* __restrict__ flags, const float* __restrict__ c_in,
                   bf16_t* __restrict__ out, int B, int n, int c_e, int c_n, int self_cond, int ld) {
  // work item = (32 consecutive pixels, one group of 8 output channels): the adjacency planes are read 128 bytes per warp,
  // every lane writes one 16-byte piece of its pixel's row
  const int groups = ld >> 3;
  const long long total = static_cast<long long>(B) * n * n;
  const int nn = n * n;
  const long long items = ((total + 31) / 32) * groups;
  const int lane = threadIdx.x & 31;
  const int ce_all = self_cond ? 2 * c_e : c_e, cn_all = self_cond ? 2 * c_n : c_n;
  for (long long it = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5); it < items; it += static_cast<long long>(gridDim.x) * 8) {
    const int grp = static_cast<int>(it % groups);
    const long long pix = (it / groups) * 32 + lane;
    if (pix >= total) continue;
    const int b = static_cast<int>(pix / nn), ij = static_cast<int>(pix - static_cast<long long>(b) * nn);
    const int i = ij / n, j = ij - i * n;
    const float ci = c_in != nullptr ? c_in[b] : 1.f;
    const bool ok = flags[b * n + i] != 0 && flags[b * n + j] != 0;
    float f[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int ch = 8 * grp + k;
      float val = 0.f;
      if (ch < ce_all) {                                   // adjacency planes: self-conditioning first (:791-794)
        const bool is_sc = self_cond && ch < c_e;
        const int c = is_sc ? ch : ch - (self_cond ? c_e : 0);
        if (is_sc) val = sc_adj != nullptr ? sc_adj[(static_cast<size_t>(b) * c_e + c) * nn + ij] : 0.f;
        else val = ci * adj[(static_cast<size_t>(b) * c_e + c) * nn + ij];
      } else if (ch < ce_all + 2 * cn_all) {               // node planes of i, then of j, masked by flag_i & flag_j (:797-800)
        const int q = ch - ce_all, side = q / cn_all, cc = q - side * cn_all;
        const size_t nrow = (static_cast<size_t>(b) * n + (side == 0 ? i : j)) * c_n;
        const bool is_sc = self_cond && cc < c_n;
        if (ok) {
          if (is_sc) val = sc_node != nullptr ? sc_node[nrow + cc] : 0.f;
          else val = ci * node[nrow + cc - (self_cond ? c_n : 0)];
        }
      }
      f[k] = val;
    }
    *reinterpret_cast<uint4*>(out + pix * ld + 8 * grp) = pack8(f);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Read-out heads: token-major head outputs -> the reference's output tensors (mask, optional EDM output
// preconditioning D = c_skip x + c_out F), and back.
//   adj: tok [B n n, ce] -> out [B, ce, n, n] masked by flag_i & flag_j       (diffusesg.py:809, :825; precond.py:102-105)
//   node: tok [B n, cn]  -> out [B, n, cn]   masked by flag_i                 (:818-822)
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
adj_out_kernel(const float* __restrict__ tok, const uint8_t* __restrict__ flags, const float* __restrict__ x_adj,
               const float* __restrict__ c_skip, const float* __restrict__ c_out, float* __restrict__ out, int B, int n,
               int c_e, int backward) {
  // forward: out = mask (c_skip x + c_out tok); backward: tok_grad (written to `out` [B n n, ce]) = mask c_out * grad (`tok` [B, ce, n, n])
  const int nn = n * n;
  const long long total = static_cast<long long>(B) * nn;
  for (long long pix = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; pix < total; pix += static_cast<long long>(gridDim.x) * 256) {
    const int b = static_cast<int>(pix / nn), ij = static_cast<int>(pix - static_cast<long long>(b) * nn);
    const int i = ij / n, j = ij - i * n;
    const bool ok = flags[b * n + i] != 0 && flags[b * n + j] != 0;
    const float co = c_out != nullptr ? c_out[b] : 1.f;
    for (int c = 0; c < c_e; ++c) {
      const size_t plane = (static_cast<size_t>(b) * c_e + c) * nn + ij;
      if (!backward) {
        float val = co * tok[pix * c_e + c];
        if (x_adj != nullptr) val += c_skip[b] * x_adj[plane];
        out[plane] = ok ? val : 0.f;
      } else {
        out[pix * c_e + c] = ok ? co * tok[plane] : 0.f;
      }
    }
  }
}
__global__ void __launch_bounds__(256)
node_out_kernel(const float* __restrict__ tok, const uint8_t* __restrict__ flags, const float* __restrict__ x_node,
                const float* __restrict__ c_skip, const float* __restrict__ c_out, float* __restrict__ out, int B, int n,
                int c_n, int backward) {
  const long long total = static_cast<long long>(B) * n * c_n;
  for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * 256) {
    const long long bi = i / c_n;
    const int b = static_cast<int>(bi / n);
    const bool ok = flags[bi] != 0;
    const float co = c_out != nullptr ? c_out[b] : 1.f;
    if (!backward) {
      float val = co * tok[i];
      if (x_node != nullptr) val += c_skip[b] * x_node[i];
      out[i] = ok ? val : 0.f;
    } else {
      out[i] = ok ? co * tok[i] : 0.f;
    }
  }
}
// masked mean over the last pair axis: pooled[b, i, :] = flag_i / n * sum_j flag_j rep[b, i, j, :]  (:812-813);
// backward: drep[b, i, j, :] += flag_i flag_j / n * dpooled[b, i, :]
__global__ void __launch_bounds__(256)
node_pool_train_kernel(const float* __restrict__ rep, const uint8_t* __restrict__ flags, float* __restrict__ pooled, int B,
                       int n, int C) {
  const int lane = threadIdx.x & 31;
  const long long rows = static_cast<long long>(B) * n;
  const long long bi = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (bi >= rows) return;
  const int b = static_cast<int>(bi / n);
  const bool live = flags[bi] != 0;
  for (int c = lane; c < C; c += 32) {
    float s = 0.f;
    if (live)
      for (int j = 0; j < n; ++j)
        if (flags[b * n + j] != 0) s += rep[(bi * n + j) * C + c];
    pooled[bi * C + c] = s / n;
  }
}
__global__ void __launch_bounds__(256)
node_pool_bwd_kernel(const float* __restrict__ dpooled, const uint8_t* __restrict__ flags, float* __restrict__ drep, int B,
                     int n, int C) {
  const int nv = C >> 2;
  const long long total = static_cast<long long>(B) * n * n * nv;
  const float inv = 1.0f / n;
  for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * 256) {
    const int v = static_cast<int>(i % nv);
    const long long pix = i / nv;
    const long long bi = pix / n;
    const int j = static_cast<int>(pix - bi * n);
    const int b = static_cast<int>(bi / n);
    if (flags[bi] == 0 || flags[b * n + j] == 0) continue;
    const float4 g = ld4(dpooled + bi * C + 4 * v);
    float* d = drep + pix * C + 4 * v;
    const float4 e = ld4(d);
    st4(d, make_float4(e.x + inv * g.x, e.y + inv * g.y, e.z + inv * g.z, e.w + inv * g.w));
  }
}

// Second layer of the adjacency read-out MLP (diffusesg.py:806-809), c_e <= 8 outputs per pixel from `embed` <= 128 hidden
// channels: far too narrow for a GEMM tile (a 64 x 64 tile would waste 90 % of its work).  One warp per pixel row, a lane
// owns channels lane + 32 k with the c_e x 4 weights in registers.
//   forward:  tok[m, c] = b[c] + sum_e h[m, e] w[c, e]
//   wgrad:    dw[c, e] += sum_m dtok[m, c] h[m, e]   (register accumulators per warp, shared memory per CTA, one atomic per
//             entry per CTA)
__global__ void __launch_bounds__(256)
adj_fc2_fwd_kernel(const bf16_t* __restrict__ h, const float* __restrict__ w, const float* __restrict__ b, float* __restrict__ tok,
                   long long M, int E, int ce) {
  const int lane = threadIdx.x & 31;
  float wv[8][4];
#pragma unroll
  for (int c = 0; c < 8; ++c)
#pragma unroll
    for (int k = 0; k < 4; ++k) wv[c][k] = (c < ce && lane + 32 * k < E) ? w[c * E + lane + 32 * k] : 0.f;
  const float bias = lane < ce ? b[lane] : 0.f;
  const long long warps = static_cast<long long>(gridDim.x) * 8;
  for (long long row = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5); row < M; row += warps) {
    float hv[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) hv[k] = lane + 32 * k < E ? __bfloat162float(h[row * E + lane + 32 * k]) : 0.f;
    float mine = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float a = 0.f;
#pragma unroll
      for (int k = 0; k < 4; ++k) a = fmaf(wv[c][k], hv[k], a);
      a = warp_sum(a);
      if (lane == c) mine = a;
    }
    if (lane < ce) tok[row * ce + lane] = mine + bias;
  }
}
__global__ void __launch_bounds__(256)
adj_fc2_wgrad_kernel(const float* __restrict__ dtok, const bf16_t* __restrict__ h, float* __restrict__ dw, long long M, int E,
                     int ce, int rows_per_cta) {
  __shared__ float sacc[8 * 128];
  for (int i = threadIdx.x; i < 8 * 128; i += 256) sacc[i] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long r0 = static_cast<long long>(blockIdx.x) * rows_per_cta, r1 = min(M, r0 + rows_per_cta);
  float acc[8][4];
#pragma unroll
  for (int c = 0; c < 8; ++c)
#pragma unroll
    for (int k = 0; k < 4; ++k) acc[c][k] = 0.f;
  for (long long row = r0 + (threadIdx.x >> 5); row < r1; row += 8) {
    float hv[4], d[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) hv[k] = lane + 32 * k < E ? __bfloat162float(h[row * E + lane + 32 * k]) : 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) d[c] = c < ce ? dtok[row * ce + c] : 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c)
#pragma unroll
      for (int k = 0; k < 4; ++k) acc[c][k] = fmaf(d[c], hv[k], acc[c][k]);
  }
#pragma unroll
  for (int c = 0; c < 8; ++c)
#pragma unroll
    for (int k = 0; k < 4; ++k) atomicAdd(&sacc[c * 128 + lane + 32 * k], acc[c][k]);
  __syncthreads();
  for (int i = threadIdx.x; i < ce * E; i += 256) {
    const int c = i / E, e = i - c * E;
    atomicAdd(&dw[i], sacc[c * 128 + e]);
  }
}

// sinusoidal noise embedding (PositionalEmbedding, diffusesg.py:507-513): [cos(x f_k) | sin(x f_k)], f_k = 10000^(-k / half)
__global__ void posemb_kernel(const float* __restrict__ labels, float* __restrict__ out, int B, int embed) {
  const int half = embed / 2;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B * half; i += gridDim.x * blockDim.x) {
    const int b = i / half, k = i - b * half;
    const float f = powf(1.0f / 10000.0f, static_cast<float>(k) / static_cast<float>(half));
    const float a = labels[b] * f;
    out[b * embed + k] = cosf(a);
    out[b * embed + half + k] = sinf(a);
  }
}

// relative-position bias: bias[h, t, u] = table[index[t, u], h] (:121-124) and its transpose-scatter
__global__ void bias_gather_kernel(const float* __restrict__ table, const int64_t* __restrict__ index, float* __restrict__ bias,
                                   int heads, int TT, int backward, float* __restrict__ dtable) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < heads * TT; i += gridDim.x * blockDim.x) {
    const int h = i / TT, tu = i - h * TT;
    const long long idx = index[tu];
    if (!backward) bias[i] = table[idx * heads + h];
    else atomicAdd(&dtable[idx * heads + h], bias[i]);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Small fp32 GEMM with arbitrary strides and an accumulate / split-K mode, for the matrices far too small or too
// oddly shaped for the tcgen05 kernel: the noise-embedding MLP and the FiLM generators (batch rows), the node
// read-out MLP ([B n] rows), the c_e / c_n wide output layers and all their gradients.
//   C[m, n] (+)= sum_k A(m, k) B(k, n) (+ bias[n]),  A(m, k) = A[m sam + k sak] (fp32 or bf16), B(k, n) = B[k sbk + n sbn]
// 64 x 64 tile, 16-deep k steps, 256 threads x (4 x 4); gridDim.z = K slices combined with atomicAdd.
// ---------------------------------------------------------------------------------------------------------
template <typename TA, typename TB>
__global__ void __launch_bounds__(256)
sgemm_kernel(const TA* __restrict__ A, long long sam, long long sak, const TB* __restrict__ Bm, long long sbk, long long sbn,
             const float* __restrict__ bias, float* __restrict__ Cm, long long ldc, int M, int N, int K, int k_per,
             int accumulate) {
  __shared__ float sA[16][65], sB[16][65];
  const int m0 = blockIdx.x * 64, n0 = blockIdx.y * 64;
  const int k_begin = blockIdx.z * k_per, k_end = min(K, k_begin + k_per);
  const int tn = threadIdx.x & 15, tm = threadIdx.x >> 4;   // thread tile: rows tm + 16 r, cols tn + 16 c
  float acc[4][4] = {};
  for (int k0 = k_begin; k0 < k_end; k0 += 16) {
    for (int i = threadIdx.x; i < 16 * 64; i += 256) {
      // A tile: choose the faster-running index to follow the smaller stride
      int kk, mm;
      if (sak <= sam) { kk = i & 15; mm = i >> 4; } else { mm = i & 63; kk = i >> 6; }
      const int m = m0 + mm, k = k0 + kk;
      sA[kk][mm] = (m < M && k < k_end) ? static_cast<float>(A[m * sam + k * sak]) : 0.f;
      int kb, nb;
      if (sbk <= sbn) { kb = i & 15; nb = i >> 4; } else { nb = i & 63; kb = i >> 6; }
      const int n = n0 + nb, k2 = k0 + kb;
      sB[kb][nb] = (n < N && k2 < k_end) ? static_cast<float>(Bm[k2 * sbk + n * sbn]) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) a[r] = sA[kk][tm + 16 * r];
#pragma unroll
      for (int c = 0; c < 4; ++c) b[c] = sB[kk][tn + 16 * c];
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] = fmaf(a[r], b[c], acc[r][c]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int m = m0 + tm + 16 * r;
    if (m >= M) continue;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int n = n0 + tn + 16 * c;
      if (n >= N) continue;
      float val = acc[r][c];
      if (bias != nullptr && blockIdx.z == 0) val += bias[n];
      float* o = Cm + static_cast<long long>(m) * ldc + n;
      if (gridDim.z > 1) atomicAdd(o, val);     // K slices meet in the output
      else if (accumulate) *o += val;           // one slice: this CTA is the element's only writer
      else *o = val;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// Window attention backward (WindowAttention.forward, diffusesg.py:108-139, with roll / window_partition /
// window_reverse :28-57, :248-267 as index arithmetic).  One CTA = one head and a contiguous chunk of (sample, window)
// pairs; per window-head, from shared memory:
//   S = Q K^T + bias (+ mask);  P = softmax(S);  dV = P^T dO;  dP = dO V^T;  dS = P o (dP - rowsum(dP o P));
//   dQ = dS K;  dK = dS^T Q;  dbias += dS   (accumulated per CTA in shared memory, one atomicAdd per entry per CTA)
// q arrives pre-scaled (the qkv weight's q rows carry head_dim^-1/2), so dQ is the gradient w.r.t. the scaled q.
// The five products run on the warp-level tensor cores (wmma m16n16k16, bf16 operands, fp32 accumulation) as 4 x 4 (x 2)
// tiles; the softmax / dS pass stays fp32, dbias accumulates the fp32 dS.  P and dS are rounded to bf16 for the second
// set of products (as the forward kernel rounds P).  Token counts that are no multiple of 16 (10 x 10 windows) are zero
// padded to TP.  Shared-memory plan per CTA (PF = fp32 pitch of S / dP, >= TP + 16):
//   sQ sK sV sDO  bf16 [TP][40]
//   sS, sD        fp32 [TP][PF]: S -> exp -> (in place, row start) P as bf16; the upper half of each row then stages
//                 the fp32 outputs dV (sS) / dQ (sD), the lower half of sS stages dK once P is dead
//   sAcc          fp32 [T][T] dbias accumulator, sTok int [TP]
// ---------------------------------------------------------------------------------------------------------
constexpr int kHd = 32, kQP = 40;
// TC: compile-time token count of the window (64 for the 8 x 8 windows of the VG geometry: every index expression and
// loop bound folds); 0 = taken from the window size at run time.
template <int TC>
__global__ void __launch_bounds__(256)
window_attention_bwd_tc_kernel(const bf16_t* __restrict__ qkv, const bf16_t* __restrict__ datt, const float* __restrict__ bias,
                               const float* __restrict__ mask, bf16_t* __restrict__ dqkv, float* __restrict__ dbias,
                               int batch, int res, int w, int shift, int heads, int items_per_cta) {
  using namespace nvcuda;
  extern __shared__ __align__(128) unsigned char smraw[];
  const int T = TC ? TC : w * w, TP = (T + 15) & ~15, NT = TP >> 4, C = heads * kHd;
  // fp32 pitch of S / dP.  P and dS are re-read as bf16 with a row stride of PF words: PF % 32 == 20 keeps the eight 16-byte
  // rows of a fragment load on distinct banks (80 gave 4-way conflicts); 10 x 10 windows keep 128 (shared-memory budget)
  const int PF = TP <= 64 ? 84 : ((TP + 16 > 80) ? TP + 16 : 80);
  const int ST = TP <= 64 ? 40 : PF / 2;          // first float of the staging half of a row (32-byte aligned, past the bf16 P)
  bf16_t* sQ = reinterpret_cast<bf16_t*>(smraw);
  bf16_t* sK = sQ + TP * kQP;
  bf16_t* sV = sK + TP * kQP;
  bf16_t* sDO = sV + TP * kQP;
  float* sS = reinterpret_cast<float*>(sDO + TP * kQP);
  float* sD = sS + TP * PF;
  float* sAcc = sD + TP * PF;
  float* sBias = sAcc + T * T;                    // this head's bias [T][T], loaded once per CTA
  int* sTok = reinterpret_cast<int*>(sBias + T * T);
  bf16_t* sPb = reinterpret_cast<bf16_t*>(sS);    // P, bf16, row pitch 2 PF
  bf16_t* sDb = reinterpret_cast<bf16_t*>(sD);    // dS
  const int LDB = 2 * PF;
  float* stV = sS + ST;                           // fp32 staging [TP][32], row pitch PF
  float* stQ = sD + ST;
  float* stK = sS;
  const int h = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nw = res / w, nW = nw * nw;
  const int total = batch * nW;
  const int item0 = blockIdx.x * items_per_cta, item1 = min(total, item0 + items_per_cta);
  const float* bh = bias + static_cast<size_t>(h) * T * T;
  for (int i = threadIdx.x; i < T * T; i += 256) { sAcc[i] = 0.f; sBias[i] = bh[i]; }
  for (int item = item0; item < item1; ++item) {
    const int b = item / nW, win = item - b * nW;
    const int wy = win / nw, wx = win - wy * nw;
    __syncthreads();
    for (int t = threadIdx.x; t < TP; t += 256) {
      const int r = t / w, c = t - r * w;
      sTok[t] = t < T ? (b * res + (wy * w + r + shift) % res) * res + (wx * w + c + shift) % res : -1;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < TP * 16; i += 256) {   // 4 matrices x 4 16-byte chunks per token
      const int t = i >> 4, m = (i >> 2) & 3, ch = i & 3;
      uint4 val = make_uint4(0u, 0u, 0u, 0u);
      const int tok = sTok[t];
      if (tok >= 0) {
        const bf16_t* p = m < 3 ? qkv + static_cast<size_t>(tok) * 3 * C + m * C + h * kHd : datt + static_cast<size_t>(tok) * C + h * kHd;
        val = *reinterpret_cast<const uint4*>(p + 8 * ch);
      }
      bf16_t* d = (m == 0 ? sQ : m == 1 ? sK : m == 2 ? sV : sDO) + t * kQP + 8 * ch;
      *reinterpret_cast<uint4*>(d) = val;
    }
    __syncthreads();
    // S = Q K^T and dP = dO V^T
    if (TC == 64) {
      // 64 tokens: eight row strips (2 products x 4 row tiles) for eight warps - the A fragments of a strip are loaded once
      const int which = warp >> 2, ti = warp & 3;
      const bf16_t* A = which == 0 ? sQ : sDO;
      const bf16_t* Bt = which == 0 ? sK : sV;
      wmma::fragment<wmma::matrix_a, 16, 16, 16, __nv_bfloat16, wmma::row_major> fa[2];
      wmma::load_matrix_sync(fa[0], A + ti * 16 * kQP, kQP);
      wmma::load_matrix_sync(fa[1], A + ti * 16 * kQP + 16, kQP);
#pragma unroll
      for (int tj = 0; tj < 4; ++tj) {
        wmma::fragment<wmma::accumulator, 16, 16, 16, float> fc;
        wmma::fill_fragment(fc, 0.f);
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
          wmma::fragment<wmma::matrix_b, 16, 16, 16, __nv_bfloat16, wmma::col_major> fb;
          wmma::load_matrix_sync(fb, Bt + tj * 16 * kQP + kk * 16, kQP);
          wmma::mma_sync(fc, fa[kk], fb, fc);
        }
        wmma::store_matrix_sync((which == 0 ? sS : sD) + ti * 16 * PF + tj * 16, fc, PF, wmma::mem_row_major);
      }
    } else
    for (int job = warp; job < 2 * NT * NT; job += 8) {
      const int which = job / (NT * NT), tile = job - which * NT * NT;
      const int ti = tile / NT, tj = tile - ti * NT;
      const bf16_t* A = which == 0 ? sQ : sDO;
      const bf16_t* Bt = which == 0 ? sK : sV;
      wmma::fragment<wmma::accumulator, 16, 16, 16, float> fc;
      wmma::fill_fragment(fc, 0.f);
#pragma unroll
      for (int kk = 0; kk < 2; ++kk) {
        wmma::fragment<wmma::matrix_a, 16, 16, 16, __nv_bfloat16, wmma::row_major> fa;
        wmma::fragment<wmma::matrix_b, 16, 16, 16, __nv_bfloat16, wmma::col_major> fb;
        wmma::load_matrix_sync(fa, A + ti * 16 * kQP + kk * 16, kQP);
        wmma::load_matrix_sync(fb, Bt + tj * 16 * kQP + kk * 16, kQP);
        wmma::mma_sync(fc, fa, fb, fc);
      }
      wmma::store_matrix_sync((which == 0 ? sS : sD) + ti * 16 * PF + tj * 16, fc, PF, wmma::mem_row_major);
    }
    __syncthreads();
    const float* mk = (mask != nullptr && shift > 0) ? mask + static_cast<size_t>(win) * T * T : nullptr;
    for (int i = warp; i < TP; i += 8) {
      float* srow = sS + i * PF;
      float* drow = sD + i * PF;
      bf16_t* prow = sPb + i * LDB;
      bf16_t* dsrow = sDb + i * LDB;
      if (i >= T) {   // padding rows: zero operands
        for (int j = lane; j < TP; j += 32) { prow[j] = __float2bfloat16_rn(0.f); dsrow[j] = __float2bfloat16_rn(0.f); }
        continue;
      }
      // the row lives in registers (<= 4 elements per lane, TP <= 128): scores + bias (+ mask), one max and one sum
      // reduction, then P and dS go back as bf16 at the start of their own rows - every fp32 read of the row is done by then
      float sv[4], dv[4];
      float mx = -INFINITY;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int j = lane + 32 * t;
        sv[t] = -INFINITY;
        dv[t] = 0.f;
        if (j < T) {
          sv[t] = srow[j] + sBias[i * T + j] + (mk != nullptr ? mk[i * T + j] : 0.f);
          dv[t] = drow[j];
          mx = fmaxf(mx, sv[t]);
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      float sum = 0.f, dun = 0.f;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const float e = (lane + 32 * t < T) ? __expf(sv[t] - mx) : 0.f;
        sv[t] = e;
        sum += e;
        dun = fmaf(e, dv[t], dun);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        sum += __shfl_xor_sync(0xffffffffu, sum, o);
        dun += __shfl_xor_sync(0xffffffffu, dun, o);
      }
      const float inv = 1.0f / sum;
      const float dot = dun * inv;
      __syncwarp();
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int j = lane + 32 * t;
        if (j < TP) {
          float pv = 0.f, ds = 0.f;
          if (j < T) {
            pv = sv[t] * inv;
            ds = pv * (dv[t] - dot);
            sAcc[i * T + j] += ds;
          }
          prow[j] = __float2bfloat16_rn(pv);
          dsrow[j] = __float2bfloat16_rn(ds);
        }
      }
    }
    __syncthreads();
    // dV = P^T dO -> stV, dQ = dS K -> stQ
    if (TC == 64) {
      // eight (product, row tile) strips: both 16-column halves of the output share the A fragment of every k step
      const int which = warp >> 2, tr = warp & 3;
      wmma::fragment<wmma::accumulator, 16, 16, 16, float> fc0, fc1;
      wmma::fill_fragment(fc0, 0.f);
      wmma::fill_fragment(fc1, 0.f);
      const bf16_t* Bm = which == 0 ? sDO : sK;
#pragma unroll
      for (int kt = 0; kt < 4; ++kt) {
        wmma::fragment<wmma::matrix_b, 16, 16, 16, __nv_bfloat16, wmma::row_major> fb0, fb1;
        wmma::load_matrix_sync(fb0, Bm + kt * 16 * kQP, kQP);
        wmma::load_matrix_sync(fb1, Bm + kt * 16 * kQP + 16, kQP);
        if (which == 0) {
          wmma::fragment<wmma::matrix_a, 16, 16, 16, __nv_bfloat16, wmma::col_major> fa;   // A(j, i) = P[i][j]
          wmma::load_matrix_sync(fa, sPb + kt * 16 * LDB + tr * 16, LDB);
          wmma::mma_sync(fc0, fa, fb0, fc0);
          wmma::mma_sync(fc1, fa, fb1, fc1);
        } else {
          wmma::fragment<wmma::matrix_a, 16, 16, 16, __nv_bfloat16, wmma::row_major> fa;   // A(i, j) = dS[i][j]
          wmma::load_matrix_sync(fa, sDb + tr * 16 * LDB + kt * 16, LDB);
          wmma::mma_sync(fc0, fa, fb0, fc0);
          wmma::mma_sync(fc1, fa, fb1, fc1);
        }
      }
      float* st = (which == 0 ? stV : stQ) + tr * 16 * PF;
      wmma::store_matrix_sync(st, fc0, PF, wmma::mem_row_major);
      wmma::store_matrix_sync(st + 16, fc1, PF, wmma::mem_row_major);
    } else
    for (int job = warp; job < 2 * NT * 2; job += 8) {
      const int which = job / (NT * 2), tile = job - which * NT * 2;
      const int tr = tile >> 1, td = tile & 1;
      wmma::fragment<wmma::accumulator, 16, 16, 16, float> fc;
      wmma::fill_fragment(fc, 0.f);
      for (int kt = 0; kt < NT; ++kt) {
        wmma::fragment<wmma::matrix_b, 16, 16, 16, __nv_bfloat16, wmma::row_major> fb;
        if (which == 0) {
          wmma::fragment<wmma::matrix_a, 16, 16, 16, __nv_bfloat16, wmma::col_major> fa;   // A(j, i) = P[i][j]
          wmma::load_matrix_sync(fa, sPb + kt * 16 * LDB + tr * 16, LDB);
          wmma::load_matrix_sync(fb, sDO + kt * 16 * kQP + td * 16, kQP);
          wmma::mma_sync(fc, fa, fb, fc);
        } else {
          wmma::fragment<wmma::matrix_a, 16, 16, 16, __nv_bfloat16, wmma::row_major> fa;   // A(i, j) = dS[i][j]
          wmma::load_matrix_sync(fa, sDb + tr * 16 * LDB + kt * 16, LDB);
          wmma::load_matrix_sync(fb, sK + kt * 16 * kQP + td * 16, kQP);
          wmma::mma_sync(fc, fa, fb, fc);
        }
      }
      wmma::store_matrix_sync((which == 0 ? stV : stQ) + tr * 16 * PF + td * 16, fc, PF, wmma::mem_row_major);
    }
    __syncthreads();
    // dK = dS^T Q -> stK (the bf16 P it overwrites is dead)
    for (int job = warp; job < NT * 2; job += 8) {
      const int tr = job >> 1, td = job & 1;
      wmma::fragment<wmma::accumulator, 16, 16, 16, float> fc;
      wmma::fill_fragment(fc, 0.f);
      for (int kt = 0; kt < NT; ++kt) {
        wmma::fragment<wmma::matrix_a, 16, 16, 16, __nv_bfloat16, wmma::col_major> fa;     // A(j, i) = dS[i][j]
        wmma::fragment<wmma::matrix_b, 16, 16, 16, __nv_bfloat16, wmma::row_major> fb;
        wmma::load_matrix_sync(fa, sDb + kt * 16 * LDB + tr * 16, LDB);
        wmma::load_matrix_sync(fb, sQ + kt * 16 * kQP + td * 16, kQP);
        wmma::mma_sync(fc, fa, fb, fc);
      }
      wmma::store_matrix_sync(stK + tr * 16 * PF + td * 16, fc, PF, wmma::mem_row_major);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < T * 48; i += 256) {   // (token, matrix, channel pair)
      const int t = i / 48, rem = i - t * 48, m = rem >> 4, d = (rem & 15) * 2;
      const float* st = (m == 0 ? stQ : m == 1 ? stK : stV) + t * PF + d;
      *reinterpret_cast<__nv_bfloat162*>(dqkv + static_cast<size_t>(sTok[t]) * 3 * C + m * C + h * kHd + d) =
          __floats2bfloat162_rn(st[0], st[1]);
    }
  }
  __syncthreads();
  float* dbh = dbias + static_cast<size_t>(h) * T * T;
  for (int i = threadIdx.x; i < T * T; i += 256) atomicAdd(&dbh[i], sAcc[i]);
}

// ---------------------------------------------------------------------------------------------------------
// Optimiser: global gradient norm (nn.utils.clip_grad_norm_, trainer_node_adj.py:174), Adam (torch.optim.Adam
// semantics incl. L2 weight decay, utils/learning_utils.py:126-145) and up to 8 exponential moving averages
// (ema_pytorch.EMA.update with update_every 1, :148-166) over ONE flat fp32 parameter buffer in one launch.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
sumsq_kernel(const float* __restrict__ g, long long n, float* __restrict__ out) {
  float s = 0.f;
  for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * 256) s += g[i] * g[i];
  __shared__ float part[8];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int k = 0; k < 8; ++k) t += part[k];
    atomicAdd(out, t);
  }
}
struct AdamArgs {
  float lr, beta1, beta2, eps, weight_decay, bc1, bc2_sqrt, max_norm;
  int n_ema;
  float ema_decay[8];
  float* ema[8];
};
__global__ void __launch_bounds__(256)
adam_ema_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n4,
                const float* __restrict__ gsumsq, AdamArgs a) {
  // n4 = elements / 4 (the flat buffer is a multiple of 4 floats); every stream is read and written once, 16 bytes at a time
  float clip = 1.f;
  if (gsumsq != nullptr && a.max_norm > 0.f) clip = fminf(1.f, a.max_norm / (sqrtf(*gsumsq) + 1e-6f));
  const float step_size = a.lr / a.bc1, inv_bc2 = 1.0f / a.bc2_sqrt;
  for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < n4; i += static_cast<long long>(gridDim.x) * 256) {
    float4 w4 = ld4(p + 4 * i);
    float w[4] = {w4.x, w4.y, w4.z, w4.w};
    if (m != nullptr) {   // m == NULL: moving averages only
      const float4 g4 = ld4(g + 4 * i), m4 = ld4(m + 4 * i), v4 = ld4(v + 4 * i);
      const float gg[4] = {g4.x, g4.y, g4.z, g4.w};
      float mm[4] = {m4.x, m4.y, m4.z, m4.w}, vv[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float gi = gg[k] * clip + a.weight_decay * w[k];
        mm[k] = a.beta1 * mm[k] + (1.f - a.beta1) * gi;
        vv[k] = a.beta2 * vv[k] + (1.f - a.beta2) * gi * gi;
        w[k] -= step_size * mm[k] / (sqrtf(vv[k]) * inv_bc2 + a.eps);
      }
      st4(m + 4 * i, make_float4(mm[0], mm[1], mm[2], mm[3]));
      st4(v + 4 * i, make_float4(vv[0], vv[1], vv[2], vv[3]));
      st4(p + 4 * i, make_float4(w[0], w[1], w[2], w[3]));
    }
#pragma unroll
    for (int k = 0; k < 8; ++k)
      if (k < a.n_ema) {   // lerp(ema, w, 1 - decay); decay 0 is ema_pytorch's plain copy
        float* e = a.ema[k] + 4 * i;
        const float d = a.ema_decay[k];
        const float4 e4 = ld4(e);
        st4(e, d == 0.f ? make_float4(w[0], w[1], w[2], w[3])
                        : make_float4(e4.x + (1.f - d) * (w[0] - e4.x), e4.y + (1.f - d) * (w[1] - e4.y),
                                      e4.z + (1.f - d) * (w[2] - e4.z), e4.w + (1.f - d) * (w[3] - e4.w)));
      }
  }
}

// weight preparation: bf16 shadows of the fp32 masters for the tcgen05 GEMMs, one launch for all matrices.
// job: src [rows, cols] fp32 -> dst [rows, ldd] bf16 (zero padded to ldd), dst_t [cols_t_rows = ldt_rows, rows]: the
// transpose with `ldt` = rows pitch (dgrad operand W^T), first `scale_elems` source elements scaled (q rows of qkv);
// dtype_f32: dst is an fp32 vector copy (the scaled qkv bias).
struct PrepJob {
  const float* src;
  void* dst;
  bf16_t* dst_t;
  int rows, cols, ldd, rows_t;   // rows_t: row count of dst_t (>= cols, zero padded)
  long long scale_elems;
  float scale;
  int dst_f32;
};
__global__ void __launch_bounds__(256)
prep_weights_kernel(const PrepJob* __restrict__ jobs) {
  const PrepJob j = jobs[blockIdx.y];
  const long long n = static_cast<long long>(j.rows) * j.ldd;
  for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * 256) {
    const int r = static_cast<int>(i / j.ldd), c = static_cast<int>(i - static_cast<long long>(r) * j.ldd);
    float val = 0.f;
    if (c < j.cols) {
      const long long s = static_cast<long long>(r) * j.cols + c;
      val = j.src[s];
      if (s < j.scale_elems) val *= j.scale;
    }
    if (j.dst_f32) static_cast<float*>(j.dst)[i] = val;
    else static_cast<bf16_t*>(j.dst)[i] = __float2bfloat16_rn(val);
    if (j.dst_t != nullptr) j.dst_t[static_cast<long long>(c) * j.rows + r] = __float2bfloat16_rn(val);
  }
  if (j.dst_t != nullptr) {  // zero rows [ldd, rows_t) of the transpose
    const long long extra = static_cast<long long>(j.rows_t - j.ldd) * j.rows;
    for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < extra; i += static_cast<long long>(gridDim.x) * 256)
      j.dst_t[static_cast<long long>(j.ldd) * j.rows + i] = __float2bfloat16_rn(0.f);
  }
}

inline unsigned grid_for(long long work, int per_block = 256, int cap_mult = 16) {
  long long g = (work + per_block - 1) / per_block;
  const long long cap = static_cast<long long>(device_sm_count()) * cap_mult;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<unsigned>(g);
}

}  // namespace
}  // namespace dsg

using namespace dsg;

extern "C" {

int dsg_tr_ln_fwd(const float* x, const float* gamma, const float* beta, void* y_bf16, float* y_f32, long long M, int C,
                  dsg_stream_t stream) {
  DSG_REQUIRE(x && gamma && beta && (y_bf16 || y_f32) && M > 0 && C > 0 && C % 4 == 0 && C <= 2048, "tr_ln_fwd: bad argument (C <= 2048)");
  const unsigned grid = grid_for(M, 8 * 4, 8);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  bf16_t* y16 = static_cast<bf16_t*>(y_bf16);
  const int nvw = (C / 4 + 31) / 32;   // float4 groups per lane
  if (nvw <= 1) ln_fwd_kernel<1><<<grid, 256, 0, st>>>(x, gamma, beta, y16, y_f32, M, C);
  else if (nvw <= 2) ln_fwd_kernel<2><<<grid, 256, 0, st>>>(x, gamma, beta, y16, y_f32, M, C);
  else if (nvw <= 3) ln_fwd_kernel<3><<<grid, 256, 0, st>>>(x, gamma, beta, y16, y_f32, M, C);
  else if (nvw <= 6) ln_fwd_kernel<6><<<grid, 256, 0, st>>>(x, gamma, beta, y16, y_f32, M, C);
  else if (nvw <= 12) ln_fwd_kernel<12><<<grid, 256, 0, st>>>(x, gamma, beta, y16, y_f32, M, C);
  else ln_fwd_kernel<16><<<grid, 256, 0, st>>>(x, gamma, beta, y16, y_f32, M, C);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_ln_bwd(const float* dy, const float* x, const float* gamma, const float* dx_add, float* dx, float* dgamma,
                  float* dbeta, long long M, int C, dsg_stream_t stream) {
  DSG_REQUIRE(dy && x && gamma && dx && dgamma && dbeta && M > 0 && C > 0 && C % 4 == 0 && C <= 2048, "tr_ln_bwd: bad argument (C <= 2048)");
  const unsigned grid = grid_for(M, 8 * 16, 4);
  const size_t smem = 2 * C * sizeof(float);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int nvw = (C / 4 + 31) / 32;   // float4 groups per lane
  if (nvw <= 1) ln_bwd_kernel<1><<<grid, 256, smem, st>>>(dy, x, gamma, dx_add, dx, dgamma, dbeta, M, C);
  else if (nvw <= 2) ln_bwd_kernel<2><<<grid, 256, smem, st>>>(dy, x, gamma, dx_add, dx, dgamma, dbeta, M, C);
  else if (nvw <= 3) ln_bwd_kernel<3><<<grid, 256, smem, st>>>(dy, x, gamma, dx_add, dx, dgamma, dbeta, M, C);
  else if (nvw <= 6) ln_bwd_kernel<6><<<grid, 256, smem, st>>>(dy, x, gamma, dx_add, dx, dgamma, dbeta, M, C);
  else if (nvw <= 12) ln_bwd_kernel<12><<<grid, 256, smem, st>>>(dy, x, gamma, dx_add, dx, dgamma, dbeta, M, C);
  else ln_bwd_kernel<16><<<grid, 256, smem, st>>>(dy, x, gamma, dx_add, dx, dgamma, dbeta, M, C);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_film_silu_fwd(const float* v, const float* film, int ldf, int off, float* out, int B, int L, int C,
                         dsg_stream_t stream) {
  DSG_REQUIRE(v && film && out && B > 0 && L > 0 && C % 4 == 0 && off % 4 == 0 && ldf % 4 == 0, "tr_film_silu_fwd: bad argument");
  const int chunks = (L + kFilmTokens - 1) / kFilmTokens;
  film_silu_fwd_kernel<<<B * chunks, 256, 0, static_cast<cudaStream_t>(stream)>>>(v, film, ldf, off, out, L, C);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_film_silu_bwd(const float* dout, const float* v, const float* film, int ldf, int off, float* dv, float* dfilm,
                         int B, int L, int C, dsg_stream_t stream) {
  DSG_REQUIRE(dout && v && film && dv && dfilm && B > 0 && L > 0 && C % 4 == 0 && off % 4 == 0 && ldf % 4 == 0 && C <= 4096,
              "tr_film_silu_bwd: bad argument");
  const int chunks = (L + kFilmBwdTokens - 1) / kFilmBwdTokens;
  film_silu_bwd_kernel<<<B * chunks, 256, 2 * C * sizeof(float), static_cast<cudaStream_t>(stream)>>>(dout, v, film, ldf, off, dv, dfilm, L, C);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_gelu(const void* pre, const void* dh, void* out, long long n, dsg_stream_t stream) {
  DSG_REQUIRE(pre && out && n > 0 && n % 8 == 0 && ((reinterpret_cast<uintptr_t>(pre) | reinterpret_cast<uintptr_t>(out) |
                                                      reinterpret_cast<uintptr_t>(dh)) & 15) == 0,
              "tr_gelu: bad argument (n %% 8 == 0, 16-byte aligned tensors)");
  if (dh == nullptr)
    gelu_fwd_kernel<<<grid_for(n / 8, 512), 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const bf16_t*>(pre), static_cast<bf16_t*>(out), n / 8);
  else
    gelu_bwd_kernel<<<grid_for(n / 8, 512), 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const bf16_t*>(dh), static_cast<const bf16_t*>(pre), static_cast<bf16_t*>(out), n / 8);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_gelu_f32(const float* pre, const float* dout, float* out, long long n, dsg_stream_t stream) {
  DSG_REQUIRE(pre && out && n > 0, "tr_gelu_f32: bad argument");
  gelu_f32_kernel<<<grid_for(n), 256, 0, static_cast<cudaStream_t>(stream)>>>(pre, dout, out, n);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_colsum(const float* src, float* out, long long M, int C, dsg_stream_t stream) {
  DSG_REQUIRE(src && out && M > 0 && C > 0, "tr_colsum: bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (C <= 32) {
    const int rows = 32768 / C;    // ~32 k elements per CTA
    colsum_narrow_kernel<<<static_cast<unsigned>((M + rows - 1) / rows), 256, 256 * C * sizeof(float), st>>>(src, out, M, C, rows);
  } else {
    const int rows = 64;
    colsum_f32_kernel<<<dim3(static_cast<unsigned>((M + rows - 1) / rows), (C + 255) / 256), 256, 0, st>>>(src, out, M, C, rows);
  }
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_precond_coef(const float* sigmas, float* out, int B, dsg_stream_t stream) {
  DSG_REQUIRE(sigmas && out && B > 0, "tr_precond_coef: bad argument");
  precond_coef_kernel<<<(B + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(sigmas, out, B);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_silu(const float* pre, const float* dout, float* out, long long n, dsg_stream_t stream) {
  DSG_REQUIRE(pre && out && n > 0, "tr_silu: bad argument");
  if (dout == nullptr) silu_fwd_kernel<<<grid_for(n), 256, 0, static_cast<cudaStream_t>(stream)>>>(pre, out, n);
  else silu_bwd_kernel<<<grid_for(n), 256, 0, static_cast<cudaStream_t>(stream)>>>(dout, pre, out, n);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_add_inplace(float* y, const float* x, long long n, dsg_stream_t stream) {
  DSG_REQUIRE(y && x && n > 0 && n % 4 == 0, "tr_add_inplace: bad argument");
  add_inplace_kernel<<<grid_for(n / 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(y, x, n / 4);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_cast_colsum(const void* src, int src_is_bf16, void* cast, float* colsum, long long M, int C, int scale_cols,
                       float scale, dsg_stream_t stream) {
  DSG_REQUIRE(src && (cast || colsum) && M > 0 && C > 0 && C % 8 == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(cast) & 15) == 0, "tr_cast_colsum: bad argument (C %% 8 == 0, 16-byte aligned)");
  const dim3 grid((C + 255) / 256, static_cast<unsigned>((M + kCsRows - 1) / kCsRows));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (src_is_bf16)
    cast_colsum_kernel<bf16_t><<<grid, 256, 0, st>>>(static_cast<const bf16_t*>(src), static_cast<bf16_t*>(cast), colsum, M, C, scale_cols, scale);
  else
    cast_colsum_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(src), static_cast<bf16_t*>(cast), colsum, M, C, scale_cols, scale);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_wgrad(const void* dy, const void* x, float* dw, long long tokens, int n_out, int x_cols, int out_cols, int ksplit,
                 int scale_rows, float row_scale, dsg_stream_t stream) {
  return launch_wgrad(dy, x, dw, tokens, n_out, x_cols, out_cols, ksplit, scale_rows, row_scale, static_cast<cudaStream_t>(stream));
}

int dsg_tr_shuffle2x2(const float* src, float* dst, int B, int H, int W, int C, int to_coarse, dsg_stream_t stream) {
  DSG_REQUIRE(src && dst && B > 0 && H > 0 && W > 0 && C % 4 == 0, "tr_shuffle2x2: bad argument");
  shuffle2x2_kernel<<<grid_for(static_cast<long long>(B) * H * W * C), 256, 0, static_cast<cudaStream_t>(stream)>>>(src, dst, B, H, W, C, to_coarse);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_copy_cols(const float* src, int lds, int scol, void* dst, int ldd, int dcol, int ncols, long long M, int dst_bf16,
                     int accumulate, dsg_stream_t stream) {
  DSG_REQUIRE(src && dst && M > 0 && ncols > 0, "tr_copy_cols: bad argument");
  const bool vec = ((ncols | lds | ldd | scol | dcol) & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(dst) & 15) == 0;
  if (vec)
    copy_cols_kernel<true><<<grid_for(M * ncols / 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(src, lds, scol, dst, ldd, dcol, ncols, M, dst_bf16, accumulate);
  else
    copy_cols_kernel<false><<<grid_for(M * ncols), 256, 0, static_cast<cudaStream_t>(stream)>>>(src, lds, scol, dst, ldd, dcol, ncols, M, dst_bf16, accumulate);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_embed_input(const float* adj, const float* node, const float* sc_adj, const float* sc_node, const uint8_t* flags,
                       const float* c_in, void* out, int B, int n, int c_e, int c_n, int self_cond, int ld,
                       dsg_stream_t stream) {
  DSG_REQUIRE(adj && node && flags && out && (self_cond ? 2 : 1) * (c_e + 2 * c_n) <= ld, "tr_embed_input: bad argument");
  DSG_REQUIRE(ld % 8 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0, "tr_embed_input: ld %% 8 == 0, 16-byte aligned output");
  embed_input_kernel<<<grid_for(static_cast<long long>(B) * n * n * (ld / 8), 256, 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      adj, node, sc_adj, sc_node, flags, c_in, static_cast<bf16_t*>(out), B, n, c_e, c_n, self_cond, ld);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_adj_out(const float* in, const uint8_t* flags, const float* x_adj, const float* c_skip, const float* c_out,
                   float* out, int B, int n, int c_e, int backward, dsg_stream_t stream) {
  DSG_REQUIRE(in && flags && out, "tr_adj_out: bad argument");
  adj_out_kernel<<<grid_for(static_cast<long long>(B) * n * n), 256, 0, static_cast<cudaStream_t>(stream)>>>(in, flags, x_adj, c_skip, c_out, out, B, n, c_e, backward);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_node_out(const float* in, const uint8_t* flags, const float* x_node, const float* c_skip, const float* c_out,
                    float* out, int B, int n, int c_n, int backward, dsg_stream_t stream) {
  DSG_REQUIRE(in && flags && out, "tr_node_out: bad argument");
  node_out_kernel<<<grid_for(static_cast<long long>(B) * n * c_n), 256, 0, static_cast<cudaStream_t>(stream)>>>(in, flags, x_node, c_skip, c_out, out, B, n, c_n, backward);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_node_pool(const float* rep, const uint8_t* flags, float* pooled, const float* dpooled, float* drep, int B, int n,
                     int C, dsg_stream_t stream) {
  DSG_REQUIRE(flags && C % 4 == 0 && ((rep && pooled) || (dpooled && drep)), "tr_node_pool: bad argument");
  if (dpooled == nullptr)
    node_pool_train_kernel<<<static_cast<unsigned>((static_cast<long long>(B) * n + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(rep, flags, pooled, B, n, C);
  else
    node_pool_bwd_kernel<<<grid_for(static_cast<long long>(B) * n * n * C / 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(dpooled, flags, drep, B, n, C);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_adj_fc2(const void* h, const float* w, const float* b, float* tok, const float* dtok, float* dw, long long M, int E,
                   int ce, dsg_stream_t stream) {
  DSG_REQUIRE(h && M > 0 && E > 0 && E <= 128 && ce > 0 && ce <= 8 && ((w && b && tok) || (dtok && dw)), "tr_adj_fc2: bad argument (embed <= 128, c_e <= 8)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtok == nullptr) {
    adj_fc2_fwd_kernel<<<grid_for(M, 8 * 8, 8), 256, 0, st>>>(static_cast<const bf16_t*>(h), w, b, tok, M, E, ce);
  } else {
    const int rows = 4096;
    adj_fc2_wgrad_kernel<<<static_cast<unsigned>((M + rows - 1) / rows), 256, 0, st>>>(dtok, static_cast<const bf16_t*>(h), dw, M, E, ce, rows);
  }
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_posemb(const float* labels, float* out, int B, int embed, dsg_stream_t stream) {
  DSG_REQUIRE(labels && out && embed % 2 == 0, "tr_posemb: bad argument");
  posemb_kernel<<<(B * embed / 2 + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(labels, out, B, embed);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_bias_gather(const float* table, const int64_t* index, float* bias, int heads, int T, int backward, float* dtable,
                       dsg_stream_t stream) {
  DSG_REQUIRE(index && bias && (backward ? dtable != nullptr : table != nullptr), "tr_bias_gather: bad argument");
  bias_gather_kernel<<<(heads * T * T + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(table, index, bias, heads, T * T, backward, dtable);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_sgemm(const void* A, int a_is_bf16, long long sam, long long sak, const void* B, int b_is_bf16, long long sbk,
                 long long sbn, const float* bias, float* C, long long ldc, int M, int N, int K, int ksplit, int accumulate,
                 dsg_stream_t stream) {
  DSG_REQUIRE(A && B && C && M > 0 && N > 0 && K > 0 && ksplit >= 1, "tr_sgemm: bad argument");
  int k_per = (K + ksplit - 1) / ksplit;
  k_per = (k_per + 15) / 16 * 16;
  const int slices = (K + k_per - 1) / k_per;
  DSG_REQUIRE(slices == 1 || accumulate, "tr_sgemm: split-K accumulates (zero C first and pass accumulate = 1)");
  const dim3 grid((M + 63) / 64, (N + 63) / 64, slices);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (a_is_bf16 && b_is_bf16)
    sgemm_kernel<bf16_t, bf16_t><<<grid, 256, 0, st>>>(static_cast<const bf16_t*>(A), sam, sak, static_cast<const bf16_t*>(B), sbk, sbn, bias, C, ldc, M, N, K, k_per, accumulate);
  else if (a_is_bf16)
    sgemm_kernel<bf16_t, float><<<grid, 256, 0, st>>>(static_cast<const bf16_t*>(A), sam, sak, static_cast<const float*>(B), sbk, sbn, bias, C, ldc, M, N, K, k_per, accumulate);
  else if (b_is_bf16)
    sgemm_kernel<float, bf16_t><<<grid, 256, 0, st>>>(static_cast<const float*>(A), sam, sak, static_cast<const bf16_t*>(B), sbk, sbn, bias, C, ldc, M, N, K, k_per, accumulate);
  else
    sgemm_kernel<float, float><<<grid, 256, 0, st>>>(static_cast<const float*>(A), sam, sak, static_cast<const float*>(B), sbk, sbn, bias, C, ldc, M, N, K, k_per, accumulate);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_window_attention_bwd(const void* qkv, const void* datt, const float* bias, const float* mask, void* dqkv,
                                float* dbias, int batch, int res, int window, int shift, int heads, dsg_stream_t stream) {
  DSG_REQUIRE(qkv && datt && bias && dqkv && dbias && res % window == 0 && shift >= 0 && shift < window,
              "tr_window_attention_bwd: bad argument");
  DSG_REQUIRE(shift == 0 || mask != nullptr, "tr_window_attention_bwd: shifted windows need the attention mask");
  const int T = window * window;
  const int TP = (T + 15) & ~15, PF = TP <= 64 ? 84 : ((TP + 16 > 80) ? TP + 16 : 80);
  const size_t smem = static_cast<size_t>(4) * TP * kQP * 2 + static_cast<size_t>(2) * TP * PF * 4 + static_cast<size_t>(2) * T * T * 4 + static_cast<size_t>(TP) * 4;
  DSG_REQUIRE(smem <= 227 * 1024, "tr_window_attention_bwd: %d-token windows do not fit shared memory (T <= 100)", T);
  static PerDeviceOnce configured;
  if (configured.first()) {
    DSG_CUDA_CHECK(cudaFuncSetAttribute(window_attention_bwd_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DSG_CUDA_CHECK(cudaFuncSetAttribute(window_attention_bwd_tc_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DSG_CUDA_CHECK(cudaFuncSetAttribute(window_attention_bwd_tc_kernel<100>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  }
  const int total = batch * (res / window) * (res / window);
  // one atomicAdd pass over dbias per CTA: keep the CTA count near two waves
  const int resident = static_cast<int>((227 * 1024) / smem) > 0 ? static_cast<int>((227 * 1024) / smem) : 1;
  int ctas_x = (device_sm_count() * (resident > 4 ? 4 : resident) * 2 + heads - 1) / heads;
  if (ctas_x > total) ctas_x = total;
  const int per = (total + ctas_x - 1) / ctas_x;
  ctas_x = (total + per - 1) / per;
  if (T == 64)
    window_attention_bwd_tc_kernel<64><<<dim3(ctas_x, heads), 256, smem, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const bf16_t*>(qkv), static_cast<const bf16_t*>(datt), bias, mask, static_cast<bf16_t*>(dqkv), dbias, batch,
        res, window, shift, heads, per);
  else if (T == 100)   // the 10 x 10 windows of the COCO-Stuff geometry
    window_attention_bwd_tc_kernel<100><<<dim3(ctas_x, heads), 256, smem, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const bf16_t*>(qkv), static_cast<const bf16_t*>(datt), bias, mask, static_cast<bf16_t*>(dqkv), dbias, batch,
        res, window, shift, heads, per);
  else
    window_attention_bwd_tc_kernel<0><<<dim3(ctas_x, heads), 256, smem, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const bf16_t*>(qkv), static_cast<const bf16_t*>(datt), bias, mask, static_cast<bf16_t*>(dqkv), dbias, batch,
        res, window, shift, heads, per);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_sumsq(const float* g, long long n, float* out, dsg_stream_t stream) {
  DSG_REQUIRE(g && out && n > 0, "tr_sumsq: bad argument");
  DSG_CUDA_CHECK(cudaMemsetAsync(out, 0, 4, static_cast<cudaStream_t>(stream)));
  sumsq_kernel<<<grid_for(n, 256, 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(g, n, out);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_adam_ema(float* p, const float* g, float* m, float* v, long long n, const float* gsumsq, float lr, float beta1,
                    float beta2, float eps, float weight_decay, int step, float max_norm, int n_ema, float* const* ema,
                    const float* ema_decay, dsg_stream_t stream) {
  DSG_REQUIRE(p && n > 0 && step >= 1 && n_ema >= 0 && n_ema <= 8 && ((g && m && v) || (!m && !v && n_ema > 0)),
              "tr_adam_ema: bad argument");
  AdamArgs a;
  memset(&a, 0, sizeof(a));
  a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.weight_decay = weight_decay; a.max_norm = max_norm;
  a.bc1 = static_cast<float>(1.0 - pow(static_cast<double>(beta1), step));
  a.bc2_sqrt = static_cast<float>(sqrt(1.0 - pow(static_cast<double>(beta2), step)));
  a.n_ema = n_ema;
  for (int k = 0; k < n_ema; ++k) { a.ema[k] = ema[k]; a.ema_decay[k] = ema_decay[k]; }
  DSG_REQUIRE(n % 4 == 0 && (reinterpret_cast<uintptr_t>(p) & 15) == 0, "tr_adam_ema: the flat buffers are multiples of 4 floats, 16-byte aligned");
  adam_ema_kernel<<<grid_for(n / 4, 256, 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(p, g, m, v, n / 4, gsumsq, a);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_prep_weights(const void* jobs_device, int n_jobs, dsg_stream_t stream) {
  DSG_REQUIRE(jobs_device && n_jobs > 0, "tr_prep_weights: bad argument");
  prep_weights_kernel<<<dim3(64, n_jobs), 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const PrepJob*>(jobs_device));
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

int dsg_tr_prep_job_bytes(void) { return static_cast<int>(sizeof(PrepJob)); }

}  // extern "C"
