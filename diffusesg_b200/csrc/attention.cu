// Shifted-window multi-head self-attention over the N x N pair grid (head_dim = 32).
//
// One CTA per (sample, window, head).  The cyclic shift, window partition and window reverse of the
// reference (model/diffusesg/diffusesg.py:246-271, :28-57) never touch memory: they are index arithmetic
// on the token gather/scatter of this kernel.  softmax(q k^T + rel_pos_bias[h] (+ shift mask[window])) v
// restates WindowAttention.forward (:108-139); q arrives pre-scaled (the 32^-0.5 factor is folded into the
// packed qkv weights).  Scores, softmax statistics and the output accumulator are fp32; q/k/v/p are bf16
// tensor-core operands (warp-level mma.sync m16n8k16: each warp owns a 16-query slab; the window tile is
// far below the 128-row tcgen05 atom, see DESIGN.md).
#include "common.cuh"
#include "kernels.h"

namespace dsg {
namespace {

constexpr int HD = 32;        // head dim
constexpr int QK_PITCH = 40;  // bf16 per q/k smem row (80 B: conflict-free fragment loads)

template <int T_PAD>
__global__ void __launch_bounds__((T_PAD / 16) * 32)
window_attention_kernel(const bf16* __restrict__ qkv, const float* __restrict__ bias, const float* __restrict__ mask,
                        bf16* __restrict__ out, int res, int w, int shift, int heads) {
  constexpr int NWARP = T_PAD / 16;
  constexpr int VT_PITCH = T_PAD + 8;
  extern __shared__ __align__(16) uint8_t att_smem[];
  bf16* sQ = reinterpret_cast<bf16*>(att_smem);
  bf16* sK = sQ + T_PAD * QK_PITCH;
  bf16* sVt = sK + T_PAD * QK_PITCH;
  int* sRow = reinterpret_cast<int*>(sVt + HD * VT_PITCH);

  const int T = w * w;
  const int nwx = res / w;
  const int nW = nwx * nwx;
  int bid = blockIdx.x;
  const int h = bid % heads; bid /= heads;
  const int win = bid % nW;
  const int b = bid / nW;
  const int wy = win / nwx, wx = win % nwx;
  const int C = heads * HD;
  const int tid = threadIdx.x;

  for (int t = tid; t < T_PAD; t += NWARP * 32) {
    int row = -1;
    if (t < T) {
      const int ty = t / w, tx = t - ty * w;
      int oy = wy * w + ty + shift; if (oy >= res) oy -= res;
      int ox = wx * w + tx + shift; if (ox >= res) ox -= res;
      row = (b * res + oy) * res + ox;
    }
    sRow[t] = row;
  }
  __syncthreads();

  // gather q, k (row-major) and v (transposed) for this head; padded tokens are zero
  for (int idx = tid; idx < T_PAD * 12; idx += NWARP * 32) {
    const int t = idx / 12;
    const int rem = idx - t * 12;
    const int part = rem >> 2, chunk = rem & 3;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    const int row = sRow[t];
    if (row >= 0)
      v = __ldg(reinterpret_cast<const uint4*>(qkv + static_cast<size_t>(row) * (3 * C) + part * C + h * HD + chunk * 8));
    if (part == 0) {
      *reinterpret_cast<uint4*>(&sQ[t * QK_PITCH + chunk * 8]) = v;
    } else if (part == 1) {
      *reinterpret_cast<uint4*>(&sK[t * QK_PITCH + chunk * 8]) = v;
    } else {
      const bf16* e = reinterpret_cast<const bf16*>(&v);
#pragma unroll
      for (int i = 0; i < 8; ++i) sVt[(chunk * 8 + i) * VT_PITCH + t] = e[i];
    }
  }
  __syncthreads();

  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t4 = lane & 3;
  const int r0 = warp * 16 + g;  // this thread's two query rows: r0 and r0 + 8
  const int r1 = r0 + 8;

  uint32_t qa[2][4];
#pragma unroll
  for (int ks = 0; ks < 2; ++ks) {
    qa[ks][0] = *reinterpret_cast<const uint32_t*>(&sQ[r0 * QK_PITCH + ks * 16 + 2 * t4]);
    qa[ks][1] = *reinterpret_cast<const uint32_t*>(&sQ[r1 * QK_PITCH + ks * 16 + 2 * t4]);
    qa[ks][2] = *reinterpret_cast<const uint32_t*>(&sQ[r0 * QK_PITCH + ks * 16 + 2 * t4 + 8]);
    qa[ks][3] = *reinterpret_cast<const uint32_t*>(&sQ[r1 * QK_PITCH + ks * 16 + 2 * t4 + 8]);
  }

  const float* bias_h = bias + static_cast<size_t>(h) * T * T;
  const float* mask_w = mask ? mask + static_cast<size_t>(win) * T * T : nullptr;
  const bool ok0 = r0 < T, ok1 = r1 < T;

  float o[4][4];
#pragma unroll
  for (int nd = 0; nd < 4; ++nd)
#pragma unroll
    for (int i = 0; i < 4; ++i) o[nd][i] = 0.f;
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;

#pragma unroll
  for (int kc = 0; kc < T_PAD; kc += 64) {
    constexpr int NT_MAX = 8;
    float s[NT_MAX][4];
#pragma unroll
    for (int nt = 0; nt < NT_MAX; ++nt) {
      if (kc + nt * 8 < T_PAD) {
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
        const int key = kc + nt * 8 + g;
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
          uint32_t kb[2];
          kb[0] = *reinterpret_cast<const uint32_t*>(&sK[key * QK_PITCH + ks * 16 + 2 * t4]);
          kb[1] = *reinterpret_cast<const uint32_t*>(&sK[key * QK_PITCH + ks * 16 + 2 * t4 + 8]);
          mma_m16n8k16_bf16(s[nt], qa[ks], kb);
        }
        const int c = kc + nt * 8 + 2 * t4;  // columns c, c + 1 (T is even, so both are valid or both padded)
        if (c < T) {
          if (ok0) {
            const float2 bv = __ldg(reinterpret_cast<const float2*>(bias_h + static_cast<size_t>(r0) * T + c));
            s[nt][0] += bv.x; s[nt][1] += bv.y;
            if (mask_w) {
              const float2 mv = __ldg(reinterpret_cast<const float2*>(mask_w + static_cast<size_t>(r0) * T + c));
              s[nt][0] += mv.x; s[nt][1] += mv.y;
            }
          }
          if (ok1) {
            const float2 bv = __ldg(reinterpret_cast<const float2*>(bias_h + static_cast<size_t>(r1) * T + c));
            s[nt][2] += bv.x; s[nt][3] += bv.y;
            if (mask_w) {
              const float2 mv = __ldg(reinterpret_cast<const float2*>(mask_w + static_cast<size_t>(r1) * T + c));
              s[nt][2] += mv.x; s[nt][3] += mv.y;
            }
          }
        } else {
          s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = -INFINITY;
        }
      }
    }
    // online softmax over this chunk of keys
    float cm0 = -INFINITY, cm1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < NT_MAX; ++nt) {
      if (kc + nt * 8 < T_PAD) {
        cm0 = fmaxf(cm0, fmaxf(s[nt][0], s[nt][1]));
        cm1 = fmaxf(cm1, fmaxf(s[nt][2], s[nt][3]));
      }
    }
    cm0 = fmaxf(cm0, __shfl_xor_sync(0xffffffffu, cm0, 1));
    cm0 = fmaxf(cm0, __shfl_xor_sync(0xffffffffu, cm0, 2));
    cm1 = fmaxf(cm1, __shfl_xor_sync(0xffffffffu, cm1, 1));
    cm1 = fmaxf(cm1, __shfl_xor_sync(0xffffffffu, cm1, 2));
    const float nm0 = fmaxf(m0, cm0), nm1 = fmaxf(m1, cm1);  // finite: every chunk holds >= 1 real key
    const float f0 = ex2_approx((m0 - nm0) * 1.4426950408889634f), f1 = ex2_approx((m1 - nm1) * 1.4426950408889634f);
    m0 = nm0; m1 = nm1;
    l0 *= f0; l1 *= f1;
#pragma unroll
    for (int nd = 0; nd < 4; ++nd) {
      o[nd][0] *= f0; o[nd][1] *= f0; o[nd][2] *= f1; o[nd][3] *= f1;
    }
#pragma unroll
    for (int nt = 0; nt < NT_MAX; ++nt) {
      if (kc + nt * 8 < T_PAD) {
        s[nt][0] = ex2_approx((s[nt][0] - m0) * 1.4426950408889634f); s[nt][1] = ex2_approx((s[nt][1] - m0) * 1.4426950408889634f);
        s[nt][2] = ex2_approx((s[nt][2] - m1) * 1.4426950408889634f); s[nt][3] = ex2_approx((s[nt][3] - m1) * 1.4426950408889634f);
        l0 += s[nt][0] + s[nt][1];
        l1 += s[nt][2] + s[nt][3];
      }
    }
    // o += p . v  (p: bf16 A fragments straight from the score registers)
#pragma unroll
    for (int kt = 0; kt < NT_MAX / 2; ++kt) {
      if (kc + kt * 16 < T_PAD) {
        uint32_t pa[4];
        pa[0] = pack_bf16x2(s[2 * kt][0], s[2 * kt][1]);
        pa[1] = pack_bf16x2(s[2 * kt][2], s[2 * kt][3]);
        pa[2] = pack_bf16x2(s[2 * kt + 1][0], s[2 * kt + 1][1]);
        pa[3] = pack_bf16x2(s[2 * kt + 1][2], s[2 * kt + 1][3]);
        const int key = kc + kt * 16 + 2 * t4;
#pragma unroll
        for (int nd = 0; nd < 4; ++nd) {
          uint32_t vb[2];
          vb[0] = *reinterpret_cast<const uint32_t*>(&sVt[(nd * 8 + g) * VT_PITCH + key]);
          vb[1] = *reinterpret_cast<const uint32_t*>(&sVt[(nd * 8 + g) * VT_PITCH + key + 8]);
          mma_m16n8k16_bf16(o[nd], pa, vb);
        }
      }
    }
  }

  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.f / l0, i1 = 1.f / l1;
  if (ok0) {
    bf16* dst = out + static_cast<size_t>(sRow[r0]) * C + h * HD + 2 * t4;
#pragma unroll
    for (int nd = 0; nd < 4; ++nd)
      *reinterpret_cast<uint32_t*>(dst + nd * 8) = pack_bf16x2(o[nd][0] * i0, o[nd][1] * i0);
  }
  if (ok1) {
    bf16* dst = out + static_cast<size_t>(sRow[r1]) * C + h * HD + 2 * t4;
#pragma unroll
    for (int nd = 0; nd < 4; ++nd)
      *reinterpret_cast<uint32_t*>(dst + nd * 8) = pack_bf16x2(o[nd][2] * i1, o[nd][3] * i1);
  }
}


// ---------------------------------------------------------------------------------------------------------
// Fast path for 64-token windows (every block of the Visual Genome geometry).
//
// One CTA = 4 warps, one head, a run of kWPC consecutive windows.  The relative-position bias of the head sits in
// registers for the whole run (32 floats per thread: exactly the score fragment layout), q/k/v of the next
// window stream into the other shared-memory buffer with cp.async while the current one is computed, v is
// consumed row-major through ldmatrix.trans, and the output tile is staged through the (already consumed) q
// buffer so that every token receives one 64-byte store.
// ---------------------------------------------------------------------------------------------------------
constexpr int kWPC = 8;

DSG_DEVICE void cp_async16(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
DSG_DEVICE void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
DSG_DEVICE void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

DSG_DEVICE void ldmatrix_x4(uint32_t (&r)[4], const void* smem_row) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(smem_u32(smem_row)));
}
DSG_DEVICE void ldmatrix_x4_trans(uint32_t (&r)[4], const void* smem_row) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(smem_u32(smem_row)));
}

// Window gw = b * nW + wy * nwx + wx of the (rolled) grid: row of its token (0, 0) before wrapping, as (b, y0, x0).
struct WinOrigin { int b_row0, y0, x0; };
// (b, wy, wx) of a window, stepped to the next window without the run-time divisions of gw / nW, win / nwx, gw % nW
// (two cursors x five divisions were ~200 of the ~640 instructions a warp spends per window)
struct WinCursor {
  int b, wy, wx, win;
  DSG_DEVICE void init(int gw, int nW, int nwx) {
    b = gw / nW;
    win = gw - b * nW;
    wy = win / nwx;
    wx = win - wy * nwx;
  }
  DSG_DEVICE void next(int nW, int nwx) {
    ++win;
    if (++wx == nwx) {
      wx = 0;
      if (++wy == nwx) { wy = 0; win = 0; ++b; }
    }
  }
  DSG_DEVICE WinOrigin origin(int res, int shift) const { return WinOrigin{b * res * res, wy * 8 + shift, wx * 8 + shift}; }
};
// token t = ty * 8 + tx of the window -> row of the un-rolled [B*res*res] token matrix (cyclic shift undone)
DSG_DEVICE int window_token_row(const WinOrigin& o, int t, int res) {
  int oy = o.y0 + (t >> 3); if (oy >= res) oy -= res;
  int ox = o.x0 + (t & 7); if (ox >= res) ox -= res;
  return o.b_row0 + oy * res + ox;
}

__global__ void __launch_bounds__(128, 5)
window_attention64_kernel(const bf16* __restrict__ qkv, const float* __restrict__ bias, const float* __restrict__ mask,
                          bf16* __restrict__ out, int res, int shift, int heads, int total_windows) {
  constexpr int T = 64;
  __shared__ __align__(16) bf16 sbuf[2][3][T * QK_PITCH];  // [buffer][q, k, v][token][40]
  const int nwx = res >> 3;
  const int nW = nwx * nwx;
  const int h = blockIdx.x % heads;
  const int w_begin = (blockIdx.x / heads) * kWPC;
  const int w_end = min(total_windows, w_begin + kWPC);
  const int C = heads * HD;
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t4 = lane & 3;
  const int r0 = warp * 16 + g, r1 = r0 + 8;

  // two threads per token: thread `tid` fetches the 32-byte half `tid & 1` of the token's q, k and v head slices
  WinCursor cur_load, cur;
  cur_load.init(w_begin, nW, nwx);
  cur = cur_load;
  auto issue_loads = [&](int buf) {  // window of the load cursor, which then advances
    const WinOrigin org = cur_load.origin(res, shift);
    cur_load.next(nW, nwx);
    const int t = tid >> 1, half = (tid & 1) * 16;
    const bf16* src = qkv + static_cast<size_t>(window_token_row(org, t, res)) * (3 * C) + h * HD + half;
#pragma unroll
    for (int part = 0; part < 3; ++part) {
      cp_async16(&sbuf[buf][part][t * QK_PITCH + half], src + part * C);
      cp_async16(&sbuf[buf][part][t * QK_PITCH + half + 8], src + part * C + 8);
    }
    cp_async_commit();
  };

  issue_loads(0);

  // relative-position bias of this head, in score-fragment layout
  float bia[8][4];
  {
    const float* bh = bias + static_cast<size_t>(h) * T * T;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const float2 a = __ldg(reinterpret_cast<const float2*>(bh + r0 * T + nt * 8 + 2 * t4));
      const float2 b = __ldg(reinterpret_cast<const float2*>(bh + r1 * T + nt * 8 + 2 * t4));
      bia[nt][0] = a.x; bia[nt][1] = a.y; bia[nt][2] = b.x; bia[nt][3] = b.y;
    }
  }

  for (int gw = w_begin; gw < w_end; ++gw) {
    const int buf = (gw - w_begin) & 1;
    if (gw + 1 < w_end) {
      issue_loads(buf ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    bf16* sQ = sbuf[buf][0];
    const bf16* sK = sbuf[buf][1];
    const bf16* sV = sbuf[buf][2];

    // A fragments of this warp's 16 query rows: matrices (rows 0-7 | 8-15) x (dims 0-7 | 8-15) of each K step
    uint32_t qa[2][4];
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
      ldmatrix_x4(qa[ks], &sQ[(warp * 16 + (lane & 15)) * QK_PITCH + ks * 16 + ((lane >> 4) << 3)]);
    float s[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      s[nt][0] = bia[nt][0]; s[nt][1] = bia[nt][1]; s[nt][2] = bia[nt][2]; s[nt][3] = bia[nt][3];
      // B fragments of keys nt*8 .. +7: matrices = dims [0,8) [8,16) [16,24) [24,32) -> (ks 0: b0 b1) (ks 1: b0 b1)
      uint32_t kb[4];
      ldmatrix_x4(kb, &sK[(nt * 8 + (lane & 7)) * QK_PITCH + ((lane >> 3) << 3)]);
      mma_m16n8k16_bf16(s[nt], qa[0], reinterpret_cast<const uint32_t(&)[2]>(kb[0]));
      mma_m16n8k16_bf16(s[nt], qa[1], reinterpret_cast<const uint32_t(&)[2]>(kb[2]));
    }
    if (mask != nullptr) {
      const float* mw = mask + static_cast<size_t>(cur.win) * T * T;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const float2 a = __ldg(reinterpret_cast<const float2*>(mw + r0 * T + nt * 8 + 2 * t4));
        const float2 b = __ldg(reinterpret_cast<const float2*>(mw + r1 * T + nt * 8 + 2 * t4));
        s[nt][0] += a.x; s[nt][1] += a.y; s[nt][2] += b.x; s[nt][3] += b.y;
      }
    }
    float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      m0 = fmaxf(m0, fmaxf(s[nt][0], s[nt][1]));
      m1 = fmaxf(m1, fmaxf(s[nt][2], s[nt][3]));
    }
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
    float l0 = 0.f, l1 = 0.f;
    constexpr float kLog2e = 1.4426950408889634f;
    const float m0s = m0 * kLog2e, m1s = m1 * kLog2e;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      s[nt][0] = ex2_approx(fmaf(s[nt][0], kLog2e, -m0s)); s[nt][1] = ex2_approx(fmaf(s[nt][1], kLog2e, -m0s));
      s[nt][2] = ex2_approx(fmaf(s[nt][2], kLog2e, -m1s)); s[nt][3] = ex2_approx(fmaf(s[nt][3], kLog2e, -m1s));
      l0 += s[nt][0] + s[nt][1];
      l1 += s[nt][2] + s[nt][3];
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);

    float o[4][4];
#pragma unroll
    for (int nd = 0; nd < 4; ++nd) o[nd][0] = o[nd][1] = o[nd][2] = o[nd][3] = 0.f;
#pragma unroll
    for (int kt = 0; kt < 4; ++kt) {
      uint32_t pa[4];
      pa[0] = pack_bf16x2(s[2 * kt][0], s[2 * kt][1]);
      pa[1] = pack_bf16x2(s[2 * kt][2], s[2 * kt][3]);
      pa[2] = pack_bf16x2(s[2 * kt + 1][0], s[2 * kt + 1][1]);
      pa[3] = pack_bf16x2(s[2 * kt + 1][2], s[2 * kt + 1][3]);
      // lanes 0-7 / 8-15 address keys kt*16 + 0..7 / 8..15 at dims n0, lanes 16-31 the same keys at dims n0 + 8
      const int krow = kt * 16 + (lane & 15);
#pragma unroll
      for (int np = 0; np < 2; ++np) {
        uint32_t vb[4];
        ldmatrix_x4_trans(vb, &sV[krow * QK_PITCH + np * 16 + ((lane >> 4) << 3)]);
        mma_m16n8k16_bf16(o[2 * np], pa, reinterpret_cast<const uint32_t(&)[2]>(vb[0]));
        mma_m16n8k16_bf16(o[2 * np + 1], pa, reinterpret_cast<const uint32_t(&)[2]>(vb[2]));
      }
    }
    const float i0 = rcp_approx(l0), i1 = rcp_approx(l1);
    const WinOrigin org_out = cur.origin(res, shift);
    cur.next(nW, nwx);
    // stage the 16 x 32 output slab of this warp in its own (consumed) q rows, then one 64-byte store per token
    __syncwarp();
#pragma unroll
    for (int nd = 0; nd < 4; ++nd) {
      *reinterpret_cast<uint32_t*>(&sQ[r0 * QK_PITCH + nd * 8 + 2 * t4]) = pack_bf16x2(o[nd][0] * i0, o[nd][1] * i0);
      *reinterpret_cast<uint32_t*>(&sQ[r1 * QK_PITCH + nd * 8 + 2 * t4]) = pack_bf16x2(o[nd][2] * i1, o[nd][3] * i1);
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int idx = lane + 32 * k;  // 16 tokens x 4 chunks
      const int t = warp * 16 + (idx >> 2), chunk = idx & 3;
      const uint4 v = *reinterpret_cast<const uint4*>(&sQ[t * QK_PITCH + chunk * 8]);
      const int row = window_token_row(org_out, t, res);
      *reinterpret_cast<uint4*>(out + static_cast<size_t>(row) * C + h * HD + chunk * 8) = v;
    }
    __syncthreads();  // everyone is done with this buffer before the loads of window gw + 2 overwrite it
  }
}

template <int T_PAD>
int launch_t(const bf16* qkv, const float* bias, const float* mask, bf16* out, int batch, int res, int window,
             int shift, int heads, cudaStream_t st) {
  const int nW = (res / window) * (res / window);
  const long long grid = static_cast<long long>(batch) * nW * heads;
  DSG_REQUIRE(grid > 0 && grid < 2147483647LL, "attention: grid out of range");
  constexpr int smem = (2 * T_PAD * QK_PITCH + HD * (T_PAD + 8)) * 2 + T_PAD * 4;
  static PerDeviceOnce configured;
  if (configured.first()) {
    DSG_CUDA_CHECK(cudaFuncSetAttribute(window_attention_kernel<T_PAD>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  }
  window_attention_kernel<T_PAD><<<static_cast<unsigned>(grid), (T_PAD / 16) * 32, smem, st>>>(qkv, bias, mask, out, res,
                                                                                            window, shift, heads);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

}  // namespace

int launch_window_attention(const bf16* qkv, const float* bias, const float* mask, bf16* out, int batch, int res,
                            int window, int shift, int heads, cudaStream_t st, int mask_canonical) {
  DSG_REQUIRE(res % window == 0 && shift >= 0 && shift < window, "attention: res %d window %d shift %d", res, window,
              shift);
  DSG_REQUIRE((shift > 0) == (mask != nullptr), "attention: a shifted block needs its mask (and only it)");
  const int T = window * window;
  DSG_REQUIRE(T % 2 == 0, "attention: odd window token count %d", T);
  const bool mask_ok = shift == 0 || (mask_canonical & ATTN_MASK_CANONICAL) != 0;
  if (mask_ok && window_attention_tc_supported(batch, res, window, shift, heads))
    return launch_window_attention_tc(qkv, bias, out, batch, res, shift, heads, st);  // 8 x 8 windows, two per tile
  // one window per tile for the other even windows up to 10 x 10 (an 8 x 8 window would fill only half of the tile)
  if (window != 8 && mask_ok && window_attention_quad_supported(batch, res, window, shift, heads))
    return launch_window_attention_quad(qkv, bias, out, batch, res, window, shift, heads, st);
  if (mask_ok && (mask_canonical & ATTN_BIAS_TOEPLITZ) != 0 &&
      window_attention_w16_supported(batch, res, window, shift, heads))
    return launch_window_attention_w16(qkv, bias, out, batch, res, shift, heads, st);  // 16 x 16 windows
  if (window == 8) {
    const long long total = static_cast<long long>(batch) * (res / 8) * (res / 8);
    const long long grid = ((total + kWPC - 1) / kWPC) * heads;
    DSG_REQUIRE(grid > 0 && grid < 2147483647LL, "attention: grid out of range");
    window_attention64_kernel<<<static_cast<unsigned>(grid), 128, 0, st>>>(qkv, bias, mask, out, res, shift, heads,
                                                                         static_cast<int>(total));
    DSG_LAUNCH_CHECK();
    return DSG_OK;
  }
  if (T <= 16) return launch_t<16>(qkv, bias, mask, out, batch, res, window, shift, heads, st);
  if (T <= 64) return launch_t<64>(qkv, bias, mask, out, batch, res, window, shift, heads, st);
  if (T <= 112) return launch_t<112>(qkv, bias, mask, out, batch, res, window, shift, heads, st);
  if (T <= 256) return launch_t<256>(qkv, bias, mask, out, batch, res, window, shift, heads, st);
  set_last_error("attention: windows of %d tokens are not supported (max 256)", T);
  return DSG_ERR_INVALID;
}

}  // namespace dsg
