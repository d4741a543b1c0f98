// Fused attention projection + residual + LayerNorm2 for the C = 192 / 384 Swin blocks:
//     x += att . W_proj^T + b_proj          (model/diffusesg/diffusesg.py:137, :272 of the reference)
//     y  = LayerNorm(x) * gamma + beta       (:275, the input of the MLP), bf16
// It replaces the proj GEMM (TMA reduce-add epilogue) followed by the LayerNorm row kernel, which read x a second time
// (4 of the LayerNorm's 6 B / element) - both are HBM-bound, so the fused kernel's traffic is what it saves.
// Measured on the B200: 126 us against 87 + 60 us at C = 384 (4.8 TB/s), 281 against 178 + 105 us at C = 192 (the
// epilogue warps do not hide the latency of the chunk pipeline there) - the denoiser schedule takes it for C = 384 only.
//
// One persistent CTA per SM walks 128-row tiles and owns FULL rows (N = C columns of tensor memory, one accumulator:
// the kernel is HBM-bound at ~1.5 KB of x traffic per row, so nothing is lost by not double buffering it):
//   warps 0..11 epilogue, thread = row: group g = warp / 4 owns the column slice [g C / 3, (g + 1) C / 3) of the
//               tile's 128 rows
//   next warp   TMA producer: A box [128 x 64] + W boxes [192 x 64] per stage, one box per lane
//   last warp   MMA issuer:   N = C as one (C = 192) or two (C = 384) tcgen05.mma of N = 192 per K step
//       pass 1: x_new = acc + b + x, stored back to global memory, row sums in registers (pivot-shifted); the
//               accumulator is released here, so the next tile's MMA phase runs under the rest of the epilogue;
//               the column slices of a row exchange (sum, sum of squares, pivot)
//       pass 2: every lane re-reads the x_new values it stored itself (L2 hits) -> normalise -> bf16 -> global memory
//   Global memory is accessed COALESCED (a warp instruction covers 4 rows x 128 B of a 32 x 32 chunk; the next chunk
//   of x is prefetched into registers) and transposed to / from the thread = row layout of tensor memory through a
//   private 32 x 36-float tile per warp (only __syncwarp): one thread reading its own 128 B per row costs the LSU 32
//   line look-ups per instruction and ran the kernel at 2.4 TB/s.
#include "common.cuh"
#include "kernels.h"

namespace dsg {
namespace {

constexpr float kPlEps = 1e-5f;  // nn.LayerNorm default

template <int C>
struct PlCfg {
  static constexpr int NB = C / 192;                      // W boxes / MMAs per K step
  static constexpr int B_STAGE = C * 64 * 2;              // W k-block: [C x 64] bf16
  static constexpr int STAGE = 16384 + B_STAGE;
  static constexpr int kStages = (C == 384) ? 2 : 4;
  static constexpr int TILE_BYTES = 32 * 36 * 4;          // per-warp transpose tile
  // epilogue groups (4 warps each) = column slices of a row.  Measured at C = 384: two groups 140 us, three 126 us,
  // four 172 us (the 576-thread CTA is capped at 96 registers and spills)
  static constexpr int NG = 3;
  static constexpr int THREADS = (4 * NG + 2) * 32;
  static constexpr int H = C / NG;                        // columns per epilogue group
  static constexpr int NCH = H / 32;                      // 32-column chunks per group
  static constexpr int PAR_FLOATS = 3 * C;                // bias, gamma, beta
  static constexpr int SMEM_BYTES = 1024 + kStages * STAGE + PAR_FLOATS * 4 + NG * 128 * 16 + 4 * NG * TILE_BYTES + 256;
  static_assert(C == 192 || C == 384, "proj_ln: C = 192 / 384");
  static_assert(SMEM_BYTES <= 227 * 1024, "proj_ln: shared memory budget");
};

struct PlParams {
  const float* bias;   // [C]
  const float* gamma;  // [C]
  const float* beta;   // [C]
  float* x;            // [M, C] fp32 residual stream, updated in place
  bf16* y;             // [M, C] bf16 LayerNorm output
  int M;
};

template <int C>
__global__ void __launch_bounds__(PlCfg<C>::THREADS, 1)
proj_ln_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, const PlParams p) {
  using G = PlCfg<C>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sA = smem;                                  // [stages][128 x 64] bf16, 128-byte swizzle
  uint8_t* sB = smem + G::kStages * 16384;             // [stages][C x 64]
  float* sBias = reinterpret_cast<float*>(smem + G::kStages * G::STAGE);
  float* sGam = sBias + C;
  float* sBet = sGam + C;
  float4* sEx = reinterpret_cast<float4*>(sBet + C);   // [groups][128 rows]: (sum, sum of squares, pivot, -)
  float* sTile = reinterpret_cast<float*>(sEx + G::NG * 128);  // [4 NG warps][32][36]
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sTile + 4 * G::NG * 32 * 36);
  uint64_t* empty_bar = full_bar + G::kStages;
  uint64_t* tfull_bar = empty_bar + G::kStages;
  uint64_t* tempty_bar = tfull_bar + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 1);

  const int warp = uniform_warp_id();
  const int lane = threadIdx.x & 31;
  constexpr int kTmaWarp = 4 * G::NG, kMmaWarp = kTmaWarp + 1;
  const int num_tiles = (p.M + 127) / 128;
  constexpr int num_kb = C / 64;

  if (warp == kTmaWarp && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
    for (int s = 0; s < G::kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(tfull_bar, 1);
    mbar_init(tempty_bar, 4 * G::NG);
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc<512>(tmem_slot);
  for (int i = threadIdx.x; i < C; i += G::THREADS) { sBias[i] = p.bias[i]; sGam[i] = p.gamma[i]; sBet[i] = p.beta[i]; }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);

  if (warp == kTmaWarp) {
    // ------------------------------------------------------------------ TMA producer (one box per lane)
    int s = 0;
    uint32_t ph = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty_bar[s], ph ^ 1);
        if (lane == 0) mbar_expect_tx(&full_bar[s], G::STAGE);
        __syncwarp();
        if (lane == 0) tma_load_2d(sA + s * 16384, &tmA, &full_bar[s], kb * 64, tile * 128);
        else if (lane <= G::NB) tma_load_2d(sB + s * G::B_STAGE + (lane - 1) * 24576, &tmW, &full_bar[s], kb * 64, (lane - 1) * 192);
        __syncwarp();
        if (++s == G::kStages) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc = umma_idesc_bf16(192);
    int s = 0;
    uint32_t ph = 0, acc_ph = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      mbar_wait(tempty_bar, acc_ph ^ 1);
      tcgen05_fence_after();
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full_bar[s], ph);
        tcgen05_fence_after();
        if (elect_one()) {
          const uint64_t da = umma_desc_sw128(smem_u32(sA + s * 16384));
#pragma unroll
          for (int nb = 0; nb < G::NB; ++nb) {
            const uint64_t db = umma_desc_sw128(smem_u32(sB + s * G::B_STAGE + nb * 24576));
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16_ss(tmem_base + nb * 192, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
          }
          umma_commit(&empty_bar[s]);
          if (kb == num_kb - 1) umma_commit(tfull_bar);
        }
        __syncwarp();
        if (++s == G::kStages) { s = 0; ph ^= 1; }
      }
      acc_ph ^= 1;
    }
  } else {
    // ------------------------------------------------------------------ epilogue: thread = row, group = column half
    const int g = warp >> 2, q = warp & 3;
    const int r = q * 32 + lane;
    const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + g * G::H;
    const int col0 = g * G::H;
    float* sT = sTile + warp * 32 * 36;
    // coalesced layout of a [32 rows x 32 cols] fp32 chunk: instruction i covers rows 4 i .. 4 i + 3, this lane the
    // 16 bytes at column 4 (lane & 7) of row 4 i + (lane >> 3)
    const int crow = lane >> 3, ccol = 4 * (lane & 7);
    uint32_t acc_ph = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const long long row0 = static_cast<long long>(tile) * 128 + q * 32;   // first row of this warp
      float* xw = p.x + row0 * C + col0 + ccol;                              // + (4 i + crow) C + 32 c
      auto load_chunk = [&](float4 (&dst)[8], int c) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int rr = 4 * i + crow;
          dst[i] = (row0 + rr < p.M) ? *reinterpret_cast<const float4*>(xw + static_cast<long long>(rr) * C + 32 * c)
                                     : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      };
      float4 xn[8];
      load_chunk(xn, 0);  // on its way before the accumulator is complete
      mbar_wait(tfull_bar, acc_ph);
      tcgen05_fence_after();
      float pivot = 0.f;
      f32x2 s1 = f2_splat(0.f), s2 = f2_splat(0.f), npiv = f2_splat(0.f);
#pragma unroll 1
      for (int c = 0; c < G::NCH; ++c) {
        uint32_t v[32];
        tmem_ld_32x32(t_row + 32 * c, v);
        // x chunk: coalesced registers -> tile -> this thread's row
#pragma unroll
        for (int i = 0; i < 8; ++i) *reinterpret_cast<float4*>(&sT[(4 * i + crow) * 36 + ccol]) = xn[i];
        if (c + 1 < G::NCH) load_chunk(xn, c + 1);
        __syncwarp();
        float4 xr[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) xr[i] = *reinterpret_cast<const float4*>(&sT[lane * 36 + 4 * i]);
        __syncwarp();
        tmem_ld_wait();
        if (c == G::NCH - 1) {  // the accumulator is drained: the MMA of the next tile runs under the second pass
          tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(tempty_bar);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 bb = *reinterpret_cast<const float4*>(&sBias[col0 + 32 * c + 4 * i]);
          // same order as the reference: (acc + bias) is the Linear output, then the residual add
          float4 o;
          o.x = (__uint_as_float(v[4 * i]) + bb.x) + xr[i].x;
          o.y = (__uint_as_float(v[4 * i + 1]) + bb.y) + xr[i].y;
          o.z = (__uint_as_float(v[4 * i + 2]) + bb.z) + xr[i].z;
          o.w = (__uint_as_float(v[4 * i + 3]) + bb.w) + xr[i].w;
          if (c == 0 && i == 0) { pivot = o.x; npiv = f2_splat(-pivot); }
          const f32x2 d0 = f2_add(f2_pack(o.x, o.y), npiv), d1 = f2_add(f2_pack(o.z, o.w), npiv);
          s1 = f2_add(s1, f2_add(d0, d1));
          s2 = f2_fma(d0, d0, f2_fma(d1, d1, s2));
          *reinterpret_cast<float4*>(&sT[lane * 36 + 4 * i]) = o;
        }
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 8; ++i) {       // x_new: tile -> coalesced stores
          const int rr = 4 * i + crow;
          const float4 o = *reinterpret_cast<const float4*>(&sT[rr * 36 + ccol]);
          if (row0 + rr < p.M) *reinterpret_cast<float4*>(xw + static_cast<long long>(rr) * C + 32 * c) = o;
        }
        __syncwarp();
      }
      // ---- row statistics over all column slices (each slice has its own pivot)
      {
        float a0, a1, b0, b1;
        f2_unpack(s1, a0, a1);
        f2_unpack(s2, b0, b1);
        sEx[g * 128 + r] = make_float4(a0 + a1, b0 + b1, pivot, 0.f);
      }
      asm volatile("bar.sync 1, %0;" ::"n"(128 * G::NG) : "memory");
      float mean, rstd;
      {
        const float4 me = sEx[g * 128 + r];
        float t1 = me.x, t2 = me.y;
#pragma unroll
        for (int o = 1; o < G::NG; ++o) {
          // re-centre the other slice's sums on this slice's pivot: sum(x - p) = S1 + n d, sum((x - p)^2) = S2 + 2 d S1 + n d^2
          const float4 ot = sEx[((g + o) % G::NG) * 128 + r];
          const float d = ot.z - me.z, n = static_cast<float>(G::H);
          t1 += ot.x + n * d;
          t2 += ot.y + 2.f * d * ot.x + n * d * d;
        }
        const float dm = t1 * (1.0f / C);
        const float var = fmaxf(t2 * (1.0f / C) - dm * dm, 0.f);
        mean = me.z + dm;
        rstd = rsqrtf(var + kPlEps);
      }
      asm volatile("bar.sync 1, %0;" ::"n"(128 * G::NG) : "memory");  // sEx may be rewritten by the next tile
      // ---- pass 2, in the coalesced layout: every lane re-reads the x_new values it stored itself in pass 1 (L2 hits),
      //      normalises them with the statistics of their rows and stores bf16 (a warp instruction = 4 rows x 64 B)
      float2* sStat = reinterpret_cast<float2*>(sT);   // this warp's tile: [32 rows] (mean, rstd)
      sStat[lane] = make_float2(mean, rstd);
      __syncwarp();
      float2 st[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) st[i] = sStat[4 * i + crow];
      __syncwarp();                                    // the tile is the transpose buffer again from the next tile on
      bf16* yw = p.y + row0 * C + col0 + ccol;
#pragma unroll 1
      for (int c = 0; c < G::NCH; ++c) {
        float4 xv[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int rr = 4 * i + crow;
          xv[i] = (row0 + rr < p.M) ? *reinterpret_cast<const float4*>(xw + static_cast<long long>(rr) * C + 32 * c)
                                    : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        const float4 gg = *reinterpret_cast<const float4*>(&sGam[col0 + 32 * c + ccol]);
        const float4 be = *reinterpret_cast<const float4*>(&sBet[col0 + 32 * c + ccol]);
        const f32x2 g01 = f2_pack(gg.x, gg.y), g23 = f2_pack(gg.z, gg.w), b01 = f2_pack(be.x, be.y), b23 = f2_pack(be.z, be.w);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int rr = 4 * i + crow;
          const f32x2 rs2 = f2_splat(st[i].y), nmr = f2_splat(-st[i].x * st[i].y);
          uint2 o;
          o.x = pack_bf16x2(f2_fma(f2_fma(f2_pack(xv[i].x, xv[i].y), rs2, nmr), g01, b01));
          o.y = pack_bf16x2(f2_fma(f2_fma(f2_pack(xv[i].z, xv[i].w), rs2, nmr), g23, b23));
          if (row0 + rr < p.M) *reinterpret_cast<uint2*>(yw + static_cast<long long>(rr) * C + 32 * c) = o;
        }
      }
      acc_ph ^= 1;
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  if (warp == kMmaWarp) tmem_dealloc<512>(tmem_base);
}

template <int C>
int launch_c(const CUtensorMap* tmA, const CUtensorMap* tmW, const PlParams& p, cudaStream_t st) {
  static PerDeviceOnce configured;
  if (configured.first()) {
    DSG_CUDA_CHECK(cudaFuncSetAttribute(proj_ln_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, PlCfg<C>::SMEM_BYTES));
  }
  const int sms = device_sm_count();
  const int tiles = (p.M + 127) / 128;
  proj_ln_kernel<C><<<tiles < sms ? tiles : sms, PlCfg<C>::THREADS, PlCfg<C>::SMEM_BYTES, st>>>(*tmA, *tmW, p);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

}  // namespace

bool proj_ln_supported(int C) { return C == 192 || C == 384; }

int launch_proj_ln(const CUtensorMap* tmA, const CUtensorMap* tmW, const float* bias, const float* gamma, const float* beta,
                   float* x, bf16* y, long long rows, int C, cudaStream_t st) {
  DSG_REQUIRE(proj_ln_supported(C) && rows > 0 && rows < 2147483647LL, "proj_ln: C=%d rows=%lld", C, rows);
  DSG_REQUIRE(x != nullptr && y != nullptr && bias != nullptr && gamma != nullptr && beta != nullptr, "proj_ln: null tensor");
  PlParams p{bias, gamma, beta, x, y, static_cast<int>(rows)};
  return C == 192 ? launch_c<192>(tmA, tmW, p, st) : launch_c<384>(tmA, tmW, p, st);
}

}  // namespace dsg
