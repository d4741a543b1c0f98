// Fused transformer MLP for sm_100a:   x += fc2(gelu(fc1(y))),  y = LayerNorm(x) in bf16   (one kernel per Swin block)
//
// Restates `x = x + self.mlp(self.norm2(x))` (model/diffusesg/diffusesg.py:275 with Mlp.forward :19-25) of the
// reference.  Unfused this is two GEMMs whose 4C-wide hidden activation makes two round trips through HBM
// (16 C bytes per token); here the hidden activation never leaves the SM.
//
// The hidden dimension is cut into chunks of HC columns that form ONE stream across the tiles of a persistent CTA
// (global chunk index g): fc1 of chunk g + 2 is issued right after fc2 of chunk g, also across a tile boundary, so
// the tensor pipe never waits for the workers and the workers never wait for the tensor pipe.
//   TMA warp           y tile [128 x C] (once per tile) and the W1 / W2 k-blocks of every chunk (5-stage ring)
//   MMA warp           acc1[g&1] = y . W1[chunk]^T  (SS mode, TMEM accumulators double buffered);
//                      acc2 += H[chunk] . W2[:, chunk]^T  (TS mode: the A operand H is read from tensor memory)
//   worker warps (16)  tcgen05.ld acc1 -> + b1 -> erf GELU -> bf16 pairs -> tcgen05.st IN PLACE over acc1 (the 16
//                      hidden columns of K step k become the 8 packed columns [16k, 16k + 8), same warp);
//                      after the last chunk of a tile: tcgen05.ld acc2 -> + b2 -> fp32 staging -> TMA reduce-add into x
// fc1 of chunk g + 2 reuses the buffer of chunk g and is issued after fc2 of chunk g by the same thread; the tensor
// pipe executes in issue order, so the chunk ring needs no "empty" barriers.  Keeping H out of shared memory frees
// 64 KB for the weight ring: with 3 stages (0.6 chunk of look-ahead) every chunk waited ~2.5 k cycles for an L2 round
// trip of its weights (430 us per launch at C = 192); 5 stages hold a whole chunk.
#include "common.cuh"
#include "kernels.h"

namespace dsg {
namespace {

constexpr int kMlpThreads = 64 + 16 * 32;  // TMA warp, MMA warp, 16 worker warps
constexpr int kWorkers = 16 * 32;

template <int C>
struct MlpCfg {
  static constexpr int HID = 4 * C;
  static constexpr int HC = 128;                        // hidden columns per chunk
  static constexpr int NCH = HID / HC;                  // 3 / 6 chunks per tile
  static constexpr int KB1 = (C + 63) / 64;             // k-blocks of fc1 (K = C)
  static constexpr int KB2 = HC / 64;                   // k-blocks of fc2 per chunk (K = HC)
  static constexpr int A_BYTES = KB1 * 16384;           // y tile, [128 x 64] bf16 per k-block
  static constexpr int H_BYTES = KB2 * 16384;
  static constexpr int STAGE_BYTES = ((HC > C) ? HC : C) * 128;  // one weight k-block: [rows x 64] bf16
  // C = 96: two y-tile buffers (the HBM latency of the next tile's y is off the critical path), 5 x 16 KB weight
  // stages (a chunk is 2 W1 + 2 W2 k-blocks, all L2 hits), two acc2 buffers so that the output of tile t runs one
  // chunk into tile t + 1, and three staging buffers: one TMA reduce per 32-column output chunk.  C = 192 does
  // not have the TMEM / smem for that.
  static constexpr bool kDefer = (C == 96);
  static constexpr int kABufs = 1;                      // y tile buffers (2 = the next tile is fetched a whole tile ahead)
  static constexpr int kStages = (C == 96) ? 6 : 5;     // weight ring: one chunk (4 / 5 k-blocks) of look-ahead
  static constexpr int kAcc2 = kDefer ? 2 : 1;
  static constexpr int kOutGroups = (C == 96) ? 3 : 2;  // column groups that write the tile output
  static constexpr int STG_BYTES = kOutGroups * 16384;  // fp32 output staging, [128 x 32] per group
  static constexpr int PAR_FLOATS = HID;                // b1
  static constexpr int SMEM_BYTES = 1024 + kABufs * A_BYTES + kStages * STAGE_BYTES + STG_BYTES + PAR_FLOATS * 4 + 256;
  static constexpr int ACC2_COL = 2 * HC;               // TMEM: acc1[0] @0, acc1[1] @HC, acc2[u] @2HC + u C
  static constexpr int CQ = HC / 4;                     // GELU columns per warp: 32
  static_assert(ACC2_COL + kAcc2 * C <= 512 && SMEM_BYTES <= 227 * 1024, "fused MLP budget");
};

struct MlpParams {
  const float* b1;   // [4C]
  const float* b2;   // [C]
  int M;
};

// byte offset of the 16-byte chunk holding elements [k, k + 8) of row r in a K-major 128-byte-swizzled operand
// made of [128 rows x 64 bf16] k-blocks (what TMA SWIZZLE_128B writes and the UMMA descriptor reads)
DSG_DEVICE uint32_t sw128_offset(int r, int k) {
  return static_cast<uint32_t>((k >> 6) * 16384 + r * 128 + ((((k & 63) >> 3) ^ (r & 7)) << 4));
}

// D[tmem] (+)= A[tmem: lane = row, one 32-bit column per pair of K elements] . B[smem descriptor]^T
DSG_DEVICE void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
DSG_DEVICE void tmem_st_32x8(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
DSG_DEVICE void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

template <int C>
// 18 warps -> 5 on the fullest SM sub-partition (16K registers each): at most 96 registers per thread
__global__ void __launch_bounds__(kMlpThreads, 1)
fused_mlp_kernel(const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmW1,
                 const __grid_constant__ CUtensorMap tmW2, const __grid_constant__ CUtensorMap tmX, const MlpParams p) {
  using G = MlpCfg<C>;
  extern __shared__ uint8_t smem_raw[];
  // round up to 1024 bytes (128-byte swizzle atoms) without casting through an integer, so that the compiler
  // keeps the shared address space and emits LDS / STS instead of generic loads and stores
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sA = smem;
  uint8_t* sW = sA + G::kABufs * G::A_BYTES;
  uint8_t* sStg = sW + G::kStages * G::STAGE_BYTES;
  float* sPar = reinterpret_cast<float*>(sStg + G::STG_BYTES);
  float* sB1 = sPar;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sPar + G::PAR_FLOATS);
  uint64_t* w_full = bars;                    // [kStages]
  uint64_t* w_empty = bars + G::kStages;      // [kStages]
  uint64_t* a_full = bars + 2 * G::kStages;   // [2] TMA -> MMA: y tile landed
  uint64_t* a_empty = a_full + 2;             // [2] MMA -> TMA: every fc1 MMA of the tile has read its sA buffer
  uint64_t* acc1_full = a_full + 4;           // [2]
  uint64_t* h_full = a_full + 8;              // [2]
  uint64_t* acc2_full = a_full + 12;          // [2]
  uint64_t* acc2_empty = a_full + 14;         // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_full + 16);

  const int warp = uniform_warp_id();
  const int lane = threadIdx.x & 31;
  // the scheduler favours the highest warp id among ready warps: the control warps take the last two ids so that
  // the 16 ALU-heavy workers (warps 0..15) cannot starve them
  constexpr int kTmaWarp = 16, kMmaWarp = 17;
  const int num_tiles = (p.M + 127) / 128;

  if (warp == kTmaWarp && lane == 0) {
    tma_prefetch_desc(&tmY);
    tma_prefetch_desc(&tmW1);
    tma_prefetch_desc(&tmW2);
    tma_prefetch_desc(&tmX);
    for (int s = 0; s < G::kStages; ++s) { mbar_init(&w_full[s], 1); mbar_init(&w_empty[s], 1); }
    for (int u = 0; u < 2; ++u) { mbar_init(&a_full[u], 1); mbar_init(&a_empty[u], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&acc1_full[b], 1); mbar_init(&h_full[b], 16); }
    for (int u = 0; u < 2; ++u) { mbar_init(&acc2_full[u], 1); mbar_init(&acc2_empty[u], 4 * G::kOutGroups); }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc<512>(tmem_slot);
  for (int i = threadIdx.x; i < G::HID; i += kMlpThreads) sB1[i] = p.b1[i];
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);
  const int my_tiles = (num_tiles > static_cast<int>(blockIdx.x)) ? (num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const int n_chunks = my_tiles * G::NCH;  // global chunk stream of this CTA

  if (warp == kTmaWarp) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      int s = 0;
      uint32_t ph = 0, n_y[2] = {0, 0};
      int y_loaded = 0;  // local tiles whose y load has been issued
      auto load_y = [&](int tl) {  // y tile of local tile tl -> sA[tl % kABufs]
        const int u = tl % G::kABufs;
        const int tile = blockIdx.x + tl * gridDim.x;
        mbar_wait(&a_empty[u], (n_y[u] & 1) ^ 1);  // every fc1 MMA of the tile that last used this buffer completed
        ++n_y[u];
        mbar_expect_tx(&a_full[u], G::A_BYTES);
        for (int kb = 0; kb < G::KB1; ++kb)
          tma_load_2d(sA + u * G::A_BYTES + kb * 16384, &tmY, &a_full[u], kb * 64, tile * 128);
      };
      auto load_fc1 = [&](int g) {  // operands of fc1 of chunk g: (y tiles, kept kABufs - 1 tiles ahead,) W1[chunk]
        const int j = g % G::NCH;
        if (j == 0) {
          const int tl = g / G::NCH;
          while (y_loaded < my_tiles && y_loaded < tl + G::kABufs) load_y(y_loaded++);
        }
        for (int kb = 0; kb < G::KB1; ++kb) {
          mbar_wait(&w_empty[s], ph ^ 1);
          mbar_expect_tx(&w_full[s], G::HC * 128);
          tma_load_2d(sW + s * G::STAGE_BYTES, &tmW1, &w_full[s], kb * 64, j * G::HC);
          if (++s == G::kStages) { s = 0; ph ^= 1; }
        }
      };
      auto load_w2 = [&](int g) {
        const int j = g % G::NCH;
        for (int kb = 0; kb < G::KB2; ++kb) {
          mbar_wait(&w_empty[s], ph ^ 1);
          mbar_expect_tx(&w_full[s], C * 128);
          tma_load_2d(sW + s * G::STAGE_BYTES, &tmW2, &w_full[s], j * G::HC + kb * 64, 0);
          if (++s == G::kStages) { s = 0; ph ^= 1; }
        }
      };
      if (n_chunks > 0) load_fc1(0);
      if (n_chunks > 1) load_fc1(1);
      for (int g = 0; g < n_chunks; ++g) {
        load_w2(g);
        if (g + 2 < n_chunks) load_fc1(g + 2);
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc1 = umma_idesc_bf16(G::HC);
    constexpr uint32_t idesc2 = umma_idesc_bf16(C);
    int s = 0;
    uint32_t ph = 0;
    uint32_t n_a[2] = {0, 0}, n_h[2] = {0, 0}, n_acc2[2] = {0, 0};  // use counters -> parities
    auto fc1 = [&](int g) {  // acc1[g & 1] = y . W1[chunk]^T
      const int b = g & 1, j = g % G::NCH;
      const int ua = (g / G::NCH) % G::kABufs;  // y buffer of this tile
      if (j == 0) {
        mbar_wait(&a_full[ua], n_a[ua] & 1);
        ++n_a[ua];
      }
      // (acc1[b] last held chunk g - 2, whose fc2 was issued before this call: the tensor pipe runs in issue order)
      tcgen05_fence_after();
      for (int kb = 0; kb < G::KB1; ++kb) {
        mbar_wait(&w_full[s], ph);
        tcgen05_fence_after();
        if (elect_one()) {
          const uint64_t da = umma_desc_sw128(smem_u32(sA + ua * G::A_BYTES + kb * 16384));
          const uint64_t db = umma_desc_sw128(smem_u32(sW + s * G::STAGE_BYTES));
          const int ksteps = ((C - kb * 64) < 64 ? (C - kb * 64) : 64) / 16;
          for (int k = 0; k < ksteps; ++k)
            umma_bf16_ss(tmem_base + b * G::HC, da + 2 * k, db + 2 * k, idesc1, (kb | k) != 0);
          umma_commit(&w_empty[s]);
        }
        __syncwarp();
        if (++s == G::kStages) { s = 0; ph ^= 1; }
      }
      if (elect_one()) {
        umma_commit(&acc1_full[b]);
        if (j == G::NCH - 1) umma_commit(&a_empty[ua]);  // the buffer may be refilled once every fc1 MMA of the tile completed
      }
      __syncwarp();
    };
    if (n_chunks > 0) fc1(0);
    if (n_chunks > 1) fc1(1);
    for (int g = 0; g < n_chunks; ++g) {
      const int j = g % G::NCH;
      const int u = G::kDefer ? ((g / G::NCH) & 1) : 0;  // acc2 buffer of this tile
      const int hb = g & 1;                               // acc1 buffer holding the GELU output of this chunk
      mbar_wait(&h_full[hb], n_h[hb] & 1);
      ++n_h[hb];
      if (j == 0) {
        mbar_wait(&acc2_empty[u], (n_acc2[u] & 1) ^ 1);  // the output phase that last used this buffer has drained it
        ++n_acc2[u];
      }
      tcgen05_fence_after();
      for (int kb = 0; kb < G::KB2; ++kb) {  // acc2 += H[chunk] . W2[:, chunk]^T
        mbar_wait(&w_full[s], ph);
        tcgen05_fence_after();
        if (elect_one()) {
          const uint64_t db = umma_desc_sw128(smem_u32(sW + s * G::STAGE_BYTES));
          for (int k = 0; k < 4; ++k)  // A = H from tensor memory: K step kb * 4 + k sits at columns [16 (..), + 8)
            umma_bf16_ts(tmem_base + G::ACC2_COL + u * C, tmem_base + hb * G::HC + (kb * 4 + k) * 16, db + 2 * k, idesc2,
                         (j | kb | k) != 0);
          umma_commit(&w_empty[s]);
        }
        __syncwarp();
        if (++s == G::kStages) { s = 0; ph ^= 1; }
      }
      if (j == G::NCH - 1) {
        if (elect_one()) umma_commit(&acc2_full[u]);
        __syncwarp();
      }
      if (g + 2 < n_chunks) fc1(g + 2);
    }
  } else {
    // ------------------------------------------------------------------ workers: GELU chunks, tile output
    const int w = warp;                     // 0..15
    const int q = warp & 3;                 // TMEM lane quarter of this warp
    const int cg = w >> 2;                  // column group 0..3
    const int r_t = q * 32 + lane;          // accumulator row owned by this thread
    // the four warps of a column group hold warp indices 4cg .. 4cg+3: elect the first as the TMA-store issuer
    const bool store_issuer = ((w & 3) == 0) && lane == 0;
    uint32_t n_acc1[2] = {0, 0}, n_acc2[2] = {0, 0};

    // tile output: acc2[u] + b2 -> swizzled fp32 staging -> TMA reduce-add into x (column groups < kOutGroups)
    auto tile_output = [&](int tile, int u) {
      if (cg >= G::kOutGroups) return;
      mbar_wait(&acc2_full[u], n_acc2[u] & 1);
      ++n_acc2[u];
      tcgen05_fence_after();
      uint8_t* buf = sStg + cg * 16384;
      constexpr int kChunks = C / 32;
#pragma unroll 1
      for (int ci = cg; ci < kChunks; ci += G::kOutGroups) {
        // the bulk reduce that last read this staging buffer must have drained it
        if (store_issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        asm volatile("bar.sync %0, 128;" ::"r"(cg + 1) : "memory");
        uint32_t r[32];
        tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + G::ACC2_COL + u * C + ci * 32, r);
        tmem_ld_wait();
        if (ci + G::kOutGroups >= kChunks) {
          tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc2_empty[u]);
        }
        uint8_t* rowp = buf + r_t * 128;
        const int sw = r_t & 7;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float4 bb = __ldg(reinterpret_cast<const float4*>(p.b2 + ci * 32 + 4 * c));
          *reinterpret_cast<float4*>(rowp + ((c ^ sw) << 4)) =
              make_float4(__uint_as_float(r[4 * c]) + bb.x, __uint_as_float(r[4 * c + 1]) + bb.y,
                          __uint_as_float(r[4 * c + 2]) + bb.z, __uint_as_float(r[4 * c + 3]) + bb.w);
        }
        fence_proxy_async_smem();
        asm volatile("bar.sync %0, 128;" ::"r"(cg + 1) : "memory");
        if (store_issuer) {
          asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];"
                       ::"l"(reinterpret_cast<uint64_t>(&tmX)), "r"(smem_u32(buf)), "r"(ci * 32), "r"(tile * 128)
                       : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
      }
    };

    int g = 0, tl = 0;  // global chunk index, local tile counter
    int prev_tile = -1;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++tl) {
      // ---- hidden chunks: acc1 -> + b1 -> GELU -> bf16 pairs, in place in tensor memory
#pragma unroll 1
      for (int j = 0; j < G::NCH; ++j, ++g) {
        const int b = g & 1;
        mbar_wait(&acc1_full[b], n_acc1[b] & 1);
        ++n_acc1[b];
        tcgen05_fence_after();
        const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + b * G::HC + cg * G::CQ;
#pragma unroll
        for (int c0 = 0; c0 < G::CQ; c0 += 16) {  // 16 hidden columns = one K step of fc2
          uint32_t r[16];
          tmem_ld_32x16(t_addr + c0, r);
          tmem_ld_wait();
          uint32_t hp[8];  // packed bf16 pairs
#pragma unroll
          for (int k = 0; k < 16; k += 4) {
            const float4 bb = *reinterpret_cast<const float4*>(&sB1[j * G::HC + cg * G::CQ + c0 + k]);
            hp[k >> 1] = gelu_bias_bf16x2(r[k], r[k + 1], bb.x, bb.y);
            hp[(k >> 1) + 1] = gelu_bias_bf16x2(r[k + 2], r[k + 3], bb.z, bb.w);
          }
          tmem_st_32x8(t_addr + c0, hp);  // in place: the first 8 of the 16 fp32 columns just read
        }
        tmem_st_wait();
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&h_full[b]);
        // deferred output of the previous tile: its last fc2 has long completed, nobody waits
        if (G::kDefer && j == 0 && prev_tile >= 0) tile_output(prev_tile, (tl - 1) & 1);
      }
      if (!G::kDefer) tile_output(tile, 0);
      prev_tile = tile;
    }
    if (G::kDefer && prev_tile >= 0) tile_output(prev_tile, (tl - 1) & 1);
    if (store_issuer) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }

  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  if (warp == kMmaWarp) tmem_dealloc<512>(tmem_base);
}

template <int C>
int launch_c(const CUtensorMap* tmY, const CUtensorMap* tmW1, const CUtensorMap* tmW2, const CUtensorMap* tmX,
             const MlpParams& p, cudaStream_t st) {
  static PerDeviceOnce configured;
  if (configured.first()) {
    DSG_CUDA_CHECK(cudaFuncSetAttribute(fused_mlp_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        MlpCfg<C>::SMEM_BYTES));
  }
  const int sms = device_sm_count();
  const int tiles = (p.M + 127) / 128;
  fused_mlp_kernel<C><<<tiles < sms ? tiles : sms, kMlpThreads, MlpCfg<C>::SMEM_BYTES, st>>>(*tmY, *tmW1, *tmW2, *tmX, p);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

}  // namespace

bool fused_mlp_supported(int C) { return C == 96 || C == 192; }
int fused_mlp_w1_box_rows(int C) { (void)C; return 128; }

int launch_fused_mlp(const CUtensorMap* tmY, const CUtensorMap* tmW1, const CUtensorMap* tmW2, const CUtensorMap* tmX,
                     const float* b1, const float* b2, long long rows, int C, cudaStream_t st) {
  DSG_REQUIRE(fused_mlp_supported(C) && rows > 0 && rows < 2147483647LL, "fused_mlp: C=%d rows=%lld", C, rows);
  MlpParams p{b1, b2, static_cast<int>(rows)};
  if (C == 96) return launch_c<96>(tmY, tmW1, tmW2, tmX, p, st);
  return launch_c<192>(tmY, tmW1, tmW2, tmX, p, st);
}

}  // namespace dsg
