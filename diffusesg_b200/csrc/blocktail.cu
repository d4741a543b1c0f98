// Fused tail of a Swin block for sm_100a (one kernel per block, C = 96):
//
//     x  = x + proj(att) + b_p                       (model/diffusesg/diffusesg.py:137, :272 of the reference)
//     y  = LayerNorm2(x)                             (:275, norm2)
//     x  = x + fc2(gelu(fc1(y) + b1)) + b2           (:275 with Mlp.forward :19-25)
//
// Unfused this is three launches (proj GEMM with a reduce-add epilogue, LayerNorm, fused MLP) that move the fp32
// residual stream through HBM three times and the bf16 LayerNorm output twice; here a 128-token tile reads att
// (bf16) and x (fp32) once and writes x once.  The residual never leaves the SM: the proj accumulator is turned
// into x_new (+ b2) IN TENSOR MEMORY (tcgen05.ld -> add -> tcgen05.st) and fc2 accumulates on top of it, so the
// final accumulator IS the block output.
//
//   warp 16  operand producer  att tile (TMA, 64-byte swizzle, 32-column k-blocks), W_proj / W1 / W2 rings
//   warp 17  MMA issuer        proj -> acc2[u] (SS);  fc1 chunk -> acc1[b] (TS, A = y);  fc2 chunk -> acc2[u] += (TS, A = H)
//   warp 18  residual mover    x tile in (TMA -> sX, L2 prefetch of the tile after) / block output out (sXo -> TMA store)
//   warps 0..15 workers        P: acc2 + b_p + x -> LN -> y (bf16 pairs in tensor memory) and x_new + b2 -> acc2
//                              G: acc1 + b1 -> GELU -> bf16 pairs, in place over acc1          (3 chunks of 128 / tile)
//                              O: final acc2 -> output staging tile
//   worker order per tile t:   G(t, 0), O(t - 1), G(t, 1), P(t + 1), G(t, 2)
//   MMA order (chunk stream):  fc2(g), fc1(g + 2), [proj(t + 1) after the first chunk of tile t]
#include "common.cuh"
#include "kernels.h"

namespace dsg {
namespace {

constexpr int kTailThreads = 19 * 32;
constexpr float kTailLnEps = 1e-5f;

template <int C>
struct TailCfg {
  static constexpr int HID = 4 * C;
  static constexpr int HC = 128;                   // hidden columns per chunk
  static constexpr int NCH = HID / HC;             // 3 chunks per tile
  static constexpr int KBN = C / 32;               // 32-column k-blocks of a K = C operand (64-byte swizzle)
  static constexpr int A_KB = 128 * 64;            // one k-block of a 128-row A operand
  static constexpr int A_BYTES = KBN * A_KB;       // att tile
  static constexpr int W1_KB = HC * 64;            // one k-block of a W1 chunk: [128 x 32] bf16
  static constexpr int W1_SLOT = KBN * W1_KB;      // W1 rows [j HC, (j + 1) HC), all of K
  static constexpr int WP_KB = C * 64;             // one k-block of W_proj: [C x 32] bf16
  static constexpr int W2_KB = C * 128;            // one k-block of a W2 chunk: [C x 64] bf16 (128-byte swizzle)
  static constexpr int W2_SLOT = (HC / 64) * W2_KB;  // W2[:, chunk]; W_proj (KBN k-blocks) shares the ring
  static constexpr int S1 = 2, S2 = 2;             // ring depths (fc1(g + 2) follows fc2(g): two chunks in flight)
  static constexpr int XB = C / 32;                // [128 x 32] fp32 boxes of the staging tile
  static constexpr int X_BYTES = XB * 16384;
  static constexpr int CW = C / 4;                 // columns per worker warp in the P / O phases
  static constexpr int PAR_FLOATS = HID + 4 * C;   // b1, b_p, b2, gamma, beta
  static constexpr int PART_BYTES = 4 * 128 * 8;   // LayerNorm partial sums: float2 [4 column groups][128 rows]
  static constexpr int SMEM_BYTES = 1024 + A_BYTES + 2 * X_BYTES + S1 * W1_SLOT + S2 * W2_SLOT + PART_BYTES +
                                    PAR_FLOATS * 4 + 512;
  // TMEM columns: acc1[b] @ b HC (two chunk buffers) | acc2[u] @ 2 HC + u C | y (bf16 pairs, the A operand of fc1).
  // Both MLP GEMMs take A from tensor memory (TS mode runs at ~93 % of the nominal MMA rate at N = 96, SS mode at
  // 80 %: tools/microbench/mma_bench.cu).  The GELU output of a chunk is written IN PLACE over its fc1 accumulator:
  // the 16 hidden columns of K step k (fp32 columns [16k, 16k + 16) of acc1[b]) become the 8 packed bf16 columns
  // [16k, 16k + 8), read and written by the same warp.  fc1 of chunk g + 2 reuses the buffer of chunk g; it is
  // issued after fc2 of chunk g by the same thread and the tensor pipe executes in issue order, so the chunk ring
  // needs no "empty" barriers.
  static constexpr int ACC2_COL = 2 * HC;
  static constexpr int Y_COL = ACC2_COL + 2 * C;
  static_assert(C % 32 == 0 && CW % 8 == 0, "tail: C must be a multiple of 32");
  static_assert(KBN * WP_KB <= W2_SLOT, "tail: W_proj must fit one W2-ring slot");
  static_assert(Y_COL + C / 2 <= 512 && SMEM_BYTES <= 227 * 1024, "tail budget");
};

struct TailParams {
  const float* bp;     // [C]   proj bias
  const float* gamma;  // [C]   norm2
  const float* beta;   // [C]
  const float* b1;     // [4C]
  const float* b2;     // [C]
  float* x;            // [M, C] fp32 residual stream (the same buffer tmX reads)
  const float* gamma_f;  // FINAL: the network's last LayerNorm (model/diffusesg/diffusesg.py:758), fused into the O phase
  const float* beta_f;
  int M;
};

// K-major operand, 64-byte swizzle, k-blocks of 32 bf16 columns: byte offset of the 16-byte chunk holding elements
// [k, k + 8) of row r (what TMA SWIZZLE_64B writes and a SWIZZLE_64B UMMA descriptor reads); kb_bytes = rows * 64
DSG_DEVICE uint32_t sw64_offset(int r, int k, int kb_bytes) {
  return static_cast<uint32_t>((k >> 5) * kb_bytes + r * 64 + (((((k & 31) >> 3) ^ (r >> 1)) & 3) << 4));
}
DSG_DEVICE uint32_t sw128_offset_1kb(int r, int k) {  // one [rows x 64] k-block, 128-byte swizzle
  return static_cast<uint32_t>(r * 128 + ((((k & 63) >> 3) ^ (r & 7)) << 4));
}

// start address >> 4 | LBO = 1 (unused) | SBO = 512 B (8 rows of 64 bytes) | version 1 | SWIZZLE_64B
DSG_DEVICE uint64_t umma_desc_sw64(uint32_t smem_addr) {
  const uint64_t lo = ((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16);
  const uint64_t hi = (512u >> 4) | (1u << 14) | (4u << 29);
  return lo | (hi << 32);
}

DSG_DEVICE void tmem_ld_32x8(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
DSG_DEVICE void tmem_st_32x8(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
DSG_DEVICE void tmem_st_32x4(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3])
               : "memory");
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
DSG_DEVICE void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// FINAL (the last block of the network): the O phase applies the final LayerNorm to the block output and stores ONLY
// its bf16 result (tmY) - the fp32 residual stream is dead after this block, so its 4 B/element write and the separate
// LayerNorm launch (4 B read + 2 B write) disappear.  The row statistics use the LN2 mean of the same row as pivot.
template <int C, bool FINAL>
__global__ void __launch_bounds__(kTailThreads, 1)
block_tail_kernel(const __grid_constant__ CUtensorMap tmAtt, const __grid_constant__ CUtensorMap tmWp,
                  const __grid_constant__ CUtensorMap tmW1, const __grid_constant__ CUtensorMap tmW2,
                  const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmY, const TailParams p) {
  using G = TailCfg<C>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sAtt = smem;
  uint8_t* sX = sAtt + G::A_BYTES;   // x tile in (TMA load -> P phase)
  uint8_t* sXo = sX + G::X_BYTES;    // block output (O phase -> TMA store); FINAL: bf16 [C / 32][128 x 32] + extras
  float2* sPartO = reinterpret_cast<float2*>(sXo + (C / 32) * 8192);               // FINAL: partial sums of the last LN
  float* sGamF = reinterpret_cast<float*>(sXo + (C / 32) * 8192 + G::PART_BYTES);  // FINAL: its gamma | beta
  float* sBetF = sGamF + C;
  static_assert((C / 32) * 8192 + G::PART_BYTES + 2 * C * 4 <= G::X_BYTES, "FINAL extras must fit the output tile");
  uint8_t* sW1 = sXo + G::X_BYTES;
  uint8_t* sW2 = sW1 + G::S1 * G::W1_SLOT;
  float2* sPart = reinterpret_cast<float2*>(sW2 + G::S2 * G::W2_SLOT);
  float* sB1 = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(sPart) + G::PART_BYTES);
  float* sBp = sB1 + G::HID;
  float* sB2 = sBp + C;
  float* sGam = sB2 + C;
  float* sBet = sGam + C;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sBet + C);
  uint64_t* w1_full = bars;                 // [S1]
  uint64_t* w1_empty = w1_full + G::S1;     // [S1]
  uint64_t* w2_full = w1_empty + G::S1;     // [S2]
  uint64_t* w2_empty = w2_full + G::S2;     // [S2]
  uint64_t* att_full = w2_empty + G::S2;    // TMA -> MMA
  uint64_t* att_empty = att_full + 1;       // MMA -> TMA: proj of the tile has read sAtt
  uint64_t* xin_full = att_full + 2;        // TMA -> workers: x tile landed in sX
  uint64_t* xin_free = att_full + 3;        // workers -> residual mover: P consumed the x tile in sX
  uint64_t* y_ready = att_full + 4;         // workers -> MMA: y (bf16, tensor memory) and x_new + b2 (acc2[u]) stored
  uint64_t* proj_full = att_full + 5;       // [2] MMA -> workers: proj accumulator of the tile complete in acc2[u]
  uint64_t* acc1_full = att_full + 7;       // [2] MMA -> workers: fc1 of the chunk complete
  uint64_t* h_full = att_full + 9;          // [2] workers -> MMA: GELU output of the chunk in place
  uint64_t* acc2_full = att_full + 11;      // [2] MMA -> workers: last fc2 of the tile complete
  uint64_t* acc2_empty = att_full + 13;     // [2] workers -> MMA: output drained, proj of tile t + 2 may overwrite
  uint64_t* out_ready = att_full + 15;      // workers -> residual mover: the output tile is in sXo
  uint64_t* out_free = att_full + 16;       // residual mover -> workers: the TMA store has read sXo
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(att_full + 17);

  const int warp = uniform_warp_id();
  const int lane = threadIdx.x & 31;
  constexpr int kTmaWarp = 16, kMmaWarp = 17, kXWarp = 18;
  const int num_tiles = (p.M + 127) / 128;
  const int my_tiles = (num_tiles > static_cast<int>(blockIdx.x)) ? (num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const int n_chunks = my_tiles * G::NCH;  // chunk stream of this CTA: g = tl * NCH + j

  if (warp == kTmaWarp && lane == 0) {
    tma_prefetch_desc(&tmAtt);
    tma_prefetch_desc(&tmWp);
    tma_prefetch_desc(&tmW1);
    tma_prefetch_desc(&tmW2);
    tma_prefetch_desc(&tmX);
    if (FINAL) tma_prefetch_desc(&tmY);
    for (int s = 0; s < G::S1; ++s) { mbar_init(&w1_full[s], 1); mbar_init(&w1_empty[s], 1); }
    for (int s = 0; s < G::S2; ++s) { mbar_init(&w2_full[s], 1); mbar_init(&w2_empty[s], 1); }
    mbar_init(att_full, 1);
    mbar_init(att_empty, 1);
    mbar_init(xin_full, 1);
    mbar_init(xin_free, 16);
    mbar_init(out_ready, 16);
    mbar_init(out_free, 1);
    mbar_init(y_ready, 16);
    for (int b = 0; b < 2; ++b) {
      mbar_init(&proj_full[b], 1);
      mbar_init(&acc1_full[b], 1);
      mbar_init(&h_full[b], 16);
      mbar_init(&acc2_full[b], 1);
      mbar_init(&acc2_empty[b], 16);
    }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc<512>(tmem_slot);
  for (int i = threadIdx.x; i < G::HID; i += kTailThreads) sB1[i] = p.b1[i];
  if (FINAL) {
    for (int i = threadIdx.x; i < C; i += kTailThreads) { sGamF[i] = p.gamma_f[i]; sBetF[i] = p.beta_f[i]; }
  }
  for (int i = threadIdx.x; i < C; i += kTailThreads) {
    sBp[i] = p.bp[i];
    sB2[i] = p.b2[i];
    sGam[i] = p.gamma[i];
    sBet[i] = p.beta[i];
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);

  if (warp == kTmaWarp) {
    // ------------------------------------------------------------------ operand producer (consumption order)
    if (elect_one()) {
      int s1 = 0, s2 = 0;
      uint32_t ph1 = 0, ph2 = 0;
      auto load_att = [&](int tl) {
        const int tile = blockIdx.x + tl * gridDim.x;
        mbar_wait(att_empty, (tl & 1) ^ 1);  // proj of tile tl - 1 has read the buffer
        mbar_expect_tx(att_full, G::A_BYTES);
        for (int kb = 0; kb < G::KBN; ++kb) tma_load_2d(sAtt + kb * G::A_KB, &tmAtt, att_full, kb * 32, tile * 128);
      };
      auto load_wp = [&]() {
        mbar_wait(&w2_empty[s2], ph2 ^ 1);
        mbar_expect_tx(&w2_full[s2], G::KBN * G::WP_KB);
        for (int kb = 0; kb < G::KBN; ++kb)
          tma_load_2d(sW2 + s2 * G::W2_SLOT + kb * G::WP_KB, &tmWp, &w2_full[s2], kb * 32, 0);
        if (++s2 == G::S2) { s2 = 0; ph2 ^= 1; }
      };
      auto load_w1 = [&](int g) {
        const int j = g % G::NCH;
        mbar_wait(&w1_empty[s1], ph1 ^ 1);
        mbar_expect_tx(&w1_full[s1], G::W1_SLOT);
        for (int kb = 0; kb < G::KBN; ++kb)
          tma_load_2d(sW1 + s1 * G::W1_SLOT + kb * G::W1_KB, &tmW1, &w1_full[s1], kb * 32, j * G::HC);
        if (++s1 == G::S1) { s1 = 0; ph1 ^= 1; }
      };
      auto load_w2 = [&](int g) {
        const int j = g % G::NCH;
        mbar_wait(&w2_empty[s2], ph2 ^ 1);
        mbar_expect_tx(&w2_full[s2], G::W2_SLOT);
        for (int kb = 0; kb < G::HC / 64; ++kb)
          tma_load_2d(sW2 + s2 * G::W2_SLOT + kb * G::W2_KB, &tmW2, &w2_full[s2], j * G::HC + kb * 64, 0);
        if (++s2 == G::S2) { s2 = 0; ph2 ^= 1; }
      };
      if (my_tiles > 0) {
        load_att(0);
        load_wp();
        load_w1(0);
        load_w1(1);
        if (my_tiles > 1) load_att(1);
      }
      for (int g = 0; g < n_chunks; ++g) {
        const int tl = g / G::NCH, j = g % G::NCH;
        load_w2(g);
        if (g + 2 < n_chunks) load_w1(g + 2);
        if (j == 0 && tl + 1 < my_tiles) load_wp();
        if (j == 1 && tl + 2 < my_tiles) load_att(tl + 2);  // proj(tl + 1) was issued one chunk ago
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc_c = umma_idesc_bf16(C);       // proj, fc2: N = C
    constexpr uint32_t idesc_h = umma_idesc_bf16(G::HC);   // fc1: N = HC
    int s1 = 0, s2 = 0;
    uint32_t ph1 = 0, ph2 = 0;
    auto proj = [&](int tl) {  // acc2[u] = att . W_proj^T   (SS mode: both operands from shared memory)
      const int u = tl & 1;
      mbar_wait(att_full, tl & 1);
      mbar_wait(&acc2_empty[u], ((tl >> 1) & 1) ^ 1);
      mbar_wait(&w2_full[s2], ph2);
      tcgen05_fence_after();
      if (elect_one()) {
        for (int kb = 0; kb < G::KBN; ++kb) {
          const uint64_t da = umma_desc_sw64(smem_u32(sAtt + kb * G::A_KB));
          const uint64_t db = umma_desc_sw64(smem_u32(sW2 + s2 * G::W2_SLOT + kb * G::WP_KB));
          for (int k = 0; k < 2; ++k)
            umma_bf16_ss(tmem_base + G::ACC2_COL + u * C, da + 2 * k, db + 2 * k, idesc_c, (kb | k) != 0);
        }
        umma_commit(&w2_empty[s2]);
        umma_commit(att_empty);
        umma_commit(&proj_full[u]);
      }
      __syncwarp();
      if (++s2 == G::S2) { s2 = 0; ph2 ^= 1; }
    };
    auto fc1 = [&](int g) {  // acc1[g & 1] = y . W1[chunk]^T   (the buffer's previous fc2 was issued earlier: in order)
      const int b = g & 1;
      if (g % G::NCH == 0) {  // first chunk of a tile: y of that tile in tensor memory, x_new + b2 in acc2[u]
        mbar_wait(y_ready, (g / G::NCH) & 1);
      }
      mbar_wait(&w1_full[s1], ph1);
      tcgen05_fence_after();
      if (elect_one()) {
        for (int kb = 0; kb < G::KBN; ++kb) {
          const uint64_t db = umma_desc_sw64(smem_u32(sW1 + s1 * G::W1_SLOT + kb * G::W1_KB));
          for (int k = 0; k < 2; ++k)
            umma_bf16_ts(tmem_base + b * G::HC, tmem_base + G::Y_COL + kb * 16 + k * 8, db + 2 * k, idesc_h, (kb | k) != 0);
        }
        umma_commit(&w1_empty[s1]);
        umma_commit(&acc1_full[b]);
      }
      __syncwarp();
      if (++s1 == G::S1) { s1 = 0; ph1 ^= 1; }
    };
    if (my_tiles > 0) {
      proj(0);
      fc1(0);
      fc1(1);
    }
    for (int g = 0; g < n_chunks; ++g) {
      const int tl = g / G::NCH, j = g % G::NCH;
      const int u = tl & 1, hb = g & 1;
      mbar_wait(&h_full[hb], (g >> 1) & 1);
      mbar_wait(&w2_full[s2], ph2);
      tcgen05_fence_after();
      if (elect_one()) {  // acc2[u] += H[chunk] . W2[:, chunk]^T   (always accumulating: acc2 holds x_new + b2)
        for (int kb = 0; kb < G::HC / 64; ++kb) {
          const uint64_t db = umma_desc_sw128(smem_u32(sW2 + s2 * G::W2_SLOT + kb * G::W2_KB));
          for (int k = 0; k < 4; ++k)
            umma_bf16_ts(tmem_base + G::ACC2_COL + u * C, tmem_base + hb * G::HC + (kb * 4 + k) * 16, db + 2 * k, idesc_c, 1u);
        }
        umma_commit(&w2_empty[s2]);
        if (j == G::NCH - 1) umma_commit(&acc2_full[u]);
      }
      __syncwarp();
      if (++s2 == G::S2) { s2 = 0; ph2 ^= 1; }
      if (g + 2 < n_chunks) fc1(g + 2);
      if (j == 0 && tl + 1 < my_tiles) proj(tl + 1);
    }
  } else if (warp == kXWarp) {
    // ------------------------------------------------------------------ residual mover
    if (elect_one()) {
      auto load_x = [&](int tl) {
        const int tile = blockIdx.x + tl * gridDim.x;
        mbar_expect_tx(xin_full, G::X_BYTES);
        for (int xb = 0; xb < G::XB; ++xb) tma_load_2d(sX + xb * 16384, &tmX, xin_full, xb * 32, tile * 128);
      };
      auto prefetch_x = [&](int tl) {  // next tile's x into L2: its load has one chunk less of slack than a tile
        const int tile = blockIdx.x + tl * gridDim.x;
        for (int xb = 0; xb < G::XB; ++xb)
          asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];"
                       ::"l"(reinterpret_cast<uint64_t>(&tmX)), "r"(xb * 32), "r"(tile * 128) : "memory");
      };
      auto store_x = [&](int tl) {
        const int tile = blockIdx.x + tl * gridDim.x;
        for (int xb = 0; xb < G::XB; ++xb) {
          if (FINAL)
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                         ::"l"(reinterpret_cast<uint64_t>(&tmY)), "r"(smem_u32(sXo + xb * 8192)), "r"(xb * 32), "r"(tile * 128)
                         : "memory");
          else
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                         ::"l"(reinterpret_cast<uint64_t>(&tmX)), "r"(smem_u32(sXo + xb * 16384)), "r"(xb * 32), "r"(tile * 128)
                         : "memory");
        }
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      };
      // worker events in time order: P(0), P(1), [O(k), P(k + 2)] for k = 0 ...
      if (my_tiles > 0) load_x(0);
      if (my_tiles > 1) prefetch_x(1);
      for (int t = 0; t < 2 && t + 1 < my_tiles; ++t) {
        mbar_wait(xin_free, t & 1);  // P(t) holds the x tile in registers
        load_x(t + 1);
        if (t + 2 < my_tiles) prefetch_x(t + 2);
      }
      for (int k = 0; k < my_tiles; ++k) {
        mbar_wait(out_ready, k & 1);
        store_x(k);
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        mbar_arrive(out_free);
        if (k + 3 < my_tiles) {
          mbar_wait(xin_free, (k + 2) & 1);
          load_x(k + 3);
          if (k + 4 < my_tiles) prefetch_x(k + 4);
        }
      }
      asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
  } else {
    // ------------------------------------------------------------------ workers
    const int q = warp & 3;            // TMEM lane quarter of this warp
    const int cg = warp >> 2;          // column group 0..3
    const int r_t = q * 32 + lane;     // accumulator row owned by this thread
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const int c0 = cg * G::CW;         // first column of this warp in the P / O phases

    // address of the 16-byte chunk holding columns [c, c + 4) of this thread's row in the fp32 staging tile
    auto sx_ptr = [&](int c) -> float4* {
      return reinterpret_cast<float4*>(sX + (c >> 5) * 16384 + r_t * 128 + (((((c & 31) >> 2)) ^ (r_t & 7)) << 4));
    };

    float mean_pre0 = 0.f, mean_pre1 = 0.f;  // FINAL: LN2 mean of this thread's row, tiles of parity 0 / 1 (pivot of O)
    // ---- P(tl): x_new = acc2 + b_p + x;  y = LN(x_new) -> tensor memory;  acc2 = x_new + b2
    auto phase_p = [&](int tl) {
      const int u = tl & 1;
      const int gt = tl * G::NCH;
      mbar_wait(&proj_full[u], (tl >> 1) & 1);
      mbar_wait(xin_full, tl & 1);
      tcgen05_fence_after();
      uint32_t v[G::CW];
#pragma unroll
      for (int i = 0; i < G::CW; i += 8) tmem_ld_32x8(t_lane + G::ACC2_COL + u * C + c0 + i, v + i);
      tmem_ld_wait();
      // packed fp32 pairs throughout: the workers are issue-bound
      const float pivot = *reinterpret_cast<const float*>(sX + r_t * 128 + ((r_t & 7) << 4));  // x[r][0]
      const f32x2 npiv = f2_splat(-pivot);
      f32x2 a[G::CW / 2];
      f32x2 s1 = f2_splat(0.f), s2 = f2_splat(0.f);
#pragma unroll
      for (int i = 0; i < G::CW; i += 4) {
        const float4 xi = *sx_ptr(c0 + i);
        const float4 bb = *reinterpret_cast<const float4*>(&sBp[c0 + i]);
        const f32x2 a0 = f2_add(f2_add(f2_pack(__uint_as_float(v[i]), __uint_as_float(v[i + 1])), f2_pack(bb.x, bb.y)),
                                f2_pack(xi.x, xi.y));
        const f32x2 a1 = f2_add(f2_add(f2_pack(__uint_as_float(v[i + 2]), __uint_as_float(v[i + 3])), f2_pack(bb.z, bb.w)),
                                f2_pack(xi.z, xi.w));
        a[i >> 1] = a0;
        a[(i >> 1) + 1] = a1;
        const f32x2 d0 = f2_add(a0, npiv), d1 = f2_add(a1, npiv);
        s1 = f2_add(s1, f2_add(d0, d1));
        s2 = f2_fma(d0, d0, f2_fma(d1, d1, s2));
      }
      {
        float s1a, s1b, s2a, s2b;
        f2_unpack(s1, s1a, s1b);
        f2_unpack(s2, s2a, s2b);
        sPart[cg * 128 + r_t] = make_float2(s1a + s1b, s2a + s2b);
      }
      // residual + fc2 bias back to tensor memory: fc2 accumulates on top of it
#pragma unroll
      for (int i = 0; i < G::CW; i += 8) {
        uint32_t w[8];
#pragma unroll
        for (int k = 0; k < 8; k += 4) {
          const float4 bb = *reinterpret_cast<const float4*>(&sB2[c0 + i + k]);
          float w0, w1, w2, w3;
          f2_unpack(f2_add(a[(i + k) >> 1], f2_pack(bb.x, bb.y)), w0, w1);
          f2_unpack(f2_add(a[((i + k) >> 1) + 1], f2_pack(bb.z, bb.w)), w2, w3);
          w[k] = __float_as_uint(w0); w[k + 1] = __float_as_uint(w1);
          w[k + 2] = __float_as_uint(w2); w[k + 3] = __float_as_uint(w3);
        }
        tmem_st_32x8(t_lane + G::ACC2_COL + u * C + c0 + i, w);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(xin_free);  // the x tile is in registers: the next one may land
      asm volatile("bar.sync 1, 512;" ::: "memory");
      float t1 = 0.f, t2 = 0.f;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 pp = sPart[k * 128 + r_t];
        t1 += pp.x;
        t2 += pp.y;
      }
      const float dm = t1 * (1.0f / C);                       // mean - pivot
      const float var = fmaxf(t2 * (1.0f / C) - dm * dm, 0.f);
      const float rstd = rsqrtf(var + kTailLnEps);
      if (FINAL) { if (u) mean_pre1 = pivot + dm; else mean_pre0 = pivot + dm; }
      const f32x2 rs2 = f2_splat(rstd);
      const f32x2 nmr = f2_splat(-(pivot + dm) * rstd);       // y = (a rstd - mean rstd) gamma + beta
#pragma unroll
      for (int i = 0; i < G::CW; i += 8) {  // y as bf16 pairs: columns [c0 + i, + 8) -> 4 tensor-memory columns
        uint32_t pk[4];
#pragma unroll
        for (int k = 0; k < 8; k += 4) {
          const float4 gg = *reinterpret_cast<const float4*>(&sGam[c0 + i + k]);
          const float4 be = *reinterpret_cast<const float4*>(&sBet[c0 + i + k]);
          pk[k >> 1] = pack_bf16x2(f2_fma(f2_fma(a[(i + k) >> 1], rs2, nmr), f2_pack(gg.x, gg.y), f2_pack(be.x, be.y)));
          pk[(k >> 1) + 1] =
              pack_bf16x2(f2_fma(f2_fma(a[((i + k) >> 1) + 1], rs2, nmr), f2_pack(gg.z, gg.w), f2_pack(be.z, be.w)));
        }
        tmem_st_32x4(t_lane + G::Y_COL + ((c0 + i) >> 1), pk);
      }
      tmem_st_wait();
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(y_ready);
    };

    // ---- O(tl): final accumulator -> output staging tile -> TMA store.  (Direct 256-bit global stores of each
    // thread's 96 contiguous bytes were measured 4x slower than staging + TMA: 32 scattered sectors per instruction.)
    auto phase_o = [&](int tl) {
      const int u = tl & 1;
      mbar_wait(&acc2_full[u], (tl >> 1) & 1);
      tcgen05_fence_after();
      uint32_t v[G::CW];
#pragma unroll
      for (int i = 0; i < G::CW; i += 8) tmem_ld_32x8(t_lane + G::ACC2_COL + u * C + c0 + i, v + i);
      tmem_ld_wait();
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc2_empty[u]);
      if (FINAL) {
        // last LayerNorm of the network on the block output: pivot-shifted one-pass statistics over the four column
        // groups of the row, then bf16 into the [128 x 32]-column chunks the adj / node heads read (64-byte swizzle)
        const float pivot = u ? mean_pre1 : mean_pre0;
        const f32x2 npiv = f2_splat(-pivot);
        f32x2 a[G::CW / 2];
        f32x2 s1 = f2_splat(0.f), s2 = f2_splat(0.f);
#pragma unroll
        for (int i = 0; i < G::CW; i += 2) {
          a[i >> 1] = f2_add(f2_pack(__uint_as_float(v[i]), __uint_as_float(v[i + 1])), npiv);
          s1 = f2_add(s1, a[i >> 1]);
          s2 = f2_fma(a[i >> 1], a[i >> 1], s2);
        }
        {
          float s1a, s1b, s2a, s2b;
          f2_unpack(s1, s1a, s1b);
          f2_unpack(s2, s2a, s2b);
          sPartO[cg * 128 + r_t] = make_float2(s1a + s1b, s2a + s2b);
        }
        asm volatile("bar.sync 2, 512;" ::: "memory");
        float t1 = 0.f, t2 = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float2 pp = sPartO[k * 128 + r_t];
          t1 += pp.x;
          t2 += pp.y;
        }
        const float dm = t1 * (1.0f / C);
        const float rstd = rsqrtf(fmaxf(t2 * (1.0f / C) - dm * dm, 0.f) + kTailLnEps);
        const f32x2 rs2 = f2_splat(rstd), nmr = f2_splat(-dm * rstd);
        if (tl > 0) mbar_wait(out_free, (tl - 1) & 1);  // the store of the previous output has read sXo
#pragma unroll
        for (int i = 0; i < G::CW; i += 8) {
          uint32_t pk[4];
#pragma unroll
          for (int k = 0; k < 8; k += 4) {
            const float4 gg = *reinterpret_cast<const float4*>(&sGamF[c0 + i + k]);
            const float4 be = *reinterpret_cast<const float4*>(&sBetF[c0 + i + k]);
            pk[k >> 1] = pack_bf16x2(f2_fma(f2_fma(a[(i + k) >> 1], rs2, nmr), f2_pack(gg.x, gg.y), f2_pack(be.x, be.y)));
            pk[(k >> 1) + 1] =
                pack_bf16x2(f2_fma(f2_fma(a[((i + k) >> 1) + 1], rs2, nmr), f2_pack(gg.z, gg.w), f2_pack(be.z, be.w)));
          }
          const int c = c0 + i;
          *reinterpret_cast<uint4*>(sXo + (c >> 5) * 8192 + r_t * 64 + (((((c & 31) >> 3)) ^ ((r_t >> 1) & 3)) << 4)) =
              make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(out_ready);
        return;
      }
      if (tl > 0) mbar_wait(out_free, (tl - 1) & 1);  // the store of the previous output has read sXo
#pragma unroll
      for (int i = 0; i < G::CW; i += 4)
        *reinterpret_cast<float4*>(sXo + ((c0 + i) >> 5) * 16384 + r_t * 128 + ((((((c0 + i) & 31) >> 2)) ^ (r_t & 7)) << 4)) =
            make_float4(__uint_as_float(v[i]), __uint_as_float(v[i + 1]), __uint_as_float(v[i + 2]), __uint_as_float(v[i + 3]));
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(out_ready);
    };

    // ---- G(g): hidden chunk  acc1 -> + b1 -> GELU -> bf16 pairs, in place (this warp's 32 columns = 2 K steps)
    auto phase_g = [&](int g) {
      const int b = g & 1, j = g % G::NCH;
      mbar_wait(&acc1_full[b], (g >> 1) & 1);
      tcgen05_fence_after();
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int col = cg * 32 + h * 16;
        uint32_t r[16];
        tmem_ld_32x16(t_lane + b * G::HC + col, r);
        tmem_ld_wait();
        uint32_t hp[8];
#pragma unroll
        for (int k = 0; k < 16; k += 4) {
          const float4 bb = *reinterpret_cast<const float4*>(&sB1[j * G::HC + col + k]);
          hp[k >> 1] = gelu_bias_bf16x2(r[k], r[k + 1], bb.x, bb.y);
          hp[(k >> 1) + 1] = gelu_bias_bf16x2(r[k + 2], r[k + 3], bb.z, bb.w);
        }
        tmem_st_32x8(t_lane + b * G::HC + col, hp);  // first half of the 16 fp32 columns just read
      }
      tmem_st_wait();
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&h_full[b]);
    };

    if (my_tiles > 0) phase_p(0);
    for (int tl = 0; tl < my_tiles; ++tl) {
      const int g0 = tl * G::NCH;
      phase_g(g0);
      if (tl > 0) phase_o(tl - 1);  // the previous tile's last fc2 completed in the shadow of the chunk above
#pragma unroll 1
      for (int j = 1; j < G::NCH - 1; ++j) phase_g(g0 + j);
      if (tl + 1 < my_tiles) {
        // y is single-buffered: every fc1 of this tile must have completed before P(tl + 1) overwrites it.  The
        // last one is waited for here (its barrier phase is consumed again, harmlessly, by G below).
        mbar_wait(&acc1_full[(g0 + G::NCH - 1) & 1], ((g0 + G::NCH - 1) >> 1) & 1);
        phase_p(tl + 1);  // fc1 of the next tile's first chunk runs while G / O below finish this tile
      }
      phase_g(g0 + G::NCH - 1);
    }
    if (my_tiles > 0) phase_o(my_tiles - 1);
  }

  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  if (warp == kMmaWarp) tmem_dealloc<512>(tmem_base);
}

template <int C>
int launch_c(const CUtensorMap* tmAtt, const CUtensorMap* tmWp, const CUtensorMap* tmW1, const CUtensorMap* tmW2,
             const CUtensorMap* tmX, const CUtensorMap* tmY, const TailParams& p, cudaStream_t st) {
  static PerDeviceOnce configured;
  if (configured.first()) {
    DSG_CUDA_CHECK(cudaFuncSetAttribute(block_tail_kernel<C, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        TailCfg<C>::SMEM_BYTES));
    DSG_CUDA_CHECK(cudaFuncSetAttribute(block_tail_kernel<C, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        TailCfg<C>::SMEM_BYTES));
  }
  const int sms = device_sm_count();
  const int tiles = (p.M + 127) / 128;
  if (tmY != nullptr)
    block_tail_kernel<C, true><<<tiles < sms ? tiles : sms, kTailThreads, TailCfg<C>::SMEM_BYTES, st>>>(
        *tmAtt, *tmWp, *tmW1, *tmW2, *tmX, *tmY, p);
  else
    block_tail_kernel<C, false><<<tiles < sms ? tiles : sms, kTailThreads, TailCfg<C>::SMEM_BYTES, st>>>(
        *tmAtt, *tmWp, *tmW1, *tmW2, *tmX, *tmX, p);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

}  // namespace

bool block_tail_supported(int C) { return C == 96; }

int launch_block_tail(const CUtensorMap* tmAtt, const CUtensorMap* tmWp, const CUtensorMap* tmW1,
                      const CUtensorMap* tmW2, const CUtensorMap* tmX, const float* bp, const float* gamma,
                      const float* beta, const float* b1, const float* b2, float* x, long long rows, int C,
                      cudaStream_t st, const CUtensorMap* tmY, const float* gamma_f, const float* beta_f) {
  DSG_REQUIRE(block_tail_supported(C) && rows > 0 && rows < 2147483647LL, "block_tail: C=%d rows=%lld", C, rows);
  DSG_REQUIRE((tmY == nullptr) == (gamma_f == nullptr) && (tmY == nullptr) == (beta_f == nullptr),
              "block_tail: the fused final LayerNorm needs its output map, gamma and beta together");
  TailParams p{bp, gamma, beta, b1, b2, x, gamma_f, beta_f, static_cast<int>(rows)};
  return launch_c<96>(tmAtt, tmWp, tmW1, tmW2, tmX, tmY, p, st);
}

}  // namespace dsg
