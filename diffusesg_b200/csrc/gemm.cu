// tcgen05 / TMEM / TMA GEMM for sm_100a:   out[M, N] = epilogue(A[M, K] . W[N, K]^T)
//
// A (activations) and W (nn.Linear weight, [out, in]) are row-major bf16 with K contiguous, i.e. both
// operands are "K-major" in UMMA terms.  One persistent CTA per SM walks 128 x BN output tiles:
//
//   warp 0      TMA producer: 128 x 64 A box + BN x 64 W box per stage (128-byte swizzle), kStages ring
//   warp 1      MMA issuer: one lane issues tcgen05.mma (M=128, N=BN, K=16) x 4 per stage; accumulators
//               live in TMEM, double buffered so the epilogue of tile i overlaps the main loop of i+1
//   warps 2..5  epilogue: tcgen05.ld (32 lanes x 32 columns per warp), bias / GELU, staged through a swizzled
//               shared-memory chunk (128 rows x 32 columns) and written with TMA bulk stores; the residual
//               epilogue x += acc + bias is a TMA reduce-add (the L2 does the read-modify-write, the tile of x is
//               never loaded by the SM); the adj read-out head epilogue writes its c_e planes directly
//
// Replaces the cuBLAS sgemm behind every nn.Linear / 1x1 conv of the reference denoiser
// (model/diffusesg/diffusesg.py:20-24 Mlp, :115 qkv, :137 proj, :334 reduction, :385/:402 breakup linears,
// :705-709 read_out, :806-809 adj head).
#include "common.cuh"
#include "kernels.h"

namespace dsg {
namespace {

constexpr int BM = 128;
constexpr int BK = 64;                    // 64 bf16 = one 128-byte swizzle row
// Epilogue groups (4 warps each): group g drains accumulator (g & 1); for the ALU-heavy epilogues (bf16 output,
// GELU, adj head) two groups share an accumulator and split its columns, so 16 warps hide the MUFU / load latency.
__host__ __device__ constexpr int epi_groups(int epi) { return (epi == EPI_RES_F32 || epi == EPI_F32) ? 2 : 4; }
__host__ __device__ constexpr int gemm_threads(int epi) { return 64 + 128 * epi_groups(epi); }
constexpr int A_STAGE_BYTES = BM * BK * 2;  // 16 KB

// PAIR: two CTAs of a 2-cluster share one 256 x BN tile (cta_group::2).  Each loads its 128 rows of A and HALF of the
// B tile, so a stage is 28 KB instead of 40 KB (BN = 192): 30 % less L2 -> SM traffic per flop and a deeper ring.
template <int BN, bool PAIR = false>
struct Cfg {
  static constexpr int kStages = PAIR ? ((BN == 256) ? 4 : (BN == 192) ? 5 : 7) : ((BN == 256) ? 3 : (BN == 192) ? 4 : 5);
  static constexpr int B_STAGE_BYTES = (PAIR ? BN / 2 : BN) * BK * 2;
  static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  static constexpr int ACC_STRIDE = (BN >= 192) ? 256 : 128;  // TMEM columns between the two accumulators
  static constexpr uint32_t TMEM_COLS = 2 * ACC_STRIDE;       // 512 / 256
  static constexpr int STAGING_BYTES = 64 * 1024;  // 2 groups x 2 x 16 KB (fp32 chunks) or 4 groups x 2 x 8 KB (bf16)
  static constexpr int BIAS_BYTES = 2 * BN * 4;     // bias slice of the current tile, per accumulator
  static constexpr int SMEM_BYTES = 1024 /*align slack*/ + kStages * STAGE_BYTES + STAGING_BYTES + BIAS_BYTES + 256 /*barriers*/;
};

static_assert(Cfg<96>::SMEM_BYTES <= 227 * 1024 && Cfg<192>::SMEM_BYTES <= 227 * 1024, "shared memory budget");
static_assert(Cfg<96, true>::SMEM_BYTES <= 227 * 1024 && Cfg<192, true>::SMEM_BYTES <= 227 * 1024, "shared memory budget");
static_assert(Cfg<256>::SMEM_BYTES <= 227 * 1024 && Cfg<256, true>::SMEM_BYTES <= 227 * 1024, "shared memory budget");

// MNM: both operands MN-major (weight gradients): tmA / tmW describe dY [tokens, N_out] and X [tokens, K_in], a stage holds
// 2 + BN / 64 TMA boxes of 64 columns x 64 tokens (8 KB each), p.M = N_out, p.N = K_in rounded up to BN, p.K = tokens.
template <int BN, int EPI, bool PAIR, bool MNM = false>
__global__ void __launch_bounds__(gemm_threads(EPI), 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
            const __grid_constant__ CUtensorMap tmO, const GemmParams p) {
  using C = Cfg<BN, PAIR>;
  static_assert(!(PAIR && EPI == EPI_ADJ_HEAD), "the adj-head epilogue is single-CTA");
  static_assert(!MNM || (!PAIR && EPI == EPI_RES_F32 && BN % 64 == 0), "MN-major operands: single-CTA split-K weight gradients");
  constexpr int kStages = C::kStages;
  extern __shared__ uint8_t smem_raw[];
  // round up to 1024 bytes (128-byte swizzle atoms) without casting through an integer, so that the compiler
  // keeps the shared address space and emits LDS / STS instead of generic loads and stores
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sA = smem;
  uint8_t* sB = smem + kStages * A_STAGE_BYTES;
  uint8_t* sOut = smem + kStages * C::STAGE_BYTES;  // staging chunks, 1024-byte aligned
  float* sBias = reinterpret_cast<float*>(sOut + C::STAGING_BYTES);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sOut + C::STAGING_BYTES + C::BIAS_BYTES);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tfull_bar = empty_bar + kStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  __shared__ float s_w2t[(EPI == EPI_ADJ_HEAD) ? 96 * 8 : 1];
  __shared__ float s_b2[8];

  const int warp = uniform_warp_id();
  const int lane = threadIdx.x & 31;
  // The warp scheduler favours the highest warp id among ready warps: the two control warps take the LAST two ids,
  // otherwise the ALU-heavy epilogue warps starve them and every hand-off gains ~1 k cycles of wake-up latency.
  constexpr int kEpiWarps = 4 * epi_groups(EPI);
  constexpr int kTmaWarp = kEpiWarps, kMmaWarp = kEpiWarps + 1;

  // tile = (block of 128 rows, or of 256 rows shared by a CTA pair) x (BN columns)
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;   // 0 = leader of the pair
  const int cta = PAIR ? (blockIdx.x >> 1) : blockIdx.x;  // tile-loop index of this CTA (pair)
  const int ncta = PAIR ? (gridDim.x >> 1) : gridDim.x;
  const int num_m = (p.M + (PAIR ? 2 * BM : BM) - 1) / (PAIR ? 2 * BM : BM);
  const int num_n = p.N / BN;
  const int num_kb = (p.K + BK - 1) / BK;
  // split-K (weight gradients: few output tiles, a contraction over every token): a work item is (output tile,
  // K slice), the slices of a tile are combined by the reduce-add epilogue.  ksplit = 1 everywhere else.
  const int ksplit = (!PAIR && p.ksplit > 1) ? p.ksplit : 1;
  const int kb_per = (num_kb + ksplit - 1) / ksplit;
  const int num_tiles = num_m * num_n * ksplit;

  if (warp == kTmaWarp && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
    if (EPI != EPI_ADJ_HEAD) tma_prefetch_desc(&tmO);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      // one arrival per epilogue warp reading accumulator a (of both CTAs of a pair: the leader's MMA warp waits)
      mbar_init(&tempty_bar[a], (PAIR ? 2 : 1) * 2 * epi_groups(EPI));
    }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) {
    if (PAIR) tmem_alloc_pair<C::TMEM_COLS>(tmem_slot);
    else tmem_alloc<C::TMEM_COLS>(tmem_slot);
  }
  if (EPI == EPI_ADJ_HEAD) {
    for (int i = threadIdx.x; i < 96 * 8; i += gemm_threads(EPI)) s_w2t[i] = p.w2t[i];
    if (threadIdx.x < 8) s_b2[threadIdx.x] = p.b2[threadIdx.x];
  }
  tcgen05_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();  // the peer's barriers exist before any multicast commit / remote arrive reaches them
  tcgen05_fence_after();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);

  if (warp == kTmaWarp) {
    // ------------------------------------------------------------------ TMA producer
    // The A box and the B box of a stage are issued by TWO lanes: one thread issuing boxes back to back is bound by
    // the TMA issue latency (~400 clk per 16 KB box = 40 B/clk per SM), two lanes in parallel reach 60 B/clk per SM
    // (tools/microbench/tma_rows_bench.cu).  Measured on the K = 384 shapes this changes nothing (still ~42 B/clk
    // per SM = 920 TFLOP/s with 128 x 192 tiles): the cap is inside the SM - an SS-mode MMA reads 10 KB of operands
    // per 96 clk from the same shared memory the TMA writes 40 KB per k-block into - not in the L2 or the issue path.
    int s = 0;
    uint32_t ph = 0;
    for (int tile = cta; tile < num_tiles; tile += ncta) {
      const int mn = tile / ksplit, kb0 = (tile - mn * ksplit) * kb_per, kb1 = min(num_kb, kb0 + kb_per);
      const int m_blk = mn / num_n, n_blk = mn % num_n;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&empty_bar[s], ph ^ 1);
        if (PAIR) {
          // this CTA's 128 rows of A and its half of the B tile; both CTAs' bytes complete on the LEADER's barrier
          if (lane == 0 && rank == 0) mbar_expect_tx(&full_bar[s], 2 * C::STAGE_BYTES);
          __syncwarp();
          const uint32_t lbar = mapa_u32(&full_bar[s], 0);
          if (lane == 0)
            tma_load_2d_pair(sA + s * A_STAGE_BYTES, &tmA, lbar, kb * BK, (m_blk * 2 + static_cast<int>(rank)) * BM);
          else if (lane == 1)
            tma_load_2d_pair(sB + s * C::B_STAGE_BYTES, &tmW, lbar, kb * BK, n_blk * BN + static_cast<int>(rank) * (BN / 2));
        } else if (MNM) {
          // one box per lane: 64 output rows / columns (inner, contiguous in memory) x 64 tokens (outer)
          if (lane == 0) mbar_expect_tx(&full_bar[s], C::STAGE_BYTES);
          __syncwarp();
          if (lane < 2) tma_load_2d(sA + s * A_STAGE_BYTES + lane * 8192, &tmA, &full_bar[s], m_blk * BM + lane * 64, kb * BK);
          else if (lane < 2 + BN / 64)
            tma_load_2d(sB + s * C::B_STAGE_BYTES + (lane - 2) * 8192, &tmW, &full_bar[s], n_blk * BN + (lane - 2) * 64, kb * BK);
        } else {
          if (lane == 0) mbar_expect_tx(&full_bar[s], C::STAGE_BYTES);
          __syncwarp();
          if (lane == 0) tma_load_2d(sA + s * A_STAGE_BYTES, &tmA, &full_bar[s], kb * BK, m_blk * BM);
          else if (lane == 1) tma_load_2d(sB + s * C::B_STAGE_BYTES, &tmW, &full_bar[s], kb * BK, n_blk * BN);
        }
        __syncwarp();
        if (++s == kStages) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == kMmaWarp && rank == 0) {
    // ------------------------------------------------------------------ MMA issuer (the leader of a pair)
    constexpr uint32_t idesc = PAIR ? umma_idesc_bf16_pair(BN) : MNM ? umma_idesc_bf16_mn(BN) : umma_idesc_bf16(BN);
    // K = 16 per MMA: two 8-row groups of the MN-major tile (2 x 1024 B), or 32 bytes inside the K-major swizzle row
    constexpr uint32_t kstep = MNM ? 128u : 2u;
    int s = 0;
    uint32_t ph = 0;
    int acc = 0;
    uint32_t acc_ph = 0;
    for (int tile = cta; tile < num_tiles; tile += ncta) {
      mbar_wait(&tempty_bar[acc], acc_ph ^ 1);
      tcgen05_fence_after();
      const uint32_t d_tmem = tmem_base + acc * C::ACC_STRIDE;
      const int kb0 = (tile % ksplit) * kb_per, kb1 = min(num_kb, kb0 + kb_per);
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&full_bar[s], ph);
        tcgen05_fence_after();
        if (elect_one()) {
          const uint64_t da = MNM ? umma_desc_sw128_mn(smem_u32(sA + s * A_STAGE_BYTES), 8192u) : umma_desc_sw128(smem_u32(sA + s * A_STAGE_BYTES));
          const uint64_t db = MNM ? umma_desc_sw128_mn(smem_u32(sB + s * C::B_STAGE_BYTES), 8192u) : umma_desc_sw128(smem_u32(sB + s * C::B_STAGE_BYTES));
          const int ksteps = min(BK, p.K - kb * BK) / 16;
          for (int k = 0; k < ksteps; ++k) {
            // advancing K by 16 bf16 = 32 bytes inside the 128-byte swizzle row: +2 in the (addr >> 4) field
            if (PAIR) umma_bf16_ss_pair(d_tmem, da + 2 * k, db + 2 * k, idesc, ((kb - kb0) | k) != 0);
            else umma_bf16_ss(d_tmem, da + kstep * k, db + kstep * k, idesc, ((kb - kb0) | k) != 0);
          }
          if (PAIR) {
            umma_commit_pair(&empty_bar[s]);
            if (kb == kb1 - 1) umma_commit_pair(&tfull_bar[acc]);
          } else {
            umma_commit(&empty_bar[s]);
            if (kb == kb1 - 1) umma_commit(&tfull_bar[acc]);
          }
        }
        __syncwarp();
        if (++s == kStages) { s = 0; ph ^= 1; }
      }
      acc ^= 1;
      if (acc == 0) acc_ph ^= 1;
    }
  } else if (warp == kMmaWarp) {
    // the peer's MMA warp only owns its half of the tensor-memory allocation
  } else {
    // ------------------------------------------------------------------ epilogue groups
    constexpr int kGroups = epi_groups(EPI);
    constexpr int kHalves = kGroups / 2;           // groups sharing one accumulator
    constexpr bool kOutBf16 = (EPI == EPI_BF16 || EPI == EPI_GELU_BF16);
    constexpr int kChunkBytes = kOutBf16 ? 128 * 64 : 128 * 128;
    const int q = warp & 3;                        // TMEM lane quarter this warp may access
    const int grp = warp >> 2;
    const int acc = grp & 1;
    const int half = grp >> 1;
    const int r_in_tile = q * 32 + lane;
    const int tig = (warp & 3) * 32 + lane;  // thread index inside the group
    const bool issuer = tig == 0;
    const int bar_id = grp + 1;
    uint8_t* sOutG = sOut + grp * 2 * kChunkBytes;
    float* sBiasA = sBias + acc * BN;
    uint32_t acc_ph = 0;
    int chunk_no = 0;  // running count of staged chunks -> staging buffer parity
    // accumulator hand-back: the leader's MMA warp counts the epilogue warps of both CTAs of a pair
    const uint32_t tempty_addr = PAIR ? mapa_u32(&tempty_bar[acc], 0) : 0u;
    auto release_acc = [&]() {
      if (PAIR) mbar_arrive_cluster(tempty_addr);
      else mbar_arrive(&tempty_bar[acc]);
    };
    for (int tile = cta + acc * ncta; tile < num_tiles; tile += 2 * ncta) {
      const int mn = tile / ksplit;
      const int m_blk = PAIR ? (mn / num_n) * 2 + static_cast<int>(rank) : mn / num_n;  // this CTA's 128-row block
      const int n_blk = mn % num_n;
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * C::ACC_STRIDE;
      if (EPI == EPI_ADJ_HEAD) {
        // columns [48 half, 48 half + 48) of the hidden layer; partial sums of the 96 -> c_e linear are combined
        // through shared memory (reusing the staging area)
        float* sPart = reinterpret_cast<float*>(sOut) + acc * 128 * 8;
        if (tile == cta + acc * ncta) {  // first tile of this group: the bias slice never changes (N == BN == 96)
          if (tig < 48) sBiasA[half * 48 + tig] = p.bias[half * 48 + tig];
          asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
        }
        const int row = m_blk * BM + r_in_tile;
        // everything the output step needs from global memory is fetched BEFORE the accumulator wait: this group
        // handles one tile at a time, so these dependent loads were ~1.5 k exposed cycles per tile
        const int n_ = p.n_img, nn_ = n_ * n_;
        const int rowc = row < p.M ? row : p.M - 1;
        int b_ = rowc / nn_, ij_ = rowc - b_ * nn_;
        if (p.perm != nullptr) {
          const int ss = p.side * p.side;
          const int img = rowc / ss, rem = rowc - img * ss;
          const int ii = rem / p.side;
          b_ = p.perm[img];
          ij_ = ii * n_ + (rem - ii * p.side);
        }
        const bool real_ = b_ >= 0;   // phantom rows of the compact layout produce no output
        if (!real_) b_ = 0;
        bool ok_ = false;
        float cs_ = 0.f, co_ = 1.f, xa_[8];
        if (half == 0) {
          const int i_ = ij_ / n_, j_ = ij_ - i_ * n_;
          ok_ = p.flags[b_ * n_ + i_] != 0 && p.flags[b_ * n_ + j_] != 0;
          if (p.x_adj != nullptr) {
            cs_ = p.c_skip[b_];
            co_ = p.c_out[b_];
#pragma unroll
            for (int c = 0; c < 8; ++c) xa_[c] = c < p.c_e ? p.x_adj[(static_cast<size_t>(b_) * p.c_e + c) * nn_ + ij_] : 0.f;
          }
        }
        mbar_wait(&tfull_bar[acc], acc_ph);
        tcgen05_fence_after();
        // packed fp32 pairs: the 8 outputs are four FFMA2 accumulators, GELU runs on column pairs
        f32x2 y2[4] = {f2_splat(0.f), f2_splat(0.f), f2_splat(0.f), f2_splat(0.f)};
#pragma unroll
        for (int c0 = 0; c0 < 48; c0 += 16) {
          uint32_t r[16];
          tmem_ld_32x16(t_row + half * 48 + c0, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; j += 2) {
            const int col = half * 48 + c0 + j;
            const float2 bb = *reinterpret_cast<const float2*>(&sBiasA[col]);
            float v0, v1;
            f2_unpack(gelu_erf2(f2_add(f2_pack(__uint_as_float(r[j]), __uint_as_float(r[j + 1])), f2_pack(bb.x, bb.y))), v0, v1);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const f32x2 vv = f2_splat(h == 0 ? v0 : v1);
              const float4 wa = *reinterpret_cast<const float4*>(&s_w2t[(col + h) * 8]);
              const float4 wb = *reinterpret_cast<const float4*>(&s_w2t[(col + h) * 8 + 4]);
              y2[0] = f2_fma(f2_pack(wa.x, wa.y), vv, y2[0]);
              y2[1] = f2_fma(f2_pack(wa.z, wa.w), vv, y2[1]);
              y2[2] = f2_fma(f2_pack(wb.x, wb.y), vv, y2[2]);
              y2[3] = f2_fma(f2_pack(wb.z, wb.w), vv, y2[3]);
            }
          }
        }
        float y[8];
#pragma unroll
        for (int c = 0; c < 4; ++c) f2_unpack(y2[c], y[2 * c], y[2 * c + 1]);
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) release_acc();
        if (half == 1) {
          *reinterpret_cast<float4*>(&sPart[r_in_tile * 8]) = make_float4(y[0], y[1], y[2], y[3]);
          *reinterpret_cast<float4*>(&sPart[r_in_tile * 8 + 4]) = make_float4(y[4], y[5], y[6], y[7]);
        }
        asm volatile("bar.sync %0, 256;" ::"r"(5 + acc) : "memory");  // both halves of this accumulator
        if (half == 0) {
          const float4 pa = *reinterpret_cast<const float4*>(&sPart[r_in_tile * 8]);
          const float4 pb = *reinterpret_cast<const float4*>(&sPart[r_in_tile * 8 + 4]);
          y[0] += pa.x + s_b2[0]; y[1] += pa.y + s_b2[1]; y[2] += pa.z + s_b2[2]; y[3] += pa.w + s_b2[3];
          y[4] += pb.x + s_b2[4]; y[5] += pb.y + s_b2[5]; y[6] += pb.z + s_b2[6]; y[7] += pb.w + s_b2[7];
          if (row < p.M && real_) {
            // row = pixel (b, i, j); zero rows/cols of padded nodes (utils/graph_utils.py:5-38), optional EDM
            // output preconditioning D = c_skip x + c_out F (model/precond/precond.py:102-104)
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              if (c < p.c_e) {
                const size_t o = (static_cast<size_t>(b_) * p.c_e + c) * nn_ + ij_;
                float val = y[c];
                if (p.x_adj != nullptr) val = __fadd_rn(__fmul_rn(cs_, xa_[c]), __fmul_rn(co_, val));
                reinterpret_cast<float*>(p.out)[o] = ok_ ? val : 0.f;
              }
            }
          }
        }
        asm volatile("bar.sync %0, 256;" ::"r"(5 + acc) : "memory");  // sPart may be overwritten by the next tile
      } else {
        // this group's share of the bias slice (its own column chunks), visible after the first chunk barrier
        if (p.bias != nullptr) {
          for (int i = tig; i < BN; i += 128)
            if (((i >> 5) % kHalves) == half) sBiasA[i] = p.bias[n_blk * BN + i];
        }
        mbar_wait(&tfull_bar[acc], acc_ph);
        tcgen05_fence_after();
        constexpr int kChunks = BN / 32;
        constexpr int kLast = ((kChunks - 1) % kHalves);  // which half owns the last chunk is irrelevant: each half
        (void)kLast;                                       // signals after ITS last chunk
#pragma unroll 1
        for (int ci = half; ci < kChunks; ci += kHalves, ++chunk_no) {
          const int c0 = ci * 32;
          uint8_t* buf = sOutG + (chunk_no & 1) * kChunkBytes;
          // the bulk store that last read this staging buffer (two chunks ago) must have drained it
          if (issuer) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
          asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
          uint32_t r[32];
          tmem_ld_32x32(t_row + c0, r);
          tmem_ld_wait();
          if (ci + kHalves >= kChunks) {  // this group's last chunk: its warps are done with the accumulator
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) release_acc();
          }
          const int col = n_blk * BN + c0;
          float v[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
          if (p.bias != nullptr) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 b = *reinterpret_cast<const float4*>(&sBiasA[c0 + j]);
              v[j] += b.x; v[j + 1] += b.y; v[j + 2] += b.z; v[j + 3] += b.w;
            }
          }
          if (EPI == EPI_GELU_BF16) {
#pragma unroll
            for (int j = 0; j < 32; j += 2) f2_unpack(gelu_erf2(f2_pack(v[j], v[j + 1])), v[j], v[j + 1]);
          }
          if (MNM) {
            if (m_blk * BM + r_in_tile < p.scale_rows) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] *= p.row_scale;
            }
          }
          if (kOutBf16) {
            // 64-byte rows, CU_TENSOR_MAP_SWIZZLE_64B: 16-byte chunk index ^= (row >> 1) & 3
            uint8_t* rowp = buf + r_in_tile * 64;
            const int sw = (r_in_tile >> 1) & 3;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              uint4 w;
              w.x = pack_bf16x2(v[8 * c], v[8 * c + 1]);
              w.y = pack_bf16x2(v[8 * c + 2], v[8 * c + 3]);
              w.z = pack_bf16x2(v[8 * c + 4], v[8 * c + 5]);
              w.w = pack_bf16x2(v[8 * c + 6], v[8 * c + 7]);
              *reinterpret_cast<uint4*>(rowp + ((c ^ sw) << 4)) = w;
            }
          } else {
            // 128-byte rows, CU_TENSOR_MAP_SWIZZLE_128B: 16-byte chunk index ^= row & 7
            uint8_t* rowp = buf + r_in_tile * 128;
            const int sw = r_in_tile & 7;
#pragma unroll
            for (int c = 0; c < 8; ++c)
              *reinterpret_cast<float4*>(rowp + ((c ^ sw) << 4)) = make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
          }
          fence_proxy_async_smem();
          asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
          if (issuer) {
            if (EPI == EPI_RES_F32) {
              asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];"
                           ::"l"(reinterpret_cast<uint64_t>(&tmO)), "r"(smem_u32(buf)), "r"(col), "r"(m_blk * BM)
                           : "memory");
            } else {
              asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                           ::"l"(reinterpret_cast<uint64_t>(&tmO)), "r"(smem_u32(buf)), "r"(col), "r"(m_blk * BM)
                           : "memory");
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
      }
      acc_ph ^= 1;
    }
    if (issuer) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }

  tcgen05_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();  // neither CTA may retire while the other can still reach its shared / tensor memory
  tcgen05_fence_after();
  if (warp == kMmaWarp) {
    if (PAIR) tmem_dealloc_pair<C::TMEM_COLS>(tmem_base);
    else tmem_dealloc<C::TMEM_COLS>(tmem_base);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess) {
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
    }
  }
  return fn;
}

int num_sms() { return device_sm_count(); }

template <int BN, int EPI>
int launch_t(const CUtensorMap* tmA, const CUtensorMap* tmW, const CUtensorMap* tmO, const GemmParams& p,
             cudaStream_t st) {
  static PerDeviceOnce configured;
  if (configured.first()) {
    DSG_CUDA_CHECK(cudaFuncSetAttribute(gemm_kernel<BN, EPI, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        Cfg<BN>::SMEM_BYTES));
  }
  const int tiles = ((p.M + BM - 1) / BM) * (p.N / BN);
  const int grid = tiles < num_sms() ? tiles : num_sms();
  gemm_kernel<BN, EPI, false><<<grid, gemm_threads(EPI), Cfg<BN>::SMEM_BYTES, st>>>(*tmA, *tmW, *tmO, p);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

// CTA-pair version: tmW must be the HALF-tile descriptor (box 64 x BN / 2)
template <int BN, int EPI>
int launch_pair(const CUtensorMap* tmA, const CUtensorMap* tmW, const CUtensorMap* tmO, const GemmParams& p,
                cudaStream_t st) {
  using K = Cfg<BN, true>;
  static PerDeviceOnce configured;
  if (configured.first()) {
    DSG_CUDA_CHECK(cudaFuncSetAttribute(gemm_kernel<BN, EPI, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        K::SMEM_BYTES));
  }
  const int tiles = ((p.M + 2 * BM - 1) / (2 * BM)) * (p.N / BN);
  const int pairs = tiles < num_sms() / 2 ? tiles : num_sms() / 2;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(gemm_threads(EPI));
  cfg.dynamicSmemBytes = K::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  DSG_CUDA_CHECK(cudaLaunchKernelEx(&cfg, gemm_kernel<BN, EPI, true>, *tmA, *tmW, *tmO, p));
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}


template <int BN>
int launch_wgrad_t(const CUtensorMap* tmA, const CUtensorMap* tmW, const CUtensorMap* tmO, const GemmParams& p, cudaStream_t st) {
  static PerDeviceOnce configured;
  if (configured.first()) {
    DSG_CUDA_CHECK(cudaFuncSetAttribute(gemm_kernel<BN, EPI_RES_F32, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        Cfg<BN>::SMEM_BYTES));
  }
  const int tiles = ((p.M + BM - 1) / BM) * (p.N / BN) * (p.ksplit > 1 ? p.ksplit : 1);
  const int grid = tiles < num_sms() ? tiles : num_sms();
  gemm_kernel<BN, EPI_RES_F32, false, true><<<grid, gemm_threads(EPI_RES_F32), Cfg<BN>::SMEM_BYTES, st>>>(*tmA, *tmW, *tmO, p);
  DSG_LAUNCH_CHECK();
  return DSG_OK;
}

}  // namespace

int make_tmap_2d(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int elem_bytes, int box_cols,
                 int box_rows);

int launch_wgrad(const void* dy, const void* x, float* dw, long long tokens, int n_out, int x_cols, int out_cols, int ksplit,
                 int scale_rows, float row_scale, cudaStream_t st) {
  DSG_REQUIRE(dy && x && dw && tokens > 0 && tokens % 16 == 0 && n_out % 8 == 0 && x_cols % 8 == 0 && out_cols > 0 &&
                  out_cols <= x_cols && (out_cols * 4) % 16 == 0,
              "wgrad: tokens %lld n_out %d x_cols %d out_cols %d (tokens %% 16, widths %% 8, 16-byte output rows)", tokens,
              n_out, x_cols, out_cols);
  const int bn = (x_cols % 192 == 0) ? 192 : 128;
  CUtensorMap ta, tw, to;
  if (int rc = make_tmap_2d(&ta, dy, tokens, n_out, 2, 64, 64)) return rc;
  if (int rc = make_tmap_2d(&tw, x, tokens, x_cols, 2, 64, 64)) return rc;
  if (int rc = make_tmap_out(&to, dw, n_out, out_cols, EPI_RES_F32)) return rc;
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.M = n_out;
  p.N = (x_cols + bn - 1) / bn * bn;
  p.K = static_cast<int>(tokens);
  p.res = dw; p.out = dw; p.ldo = p.N; p.bn = bn;
  p.scale_rows = scale_rows; p.row_scale = row_scale;
  const int num_kb = (p.K + BK - 1) / BK;
  if (ksplit > 1) {
    const int per = (num_kb + ksplit - 1) / ksplit;
    p.ksplit = (num_kb + per - 1) / per;
  }
  return bn == 192 ? launch_wgrad_t<192>(&ta, &tw, &to, p, st) : launch_wgrad_t<128>(&ta, &tw, &to, p, st);
}

int make_tmap_2d(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int elem_bytes, int box_cols,
                 int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (fn == nullptr) {
    set_last_error("cuTensorMapEncodeTiled is not available from the CUDA driver");
    return DSG_ERR_CUDA;
  }
  const int inner = box_cols * elem_bytes;
  DSG_REQUIRE((elem_bytes == 2 || elem_bytes == 4) && (inner == 64 || inner == 128),
              "make_tmap_2d: box of %d x %d-byte elements (inner extent must be 64 or 128 bytes)", box_cols, elem_bytes);
  DSG_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0 && (cols * elem_bytes) % 16 == 0 && box_rows > 0 &&
                  box_rows <= 256,
              "make_tmap_2d: unaligned base/pitch or bad box (rows=%lld cols=%lld box_rows=%d)", (long long)rows,
              (long long)cols, box_rows);
  const cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  const cuuint64_t gstride[1] = {static_cast<cuuint64_t>(cols) * elem_bytes};
  const cuuint32_t box[2] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows)};
  const cuuint32_t estride[2] = {1, 1};
  const CUresult r = fn(map, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                        const_cast<void*>(base), gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        inner == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld cols=%lld box=%dx%d)", (int)r,
                   (long long)rows, (long long)cols, box_cols, box_rows);
    return DSG_ERR_CUDA;
  }
  return DSG_OK;
}

// bf16 tensor [d2][d1][d0] (d0 contiguous, byte strides s1 / s2 of d1 / d2), box b0 x b1 x b2, 64-byte swizzle
// (b0 must be 32 elements).  Used for the 8 x 8-token window boxes of the tcgen05 attention kernel.
int make_tmap_3d_bf16(CUtensorMap* map, const void* base, int64_t d0, int64_t d1, int64_t d2, int64_t s1, int64_t s2, int b0,
                      int b1, int b2) {
  EncodeTiledFn fn = get_encode_fn();
  if (fn == nullptr) {
    set_last_error("cuTensorMapEncodeTiled is not available from the CUDA driver");
    return DSG_ERR_CUDA;
  }
  DSG_REQUIRE(b0 == 32 && (reinterpret_cast<uintptr_t>(base) & 15) == 0 && s1 % 16 == 0 && s2 % 16 == 0 && b1 > 0 &&
                  b1 <= 256 && b2 > 0 && b2 <= 256,
              "make_tmap_3d_bf16: bad box / strides");
  const cuuint64_t gdim[3] = {static_cast<cuuint64_t>(d0), static_cast<cuuint64_t>(d1), static_cast<cuuint64_t>(d2)};
  const cuuint64_t gstride[2] = {static_cast<cuuint64_t>(s1), static_cast<cuuint64_t>(s2)};
  const cuuint32_t box[3] = {static_cast<cuuint32_t>(b0), static_cast<cuuint32_t>(b1), static_cast<cuuint32_t>(b2)};
  const cuuint32_t estride[3] = {1, 1, 1};
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), gdim, gstride, box, estride,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled (3d) failed with CUresult %d", (int)r);
    return DSG_ERR_CUDA;
  }
  return DSG_OK;
}

int make_tmap_bf16(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int box_rows) {
  return make_tmap_2d(map, base, rows, cols, 2, BK, box_rows);
}

int make_tmap_out(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int epi) {
  const bool bf = (epi == EPI_BF16 || epi == EPI_GELU_BF16);
  return make_tmap_2d(map, base, rows, cols, bf ? 2 : 4, 32, BM);
}

int gemm_block_n(int N) { return (N % 192 == 0) ? 192 : 96; }

int gemm_choose_bn(long long rows, int N, int K, int epi, bool pair) {
  const int bn0 = gemm_block_n(N);
  if (N % 256 != 0 || K < 384 || epi == EPI_ADJ_HEAD) return bn0;
  auto fill = [&](int bn) {  // how full the waves of a persistent launch are
    const long long tiles = ((rows + (pair ? 255 : 127)) / (pair ? 256 : 128)) * (N / bn);
    const long long slots = pair ? num_sms() / 2 : num_sms();
    const long long waves = (tiles + slots - 1) / slots;
    return static_cast<double>(tiles) / static_cast<double>(waves * slots);
  };
  return fill(256) * 1.08 > fill(bn0) ? 256 : bn0;
}

// CTA pairs cut the operand bytes a CTA's shared memory takes in (and serves to the tensor core) per flop by 30 %,
// which is what bounds the single-CTA tiles at ~42 B/clk per SM = 40 KB per 128 x 192 x 64 step -> ~920 TFLOP/s
// (not the L2: a TMA-only microbenchmark reaches 60 B/clk per SM from L2).  Measured (same box, A/B):
// +10..18 % for K >= 768; at K = 384 +3..10 % for the plain bf16 epilogue (qkv), -8 % for fc1 (its GELU epilogue
// is the co-bound and loses its slack), -2 % for the HBM-bound residual epilogue; K <= 192 shapes are HBM-bound.
bool gemm_use_pair(long long rows, int K, int epi) {
  return epi != EPI_ADJ_HEAD && rows >= 256 && (K >= 768 || (K >= 384 && epi == EPI_BF16));
}

int launch_gemm(const CUtensorMap* tmA, const CUtensorMap* tmW, const CUtensorMap* tmO, int epi, const GemmParams& p,
                cudaStream_t st, bool pair) {
  DSG_REQUIRE(p.M > 0 && p.N > 0 && p.K > 0 && p.N % 96 == 0 && p.K % 16 == 0,
              "gemm: unsupported shape M=%d N=%d K=%d (N %% 96 == 0 and K %% 16 == 0 required)", p.M, p.N, p.K);
  DSG_REQUIRE(p.out != nullptr, "gemm: null output");
  DSG_REQUIRE(p.ksplit <= 1, "gemm: split-K (ksplit %d) is only for the MN-major weight-gradient GEMM", p.ksplit);
  const int bn = p.bn ? p.bn : gemm_block_n(p.N);
  DSG_REQUIRE(p.N % bn == 0 && (bn == 96 || bn == 192 || bn == 256), "gemm: tile width %d for N = %d", bn, p.N);
  if (epi == EPI_ADJ_HEAD) {
    DSG_REQUIRE(p.N == 96 && p.c_e >= 1 && p.c_e <= 8 && p.w2t && p.b2 && p.flags && p.n_img > 0,
                "gemm: adj-head epilogue needs N == 96, c_e <= 8 and the head tensors");
    return launch_t<96, EPI_ADJ_HEAD>(tmA, tmW, tmO, p, st);
  }
  DSG_REQUIRE(p.ldo % 8 == 0, "gemm: ldo must be a multiple of 8");
  DSG_REQUIRE(tmO != nullptr && p.ldo == p.N, "gemm: output tensor map missing or ldo != N");
  if (epi == EPI_RES_F32)
    DSG_REQUIRE(p.res == p.out, "gemm: the residual epilogue accumulates in place (res must alias out)");
  if (pair) {  // CTA pairs: tmW is the half-tile descriptor
    if (bn == 256) {
      switch (epi) {
        case EPI_BF16: return launch_pair<256, EPI_BF16>(tmA, tmW, tmO, p, st);
        case EPI_GELU_BF16: return launch_pair<256, EPI_GELU_BF16>(tmA, tmW, tmO, p, st);
        case EPI_RES_F32: return launch_pair<256, EPI_RES_F32>(tmA, tmW, tmO, p, st);
        case EPI_F32: return launch_pair<256, EPI_F32>(tmA, tmW, tmO, p, st);
      }
    } else if (bn == 192) {
      switch (epi) {
        case EPI_BF16: return launch_pair<192, EPI_BF16>(tmA, tmW, tmO, p, st);
        case EPI_GELU_BF16: return launch_pair<192, EPI_GELU_BF16>(tmA, tmW, tmO, p, st);
        case EPI_RES_F32: return launch_pair<192, EPI_RES_F32>(tmA, tmW, tmO, p, st);
        case EPI_F32: return launch_pair<192, EPI_F32>(tmA, tmW, tmO, p, st);
      }
    } else {
      switch (epi) {
        case EPI_BF16: return launch_pair<96, EPI_BF16>(tmA, tmW, tmO, p, st);
        case EPI_GELU_BF16: return launch_pair<96, EPI_GELU_BF16>(tmA, tmW, tmO, p, st);
        case EPI_RES_F32: return launch_pair<96, EPI_RES_F32>(tmA, tmW, tmO, p, st);
        case EPI_F32: return launch_pair<96, EPI_F32>(tmA, tmW, tmO, p, st);
      }
    }
  }
  if (bn == 256) {
    switch (epi) {
      case EPI_BF16: return launch_t<256, EPI_BF16>(tmA, tmW, tmO, p, st);
      case EPI_GELU_BF16: return launch_t<256, EPI_GELU_BF16>(tmA, tmW, tmO, p, st);
      case EPI_RES_F32: return launch_t<256, EPI_RES_F32>(tmA, tmW, tmO, p, st);
      case EPI_F32: return launch_t<256, EPI_F32>(tmA, tmW, tmO, p, st);
    }
  } else if (bn == 192) {
    switch (epi) {
      case EPI_BF16: return launch_t<192, EPI_BF16>(tmA, tmW, tmO, p, st);
      case EPI_GELU_BF16: return launch_t<192, EPI_GELU_BF16>(tmA, tmW, tmO, p, st);
      case EPI_RES_F32: return launch_t<192, EPI_RES_F32>(tmA, tmW, tmO, p, st);
      case EPI_F32: return launch_t<192, EPI_F32>(tmA, tmW, tmO, p, st);
    }
  } else {
    switch (epi) {
      case EPI_BF16: return launch_t<96, EPI_BF16>(tmA, tmW, tmO, p, st);
      case EPI_GELU_BF16: return launch_t<96, EPI_GELU_BF16>(tmA, tmW, tmO, p, st);
      case EPI_RES_F32: return launch_t<96, EPI_RES_F32>(tmA, tmW, tmO, p, st);
      case EPI_F32: return launch_t<96, EPI_F32>(tmA, tmW, tmO, p, st);
    }
  }
  set_last_error("gemm: unknown epilogue %d", epi);
  return DSG_ERR_INVALID;
}

}  // namespace dsg
