// tcgen05 / TMEM / TMA dense-layer GEMM for sm_100a with fused epilogues.
//
//   D[M,N] = sum_k A(m,k) * B(n,k)      A, B bf16, fp32 accumulation in TMEM
//
// Each operand is consumed in the layout it already has in HBM - no transposed copies anywhere:
//   K-major  : element (r,k) at r*ld + k   (row-major [M|N, K]);  TMA box 64(K) x rows, UMMA K-major descriptor
//   MN-major : element (r,k) at k*ld + r   (row-major [K, M|N]);  TMA boxes 64(MN) x 64(K), UMMA MN-major descriptor
//
// One kernel covers every dense contraction of the tabular-DNN step (the TF ops behind nn_layer,
// res/ssgd_monitor.py:57-71, and their gradients built by opt.minimize, :142):
//   EPI_FWD : Z = A_{l-1} W_l        A K-major [rows,in], B = W_l [in,out] MN-major; +bias, activation -> A_l (bf16)
//   EPI_DA  : dA = dZ_l W_l^T        A K-major [rows,out], B = W_l [in,out] K-major; *act'(A_{l-1}) -> dZ_{l-1},
//                                    column sums -> db_{l-1}
//   EPI_DW  : dW_l = A_{l-1}^T dZ_l  A = A_{l-1} [rows,in] MN-major, B = dZ_l [rows,out] MN-major; split-K over the
//                                    batch, fp32 red.add into the flat gradient
//   EPI_F32 : plain fp32 store (kernel-level parity test hook)
//   EPI_FWD_OUT : last hidden layer of a TRAINING step, output layer fused into the epilogue (K2 + K3 + K4 + output
//                 backward in one kernel; needs N = h_L <= BN so a CTA holds whole rows of A_L in TMEM):
//                 pass 1  a = act(acc + bias), z = a . w_o + b_o, y_hat = sigmoid(z), loss term, d z_hat
//                 pass 2  (accumulator re-read from TMEM) dZ_L = dz * w_o * act'(a) -> bf16, db_L / dw_o column sums,
//                         db_o, loss sum.  A_L itself never goes to HBM.
//
// Two tile configurations (template CG):
//   CG = 1 : one CTA owns a 128 x BN tile (tcgen05.mma.cta_group::1, M = 128)         - small / narrow problems
//   CG = 2 : a CTA PAIR (cluster of 2 on one TPC) owns a 256 x BN tile: tcgen05.mma.cta_group::2 with M = 256.
//            Each CTA stages its own 128 rows of A and HALF of the B tile, so every byte fetched from L2 feeds
//            twice the MMA work of CG = 1 - the 128x128 single-CTA tile is L2->SM bandwidth bound at ~45 % of the
//            tensor peak on this part (measured, DESIGN.md), the pair tile is not.
//
// Structure (persistent, one CTA per SM, 320 threads):
//   warp 0     : TMA producer   - cp.async.bulk.tensor 128B-swizzled tiles into a STAGES-deep smem ring
//   warp 1     : MMA issuer     - one thread (of the leader CTA when CG = 2) issues tcgen05.mma, commits to mbarriers
//   warps 2..9 : epilogue       - tcgen05.ld the accumulator (double-buffered in TMEM) and apply the epilogue;
//                                 two warps per TMEM lane quarter, each taking every other 32-column chunk
// M/N/K tails need no special code on the load side: TMA zero-fills out-of-bounds box elements.
#pragma once
#include <cuda.h>
#include "common.cuh"
#include "ptx.cuh"
#include "kernels.cuh"

namespace sb {

enum { EPI_FWD = 0, EPI_DA = 1, EPI_DW = 2, EPI_F32 = 3, EPI_FWD_OUT = 4 };

struct GemmTcParams {
  int M, N, K;
  int kb_per_split;  // k-blocks (of 64) per split
  int split_k;       // number of splits actually used (all non-empty)
  // EPI_FWD
  const float* bias;  // [N]
  int act;            // FWD: activation applied; DA: activation whose derivative is applied
  __nv_bfloat16* out;  // [M, ld_out] row-major (FWD, DA)
  int ld_out;
  // EPI_DA
  const __nv_bfloat16* aux;  // activation output A_{l-1} [M, ld_aux]
  int ld_aux;
  float* colsum;  // [N] fp32, atomically accumulated (bias gradient), nullable
  // EPI_DW / EPI_F32
  float* accum;  // [M, ld_acc] fp32
  int ld_acc;
  int acc_vec4;  // 1 if 16-byte aligned rows -> red.global.add.v4.f32
  // EPI_FWD_OUT (output layer + loss + its backward, res/ssgd_monitor.py:121,129)
  const float* wo;          // [N] output-layer weights (fp32)
  const float* bo;          // [1]
  const BatchDesc* desc;    // y, w of the current batch
  float* scal;              // SCAL_LOSS_SUM / SCAL_NNZ
  int loss;                 // sb_loss
  float *g_wo, *g_bo, *g_bL;  // gradient slots: dw_o [N], db_o [1], db_L [N]
  const BatchDesc* a_rows;  // non-null: operand A lives in the HBM-resident set; add a_rows->row0 to its row coordinate
  // optional: the epilogue warps clear this buffer (16-byte units) while they wait for their first accumulator.  Used by
  // the layer-0 forward GEMM of a resident step to clear the step's gradient buffer (no memset node on the chain).
  float4* zero_buf;
  long long zero_n4;
  unsigned long long* trace;  // debug: CTA 0 writes %globaltimer stamps of its pipeline milestones (nullable)
  // Split-precision modes (SB_PREC_FP32_TC / SB_PREC_BF16X2, net.cuh): every fp32 operand value is held as np bf16 PARTS
  // v = p0 + p1 (+ p2) in np equally shaped arrays; the contraction is then a plain bf16 GEMM over an EXTENDED K axis that
  // walks the part pairs (a_i, b_j) with i + j < np one after the other, all accumulating into the same fp32 TMEM tile:
  //   np = 2 : a0b0 + a0b1 + a1b0                        (relative error ~2^-17 per product)
  //   np = 3 : a0b0 + a0b1 + a1b0 + a0b2 + a1b1 + a2b0   (~2^-24: fp32-class, what TF-CPU's fp32 GEMM delivers)
  // The MMA issuer does not know about it; the TMA producer picks the pair's tensor maps per k-block.
  int np;                     // parts per value in `out` / `aux` (1 = plain bf16)
  int n_pairs;                // part pairs accumulated (1, 3 or 6); 0 is read as 1
  unsigned char pair_a[6], pair_b[6];
  long long out_ps, aux_ps;   // element stride between consecutive parts of `out` / `aux`
  // EPI_FWD, nullable: fp32 [M, ld_add] added to the pre-activation before bias + activation.  Wide+deep first layer:
  // the sum of the embedding rows of the row's categorical values, i.e. the one-hot block of Z_0 = X W_0 evaluated as a
  // gather (oracle/wide_deep.py) while this GEMM contracts only the dense columns.
  const float* addend;
  int ld_add;
};

// tensor maps of the parts of both operands (one kernel parameter, 768 B)
struct TmapSet {
  CUtensorMap a[3];
  CUtensorMap b[3];
  CUtensorMap o;   // TMA-staged epilogues: the bf16 output matrix [M, N] (box 64 columns x 128 rows, 128-byte swizzle)
  CUtensorMap x;   // EPI_DA: A_{l-1} [M, N], same box
};

// bytes of TMA staging the epilogue of an instantiation needs: the plain-bf16 forward and dA epilogues move their global
// data through 128 x 64 bf16 tiles (16 KB) with TMA - output tile double-buffered, dA additionally its A_{l-1} tile
__host__ __device__ constexpr int epi_tma_bytes(int EPI, bool GENERIC) {
  return GENERIC ? 0 : (EPI == 0 /*EPI_FWD*/ ? 2 * 16384 : (EPI == 1 /*EPI_DA*/ ? 4 * 16384 : 0));
}

template <int BN, int CG, int XB = 0>
struct GemmTcCfg {
  static_assert(CG == 1 || CG == 2, "cta group");
  static_assert(BN == 64 || BN == 128 || BN == 256, "tile N");
  static_assert(CG == 1 || BN >= 128, "pair tiles need BN >= 128 (each CTA stages BN/2 >= 64 rows of B)");
  static constexpr int BM = 128;        // rows of the tile owned by ONE CTA
  static constexpr int TILE_M = BM * CG;  // rows of the (pair) tile
  static constexpr int BK = 64;         // 64 bf16 = 128 B = one swizzle row
  static constexpr int BN_CTA = BN / CG;  // B rows staged by one CTA
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = BN_CTA * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  // shared memory besides the operand ring: align slack, barriers, epilogue scratch, bias (+ w_o), per-warp transpose tiles
  // (only the epilogues without TMA staging use them), column-sum accumulators, TMA staging tiles (XB)
  static constexpr int TR_BYTES = XB > 0 ? 0 : 8 * 2048;
  static constexpr int FIXED_BYTES = 1024 + 256 + 2048 + 2048 + TR_BYTES + 4096 + XB;
  static constexpr int RING_BUDGET = (XB > 0 ? 232448 - FIXED_BYTES : 200 * 1024);   // (the un-staged kernels keep their round-1 depth)
  static constexpr int STAGES = RING_BUDGET / STAGE_BYTES > 8 ? 8 : RING_BUDGET / STAGE_BYTES;
  static constexpr int TMEM_COLS = (2 * BN <= 32) ? 32 : (2 * BN <= 64 ? 64 : (2 * BN <= 128 ? 128 : (2 * BN <= 256 ? 256 : 512)));
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + FIXED_BYTES;
  static_assert(SMEM_BYTES <= 232448, "shared memory budget");
  // Epilogue warps.  The dA epilogue (the longest: A_{l-1} tile in, act', column sums, dZ tile out) runs SIXTEEN warps in two
  // groups of eight that work on alternate 64-column blocks (cfg2 dA_1 19.7 -> 18.8 us, dA_2 7.9 -> 6.8 us; the forward
  // epilogue gained nothing and keeps eight: 320 threads x <= 115 registers leave room for an exchange block on the same SM,
  // see xchg_p2p.cuh).
  static constexpr int EPI_WARPS = XB >= 4 * 16384 ? 16 : 8;
  static constexpr int EPI_GROUPS = EPI_WARPS / 8;
  static constexpr int EPI_THREADS = 32 * EPI_WARPS;
  static constexpr int THREADS = 64 + EPI_THREADS;
};

// ---- epilogue element functions, specialised per activation so the switch is hoisted out of the element loop
template <int ACT>
__device__ __forceinline__ void epi_fwd_chunk(float (&v)[32], const float (&b)[32]) {
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = act_apply(v[j] + b[j], ACT);
}
template <int ACT>
__device__ __forceinline__ void epi_da_chunk(float (&v)[32], const __nv_bfloat16* ah) {
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] *= act_grad_from_out(__bfloat162float(ah[j]), ACT);
}

// ACT_T: activation fixed at compile time (EPI_FWD_OUT: its two-pass epilogue with every activation variant inlined was
// 7.4 k instructions and spent 38 % of its warp samples waiting for instruction fetch, profiles/ncu_r01_*), or
// SB_ACT_AT_RUNTIME = read p.act.
constexpr int SB_ACT_AT_RUNTIME = -100;

// GENERIC = false: the plain-bf16 epilogues (performance mode; their instruction footprint decides the epilogue speed - a
// 7.4 k-instruction epilogue spent 38 % of its issue slots waiting for instruction fetch).  GENERIC = true adds the cold
// features at compile time: split-precision part stores / loads (np > 1) and the fp32 addend of the wide+deep first layer.
template <int BN, int EPI, bool A_MN, bool B_MN, int CG, int ACT_T = SB_ACT_AT_RUNTIME, bool GENERIC = false>
__global__ void __launch_bounds__((GemmTcCfg<BN, CG, epi_tma_bytes(EPI, GENERIC)>::THREADS), 1)
gemm_tc_kernel(const __grid_constant__ TmapSet tms, const GemmTcParams p) {
  using Cfg = GemmTcCfg<BN, CG, epi_tma_bytes(EPI, GENERIC)>;
  constexpr bool TMA_EPI = epi_tma_bytes(EPI, GENERIC) > 0;
  const int act_sel = (ACT_T == SB_ACT_AT_RUNTIME) ? p.act : ACT_T;
  constexpr int BM = Cfg::BM, BK = Cfg::BK, STAGES = Cfg::STAGES, TILE_M = Cfg::TILE_M, BN_CTA = Cfg::BN_CTA;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;  // SWIZZLE_128B needs 1024 B alignment
  const uint32_t xbuf_base = smem_base + STAGES * Cfg::STAGE_BYTES;            // TMA staging tiles (1024-byte aligned)
  const uint32_t bar_base = xbuf_base + epi_tma_bytes(EPI, GENERIC);
  // barrier layout (8 B each): full[STAGES], empty[STAGES], tmem_full[2], tmem_empty[2], then tmem base slot.
  // CG = 2: full[] and tmem_empty[] are only used in the leader CTA (rank 0); empty[] / tmem_full[] in both.
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 4);
  auto smem_a = [&](int s) { return smem_base + s * Cfg::STAGE_BYTES; };
  auto smem_b = [&](int s) { return smem_base + s * Cfg::STAGE_BYTES + Cfg::A_BYTES; };

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const bool tracing = p.trace != nullptr && blockIdx.x == 0;
  auto stamp = [&](int slot) { if (tracing) p.trace[slot] = globaltimer_ns(); };
  if (threadIdx.x == 0) stamp(0);  // kernel entry
  const uint32_t rank = (CG == 2) ? cluster_ctarank() : 0u;  // CTA rank inside the pair
  const bool leader = rank == 0;

  const int n_pairs = p.n_pairs > 0 ? p.n_pairs : 1;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tms.a[0]);
    tma_prefetch_desc(&tms.b[0]);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), CG);  // CG = 2: leader producer's arrive.expect_tx + peer producer's remote arrive
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), Cfg::EPI_WARPS * CG);  // one arrival per epilogue warp (of both CTAs)
    }
    fence_barrier_init();
  }
  __syncwarp();
  if constexpr (CG == 2) cluster_sync_all();  // both CTAs alive before the pair-wide TMEM allocation
  if (warp == 2) {
    if constexpr (CG == 2) tmem_alloc_cg2<Cfg::TMEM_COLS>(tmem_slot);
    else tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  }
  tcgen05_fence_before();
  if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  // PDL: everything above (barrier init, TMEM allocation, descriptor prefetch) overlapped the previous kernel's tail;
  // from here on global memory written by it is touched.
  if (threadIdx.x == 0) stamp(1);  // setup done
  pdl_wait();
  pdl_launch_dependents();
  if (threadIdx.x == 0) stamp(2);  // dependencies resolved

  const int tiles_m = (p.M + TILE_M - 1) / TILE_M;
  const int tiles_n = (p.N + BN - 1) / BN;
  const int n_tiles = tiles_m * tiles_n;
  const int n_work = n_tiles * p.split_k;
  const int part_kb = (p.K + BK - 1) / BK;         // k-blocks of ONE part pair
  const int total_kb = part_kb * n_pairs;          // extended K axis: the pairs one after the other
  const int w_first = (CG == 2) ? (blockIdx.x >> 1) : blockIdx.x;   // work items are per CTA (CG=1) or per pair (CG=2)
  const int w_step = (CG == 2) ? (gridDim.x >> 1) : gridDim.x;

  if (warp == 0) {
    // ================= TMA producer (every CTA) =================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const int a_row0 = (p.a_rows != nullptr) ? p.a_rows->row0 : 0;  // batch position inside the resident set
      for (int w = w_first; w < n_work; w += w_step) {
        const int tile = w % n_tiles, ks = w / n_tiles;
        const int tm = tile / tiles_n, tn = tile % tiles_n;
        const int kb0 = ks * p.kb_per_split;
        const int kb1 = min(total_kb, kb0 + p.kb_per_split);
        const int m0 = tm * TILE_M + static_cast<int>(rank) * BM;      // this CTA's rows of A
        const int n0 = tn * BN + static_cast<int>(rank) * BN_CTA;      // this CTA's share of the B tile
        for (int kbx = kb0; kbx < kb1; ++kbx) {
          const int pp = (n_pairs > 1) ? kbx / part_kb : 0;     // which part pair this k-block belongs to
          const int kb = kbx - pp * part_kb;
          const CUtensorMap* tmA = &tms.a[n_pairs > 1 ? p.pair_a[pp] : 0];
          const CUtensorMap* tmB = &tms.b[n_pairs > 1 ? p.pair_b[pp] : 0];
          mbar_wait(empty_bar(stage), phase ^ 1);
          const uint32_t fb = full_bar(stage);
          if (leader) mbar_arrive_expect_tx(fb, Cfg::STAGE_BYTES * CG);
          auto load = [&](uint32_t dst, const CUtensorMap* tm_, int c0, int c1) {
            if constexpr (CG == 2) tma_load_2d_cg2(dst, tm_, fb, c0, c1);
            else tma_load_2d(dst, tm_, fb, c0, c1);
          };
          if constexpr (A_MN) {
#pragma unroll
            for (int i = 0; i < BM / 64; ++i)  // 64(MN) x 64(K) boxes, 8 KB each, side by side along MN
              load(smem_a(stage) + i * 8192, tmA, m0 + i * 64, kb * BK + a_row0);   // rows of the set = K here
          } else {
            load(smem_a(stage), tmA, kb * BK, m0 + a_row0);
          }
          if constexpr (B_MN) {
#pragma unroll
            for (int i = 0; i < BN_CTA / 64; ++i)
              load(smem_b(stage) + i * 8192, tmB, n0 + i * 64, kb * BK);
          } else {
            load(smem_b(stage), tmB, kb * BK, n0);
          }
          if constexpr (CG == 2) {
            if (!leader) mbar_arrive_cluster(fb, 0);  // second arrival on the leader's full barrier
          }
          if (kbx == kb0 && w == w_first) stamp(3);  // first TMA issued
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();   // the whole warp reaches the final block barrier together (bar.sync counts warps, not lanes)
  } else if (warp == 1) {
    // ================= MMA issuer (leader CTA only when CG = 2) =================
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = make_idesc_bf16(TILE_M, BN, A_MN ? 1u : 0u, B_MN ? 1u : 0u);
      // descriptor step for 16 elements along K: K-major = 32 B inside the swizzle row; MN-major = 16 rows of 128 B
      constexpr uint32_t a_kstep = A_MN ? (2048u >> 4) : (32u >> 4);
      constexpr uint32_t b_kstep = B_MN ? (2048u >> 4) : (32u >> 4);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int w = w_first; w < n_work; w += w_step, ++it) {
        const int ks = w / n_tiles;
        const int kb0 = ks * p.kb_per_split;
        const int kb1 = min(total_kb, kb0 + p.kb_per_split);
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1);  // epilogue(s) have drained this accumulator
        tcgen05_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar(stage), phase);  // TMA bytes of both CTAs have landed
          tcgen05_fence_after();
          if (kb == kb0 && w == w_first) stamp(4);  // first stage landed
          const uint64_t da = A_MN ? make_mnmajor_sw128_desc(smem_a(stage), 8192u) : make_kmajor_sw128_desc(smem_a(stage));
          const uint64_t db = B_MN ? make_mnmajor_sw128_desc(smem_b(stage), 8192u) : make_kmajor_sw128_desc(smem_b(stage));
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint32_t accumulate = (kb > kb0 || k > 0) ? 1u : 0u;
            if constexpr (CG == 2) umma_bf16_cg2(tmem_d, da + a_kstep * k, db + b_kstep * k, idesc, accumulate);
            else umma_bf16(tmem_d, da + a_kstep * k, db + b_kstep * k, idesc, accumulate);
          }
          // frees the smem slot (in both CTAs) once these MMAs have read it
          if constexpr (CG == 2) umma_commit_cg2(empty_bar(stage)); else umma_commit(empty_bar(stage));
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        // accumulator complete -> epilogue (of both CTAs)
        if constexpr (CG == 2) umma_commit_cg2(tfull_bar(acc)); else umma_commit(tfull_bar(acc));
        if (w == w_first) stamp(5);  // all MMAs of the first tile issued
      }
    }
    __syncwarp();
  } else {
    // ================= epilogue warps (2..9), every CTA: its own 128 rows x BN columns =================
    const int quarter = warp & 3;        // TMEM lane quarter this warp may access
    const int half = ((warp - 2) >> 2) & 1;    // which of the two warps (of a group) sharing the quarter
    const int grp = (warp - 2) >> 3;           // TMA-staged epilogues: group 0 / 1 takes the even / odd 64-column blocks
    const int et = static_cast<int>(threadIdx.x) - 64;   // 0 .. EPI_THREADS-1 over all epilogue warps
    constexpr int ET = Cfg::EPI_THREADS;
    constexpr int NGRP = Cfg::EPI_GROUPS;
    auto bar_all = [&]() { asm volatile("bar.sync 1, %0;" ::"n"(Cfg::EPI_THREADS) : "memory"); };    // every epilogue warp
    auto bar_grp = [&]() { asm volatile("bar.sync %0, 256;" ::"r"(2 + grp) : "memory"); };              // the eight warps of a group
    if (p.zero_buf != nullptr) {
      // idle time before the first accumulator completes: clear the step's gradient buffer (read by nobody before the
      // next kernel boundary)
      const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
      for (long long i = static_cast<long long>(blockIdx.x) * ET + et; i < p.zero_n4; i += static_cast<long long>(gridDim.x) * ET) p.zero_buf[i] = z4;
    }
    // EPI_FWD_OUT: bias and w_o of the (single) n-tile staged in shared memory once, before the accumulator wait, so the
    // two epilogue passes read them with broadcast ld.shared instead of dependent global loads
    const uint32_t sm_vec = bar_base + 8u * (2 * STAGES + 4) + 16u + 2048u;   // [bias BN floats][w_o BN floats]
    // Coalescing: tcgen05.ld hands thread t the 32 columns of ROW t, so a direct 16-byte access per thread touches 32
    // different rows (32 L1 wavefronts per instruction).  Every global access of the epilogue therefore goes through a
    // warp-private 32 x 64 B tile in shared memory (16-byte pieces XOR-swizzled by row pair -> conflict-free on both
    // sides): on the global side lane l handles piece (l & 3) of rows 8 i + (l >> 2), i = 0..3, i.e. four lanes cover
    // 64 contiguous bytes of a row and one instruction touches 8 rows instead of 32.
    const uint32_t sm_stage = sm_vec + 2048u + static_cast<uint32_t>(warp - 2) * 2048u;
    // Column sums (bias gradients; dw_o of the fused output layer) are accumulated per CTA in shared memory and flushed to
    // the flat gradient ONCE per tile and column: one red.global per column per 128 rows instead of one per 32 rows.  With
    // one red per warp and chunk, the 8192 x 1024 dA GEMM of cfg2 sent 262 k reds to 32 cache lines and spent 3/4 of its time
    // waiting for the L2 atomic units (tensor pipe 25 % active, profiles/ncu_r01_cfg2_gemm_full.txt).
    // layout: [buffer (tile parity)][array 0: db | array 1: dw_o][BN] floats
    const uint32_t sm_col = sm_vec + 2048u + static_cast<uint32_t>(Cfg::TR_BYTES);
    // TMA-staged epilogue (plain-bf16 forward / dA): the 128 x BN tile leaves in 64-column blocks.  Block k: every thread
    // writes the 32 bf16 of its row-chunk as four 16-byte pieces into the 128-byte-swizzled 128 x 64 tile xo[k & 1] (the layout
    // the output tensor map expects; a quarter-warp covers all 32 banks), one thread issues cp.async.bulk.tensor (store) for
    // the tile; dA additionally gets its A_{l-1} block by TMA load into xa[k & 1] (issued two blocks ahead) and reads it back
    // with the same swizzle.  No ld.shared / st.global per element, no transposes, M / N tails clipped by the tensor map.
    auto xo = [&](int b) { return xbuf_base + static_cast<uint32_t>(b) * 16384u; };
    auto xa = [&](int b) { return xbuf_base + 32768u + static_cast<uint32_t>(b) * 16384u; };
    auto aux_bar = [&](int b) { return bar_base + 8u * (2 * STAGES + 4) + 16u + 8u * static_cast<uint32_t>(b); };   // (scratch of EPI_FWD_OUT, unused here)
    const int rt = quarter * 32 + lane;                                   // row of this thread inside the CTA's 128 rows
    auto piece = [&](int half_, int i) { return static_cast<uint32_t>(rt) * 128u + static_cast<uint32_t>(((half_ * 4 + i) ^ (rt & 7)) << 4); };
    const bool xthread = (((warp - 2) & 7) == 0 && lane == 0);            // first lane of a group: issues its TMA loads / stores
    unsigned xblk = 0;                                                    // 64-column blocks processed so far by this GROUP
    if constexpr (TMA_EPI && EPI == EPI_DA) {
      if (warp == 2 && lane == 0) { mbar_init(aux_bar(0), 1); mbar_init(aux_bar(1), 1); fence_barrier_init(); }
      bar_all();
    }
    auto col_slot = [&](int buf, int arr, int j) { return sm_col + static_cast<uint32_t>(((buf * 2 + arr) * BN + j) * 4); };
    auto red_shared = [](uint32_t a, float v) { asm volatile("red.shared.add.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); };
    if constexpr (EPI == EPI_DA || EPI == EPI_FWD_OUT) {
      for (int j = et; j < 4 * BN; j += ET) asm volatile("st.shared.f32 [%0], %1;" ::"r"(sm_col + static_cast<uint32_t>(j) * 4u), "f"(0.f) : "memory");
      bar_all();
    }
    // after every epilogue warp has added its sums of tile `it`: one thread per column flushes and clears buffer it & 1
    auto flush_cols = [&](int it_, int tn_, float* dst0, float* dst1) {
      bar_all();
      for (int j = et; j < BN; j += ET) {
        const int col = tn_ * BN + j;
#pragma unroll
        for (int arr = 0; arr < 2; ++arr) {
          float* dst = arr == 0 ? dst0 : dst1;
          if (dst == nullptr) continue;
          float vsum;
          asm volatile("ld.shared.f32 %0, [%1];" : "=f"(vsum) : "r"(col_slot(it_ & 1, arr, j)) : "memory");
          asm volatile("st.shared.f32 [%0], %1;" ::"r"(col_slot(it_ & 1, arr, j)), "f"(0.f) : "memory");
          if (col < p.N && vsum != 0.f) red_add_f32(dst + col, vsum);
        }
      }
    };
    const int lrow = lane >> 2, lpc = lane & 3;
    auto stg = [&](int r, int pc) { return sm_stage + static_cast<uint32_t>(r) * 64u + static_cast<uint32_t>((pc ^ ((r >> 1) & 3)) << 4); };
    auto sts4 = [](uint32_t a, const uint4& v) {
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
    };
    auto lds4 = [](uint32_t a) {
      uint4 v;
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
      return v;
    };
    auto row_to_lanes = [&](const uint4 (&mine)[4], uint4 (&out)[4]) {   // thread-owns-row -> lane-coalesced
#pragma unroll
      for (int q = 0; q < 4; ++q) sts4(stg(lane, q), mine[q]);
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 4; ++i) out[i] = lds4(stg(8 * i + lrow, lpc));
      __syncwarp();
    };
    auto lanes_to_row = [&](const uint4 (&in)[4], uint4 (&mine)[4]) {    // lane-coalesced -> thread-owns-row
#pragma unroll
      for (int i = 0; i < 4; ++i) sts4(stg(8 * i + lrow, lpc), in[i]);
      __syncwarp();
#pragma unroll
      for (int q = 0; q < 4; ++q) mine[q] = lds4(stg(lane, q));
      __syncwarp();
    };
    if constexpr (EPI == EPI_FWD_OUT) {
#pragma unroll
      for (int j = et; j < 2 * BN; j += ET) {
        const int col = (j < BN) ? j : j - BN;
        const float* src = (j < BN) ? p.bias : p.wo;
        const float v = (col < p.N) ? __ldg(src + col) : 0.f;
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(sm_vec + static_cast<uint32_t>(j) * 4u), "f"(v) : "memory");
      }
      bar_all();
    }
    int it = 0;
    for (int w = w_first; w < n_work; w += w_step, ++it) {
      const int tile = w % n_tiles;
      const int tm = tile / tiles_n, tn = tile % tiles_n;
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int row = tm * TILE_M + static_cast<int>(rank) * BM + quarter * 32 + lane;  // output row of this thread
      const bool row_ok = row < p.M;
      // operands of the epilogue that do not depend on the accumulator are fetched BEFORE waiting for it (the epilogue
      // warps idle during the main loop): per-row label / weight / n_nz / b_o of the fused output layer, and the first
      // chunk of A_{l-1} of the dA epilogue (the next chunk's is fetched while the current one is processed)
      float pre_y = 0.f, pre_w = 0.f, pre_nnz = 0.f, pre_bo = 0.f;
      // dA epilogue: A_{l-1} of EVERY chunk this warp will handle is fetched before the accumulator wait (the loads do not
      // depend on it) and kept in registers as a shift queue, so that one L2 / HBM latency is paid per tile instead of one
      // per 32-column chunk (the chunk-ahead prefetch left this epilogue latency bound: 5 us per 256 x 256 tile at cfg2)
      constexpr int AUXQ = (EPI == EPI_DA && !TMA_EPI) ? (BN / 64 > 0 ? BN / 64 : 1) : 1;
      uint4 aux_q[AUXQ][4];
      const int row_base = tm * TILE_M + static_cast<int>(rank) * BM + quarter * 32;   // first row of this warp's 32
      // store a 32 x 64 B tile held one-row-per-thread (4 pieces each) to a row-major bf16 matrix, coalesced
      auto store_rows_bf16 = [&](const uint4 (&mine)[4], __nv_bfloat16* base, int ld, int col0_, bool all_cols) {
        uint4 oc[4];
        row_to_lanes(mine, oc);
        const int gc = col0_ + 8 * lpc;
        if (all_cols || gc < ld) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int gr = row_base + 8 * i + lrow;
            if (gr < p.M) *reinterpret_cast<uint4*>(base + static_cast<size_t>(gr) * ld + gc) = oc[i];
          }
        }
      };
      // split-precision output: part 0 = bf16(v), part k = bf16(v - sum of the previous parts); np = 1 is the plain store.
      // x is left untouched (the residual of part k is re-derived from x: at most two extra cvt + sub per element).
      auto store_parts = [&](const float (&x)[32], __nv_bfloat16* base, long long ps, int ld, int col0_, bool all_cols) {
        const int np_ = GENERIC ? p.np : 1;
#pragma unroll 1
        for (int part = 0; part < np_; ++part) {
          auto res = [&](float r) {
            if constexpr (GENERIC) {
              for (int i = 0; i < part; ++i) r -= __bfloat162float(__float2bfloat16_rn(r));
            }
            return r;
          };
          uint4 o[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            o[q].x = pack_bf16x2(res(x[q * 8 + 0]), res(x[q * 8 + 1]));
            o[q].y = pack_bf16x2(res(x[q * 8 + 2]), res(x[q * 8 + 3]));
            o[q].z = pack_bf16x2(res(x[q * 8 + 4]), res(x[q * 8 + 5]));
            o[q].w = pack_bf16x2(res(x[q * 8 + 6]), res(x[q * 8 + 7]));
          }
          store_rows_bf16(o, base + part * ps, ld, col0_, all_cols);
        }
      };
      auto load_aux = [&](int c, uint4 (&a)[4], int part = 0) {   // lane-coalesced fetch of chunk c of A_{l-1}; zeros outside
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = make_uint4(0, 0, 0, 0);
        const int gc = tn * BN + c * 32 + 8 * lpc;
        if (c < BN / 32 && tn * BN + c * 32 < p.N && gc < p.ld_aux) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int gr = row_base + 8 * i + lrow;
            if (gr < p.M) a[i] = __ldg(reinterpret_cast<const uint4*>(p.aux + part * p.aux_ps + static_cast<size_t>(gr) * p.ld_aux + gc));
          }
        }
      };
      if constexpr (EPI == EPI_FWD_OUT) {
        if (row_ok) { pre_y = __ldg(p.desc->y + row); pre_w = __ldg(p.desc->w + row); }
        pre_nnz = p.scal[SCAL_NNZ];
        pre_bo = __ldg(p.bo);
      }
      if constexpr (EPI == EPI_DA && !TMA_EPI) {
#pragma unroll
        for (int i = 0; i < AUXQ; ++i) load_aux(half + 2 * i, aux_q[i]);
      }
      // blocks of 64 columns this tile really has (the same number for every warp: the block loop contains barriers)
      const int tile_cols = (p.N - tn * BN) < BN ? (p.N - tn * BN) : BN;
      const int nblk = (tile_cols + 63) / 64;
      const int x_row0 = tm * TILE_M + static_cast<int>(rank) * BM;      // TMA row coordinate of this CTA's 128 rows
      if constexpr (TMA_EPI && EPI == EPI_DA) {
        if constexpr (NGRP == 2) {
          if (xthread && grp < nblk) {       // A_{l-1} of this group's first block (its buffer is free: the group has left the previous tile)
            mbar_arrive_expect_tx(aux_bar(grp), 16384u);
            tma_load_2d(xa(grp), &tms.x, aux_bar(grp), tn * BN + grp * 64, x_row0);
          }
        } else {
          if (xthread) {
            for (int k = 0; k < 2 && k < nblk; ++k) {       // A_{l-1} of the first two blocks (buffers free: every warp has left the previous tile)
              const int b = (xblk + k) & 1;
              mbar_arrive_expect_tx(aux_bar(b), 16384u);
              tma_load_2d(xa(b), &tms.x, aux_bar(b), tn * BN + k * 64, x_row0);
            }
          }
        }
      }
      const uint32_t sm_bias = sm_vec + static_cast<uint32_t>(it & 1) * (BN * 4u);   // EPI_FWD: this tile's bias, double-buffered
      if constexpr (EPI == EPI_FWD) {
        // (a warp reaches this barrier only after finishing the previous tile, so buffer it & 1 is no longer read)
#pragma unroll
        for (int j = et; j < BN; j += ET) {
          const int col = tn * BN + j;
          const float bv = (col < p.N) ? __ldg(p.bias + col) : 0.f;
          asm volatile("st.shared.f32 [%0], %1;" ::"r"(sm_bias + static_cast<uint32_t>(j) * 4u), "f"(bv) : "memory");
        }
        bar_all();
      }
      mbar_wait(tfull_bar(acc), acc_phase);
      tcgen05_fence_after();
      if (w == w_first && warp == 2 && lane == 0) stamp(6);  // first accumulator complete
      if constexpr (EPI == EPI_FWD_OUT) {
        // ---------- fused output layer (tiles_n == 1: this CTA's TMEM holds complete rows of A_L) ----------
        const uint32_t zs = bar_base + 8u * (2 * STAGES + 4) + 16u + static_cast<uint32_t>(it & 1) * 1024u;  // zpart[2][128]
        const int rl = quarter * 32 + lane;
        // 32 consecutive fp32 of the staged bias (which = 0) / w_o (which = 1): 8 broadcast 16-byte ld.shared
        auto load_vec32 = [&](int which, int col0, float (&o)[32]) {
          const uint32_t a = sm_vec + static_cast<uint32_t>(which * BN + col0) * 4u;
#pragma unroll
          for (int q = 0; q < 8; ++q)
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                         : "=f"(o[4 * q]), "=f"(o[4 * q + 1]), "=f"(o[4 * q + 2]), "=f"(o[4 * q + 3])
                         : "r"(a + 16u * q));
        };
        auto load_act = [&](int c, float (&v)[32]) {   // a = act(acc + bias) for chunk c; 0 beyond N
          const int col0 = c * 32;
          uint32_t raw[32];
          tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * BN + c * 32, raw);
          tmem_ld_wait();
          float b[32];
          load_vec32(0, col0, b);
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(raw[j]);
          switch (act_sel) {
            case SB_ACT_RELU: epi_fwd_chunk<SB_ACT_RELU>(v, b); break;
            case SB_ACT_SIGMOID: epi_fwd_chunk<SB_ACT_SIGMOID>(v, b); break;
            case SB_ACT_TANH: epi_fwd_chunk<SB_ACT_TANH>(v, b); break;
            case SB_ACT_LEAKYRELU: epi_fwd_chunk<SB_ACT_LEAKYRELU>(v, b); break;
            default: epi_fwd_chunk<SB_ACT_NONE>(v, b); break;
          }
          if (col0 + 32 > p.N) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (col0 + j >= p.N) v[j] = 0.f;
          }
        };
        // pass 1: partial dot product of this thread's row with w_o over this warp's chunks
        float zp = 0.f;
#pragma unroll 1
        for (int c = half; c < BN / 32; c += 2) {
          if (c * 32 >= p.N) break;
          float v[32], wv[32];
          load_act(c, v);
          load_vec32(1, c * 32, wv);
#pragma unroll
          for (int j = 0; j < 32; ++j) zp = fmaf(v[j], wv[j], zp);
        }
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(zs + static_cast<uint32_t>(half * 128 + rl) * 4u), "f"(zp) : "memory");
        asm volatile("bar.sync 1, 256;" ::: "memory");   // the 8 epilogue warps only
        float z0, z1;
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(z0) : "r"(zs + static_cast<uint32_t>(rl) * 4u) : "memory");
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(z1) : "r"(zs + static_cast<uint32_t>(128 + rl) * 4u) : "memory");
        const float z = z0 + z1 + pre_bo;
        float dz = 0.f, lossv = 0.f;
        if (row_ok) {
          const float nnz = pre_nnz;
          const float inv_nnz = nnz > 0.f ? 1.f / nnz : 0.f;
          const float yh = sigmoidf_stable(z);
          const float y = pre_y, wgt = pre_w;
          if (p.loss == SB_LOSS_MSE) {
            const float d = yh - y;
            lossv = wgt * d * d;
            dz = 2.f * wgt * d * yh * (1.f - yh) * inv_nnz;
          } else {
            lossv = wgt * (fmaxf(z, 0.f) - z * y + log1pf(expf(-fabsf(z))));
            dz = wgt * (yh - y) * inv_nnz;
          }
        }
        if (half == 0) {
          const float ls = warp_sum(lossv), ds = warp_sum(dz);
          if (lane == 0) { atomicAdd(p.scal + SCAL_LOSS_SUM, ls); atomicAdd(p.g_bo, ds); }
        }
        // pass 2: rank-1 backward of the output layer through act'
#pragma unroll 1
        for (int c = half; c < BN / 32; c += 2) {
          const int col0 = c * 32;
          if (col0 >= p.N) break;
          float v[32], g[32];
          load_act(c, v);
          load_vec32(1, col0, g);      // g starts as w_o (0 beyond N)
          switch (act_sel) {
#define SB_G(ACT) _Pragma("unroll") for (int j = 0; j < 32; ++j) g[j] = dz * g[j] * act_grad_from_out(v[j], ACT);
            case SB_ACT_RELU: SB_G(SB_ACT_RELU) break;
            case SB_ACT_SIGMOID: SB_G(SB_ACT_SIGMOID) break;
            case SB_ACT_TANH: SB_G(SB_ACT_TANH) break;
            case SB_ACT_LEAKYRELU: SB_G(SB_ACT_LEAKYRELU) break;
            default: SB_G(SB_ACT_NONE) break;
#undef SB_G
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] *= dz;          // dz * a  -> dw_o contributions (0 for rows >= M)
          store_parts(g, p.out, p.out_ps, p.ld_out, col0, false);       // dZ_L (bf16, or its parts)
          const float sb_ = warp_colsum_32x32(g, lane);
          const float sw_ = warp_colsum_32x32(v, lane);
          red_shared(col_slot(it & 1, 0, col0 + lane), sb_);       // columns beyond N carry zeros
          red_shared(col_slot(it & 1, 1, col0 + lane), sw_);
        }
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) {
          if constexpr (CG == 2) mbar_arrive_cluster(tempty_bar(acc), 0);
          else mbar_arrive(tempty_bar(acc));
        }
        flush_cols(it, 0, p.g_bL, p.g_wo);
        continue;
      }
#pragma unroll 1
      for (int c = TMA_EPI ? 2 * grp + half : half; c < BN / 32; c += (TMA_EPI ? 2 * NGRP : 2)) {
        const int col0 = tn * BN + c * 32;
        if constexpr (TMA_EPI) {
          if ((c >> 1) >= nblk) break;          // same trip count for the eight warps of a group
        } else {
          if (col0 >= p.N) break;  // whole chunk out of range (warp-uniform)
        }
        const bool chunk_ok = col0 < p.N;       // (TMA path: a warp whose 32 columns lie beyond N only joins the barriers)
        uint32_t raw[32];
        if (chunk_ok) {
          tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * BN + c * 32, raw);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) raw[j] = 0u;
        }
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(raw[j]);
        const bool full = col0 + 32 <= p.N;  // warp-uniform fast path
        // staging tiles: two groups -> each owns one output and one A_{l-1} tile; one group -> it alternates between two
        const int xb = NGRP == 2 ? grp : static_cast<int>(xblk & 1u);

        if constexpr (EPI == EPI_FWD) {
          if (GENERIC && p.addend != nullptr && row_ok) {
            const float* ad = p.addend + static_cast<size_t>(row) * p.ld_add + col0;
            if (full && (p.ld_add & 3) == 0) {
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                const float4 a4 = __ldg(reinterpret_cast<const float4*>(ad) + q);
                v[4 * q] += a4.x; v[4 * q + 1] += a4.y; v[4 * q + 2] += a4.z; v[4 * q + 3] += a4.w;
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (col0 + j < p.N) v[j] += __ldg(ad + j);
            }
          }
          float b[32];   // staged before the accumulator wait (0 beyond N)
#pragma unroll
          for (int q = 0; q < 8; ++q)
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                         : "=f"(b[4 * q]), "=f"(b[4 * q + 1]), "=f"(b[4 * q + 2]), "=f"(b[4 * q + 3])
                         : "r"(sm_bias + static_cast<uint32_t>(c * 32 + 4 * q) * 4u));
          switch (act_sel) {
            case SB_ACT_RELU: epi_fwd_chunk<SB_ACT_RELU>(v, b); break;
            case SB_ACT_SIGMOID: epi_fwd_chunk<SB_ACT_SIGMOID>(v, b); break;
            case SB_ACT_TANH: epi_fwd_chunk<SB_ACT_TANH>(v, b); break;
            case SB_ACT_LEAKYRELU: epi_fwd_chunk<SB_ACT_LEAKYRELU>(v, b); break;
            default: epi_fwd_chunk<SB_ACT_NONE>(v, b); break;
          }
        } else if constexpr (EPI == EPI_DA) {
          // multiply by act'(A_{l-1}[row, col]) read as bf16 (64 B per thread per chunk, fetched one chunk ahead)
          uint4 a4[4];
          if constexpr (TMA_EPI) {
            mbar_wait(aux_bar(xb), (NGRP == 2 ? xblk : (xblk >> 1)) & 1u);   // this block's A_{l-1} tile has landed
#pragma unroll
            for (int i = 0; i < 4; ++i) a4[i] = lds4(xa(xb) + piece(half, i));
          } else {
            lanes_to_row(aux_q[0], a4);
#pragma unroll
            for (int i = 0; i + 1 < AUXQ; ++i) {
#pragma unroll
              for (int k = 0; k < 4; ++k) aux_q[i][k] = aux_q[i + 1][k];
            }
          }
          __nv_bfloat16* ah = reinterpret_cast<__nv_bfloat16*>(a4);
          if (GENERIC && p.np > 1 && (act_sel == SB_ACT_SIGMOID || act_sel == SB_ACT_TANH)) {
            // act' needs the VALUE of A_{l-1}: add the lower parts (fetched here, not prefetched: the split modes are the
            // parity modes).  relu / leaky relu only look at the sign, which part 0 carries.
            float af[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) af[j] = __bfloat162float(ah[j]);
            for (int part = 1; part < p.np; ++part) {
              uint4 lo_l[4], lo_r[4];
              load_aux(c, lo_l, part);
              lanes_to_row(lo_l, lo_r);
              const __nv_bfloat16* lh = reinterpret_cast<const __nv_bfloat16*>(lo_r);
#pragma unroll
              for (int j = 0; j < 32; ++j) af[j] += __bfloat162float(lh[j]);
            }
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] *= act_grad_from_out(af[j], act_sel);
          } else
          switch (act_sel) {
            case SB_ACT_RELU: epi_da_chunk<SB_ACT_RELU>(v, ah); break;
            case SB_ACT_SIGMOID: epi_da_chunk<SB_ACT_SIGMOID>(v, ah); break;
            case SB_ACT_TANH: epi_da_chunk<SB_ACT_TANH>(v, ah); break;
            case SB_ACT_LEAKYRELU: epi_da_chunk<SB_ACT_LEAKYRELU>(v, ah); break;
            default: break;
          }
          if (!row_ok || !full) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (!row_ok || col0 + j >= p.N) v[j] = 0.f;
          }
        }

        if constexpr (EPI == EPI_FWD || EPI == EPI_DA) {
          if constexpr (TMA_EPI) {
            uint4 o[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              o[q].x = pack_bf16x2(v[q * 8 + 0], v[q * 8 + 1]);
              o[q].y = pack_bf16x2(v[q * 8 + 2], v[q * 8 + 3]);
              o[q].z = pack_bf16x2(v[q * 8 + 4], v[q * 8 + 5]);
              o[q].w = pack_bf16x2(v[q * 8 + 6], v[q * 8 + 7]);
            }
            if (xthread) {                                         // the last store out of this tile has finished reading it ...
              if constexpr (NGRP == 2) tma_store_wait_read<0>(); else tma_store_wait_read<1>();
            }
            bar_grp();                                             // (B) ... which every warp of the group may now overwrite
#pragma unroll
            for (int q = 0; q < 4; ++q) sts4(xo(xb) + piece(half, q), o[q]);
            fence_proxy_async();                                   // generic-proxy writes -> visible to the TMA engine
            bar_grp();                                             // (A) the block's tile is complete; A_{l-1} tile consumed
            if (xthread) {
              tma_store_2d(&tms.o, xo(xb), tn * BN + (c >> 1) * 64, x_row0);
              tma_store_commit();
              if constexpr (EPI == EPI_DA) {
                if ((c >> 1) + 2 < nblk) {                         // A_{l-1} of the group's next block, into the tile just consumed
                  mbar_arrive_expect_tx(aux_bar(xb), 16384u);
                  tma_load_2d(xa(xb), &tms.x, aux_bar(xb), tn * BN + ((c >> 1) + 2) * 64, x_row0);
                }
              }
            }
            ++xblk;
          } else {
            // row-major bf16 (ld_out is a multiple of 8, pad columns belong to the buffer); split modes: np part arrays
            store_parts(v, p.out, p.out_ps, p.ld_out, col0, full);
          }
          if constexpr (EPI == EPI_DA) {
            if (p.colsum != nullptr) {
              // bias gradient: per-column sum over this warp's 32 rows, accumulated per CTA in shared memory
              const float s = warp_colsum_32x32(v, lane);
              red_shared(col_slot(it & 1, 0, c * 32 + lane), s);     // columns beyond N / rows beyond M were zeroed above
            }
          }
        } else if constexpr (EPI == EPI_DW) {
          if (p.acc_vec4 && full) {
            // fp32 rows are 128 B per 32-column chunk: two 64-byte halves through the transpose tile, then
            // red.global.add.v4.f32 with four lanes per 64 contiguous bytes
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              uint4 mine[4], oc[4];
#pragma unroll
              for (int q = 0; q < 4; ++q)
                mine[q] = make_uint4(__float_as_uint(v[16 * h + 4 * q]), __float_as_uint(v[16 * h + 4 * q + 1]),
                                     __float_as_uint(v[16 * h + 4 * q + 2]), __float_as_uint(v[16 * h + 4 * q + 3]));
              row_to_lanes(mine, oc);
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const int gr = row_base + 8 * i + lrow;
                if (gr < p.M)
                  red_add_v4_f32(p.accum + static_cast<size_t>(gr) * p.ld_acc + col0 + 16 * h + 4 * lpc, __uint_as_float(oc[i].x),
                                 __uint_as_float(oc[i].y), __uint_as_float(oc[i].z), __uint_as_float(oc[i].w));
              }
            }
          } else if (row_ok) {
            float* gp = p.accum + static_cast<size_t>(row) * p.ld_acc + col0;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (col0 + j < p.N) red_add_f32(gp + j, v[j]);
          }
        } else {  // EPI_F32
          if (row_ok) {
            float* gp = p.accum + static_cast<size_t>(row) * p.ld_acc + col0;
            if (p.split_k == 1) {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (col0 + j < p.N) gp[j] = v[j];
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (col0 + j < p.N) red_add_f32(gp + j, v[j]);
            }
          }
        }
      }
      // release the accumulator back to the MMA warp: one arrival per warp on the leader's barrier
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (CG == 2) mbar_arrive_cluster(tempty_bar(acc), 0);
        else mbar_arrive(tempty_bar(acc));
      }
      if constexpr (EPI == EPI_DA) {
        if (p.colsum != nullptr) flush_cols(it, tn, p.colsum, nullptr);
      }
      if (w == w_first && warp == 2 && lane == 0) stamp(7);  // first tile's epilogue done
    }
  }

  if constexpr (TMA_EPI) {
    if (warp >= 2 && ((warp - 2) & 7) == 0 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // the last tiles are in global memory
  }
  tcgen05_fence_before();
  if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
  if (threadIdx.x == 0) stamp(8);  // all roles finished
  // in-graph kernel span: slot 2 (dependencies resolved, CTA 0) .. slot 10 (latest exit over ALL CTAs; %globaltimer only
  // grows, so atomicMax needs no reset between steps)
  if (p.trace != nullptr && threadIdx.x == 0) atomicMax(p.trace + 10, static_cast<unsigned long long>(globaltimer_ns()));
  if (warp == 2) {
    tcgen05_fence_after();
    if constexpr (CG == 2) tmem_dealloc_cg2<Cfg::TMEM_COLS>(tmem_base);
    else tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiled get_encode_tiled();

// Tensor map of a row-major bf16 matrix [rows, cols] with leading dimension ld (elements):
// box = 64 columns x box_rows rows, 128-byte swizzle.  cols/rows are the LOGICAL extents (TMA zero-fills beyond
// them), ld*2 must be a multiple of 16 bytes.  K-major operand: box_rows = rows one CTA stages (128 for A,
// BN / CG for B); MN-major operand: 64.
int make_tmap_bf16(CUtensorMap* out, const void* base, int rows, int cols, int ld, int box_rows);
// the same map for each of np part arrays that lie part_stride ELEMENTS apart (np = 1: just the one)
int make_tmaps_bf16(CUtensorMap* out3, const void* base, long long part_stride, int np, int rows, int cols, int ld, int box_rows);
// fills n_pairs / pair_a / pair_b of p for np parts per operand
void set_part_pairs(GemmTcParams* p, int np);

// Tile configuration chosen per problem.
struct GemmPlan {
  int cg;            // 1 or 2
  int bn;            // 64 / 128 / 256
  int split_k, kb_per_split;
  int grid;          // CTAs to launch (a multiple of cg)
};
GemmPlan plan_gemm(int M, int N, int K, int num_sms, bool allow_split);

// launch_gemm_tc<EPI, A_MN, B_MN>(plan, tmA, tmB, params, stream, pdl) lives in gemm_tc_launch.cuh

}  // namespace sb
