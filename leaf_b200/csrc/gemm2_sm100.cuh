// CTA-pair (cta_group::2) version of the tower GEMM: two CTAs on the two SMs of a TPC compute one 256x256 tile.
//
// Why: with 128x256 tiles per SM the operand traffic is 48 KB per 4.2 MFLOP (85 FLOP/B); 148 SMs at tensor peak
// would pull ~26 TB/s out of L2, more than twice what the L2 delivers, and ncu showed the 1-CTA kernel stuck near
// 1.0-1.1 PFLOP/s (profiles/r1, r2). In a pair each CTA stages its own 128 rows of A and only HALF of the B tile
// (128 of the 256 weight rows); tcgen05.mma.cta_group::2 (M256 N256 K16) reads both halves, so a CTA moves 32 KB per
// 4.2 MFLOP (131 FLOP/B); the ring holds 5 stages and 40 KB are left for the 16 epilogue warps' staging buffers.
//
// Protocol (per stage s; "leader" = CTA rank 0 of the pair):
//   producers (warp WARP_TMA = 16 of BOTH CTAs) wait on their local empty[s], then TMA their A and B boxes into local smem with
//     cp.async.bulk.tensor...cta_group::2, whose complete_tx lands on the LEADER's full[s]; the leader's producer
//     arms full[s] with the bytes of both CTAs;
//   the leader's MMA thread waits full[s], issues 4 MMAs, then tcgen05.commit...multicast::cluster arrives on empty[s]
//     of both CTAs (and on tmem_full[acc] of both after the last k-block);
//   epilogue warps of both CTAs drain their own 128 TMEM lanes and arrive (remotely for the peer) on the leader's
//     tmem_empty[acc] (count 2 x 16 warps).
#pragma once
#include "gemm_sm100.cuh"

namespace leaf {

constexpr int GEMM2_BM = 256;                 // per pair (128 per CTA)
constexpr int GEMM2_STAGES = 5;
constexpr uint32_t GEMM2_A_BYTES = 128 * GEMM_BK * 2;
constexpr uint32_t GEMM2_B_BYTES = 128 * GEMM_BK * 2;
constexpr uint32_t GEMM2_STAGE_BYTES = GEMM2_A_BYTES + GEMM2_B_BYTES;
constexpr uint32_t GEMM2_SMEM_BYTES = GEMM2_STAGES * GEMM2_STAGE_BYTES + EPI_WARPS * EPI_STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
// Warp roles. The warp scheduler favours the highest warp id of an SM sub-partition (B300_MICROARCH.md), and the single
// MMA-issuing thread must never queue behind the 4 epilogue warps it shares a sub-partition with (ncu r6: with the issuer
// on warp 1 the GELU GEMM ran the tensor pipe at 63 % although neither the TMA ring nor the epilogue was late).
constexpr int WARP_TMA = EPI_WARPS, WARP_MMA = EPI_WARPS + 1, WARP_TMEM = EPI_WARPS + 2;   // epilogue = warps 0..15
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;   // shared::cluster address of the same offset in CTA rank 0 of a pair

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t smem_dst, const CUtensorMap* tmap, uint32_t bar_leader, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar_leader), "r"(x), "r"(y)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t smem_dst, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(static_cast<uint16_t>(3)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar_local) {
  // default semantics (as CUTLASS' umma_arrive_2x1SM_sm0): what is ordered is the TMEM read, already fenced with
  // tcgen05.wait::ld + tcgen05.fence::before_thread_sync; .release.cluster cost a membar per tile and warp (ncu r6)
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar_local & PEER_BIT_MASK) : "memory");
}

template <int EPI>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm2_bf16_tn_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                     const GemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + GEMM2_STAGES * GEMM2_STAGE_BYTES + EPI_WARPS * EPI_STAGE_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (GEMM2_STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * GEMM2_STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * GEMM2_STAGES + 2 + s); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * GEMM2_STAGES + 4);
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_gen =
      reinterpret_cast<volatile uint32_t*>(smem_gen + GEMM2_STAGES * GEMM2_STAGE_BYTES + EPI_WARPS * EPI_STAGE_BYTES +
                                           8u * (2 * GEMM2_STAGES + 4));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int M = p.m_dev ? min(*p.m_dev, p.M) : p.M;
  const int m_tiles = (M + GEMM2_BM - 1) / GEMM2_BM;
  const int n_tiles = (p.N + GEMM_BN - 1) / GEMM_BN;
  const int k_blocks = (p.K + GEMM_BK - 1) / GEMM_BK;
  // split-K: the k-blocks of an output tile are divided over `split` consecutive work units (GemmParams::split_k)
  const int split = ((EPI == EPI_F32_SPLITK || EPI == EPI_F32_SPLITK_DET) && p.split_k > 1) ? p.split_k : 1;
  const int kpb = (k_blocks + split - 1) / split;
  const int total_tiles = m_tiles * n_tiles * split;

  if (warp == WARP_TMA && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp == WARP_MMA && lane == 0) {
    for (int s = 0; s < GEMM2_STAGES; ++s) {
      mbar_init(full_bar(s), 1);           // leader producer's arrive.expect_tx (peer's copy of the barrier is unused)
      mbar_init(empty_bar(s), 1);          // one multicast commit from the leader's MMA thread
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);          // multicast commit
      mbar_init(tempty_bar(s), 2 * EPI_WARPS);   // every epilogue warp of both CTAs (leader's copy is the one waited on)
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == WARP_TMEM) tmem_alloc_2sm(tmem_slot, 512);
  tc_fence_before();
  cluster_sync_all();                       // barriers of both CTAs initialised, TMEM allocated
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;
  // Everything above overlapped the previous kernel's tail (engine.cu launches every GEMM with programmatic stream
  // serialization); its output is read below. The GEMM itself never calls pdl_trigger(): a LayerNorm / attention grid that
  // becomes resident next to still-draining GEMM CTAs keeps those SMs in the GEMM's shared-memory carve-out (almost no L1)
  // for its whole run - the attack step lost 5 ms of 157 with a trigger here, at the start or at the end of the kernel
  // (profiles/r2_25_pdl_ab.txt).
  pdl_wait();

  // The producer and the MMA issuer run as WHOLE warps with warp-uniform state and elect one lane only for the
  // asynchronous instructions themselves. Written as `if (lane == 0) { loop }` the same code compiled to ~130
  // dependent SASS instructions per k-block (ELECT + R2UR per descriptor word), which at ~5 cycles each is MORE than
  // the 512 tensor-pipe cycles of the 4 MMAs it issues: the issuing thread, not TMA or the epilogue, capped the
  // tensor pipe at 63-81 % (ncu source page, profiles/r6).
  if (warp == WARP_TMA) {
    // ===== TMA producer (both CTAs) =====
    int stage = 0;
    uint32_t phase = 0;
    const int a_row_off = static_cast<int>(rank) * 128;
    for (int tile = pair; tile < total_tiles; tile += n_pairs) {
      const int mn = tile / split, kb0 = (tile - mn * split) * kpb, kb1 = min(k_blocks, kb0 + kpb);
      const int m_blk = mn / n_tiles, n_blk = mn - m_blk * n_tiles;
      const int a_row = m_blk * GEMM2_BM + a_row_off, b_row = n_blk * GEMM_BN + a_row_off;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(empty_bar(stage), phase ^ 1);
        if (elect_one()) {
          const uint32_t sa = smem_base + stage * GEMM2_STAGE_BYTES;
          const uint32_t fb = full_bar(stage) & PEER_BIT_MASK;
          if (leader) mbar_arrive_expect_tx(full_bar(stage), p.tx_bytes);
          if (p.mn_major & GEMM_A_MN) {        // operand stored [K, MN]: two 64 (MN) x 64 (k) boxes
            tma_load_2d_2sm(sa, &tmap_a, fb, a_row, kb * GEMM_BK);
            tma_load_2d_2sm(sa + GEMM_MN_LBO, &tmap_a, fb, a_row + 64, kb * GEMM_BK);
          } else {
            tma_load_2d_2sm(sa, &tmap_a, fb, kb * GEMM_BK, a_row);
          }
          if (p.mn_major & GEMM_B_MN) {
            tma_load_2d_2sm(sa + GEMM2_A_BYTES, &tmap_b, fb, b_row, kb * GEMM_BK);
            tma_load_2d_2sm(sa + GEMM2_A_BYTES + GEMM_MN_LBO, &tmap_b, fb, b_row + 64, kb * GEMM_BK);
          } else {
            tma_load_2d_2sm(sa + GEMM2_A_BYTES, &tmap_b, fb, kb * GEMM_BK, b_row);
          }
        }
        __syncwarp();
        if (++stage == GEMM2_STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == WARP_MMA) {
    // ===== MMA issuer: the leader CTA's warp, one elected lane issues =====
    if (leader) {
      const bool a_mn = p.mn_major & GEMM_A_MN, b_mn = p.mn_major & GEMM_B_MN;
      const uint32_t idesc = make_idesc_bf16(GEMM2_BM, GEMM_BN) | (a_mn ? IDESC_A_MN_MAJOR : 0u) | (b_mn ? IDESC_B_MN_MAJOR : 0u);
      // stage 0 descriptors; + k-step per UMMA_K (32 B along a K-major row, 2 KB = 16 lines of an MN-major tile), + stage bytes >> 4 per stage
      const uint64_t adesc0 = a_mn ? make_smem_desc_mn_sw128(smem_base, GEMM_MN_LBO, GEMM_MN_SBO) : make_smem_desc_sw128(smem_base);
      const uint64_t bdesc0 = b_mn ? make_smem_desc_mn_sw128(smem_base + GEMM2_A_BYTES, GEMM_MN_LBO, GEMM_MN_SBO)
                                   : make_smem_desc_sw128(smem_base + GEMM2_A_BYTES);
      const uint64_t ak = a_mn ? (GEMM_MN_KSTEP >> 4) : 2u, bk = b_mn ? (GEMM_MN_KSTEP >> 4) : 2u;
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = pair; tile < total_tiles; tile += n_pairs) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * GEMM_BN);
        const int kb0 = (tile % split) * kpb, kb1 = min(k_blocks, kb0 + kpb);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t adesc = adesc0 + static_cast<uint64_t>(stage * (GEMM2_STAGE_BYTES >> 4));
            const uint64_t bdesc = bdesc0 + static_cast<uint64_t>(stage * (GEMM2_STAGE_BYTES >> 4));
            umma_bf16_2sm(d_tmem, adesc, bdesc, idesc, kb != kb0 ? 1u : 0u);
            umma_bf16_2sm(d_tmem, adesc + ak, bdesc + bk, idesc, 1u);
            umma_bf16_2sm(d_tmem, adesc + 2 * ak, bdesc + 2 * bk, idesc, 1u);
            umma_bf16_2sm(d_tmem, adesc + 3 * ak, bdesc + 3 * bk, idesc, 1u);
            umma_commit_2sm(empty_bar(stage));
            if (kb == kb1 - 1) umma_commit_2sm(tfull_bar(acc));
          }
          __syncwarp();
          if (++stage == GEMM2_STAGES) { stage = 0; phase ^= 1; }
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp < EPI_WARPS) {
    // ===== epilogue (both CTAs): this CTA's 128 rows of the 256-row tile =====
    const int quad = warp & 3;
    const int part = warp >> 2;                // which 64 accumulator columns
    uint8_t* stage_buf = smem_gen + GEMM2_STAGES * GEMM2_STAGE_BYTES + warp * EPI_STAGE_BYTES;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = pair; tile < total_tiles; tile += n_pairs) {
      const int mn = tile / split;
      const int m_blk = mn / n_tiles, n_blk = mn % n_tiles;
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
      const int row0 = m_blk * GEMM2_BM + static_cast<int>(rank) * 128 + quad * 32;
#pragma unroll 1
      for (int c = 0; c < 64; c += 32) {
        const int col0 = n_blk * GEMM_BN + part * 64 + c;
        if (col0 >= p.N) break;
        ResidualRegs res;
        if (row0 < M) epilogue_load_residual<EPI>(p, res, lane, row0, col0, M);
        uint32_t v[32];
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) +
                               static_cast<uint32_t>(acc * GEMM_BN + part * 64 + c);
        tmem_ld32(taddr, v);
        tmem_ld_wait();
        if constexpr (EPI == EPI_F32_SPLITK_DET) {
          // this work unit's partial sums, [column][lane] in the warp's region of the unit's tile (coalesced)
          if (row0 < M) {
            float* w = p.ws + static_cast<size_t>(tile) * (GEMM2_BM * GEMM_BN) + ((rank * EPI_WARPS + warp) * 2 + (c >> 5)) * 1024 + lane;
#pragma unroll
            for (int j = 0; j < 32; ++j) w[j * 32] = __uint_as_float(v[j]);
          }
        } else {
          if (row0 < M) epilogue_chunk<EPI>(p, v, res, stage_buf, lane, row0, col0, M);      // warp-uniform
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(tempty_bar(acc));
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      if constexpr (EPI == EPI_F32_SPLITK_DET) {
        // The last of the `split` units of this output tile to reach this warp's region adds the partials to C in split order.
        int* ctr = p.cnt + mn * (2 * EPI_WARPS) + rank * EPI_WARPS + warp;
        __threadfence();
        __syncwarp();
        int old = 0;
        if (lane == 0) old = atomicAdd(ctr, 1);
        old = __shfl_sync(0xffffffffu, old, 0);
        if (old == split - 1) {
          __threadfence();
          if (row0 < M) {
#pragma unroll 1
            for (int c = 0; c < 64; c += 32) {
              const int col0 = n_blk * GEMM_BN + part * 64 + c;
              if (col0 >= p.N) break;
              const float* w = p.ws + static_cast<size_t>(mn) * split * (GEMM2_BM * GEMM_BN) + ((rank * EPI_WARPS + warp) * 2 + (c >> 5)) * 1024 + lane;
              float f[32];
#pragma unroll
              for (int j = 0; j < 32; ++j) f[j] = __ldcg(w + j * 32);
#pragma unroll 1
              for (int u = 1; u < split; ++u) {
                w += GEMM2_BM * GEMM_BN;
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] += __ldcg(w + j * 32);
              }
              uint32_t v[32];
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(f[j]);
              ResidualRegs res;                                   // C = C + sum, through the staged fp32 store
              epilogue_load_residual<EPI_F32_RESIDUAL>(p, res, lane, row0, col0, M);
              epilogue_chunk<EPI_F32_RESIDUAL>(p, v, res, stage_buf, lane, row0, col0, M);
            }
          }
          if (lane == 0) *ctr = 0;
        }
      }
      if constexpr (EPI == EPI_BF16_ACTBWD_DET) {
        // The last 32-row chunk to finish these 64 columns adds every chunk's column sums to C2 in row order.
        if (p.C2 && row0 < M && n_blk * GEMM_BN + part * 64 < p.N) {
          int* ctr = p.cnt + n_blk * 4 + part;
          __threadfence();
          __syncwarp();
          int old = 0;
          if (lane == 0) old = atomicAdd(ctr, 1);
          old = __shfl_sync(0xffffffffu, old, 0);
          const int chunks = (M + 31) >> 5;
          if (old == chunks - 1) {
            __threadfence();
#pragma unroll 1
            for (int c = 0; c < 64; c += 32) {
              const int col = n_blk * GEMM_BN + part * 64 + c + lane;
              if (col < p.N) {
                reinterpret_cast<float*>(p.C2)[col] += ordered_sum<16>(p.ws + col, p.N, chunks);
              }
            }
            if (lane == 0) *ctr = 0;
          }
        }
      }
    }
  }

  tc_fence_before();
  cluster_sync_all();                       // nobody may still be reading the peer's smem / TMEM
  if (warp == WARP_TMEM) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}

}  // namespace leaf
