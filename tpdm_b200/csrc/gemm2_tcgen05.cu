// tpdm_b200 -- CTA-pair (cta_group::2) variant of the bf16 GEMM: a cluster of two CTAs computes a 256 x 256 output tile.
//
// Why: with one CTA per 128 x 256 tile the tensor core reads 12 KB of operands from shared memory per 128-cycle MMA
// (96 B/clk) while TMA writes the same 96 B/clk into the ring -- 192 B/clk against the SM's 128 B/clk of shared-memory
// bandwidth, i.e. a hard ~67 % ceiling on tensor-pipe activity (ncu: 67-71 %, profiles/r01_gemm_ncu.txt).  In a pair each
// CTA stages its own 128 rows of A but only HALF of the tile's W rows; tcgen05.mma.cta_group::2 (M = 256) reads A from
// both CTAs and each half of B from the CTA that holds it: 64 + 64 B/clk per SM.  Stages shrink to 32 KB, so the ring is 6 deep.
//
// Roles per CTA (320 threads: TMA warp, MMA warp, 8 epilogue warps) follow gemm_tcgen05.cu; differences:
//   * TMA loads of BOTH CTAs complete on the LEADER's full barrier (cp.async.bulk.tensor ... cta_group::2, barrier address
//     mapped with mapa); the leader's barrier expects one arrive.expect_tx per CTA;
//   * only the leader's warp 1 issues MMAs; tcgen05.commit multicasts to both CTAs' empty / tmem_full barriers;
//   * the epilogue warps of both CTAs release the accumulator on the leader's tmem_empty barrier (count 16);
//   * TMEM is allocated / freed with the cta_group::2 forms by one warp of each CTA; cluster barriers bracket the kernel.
#include <cuda_bf16.h>

#include "common.cuh"
#include "gemm_epilogue.cuh"
#include "host.h"

namespace tpdm {

namespace {

constexpr int BM = 128;
constexpr int BN2 = 256;
#ifndef TPDM_GEMM2_BK
#define TPDM_GEMM2_BK 64
#endif
constexpr int BK = TPDM_GEMM2_BK;   // k-block per pipeline stage: 64 (one 128-byte swizzle atom row) or 128 (two, side by side)
constexpr int kSub = BK / 64;       // 64-wide TMA boxes per operand and stage
// E4M3 instantiation: a 128-byte swizzle row holds 128 one-byte elements, so every byte offset, stage size and ring depth below is
// unchanged and only the element counts along K double (a stage covers 2 * BK elements, each MMA K = 32)
template <bool kFp8>
constexpr int kElemsPerRow = kFp8 ? 128 : 64;
constexpr int kStages2 = BK == 64 ? 5 : 3;
constexpr int kEpiWarps2 = 8;   // two warps per TMEM lane quarter, each draining half of the tile's columns
constexpr int kThreads2 = 64 + 32 * kEpiWarps2;
constexpr int kABytes2 = BM * BK * 2;
constexpr int kBBytes2 = (BN2 / 2) * BK * 2;
constexpr int kStageBytes2 = kABytes2 + kBBytes2;
constexpr int kRing2 = kStages2 * kStageBytes2;
constexpr int kEpi2 = kEpiWarps2 * 32 * kStagePad * 4 + kEpiWarps2 * 2 * (BN2 / 2) * 4;
constexpr int kBarOff2 = kRing2 + kEpi2;
constexpr int kSmem2 = kBarOff2 + 256 + 1024;

// -DTPDM_GEMM_TRACE: clock64() stamps of the leader CTA's MMA warp (cluster 0): per k-block {before the full-barrier wait, after it,
// after the issue + commit}, and per tile the wait for a free accumulator; read back with tpdm_gemm_trace_read (tools/gemm_trace.py)
#ifdef TPDM_GEMM_TRACE
__device__ long long g_gemm_trace[4096];
__device__ int g_gemm_trace_n;
#endif

struct Gemm2Params {
  GemmOp op[2];
  int n_ops;
  int tiles0, total_tiles;  // pair tiles of op 0 / of all ops
  const int* skip;
  const int* bmask;
  int bslots;
};

struct PairCoord {
  int g, b, mtp, nt;
};

__device__ __forceinline__ PairCoord decode_pair(const Gemm2Params& P, int tile) {
  PairCoord t;
  t.g = (P.n_ops > 1 && tile >= P.tiles0) ? 1 : 0;
  const int local = tile - (t.g ? P.tiles0 : 0);
  const GemmOp& G = P.op[t.g];
  const int tiles_mp = (G.rows_per_batch + 2 * BM - 1) / (2 * BM);
  const int m_idx = local / G.tiles_n;  // N fastest, see gemm_tcgen05.cu
  t.nt = local - m_idx * G.tiles_n;
  t.b = m_idx / tiles_mp;
  t.mtp = m_idx - t.b * tiles_mp;
  return t;
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(const void* p, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_expect_tx_cluster(uint32_t cluster_addr, uint32_t bytes) {
  // default semantics (no cluster-scope release): the producer publishes nothing of its own; a .release.cluster here costs an
  // ERRBAR per k-block on the critical path of the TMA issue (measured: tensor pipe 35 % instead of >80 %)
  asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;" ::"r"(cluster_addr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma2_load_3d(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma2_load_2d(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma2_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// The same two instructions for a CONVERGED warp: every lane executes the statement with identical (warp-uniform) operands and one
// elected lane issues.  Inside `if (lane == 0)` the compiler cannot use the uniform datapath and wraps every UTCHMMA in a
// "waterfall" loop (ELECT / R2UR / PLOP3 / BRA.U.ANY, ~13 instructions and a dependent branch per MMA); in converged code the
// descriptors live in uniform registers and an MMA costs a UIADD3 or two.
__device__ __forceinline__ void umma2_ss_elect(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma2_ss_elect_e4m3(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma2_commit_multicast_elect(uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}\n" ::"r"(smem_u32(bar)),
      "h"(static_cast<uint16_t>(3))
      : "memory");
}
// arrives on the barrier at this shared-memory offset in BOTH CTAs of the pair once the MMAs issued so far have retired
__device__ __forceinline__ void umma2_commit_multicast(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n" ::"r"(smem_u32(bar)),
               "h"(static_cast<uint16_t>(3))
               : "memory");
}

// kFp8: E4M3 x E4M3 -> fp32 (kind::f8f6f4) with the scaled epilogue; otherwise bf16 x bf16 -> fp32 (kind::f16)
template <bool kFp8>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads2, 1) gemm2_bf16_tcgen05_kernel(const __grid_constant__ Gemm2Params P) {
  constexpr int kRowElems = kElemsPerRow<kFp8>;
  constexpr int kStageK = kSub * kRowElems;  // K elements per stage
  pdl_launch_dependents();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float* epi_stage = reinterpret_cast<float*>(smem + kRing2);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kBarOff2);  // used in the leader CTA only
  uint64_t* empty_bar = full_bar + kStages2;                          // one set per CTA
  uint64_t* tmem_full = empty_bar + kStages2;                         // one set per CTA
  uint64_t* tmem_empty = tmem_full + 2;                               // used in the leader CTA only
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < P.n_ops; ++i) {
      tma_prefetch_desc(&P.op[i].tmA);
      tma_prefetch_desc(&P.op[i].tmB2);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kStages2; ++i) {
      mbar_init(&full_bar[i], 2);  // one arrive.expect_tx from the producer of each CTA
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 2 * kEpiWarps2);  // epilogue warps of both CTAs
    }
    fence_barrier_init();
  }
  pdl_wait();
  if (P.skip != nullptr && *P.skip != 0) return;  // uniform over the grid, so both CTAs of a pair leave together
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;\n" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();  // barriers of both CTAs initialised, TMEM allocated, before any remote arrive / TMA / MMA
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (both CTAs)
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = cluster_id; tile < P.total_tiles; tile += num_clusters) {
        const PairCoord tc = decode_pair(P, tile);
        if (P.bmask != nullptr && P.bmask[tc.b % P.bslots] == 0) continue;
        const GemmOp& G = P.op[tc.g];
        const int nkb = (G.K + kStageK - 1) / kStageK;
        const int m0 = tc.mtp * 2 * BM + static_cast<int>(rank) * BM;
        const int nb0 = tc.nt * BN2 + static_cast<int>(rank) * (BN2 / 2);
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait_backoff(&empty_bar[stage], phase ^ 1);
          uint8_t* sA = smem + stage * kStageBytes2;
          uint8_t* sB = sA + kABytes2;
          const uint32_t leader_full = map_to_cta(&full_bar[stage], 0);
          mbar_arrive_expect_tx_cluster(leader_full, kStageBytes2);
#pragma unroll
          for (int h = 0; h < kSub; ++h) {
            tma2_load_3d(sA + h * (BM * 128), &G.tmA, leader_full, kb * kStageK + h * kRowElems, m0, tc.b);
            tma2_load_2d(sB + h * ((BN2 / 2) * 128), &G.tmB2, leader_full, kb * kStageK + h * kRowElems, nb0);
          }
          if (++stage == kStages2) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA only)
    if (rank == 0) {
      constexpr uint32_t idesc = kFp8 ? make_idesc_e4m3(2 * BM, BN2) : make_idesc_bf16(2 * BM, BN2);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = cluster_id; tile < P.total_tiles; tile += num_clusters) {
        const PairCoord tc = decode_pair(P, tile);
        if (P.bmask != nullptr && P.bmask[tc.b % P.bslots] == 0) continue;
        const GemmOp& G = P.op[tc.g];
        const int nkb = (G.K + kStageK - 1) / kStageK;
#ifdef TPDM_GEMM_TRACE
        const bool tr = cluster_id == 0 && lane == 0;
        long long tq0 = 0;
        if (tr) tq0 = clock64();
#endif
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
#ifdef TPDM_GEMM_TRACE
        if (tr && g_gemm_trace_n + 4 <= 4096) {
          g_gemm_trace[g_gemm_trace_n++] = -1;          // tile marker
          g_gemm_trace[g_gemm_trace_n++] = tq0;
          g_gemm_trace[g_gemm_trace_n++] = clock64();
          g_gemm_trace[g_gemm_trace_n++] = nkb;
        }
#endif
        const uint32_t d_tmem = tmem_base + acc * BN2;
        for (int kb = 0; kb < nkb; ++kb) {
#ifdef TPDM_GEMM_TRACE
          long long t0 = 0, t1 = 0;
          if (tr) t0 = clock64();
#endif
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
#ifdef TPDM_GEMM_TRACE
          if (tr) t1 = clock64();
#endif
          {
            const uint32_t a_base = smem_u32(smem + stage * kStageBytes2);
            const uint32_t b_base = a_base + kABytes2;
            // descriptors of the stage once; the 32-byte k steps (16 bf16 or 32 E4M3 elements) advance the 14-bit start-address
            // field (units of 16 B)
            const uint64_t adesc0 = make_smem_desc_sw128(a_base, 16, 1024), bdesc0 = make_smem_desc_sw128(b_base, 16, 1024);
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
              const uint32_t ao = ((k / 4) * (BM * 128) + (k % 4) * 32) >> 4, bo = ((k / 4) * ((BN2 / 2) * 128) + (k % 4) * 32) >> 4;
              if constexpr (kFp8)
                umma2_ss_elect_e4m3(d_tmem, adesc0 + ao, bdesc0 + bo, idesc, (kb | k) != 0 ? 1u : 0u);
              else
                umma2_ss_elect(d_tmem, adesc0 + ao, bdesc0 + bo, idesc, (kb | k) != 0 ? 1u : 0u);
            }
            umma2_commit_multicast_elect(&empty_bar[stage]);
            if (kb == nkb - 1) umma2_commit_multicast_elect(&tmem_full[acc]);
          }
#ifdef TPDM_GEMM_TRACE
          if (tr && g_gemm_trace_n + 3 <= 4096) {
            g_gemm_trace[g_gemm_trace_n++] = t0;
            g_gemm_trace[g_gemm_trace_n++] = t1;
            g_gemm_trace[g_gemm_trace_n++] = clock64();
          }
#endif
          __syncwarp();
          if (++stage == kStages2) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (warps 2..9, both CTAs; own 128 rows)
    // The epilogue, not the MMA, bounds the K = 1536 GEMMs (measured with K = 64: ~8.5 us per 128 x 256 tile with 4 warps
    // against 7 us of MMA), so each TMEM lane quarter is drained by two warps: columns [0,128) and [128,256).
    const int q = warp & 3;
    const int hh = (warp - 2) >> 2;
    float* st = epi_stage + (warp - 2) * 32 * kStagePad;
    float* sbias = epi_stage + kEpiWarps2 * 32 * kStagePad + (warp - 2) * 2 * (BN2 / 2);
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = cluster_id; tile < P.total_tiles; tile += num_clusters) {
      const PairCoord tc = decode_pair(P, tile);
        if (P.bmask != nullptr && P.bmask[tc.b % P.bslots] == 0) continue;
      const GemmOp& G = P.op[tc.g];
      const int n0 = tc.nt * BN2;
      const int row_base = tc.mtp * 2 * BM + static_cast<int>(rank) * BM + q * 32;
      gemm_epilogue_tile<BN2, kFp8>(
          G, tc.b, row_base, n0, tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BN2, st, sbias, lane, hh * (BN2 / 64), (hh + 1) * (BN2 / 64),
          [&]() { mbar_wait_backoff(&tmem_full[acc], acc_phase); },
          [&]() {
            if (lane == 0) mbar_arrive_cluster(map_to_cta(&tmem_empty[acc], 0));
          });
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  }

  __syncwarp();
  tc_fence_before();
  cluster_sync_all();  // nobody leaves while the peer may still signal our barriers or the leader's MMAs read our smem
  if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;\n" ::"r"(tmem_base) : "memory");
}

}  // namespace

#ifdef TPDM_GEMM_TRACE
extern "C" int tpdm_gemm_trace_read(long long* host, int* n, int reset) {
  int cnt = 0;
  if (cudaMemcpyFromSymbol(&cnt, g_gemm_trace_n, sizeof(int)) != cudaSuccess) return -1;
  if (cudaMemcpyFromSymbol(host, g_gemm_trace, sizeof(long long) * 4096) != cudaSuccess) return -1;
  *n = cnt;
  if (reset) {
    cnt = 0;
    cudaMemcpyToSymbol(g_gemm_trace_n, &cnt, sizeof(int));
  }
  return 0;
}
#endif

int gemm2_launch(const GemmOp* ops, int n_ops, cudaStream_t stream) {
  TPDM_CHECK(n_ops >= 1 && n_ops <= 2, TPDM_ERR_ARG, "gemm2_launch: 1 or 2 ops per launch");
  Gemm2Params P;
  P.n_ops = n_ops;
  P.total_tiles = 0;
  P.tiles0 = 0;
  P.skip = skip_flag();
  P.bmask = batch_mask();
  P.bslots = batch_mask_slots();
  double flops = 0;
  const bool fp8 = ops[0].fp8 != 0;
  for (int i = 0; i < n_ops; ++i) {
    TPDM_CHECK(ops[i].conv == 0 && ops[i].block_n == 256, TPDM_ERR_ARG, "gemm2_launch: plain GEMMs with 256-wide N tiles only");
    TPDM_CHECK((ops[i].fp8 != 0) == fp8, TPDM_ERR_ARG, "gemm2_launch: grouped ops must share the operand type");
    P.op[i] = ops[i];
    const int tiles_mp = (ops[i].rows_per_batch + 2 * BM - 1) / (2 * BM);
    const int t = ops[i].batch * tiles_mp * ops[i].tiles_n;
    if (i == 0) P.tiles0 = t;
    P.total_tiles += t;
    flops += 2.0 * ops[i].batch * ops[i].rows_per_batch * static_cast<double>(ops[i].N) * ops[i].K;
  }
  if (n_ops == 1) P.op[1] = ops[0];
  static bool attr_set[2] = {false, false};
  if (!attr_set[fp8]) {
    TPDM_CUDA_OK(cudaFuncSetAttribute(fp8 ? gemm2_bf16_tcgen05_kernel<true> : gemm2_bf16_tcgen05_kernel<false>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem2));
    attr_set[fp8] = true;
  }
  const int max_clusters = num_sms() / 2;
  const int clusters = P.total_tiles < max_clusters ? P.total_tiles : max_clusters;
  prof_begin(0, flops, stream);
  TPDM_CUDA_OK(launch_pdl(fp8 ? gemm2_bf16_tcgen05_kernel<true> : gemm2_bf16_tcgen05_kernel<false>, dim3(2 * clusters), dim3(kThreads2), kSmem2,
                          stream, P));
  prof_end(stream);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace tpdm
