// tpdm_b200 -- persistent, warp-specialised bf16 GEMM on tcgen05 tensor cores (sm_100a).
//
//   out = epilogue( A[rows x K] . W[N x K]^T )        fp32 accumulation in TMEM
//
// Replaces every nn.Linear on the MMDiT path (diffusers to_q/to_k/to_v, add_*_proj, to_out, to_add_out, ff.net.*,
// context_embedder, proj_out; call sites /root/reference/src/models/stable_diffusion_3/transformer_sd3.py:337,361,374)
// and, in conv mode, TimePredictor.conv1 (modeling_sd3_pnt.py:88,104) as a 9-tap implicit GEMM.
//
// Structure (one CTA per SM, 192 threads):
//   warp 0     TMA producer: A tile 128x64 and W tile BNx64 (bf16, 128B swizzle) into a 4-stage smem ring
//   warp 1     MMA issuer: one elected lane issues 4 x tcgen05.mma (128 x BN x 16) per stage into a double-buffered
//              TMEM accumulator (2 x BN columns), tcgen05.commit releases the smem stage / signals the epilogue
//   warps 2-5  epilogue: tcgen05.ld 32 rows x 32 cols per warp, transpose through padded smem so that global traffic is
//              row-contiguous, then bias / GELU-tanh / gate*x + fp32 residual
// Up to two independent problems (image stream + text stream) share one launch so the small text GEMM fills the tail wave.
#include <cuda_bf16.h>
#include <stdlib.h>

#include "common.cuh"
#include "gemm_epilogue.cuh"
#include "host.h"

namespace tpdm {

namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int kStages = 4;
constexpr int kGemmThreads = 192;
constexpr int kABytes = BM * BK * 2;

struct GemmParams {
  GemmOp op[2];
  int n_ops;
  int total_tiles;
  const int* skip;
  const int* bmask;  // set_batch_mask: tiles of inactive batch entries are skipped by every role
  int bslots;
};

template <int BN>
struct GemmSmem {
  static constexpr int kBBytes = BN * BK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kRing = kStages * kStageBytes;
  static constexpr int kEpi = 4 * 32 * kStagePad * 4 + 4 * 2 * BN * 4;  // transpose staging + per-warp bias / gate vectors of the tile
  static constexpr int kBarOff = kRing + kEpi;
  static constexpr int kTotal = kBarOff + 256 + 1024;  // + barriers + alignment slack
};

struct TileCoord {
  int g, b, mt, nt, ks;
};

__device__ __forceinline__ TileCoord decode_tile(const GemmParams& P, int tile) {
  TileCoord t;
  t.g = (P.n_ops > 1 && tile >= P.op[0].num_tiles) ? 1 : 0;
  int local = tile - (t.g ? P.op[0].num_tiles : 0);
  const GemmOp& G = P.op[t.g];
  // N fastest: the n-tiles that share an A row-block run in the same wave, so A is fetched from DRAM once (the others hit
  // L2) and the weight matrix -- the operand every CTA re-reads -- stays L2 resident.  (M fastest re-read A once per wave:
  // ncu showed 408 MB of DRAM reads for FF2 against 170 MB algorithmic.)
  const int per_split = G.num_tiles / G.ksplit;
  t.ks = local / per_split;  // K range of a split-K op (0 otherwise)
  local -= t.ks * per_split;
  int m_idx = local / G.tiles_n;
  t.nt = local - m_idx * G.tiles_n;
  t.b = m_idx / G.tiles_m_per_batch;
  t.mt = m_idx % G.tiles_m_per_batch;
  return t;
}

template <int BN>
__global__ void __launch_bounds__(kGemmThreads, 1) gemm_bf16_tcgen05_kernel(const __grid_constant__ GemmParams P) {
  using L = GemmSmem<BN>;
  pdl_launch_dependents();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float* epi_stage = reinterpret_cast<float*>(smem + L::kRing);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full = empty_bar + kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < P.n_ops; ++i) {
      tma_prefetch_desc(&P.op[i].tmA);
      tma_prefetch_desc(&P.op[i].tmB);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 4);  // one arrive per epilogue warp
    }
    fence_barrier_init();
  }
  pdl_wait();
  if (P.skip != nullptr && *P.skip != 0) return;
  if (warp == 2) {
    tmem_alloc<2 * BN>(tmem_slot);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < P.total_tiles; tile += gridDim.x) {
        const TileCoord tc = decode_tile(P, tile);
        if (P.bmask != nullptr && P.bmask[tc.b % P.bslots] == 0) continue;
        const GemmOp& G = P.op[tc.g];
        const int nkb_all = (G.K + BK - 1) / BK, kps = (nkb_all + G.ksplit - 1) / G.ksplit;
        const int kb0 = tc.ks * kps, nkb = kb0 + kps < nkb_all ? kb0 + kps : nkb_all;
        for (int kb = kb0; kb < nkb; ++kb) {
          mbar_wait_backoff(&empty_bar[stage], phase ^ 1);
          uint8_t* sA = smem + stage * L::kStageBytes;
          uint8_t* sB = sA + kABytes;
          mbar_arrive_expect_tx(&full_bar[stage], L::kStageBytes);
          if (G.conv == 2) {
            // conv1 weight gradient: K runs over (sample, 64-pixel block); A = dY^T [sample][oc][pix],
            // B = X (NCHW) shifted by the tile's tap: 64 consecutive pixels of `BN` channels per k-block
            const int sample = kb / G.kb_per_tap, pblk = kb - sample * G.kb_per_tap;
            const int tap = tc.nt / G.wg_ctiles, c0 = (tc.nt - tap * G.wg_ctiles) * BN;
            tma_load_3d(sA, &G.tmA, &full_bar[stage], pblk * BK, 0, sample);
            // B: pixels (y, x) are one flattened, contiguous dimension, so a 64-pixel block is always a 128-byte inner
            // box; the row shift (ky) is +-g pixels with zero fill past either end, the column shift (kx) selects one of
            // three pre-shifted copies so the innermost (swizzled) coordinate stays 16-byte aligned
            tma_load_4d(sB, &G.tmB, &full_bar[stage], pblk * BK + (tap / 3 - 1) * G.wg_px, c0, tap % 3, sample);
            if (++stage == kStages) {
              stage = 0;
              phase ^= 1;
            }
            continue;
          }
          if (G.conv) {
            const int tap = kb / G.kb_per_tap;
            const int c0 = (kb - tap * G.kb_per_tap) * BK;
            const int yt = tc.mt / G.conv_xt, xt = tc.mt - yt * G.conv_xt;
            tma_load_4d(sA, &G.tmA, &full_bar[stage], c0, xt * G.conv_bx + tap % 3 - 1, yt * G.conv_by + tap / 3 - 1, tc.b);
          } else {
            tma_load_3d(sA, &G.tmA, &full_bar[stage], kb * BK, tc.mt * BM, tc.b);
          }
          tma_load_2d(sB, &G.tmB, &full_bar[stage], kb * BK, tc.nt * BN);
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc = make_idesc_bf16(BM, BN);
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < P.total_tiles; tile += gridDim.x) {
      const TileCoord tc = decode_tile(P, tile);
        if (P.bmask != nullptr && P.bmask[tc.b % P.bslots] == 0) continue;
      const GemmOp& G = P.op[tc.g];
      const int nkb_all = (G.K + BK - 1) / BK, kps = (nkb_all + G.ksplit - 1) / G.ksplit;
      const int kb0 = tc.ks * kps, nkb = kb0 + kps < nkb_all ? kb0 + kps : nkb_all;
      mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * BN;
      for (int kb = kb0; kb < nkb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        {
          // converged warp, one elected lane per instruction (umma_ss_elect in common.cuh): no waterfall loop around the MMAs
          const uint32_t a_base = smem_u32(smem + stage * L::kStageBytes);
          const uint32_t b_base = a_base + kABytes;
          const uint64_t adesc0 = make_smem_desc_sw128(a_base, 16, 1024), bdesc0 = make_smem_desc_sw128(b_base, 16, 1024);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k)
            umma_ss_elect(d_tmem, adesc0 + ((k * 32) >> 4), bdesc0 + ((k * 32) >> 4), idesc, (kb != kb0 || k != 0) ? 1u : 0u);
          umma_commit_elect(&empty_bar[stage]);
          if (kb == nkb - 1) umma_commit_elect(&tmem_full[acc]);
        }
        __syncwarp();
        if (++stage == kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (warps 2..5)
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    float* st = epi_stage + (warp - 2) * 32 * kStagePad;
    float* sbias = epi_stage + 4 * 32 * kStagePad + (warp - 2) * 2 * BN;  // [0,BN) bias, [BN,2BN) gate of the current tile
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < P.total_tiles; tile += gridDim.x) {
      const TileCoord tc = decode_tile(P, tile);
        if (P.bmask != nullptr && P.bmask[tc.b % P.bslots] == 0) continue;
      const GemmOp& G = P.op[tc.g];
      const int n0 = tc.nt * BN;
      const int row_base = tc.mt * BM + q * 32;
      gemm_epilogue_tile<BN>(
          G, tc.b + tc.ks * G.batch, row_base, n0, tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BN, st, sbias, lane, 0, BN / 32,
          [&]() { mbar_wait_backoff(&tmem_full[acc], acc_phase); }, [&]() { if (lane == 0) mbar_arrive(&tmem_empty[acc]); });
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<2 * BN>(tmem_base);
}

template <int BN>
int launch_impl(const GemmParams& P, cudaStream_t stream) {
  static bool attr_set = false;
  if (!attr_set) {
    TPDM_CUDA_OK(cudaFuncSetAttribute(gemm_bf16_tcgen05_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      GemmSmem<BN>::kTotal));
    attr_set = true;
  }
  int grid = P.total_tiles < num_sms() ? P.total_tiles : num_sms();
  double flops = 0;
  for (int i = 0; i < P.n_ops; ++i) flops += 2.0 * P.op[i].batch * P.op[i].rows_per_batch * static_cast<double>(P.op[i].N) * P.op[i].K;
  prof_begin(0, flops, stream);
  TPDM_CUDA_OK(launch_pdl(gemm_bf16_tcgen05_kernel<BN>, dim3(grid), dim3(kGemmThreads), GemmSmem<BN>::kTotal, stream, P));
  prof_end(stream);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int finish_op(GemmOp* op, const void* W, int N, int K, int epi, void* out, long long out_batch_stride, int ldo,
              const float* bias, const float* gate, int gate_stride) {
  op->N = N;
  op->K = K;
  op->block_n = N <= 128 ? 128 : 256;
  op->tiles_n = (N + op->block_n - 1) / op->block_n;
  op->num_tiles = op->batch * op->tiles_m_per_batch * op->tiles_n;
  op->epi = epi;
  op->out = out;
  op->out_batch_stride = out_batch_stride;
  op->ldo = ldo;
  op->bias = bias;
  op->gate = gate;
  op->gate_stride = gate_stride;
  TPDM_CHECK(K % 8 == 0, TPDM_ERR_SHAPE, "gemm: K=%d must be a multiple of 8", K);
  TPDM_CHECK(N % 8 == 0 && ldo % 8 == 0, TPDM_ERR_SHAPE, "gemm: N=%d and ldo=%d must be multiples of 8 (16-byte row segments)", N, ldo);
  TPDM_CHECK((reinterpret_cast<uintptr_t>(out) & 15) == 0 && (reinterpret_cast<uintptr_t>(bias) & 15) == 0 &&
                 (reinterpret_cast<uintptr_t>(gate) & 15) == 0 && gate_stride % 4 == 0,
             TPDM_ERR_ARG, "gemm: out / bias / gate must be 16-byte aligned");
  TPDM_CHECK(epi != EPI_GATE_RESIDUAL || gate != nullptr, TPDM_ERR_ARG, "gemm: gate pointer required");
  uint64_t dims[2] = {static_cast<uint64_t>(K), static_cast<uint64_t>(N)};
  uint64_t strides[1] = {static_cast<uint64_t>(K) * 2};
  uint32_t box[2] = {BK, static_cast<uint32_t>(op->block_n)};
  TPDM_TRY(encode_tmap_bf16(&op->tmB, W, 2, dims, strides, box));
  uint32_t box2[2] = {BK, 128};
  return encode_tmap_bf16(&op->tmB2, W, 2, dims, strides, box2);
}

}  // namespace

int gemm_op_init(GemmOp* op, const void* A, long long a_row_stride, long long a_batch_stride, int rows_per_batch, int batch,
                 int K, const void* W, int N, int epi, void* out, long long out_batch_stride, int ldo, const float* bias,
                 const float* gate, int gate_stride) {
  *op = GemmOp{};
  TPDM_CHECK(rows_per_batch > 0 && batch > 0 && K > 0 && N > 0, TPDM_ERR_SHAPE, "gemm: empty problem");
  op->rows_per_batch = rows_per_batch;
  op->batch = batch;
  op->tiles_m_per_batch = (rows_per_batch + BM - 1) / BM;
  op->conv = 0;
  uint64_t dims[3] = {static_cast<uint64_t>(K), static_cast<uint64_t>(rows_per_batch), static_cast<uint64_t>(batch)};
  uint64_t strides[2] = {static_cast<uint64_t>(a_row_stride) * 2,
                         static_cast<uint64_t>(batch > 1 ? a_batch_stride : a_row_stride * rows_per_batch) * 2};
  uint32_t box[3] = {BK, BM, 1};
  TPDM_TRY(encode_tmap_bf16(&op->tmA, A, 3, dims, strides, box));
  return finish_op(op, W, N, K, epi, out, out_batch_stride, ldo, bias, gate, gate_stride);
}

int gemm_op_init_fp8(GemmOp* op, const void* A, long long a_row_stride, long long a_batch_stride, const float* a_scale, int rows_per_batch,
                     int batch, int K, const void* W, const float* w_scale, int N, int epi, void* out, long long out_batch_stride, int ldo,
                     const float* bias) {
  *op = GemmOp{};
  TPDM_CHECK(rows_per_batch > 0 && batch > 0 && K > 0 && N > 0, TPDM_ERR_SHAPE, "gemm fp8: empty problem");
  TPDM_CHECK(epi == EPI_BIAS_BF16 || epi == EPI_BIAS_F32 || epi == EPI_BIAS_GELU_BF16, TPDM_ERR_ARG, "gemm fp8: epilogue %d unsupported", epi);
  TPDM_CHECK(N > 128, TPDM_ERR_SHAPE, "gemm fp8: N=%d must exceed 128 (CTA-pair kernel, 256-wide N tiles)", N);
  TPDM_CHECK(K % 16 == 0 && a_row_stride % 16 == 0, TPDM_ERR_SHAPE, "gemm fp8: K=%d and the A row stride must be multiples of 16", K);
  TPDM_CHECK(a_scale != nullptr && w_scale != nullptr && (reinterpret_cast<uintptr_t>(w_scale) & 15) == 0, TPDM_ERR_ARG,
             "gemm fp8: a_scale and a 16-byte aligned w_scale are required");
  op->rows_per_batch = rows_per_batch;
  op->batch = batch;
  op->tiles_m_per_batch = (rows_per_batch + BM - 1) / BM;
  op->conv = 0;
  op->fp8 = 1;
  op->a_scale = a_scale;
  op->w_scale = w_scale;
  op->N = N;
  op->K = K;
  op->block_n = 256;
  op->tiles_n = (N + 255) / 256;
  op->num_tiles = batch * op->tiles_m_per_batch * op->tiles_n;
  op->epi = epi;
  op->out = out;
  op->out_batch_stride = out_batch_stride;
  op->ldo = ldo;
  op->bias = bias;
  TPDM_CHECK(N % 8 == 0 && ldo % 8 == 0, TPDM_ERR_SHAPE, "gemm fp8: N=%d and ldo=%d must be multiples of 8 (16-byte row segments)", N, ldo);
  TPDM_CHECK((reinterpret_cast<uintptr_t>(out) & 15) == 0 && (reinterpret_cast<uintptr_t>(bias) & 15) == 0, TPDM_ERR_ARG,
             "gemm fp8: out / bias must be 16-byte aligned");
  // a 128-byte swizzle row is 128 E4M3 elements: boxes {128, rows}
  uint64_t dims[3] = {static_cast<uint64_t>(K), static_cast<uint64_t>(rows_per_batch), static_cast<uint64_t>(batch)};
  uint64_t strides[2] = {static_cast<uint64_t>(a_row_stride), static_cast<uint64_t>(batch > 1 ? a_batch_stride : a_row_stride * rows_per_batch)};
  uint32_t box[3] = {128, BM, 1};
  TPDM_TRY(encode_tmap(&op->tmA, CU_TENSOR_MAP_DATA_TYPE_UINT8, A, 3, dims, strides, box));
  uint64_t wdims[2] = {static_cast<uint64_t>(K), static_cast<uint64_t>(N)};
  uint64_t wstrides[1] = {static_cast<uint64_t>(K)};
  uint32_t wbox[2] = {128, 128};
  return encode_tmap(&op->tmB2, CU_TENSOR_MAP_DATA_TYPE_UINT8, W, 2, wdims, wstrides, wbox);
}

int gemm_op_init_conv3x3(GemmOp* op, const void* X, int batch, int g, int C, const void* W, int N, int epi, void* out,
                         int ldo, const float* bias) {
  *op = GemmOp{};
  TPDM_CHECK(g >= 8 && g <= 128 && (g & (g - 1)) == 0, TPDM_ERR_SHAPE, "conv3x3: grid side %d must be a power of two in [8,128]", g);
  TPDM_CHECK(C % BK == 0, TPDM_ERR_SHAPE, "conv3x3: C=%d must be a multiple of 64", C);
  op->rows_per_batch = g * g;
  op->batch = batch;
  op->tiles_m_per_batch = (g * g + BM - 1) / BM;
  op->conv = 1;
  op->conv_by = BM / g;
  op->conv_bx = g;
  op->conv_xt = 1;
  op->kb_per_tap = C / BK;
  uint64_t dims[4] = {static_cast<uint64_t>(C), static_cast<uint64_t>(g), static_cast<uint64_t>(g), static_cast<uint64_t>(batch)};
  uint64_t strides[3] = {static_cast<uint64_t>(C) * 2, static_cast<uint64_t>(C) * g * 2, static_cast<uint64_t>(C) * g * g * 2};
  uint32_t box[4] = {BK, static_cast<uint32_t>(g), static_cast<uint32_t>(BM / g), 1};
  TPDM_TRY(encode_tmap_bf16(&op->tmA, X, 4, dims, strides, box));
  return finish_op(op, W, N, 9 * C, epi, out, static_cast<long long>(g) * g * ldo, ldo, bias, nullptr, 0);
}

int gemm_op_init_conv3x3_hw(GemmOp* op, const void* X, int batch, int H, int Wd, int C, const void* W, int N, int epi, void* out,
                            int ldo, const float* bias, const void* res) {
  *op = GemmOp{};
  const int bx = Wd < BM ? Wd : BM;
  TPDM_CHECK(H > 0 && Wd >= 8 && (Wd >= BM ? Wd % BM == 0 : (Wd & (Wd - 1)) == 0), TPDM_ERR_SHAPE,
             "conv3x3: image width %d must be a multiple of 128 or a power of two in [8,128)", Wd);
  TPDM_CHECK(C % BK == 0, TPDM_ERR_SHAPE, "conv3x3: C=%d must be a multiple of 64", C);
  TPDM_CHECK(epi != EPI_BIAS_ADD_BF16 || (res != nullptr && (reinterpret_cast<uintptr_t>(res) & 15) == 0), TPDM_ERR_ARG,
             "conv3x3: the add epilogue needs a 16-byte aligned addend");
  op->rows_per_batch = H * Wd;
  op->batch = batch;
  op->tiles_m_per_batch = (H * Wd + BM - 1) / BM;
  op->conv = 1;
  op->conv_bx = bx;
  op->conv_by = BM / bx;
  op->conv_xt = Wd / bx;
  op->kb_per_tap = C / BK;
  op->res = res;
  uint64_t dims[4] = {static_cast<uint64_t>(C), static_cast<uint64_t>(Wd), static_cast<uint64_t>(H), static_cast<uint64_t>(batch)};
  uint64_t strides[3] = {static_cast<uint64_t>(C) * 2, static_cast<uint64_t>(C) * Wd * 2, static_cast<uint64_t>(C) * Wd * H * 2};
  uint32_t box[4] = {BK, static_cast<uint32_t>(bx), static_cast<uint32_t>(BM / bx), 1};
  TPDM_TRY(encode_tmap_bf16(&op->tmA, X, 4, dims, strides, box));
  return finish_op(op, W, N, 9 * C, epi, out, static_cast<long long>(H) * Wd * ldo, ldo, bias, nullptr, 0);
}

int gemm_op_init_conv3x3_wgrad(GemmOp* op, const void* dYt, const void* Xnchw, int samples, int g, int C, int M, float* dW) {
  *op = GemmOp{};
  TPDM_CHECK(g >= 8 && g <= 128 && (g & (g - 1)) == 0, TPDM_ERR_SHAPE, "conv3x3 wgrad: grid side %d must be a power of two in [8,128]", g);
  TPDM_CHECK(C % 256 == 0 && M <= BM && M % 8 == 0, TPDM_ERR_SHAPE, "conv3x3 wgrad: C=%d must be a multiple of 256 and M=%d <= 128", C, M);
  const int P = g * g;
  op->rows_per_batch = M;
  op->batch = 1;
  op->tiles_m_per_batch = 1;
  op->conv = 2;
  op->wg_px = g;                  // pixels per image row (= the flattened shift of one row)
  op->wg_ctiles = C / 256;
  op->kb_per_tap = P / BK;        // k-blocks per sample
  op->N = 9 * C;
  op->K = samples * P;
  op->block_n = 256;
  op->tiles_n = 9 * (C / 256);
  op->num_tiles = op->tiles_n;
  op->epi = EPI_BIAS_F32;
  op->out = dW;
  op->out_batch_stride = 0;
  op->ldo = 9 * C;
  uint64_t adims[3] = {static_cast<uint64_t>(P), static_cast<uint64_t>(M), static_cast<uint64_t>(samples)};
  uint64_t astr[2] = {static_cast<uint64_t>(P) * 2, static_cast<uint64_t>(P) * M * 2};
  uint32_t abox[3] = {BK, BM, 1};
  TPDM_TRY(encode_tmap_bf16(&op->tmA, dYt, 3, adims, astr, abox));
  uint64_t bdims[4] = {static_cast<uint64_t>(P), static_cast<uint64_t>(C), 3, static_cast<uint64_t>(samples)};
  uint64_t bstr[3] = {static_cast<uint64_t>(P) * 2, static_cast<uint64_t>(P) * C * 2, static_cast<uint64_t>(P) * C * 3 * 2};
  uint32_t bbox[4] = {BK, 256, 1, 1};
  return encode_tmap_bf16(&op->tmB, Xnchw, 4, bdims, bstr, bbox);
}

int gemm_op_set_ksplit(GemmOp* op, int ksplit) {
  const int nkb = (op->K + BK - 1) / BK;
  TPDM_CHECK(ksplit >= 1 && ksplit <= nkb, TPDM_ERR_ARG, "gemm: ksplit %d outside [1, %d]", ksplit, nkb);
  TPDM_CHECK(ksplit == 1 || (op->epi == EPI_BIAS_F32 && op->bias == nullptr && op->conv != 2 && op->block_n == 128), TPDM_ERR_ARG,
             "gemm: split K needs a bias-free fp32 output on the 128-wide 1-CTA kernel");
  TPDM_CHECK((nkb + ksplit - 1) / ksplit * (ksplit - 1) < nkb, TPDM_ERR_ARG, "gemm: ksplit %d leaves an empty K range", ksplit);
  op->num_tiles = op->num_tiles / op->ksplit * ksplit;
  op->ksplit = ksplit;
  return 0;
}

int gemm_launch(const GemmOp* ops, int n_ops, cudaStream_t stream) {
  TPDM_CHECK(n_ops >= 1 && n_ops <= 2, TPDM_ERR_ARG, "gemm_launch: 1 or 2 ops per launch");
  GemmParams P;
  P.n_ops = n_ops;
  P.total_tiles = 0;
  P.skip = skip_flag();
  P.bmask = batch_mask();
  P.bslots = batch_mask_slots();
  for (int i = 0; i < n_ops; ++i) {
    P.op[i] = ops[i];
    P.total_tiles += ops[i].num_tiles;
    TPDM_CHECK(ops[i].block_n == ops[0].block_n && ops[i].fp8 == ops[0].fp8, TPDM_ERR_ARG, "gemm_launch: grouped ops must share the N tile and operand type");
  }
  if (n_ops == 1) P.op[1] = ops[0];
  if (ops[0].fp8) return gemm2_launch(ops, n_ops, stream);  // E4M3 operands exist only in the CTA-pair kernel
  // plain GEMMs with 256-wide N tiles go to the CTA-pair kernel (TPDM_GEMM_2CTA=0 forces the 1-CTA kernel)
  static const bool pair = getenv("TPDM_GEMM_2CTA") == nullptr || atoi(getenv("TPDM_GEMM_2CTA")) != 0;
  bool plain = ops[0].block_n == 256;
  for (int i = 0; i < n_ops; ++i) plain = plain && ops[i].conv == 0;
  if (pair && plain) return gemm2_launch(ops, n_ops, stream);
  return ops[0].block_n == 128 ? launch_impl<128>(P, stream) : launch_impl<256>(P, stream);
}

}  // namespace tpdm
