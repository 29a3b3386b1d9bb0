// tpdm_b200 -- bandwidth-bound kernels of the TPDM step (sm_100a): vectorised, coalesced, warp-shuffle reduced.
// Each kernel names the reference code it replaces (paths relative to /root/reference).
#include <curand_kernel.h>
#include <math.h>
#include <cstdlib>

#include "common.cuh"
#include "host.h"
#include "kernels.h"

namespace tpdm {

namespace {

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ uint4 ldg_nc_u4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ float bf16lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }

// token n of a g x g grid -> pixel index after reshape_hidden_states_to_2d (modeling_sd3_pnt.py:33-54)
__device__ __forceinline__ int scramble_pixel(int n, int g) {
  const int y = 2 * (n / (2 * g)) + ((n & 3) >> 1);
  const int x = 2 * ((n % (2 * g)) >> 2) + (n & 1);
  return y * g + x;
}

// ------------------------------------------------------------------------------------------------------------
__global__ void cast_bf16_kernel(const float* __restrict__ in, bf16* __restrict__ out, long long n) {
  long long i = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x * 4;
  for (; i + 3 < n; i += stride) {
    float4 v = ld4(in + i);
    uint2 w;
    w.x = pack_bf16x2(v.x, v.y);
    w.y = pack_bf16x2(v.z, v.w);
    *reinterpret_cast<uint2*>(out + i) = w;
  }
  if (i < n)
    for (long long k = i; k < n && k < i + 4; ++k) out[k] = __float2bfloat16(in[k]);
}

// diffusers get_timestep_embedding (call site transformer_sd3.py:336)
__global__ void timestep_embedding_kernel(const float* __restrict__ t, int t_stride, float scale, float* __restrict__ out, int Bt,
                                          int rep) {
  const int b = blockIdx.x;
  const int i = threadIdx.x;  // 0..127
  const float ts = t[(b % (Bt / rep)) * t_stride] * scale;
  const float f = expf(-logf(10000.0f) * static_cast<float>(i) / 128.0f);
  const float a = ts * f;
  out[b * 256 + i] = cosf(a);
  out[b * 256 + 128 + i] = sinf(a);
}

// ------------------------------------------------------------------------------------------------------------
// GEMV family: adaLN modulation linears of all blocks in one launch, time/text embedders, TPM norm1.linear
// (diffusers AdaLayerNormZero/Continuous .linear, TimestepEmbedding, PixArtAlphaTextProjection; K6/K4 of SURVEY 2.2)
// ------------------------------------------------------------------------------------------------------------
constexpr int kGemvRowsPerWarp = 4;
constexpr int kGemvWarps = 8;

// One warp owns kGemvRowsPerWarp consecutive weight rows and streams them TOGETHER (4 independent 16-byte loads per lane
// and k-step, unrolled x2 -> 8 loads in flight per lane) so HBM latency is covered by memory-level parallelism rather
// than occupancy.  act(x) for NB batch rows is staged once per block in shared memory.
template <typename WT, int NB, int WARPS = kGemvWarps>
__global__ void __launch_bounds__(WARPS * 32) gemv_kernel(const WT* __restrict__ W, const float* __restrict__ bias,
                                                                const float* __restrict__ x, int ldx,
                                                                const float* __restrict__ addend, float* __restrict__ y, int ldy,
                                                                int Bt, int J, int K, int act) {
  extern __shared__ float xs[];  // [NB][K]
  constexpr int EPL = 16 / sizeof(WT);  // elements per 16-byte load
  constexpr int R = kGemvRowsPerWarp;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int b0 = 0; b0 < Bt; b0 += NB) {
    const int nb = min(NB, Bt - b0);
    __syncthreads();
    for (int i = threadIdx.x; i < NB * K; i += blockDim.x) {
      const int bb = i / K, k = i - bb * K;
      float v = bb < nb ? x[static_cast<long long>(b0 + bb) * ldx + k] : 0.f;
      xs[i] = act ? silu_f(v) : v;
    }
    __syncthreads();
    // grid-stride over row groups: act(x) is staged once per block, not once per 32 rows (13 800 short-lived blocks spent
    // a third of their life on that staging and reached 64 % of the HBM rate)
    for (int j0 = (blockIdx.x * WARPS + warp) * R; j0 < J; j0 += gridDim.x * WARPS * R) {
    float acc[R][NB];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int bb = 0; bb < NB; ++bb) acc[r][bb] = 0.f;
    const WT* wrow[R];
#pragma unroll
    for (int r = 0; r < R; ++r) wrow[r] = W + static_cast<long long>(min(j0 + r, J - 1)) * K;
#pragma unroll 2
    for (int k = lane * EPL; k < K; k += 32 * EPL) {
      uint4 raw[R];
#pragma unroll
      for (int r = 0; r < R; ++r) raw[r] = ldg_nc_u4(wrow[r] + k);
      float xv[NB][EPL];
#pragma unroll
      for (int bb = 0; bb < NB; ++bb)
#pragma unroll
        for (int e = 0; e < EPL; e += 4) {
          const float4 t = *reinterpret_cast<const float4*>(xs + bb * K + k + e);
          xv[bb][e] = t.x; xv[bb][e + 1] = t.y; xv[bb][e + 2] = t.z; xv[bb][e + 3] = t.w;
        }
#pragma unroll
      for (int r = 0; r < R; ++r) {
        float w[EPL];
        if constexpr (sizeof(WT) == 2) {
          w[0] = bf16lo(raw[r].x); w[1] = bf16hi(raw[r].x); w[2] = bf16lo(raw[r].y); w[3] = bf16hi(raw[r].y);
          w[4] = bf16lo(raw[r].z); w[5] = bf16hi(raw[r].z); w[6] = bf16lo(raw[r].w); w[7] = bf16hi(raw[r].w);
        } else {
          w[0] = __uint_as_float(raw[r].x); w[1] = __uint_as_float(raw[r].y); w[2] = __uint_as_float(raw[r].z);
          w[3] = __uint_as_float(raw[r].w);
        }
#pragma unroll
        for (int bb = 0; bb < NB; ++bb)
#pragma unroll
          for (int e = 0; e < EPL; ++e) acc[r][bb] = fmaf(w[e], xv[bb][e], acc[r][bb]);
      }
    }
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int bb = 0; bb < NB; ++bb) {
        const float sum = warp_sum(acc[r][bb]);
        const int j = j0 + r;
        if (lane == 0 && j < J && bb < nb) {
          const long long o = static_cast<long long>(b0 + bb) * ldy + j;
          y[o] = sum + (bias ? bias[j] : 0.f) + (addend ? addend[o] : 0.f);
        }
      }
    }
  }
}

template <typename WT, int NB, int WARPS = kGemvWarps>
int gemv_launch_nb(const WT* W, const float* bias, const float* x, int ldx, const float* addend, float* y, int ldy, int Bt, int J, int K,
                   int act, cudaStream_t s) {
  const size_t smem = static_cast<size_t>(NB) * K * sizeof(float);
  TPDM_CHECK(smem <= 160 * 1024, TPDM_ERR_SHAPE, "gemv: K=%d too large", K);
  static bool attr_set = false;
  if (smem > 48 * 1024 && !attr_set) {
    TPDM_CUDA_OK(cudaFuncSetAttribute(gemv_kernel<WT, NB, WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    attr_set = true;
  }
  const int rows_per_block = WARPS * kGemvRowsPerWarp;
  const int want = (J + rows_per_block - 1) / rows_per_block, cap = 6 * num_sms();
  gemv_kernel<WT, NB, WARPS><<<want < cap ? want : cap, WARPS * 32, smem, s>>>(W, bias, x, ldx, addend, y, ldy, Bt, J, K, act);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

template <typename WT>
int gemv_launch(const WT* W, const float* bias, const float* x, int ldx, const float* addend, float* y, int ldy, int Bt, int J, int K,
                int act, cudaStream_t s) {
  constexpr int EPL = 16 / sizeof(WT);
  TPDM_CHECK(K % EPL == 0 && K % 4 == 0, TPDM_ERR_SHAPE, "gemv: K=%d must be a multiple of %d", K, EPL);
  if (Bt <= 2) return gemv_launch_nb<WT, 2>(W, bias, x, ldx, addend, y, ldy, Bt, J, K, act, s);
  if (Bt <= 4) return gemv_launch_nb<WT, 4>(W, bias, x, ldx, addend, y, ldy, Bt, J, K, act, s);
  return gemv_launch_nb<WT, 8>(W, bias, x, ldx, addend, y, ldy, Bt, J, K, act, s);
}

// ------------------------------------------------------------------------------------------------------------
// PatchEmbed (diffusers; call site transformer_sd3.py:334) + hidden_states_1 tap (:335)
// ------------------------------------------------------------------------------------------------------------
constexpr int kPatchTok = 32;

__global__ void __launch_bounds__(256) patchify_kernel(const float* __restrict__ lat, const float* __restrict__ Wp,
                                                       const float* __restrict__ bias, const float* __restrict__ pos, int pos_max,
                                                       float* __restrict__ x, int Bl, int dup, int C, int Hl, int Wl, int D,
                                                       float* __restrict__ h1_out, bf16* __restrict__ tpm_x) {
  extern __shared__ float in_s[];  // [kPatchTok][C*4]
  const int gw = Wl / 2, gh = Hl / 2, N = gw * gh;
  const int KK = C * 4;
  const int bl = blockIdx.y;
  const int n0 = blockIdx.x * kPatchTok;
  for (int i = threadIdx.x; i < kPatchTok * KK; i += blockDim.x) {
    const int t = i / KK, k = i - t * KK;
    const int c = k >> 2, p = (k >> 1) & 1, q = k & 1;
    const int n = n0 + t;
    const int ty = n / gw, tx = n - ty * gw;
    in_s[i] = lat[((static_cast<long long>(bl) * C + c) * Hl + 2 * ty + p) * Wl + 2 * tx + q];
  }
  // per-token element offsets, computed once per block (the divisions, the scramble and the 64-bit address arithmetic
  // used to be redone by every thread for every token: 200 instructions per token and warp, half of them for this)
  __shared__ int pos_off[kPatchTok], x_off[kPatchTok], tpm_off[kPatchTok];
  const int top = (pos_max - gh) / 2, left = (pos_max - gw) / 2;
  if (threadIdx.x < kPatchTok) {
    const int n = n0 + threadIdx.x;
    const int ty = n / gw, tx = n - ty * gw;
    pos_off[threadIdx.x] = ((top + ty) * pos_max + left + tx) * D;
    x_off[threadIdx.x] = n * D;
    tpm_off[threadIdx.x] = scramble_pixel(n, gw) * (2 * D);
  }
  // this block's 256 output channels: weights staged TRANSPOSED in shared memory (ws[k][d], row padded to 257 floats so that
  // both the staging stores and the per-k reads are conflict-free).  Keeping the 64 weights of a channel in registers cost
  // 128 registers per thread, two resident blocks per SM and a 2.6-wave tail (69 us); with 8 accumulators per thread the
  // kernel fits three blocks per SM.
  float* ws = in_s + kPatchTok * 64;  // [64][257]
  const int d = blockIdx.z * blockDim.x + threadIdx.x;
  if (d < D) {
    const float* wr = Wp + static_cast<long long>(d) * 64;
#pragma unroll 4
    for (int k = 0; k < 64; k += 4) {
      const float4 v = ld4(wr + k);
      ws[(k + 0) * 257 + threadIdx.x] = v.x;
      ws[(k + 1) * 257 + threadIdx.x] = v.y;
      ws[(k + 2) * 257 + threadIdx.x] = v.z;
      ws[(k + 3) * 257 + threadIdx.x] = v.w;
    }
  }
  __syncthreads();
  if (d >= D) return;
  const float bs = bias[d];
  // output pointers resolved once per thread; inside the token loop a store is one 32-bit offset away (the generic form --
  // 64-bit index arithmetic and a run-time `dup` loop per token -- made address code 3x the FMA count)
  const long long xb = static_cast<long long>(bl) * N * D + d, xdup = static_cast<long long>(Bl) * N * D;
  float* const x0 = x + xb;
  float* const x1 = dup > 1 ? x0 + xdup : nullptr;
  float* const h0 = h1_out ? h1_out + xb : nullptr;
  float* const h1 = (h1_out && dup > 1) ? h1_out + xb + xdup : nullptr;
  bf16* const tpm_b = tpm_x ? tpm_x + static_cast<long long>(bl) * N * (2 * D) + d : nullptr;
  const float* const posd = pos + d;
  const float* wcol = ws + threadIdx.x;
  for (int t0 = 0; t0 < kPatchTok; t0 += 8) {
    float pv[8], acc[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      pv[u] = posd[pos_off[t0 + u]];   // eight independent loads in flight under the FMA block
      acc[u] = bs;
    }
#pragma unroll 4
    for (int k = 0; k < 16; ++k) {
      const float w0 = wcol[(4 * k + 0) * 257], w1 = wcol[(4 * k + 1) * 257], w2 = wcol[(4 * k + 2) * 257], w3 = wcol[(4 * k + 3) * 257];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const float4 v = *reinterpret_cast<const float4*>(in_s + (t0 + u) * 64 + 4 * k);  // broadcast LDS.128
        acc[u] = fmaf(w0, v.x, acc[u]);
        acc[u] = fmaf(w1, v.y, acc[u]);
        acc[u] = fmaf(w2, v.z, acc[u]);
        acc[u] = fmaf(w3, v.w, acc[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const float r_ = acc[u] + pv[u];
      const int o = x_off[t0 + u];
      x0[o] = r_;
      if (x1) x1[o] = r_;
      if (h0) h0[o] = r_;
      if (h1) h1[o] = r_;
      if (tpm_b) tpm_b[tpm_off[t0 + u]] = __float2bfloat16(r_);
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// LayerNorm + adaLN modulation (diffusers AdaLayerNormZero.forward, norm2 + modulate in JointTransformerBlock.forward,
// AdaLayerNormContinuous; K7/K13).  One warp per token row, fp32 statistics, two-pass variance.
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void row_stats(const float* __restrict__ row, int D, int lane, float& mean, float& rstd) {
  float s = 0.f;
  for (int k = lane * 4; k < D; k += 128) {
    float4 v = ld4(row + k);
    s += (v.x + v.y) + (v.z + v.w);
  }
  mean = warp_sum(s) / D;
  float ss = 0.f;
  for (int k = lane * 4; k < D; k += 128) {
    float4 v = ld4(row + k);
    const float a = v.x - mean, b = v.y - mean, c = v.z - mean, d = v.w - mean;
    ss += (a * a + b * b) + (c * c + d * d);
  }
  rstd = rsqrtf(warp_sum(ss) / D + 1e-6f);
}

struct LnParams {
  LnSeg seg[2];
  int nseg, D;
  long long blocks0, blocks_total;  // blocks of segment 0 / of both segments
  const int* skip;
  const int* bmask;
  int bslots;
};

// One block = 32 consecutive token rows of ONE batch entry of one stream: the batch entry's shift / scale vectors are
// staged in shared memory once per block, each warp then streams 4 rows (row kept in registers when D = 128 * VPL, read
// once with no-allocate loads; VPL = 0 is the generic route that re-reads the row through L1 for the statistics).
constexpr int kLnRowsPerBlock = 32;

__device__ __forceinline__ float4 ld4_stream(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}

// kFp8: the modulated row is written as E4M3 codes + one row scale (S.out8 / S.out_scale) instead of bf16
template <int VPL, bool kFp8 = false>
__global__ void __launch_bounds__(256) ln_modulate_kernel(const __grid_constant__ LnParams P) {
  pdl_launch_dependents();
  pdl_wait();
  if (P.skip != nullptr && *P.skip != 0) return;
  extern __shared__ float ln_mod[];  // [D] shift, [D] scale
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int si = static_cast<long long>(blockIdx.x) >= P.blocks0 ? 1 : 0;
  const LnSeg& S = P.seg[si];
  const int blk = blockIdx.x - (si ? static_cast<int>(P.blocks0) : 0);
  const int rb_per_batch = (S.rows + kLnRowsPerBlock - 1) / kLnRowsPerBlock;
  const int b = blk / rb_per_batch, r0 = (blk - b * rb_per_batch) * kLnRowsPerBlock;
  if (P.bmask != nullptr && P.bmask[b % P.bslots] == 0) return;  // emptied queue slot (uniform over the block)
  const float* sh = S.shift + static_cast<long long>(b) * S.mod_stride;
  const float* sc = S.scale + static_cast<long long>(b) * S.mod_stride;
  for (int k = threadIdx.x * 4; k < P.D; k += 256 * 4) {
    *reinterpret_cast<float4*>(ln_mod + k) = ld4(sh + k);
    float4 c = ld4(sc + k);
    c.x += 1.f; c.y += 1.f; c.z += 1.f; c.w += 1.f;
    *reinterpret_cast<float4*>(ln_mod + P.D + k) = c;
  }
  __syncthreads();
  for (int rr = warp; rr < kLnRowsPerBlock; rr += 8) {
    const int r = r0 + rr;
    if (r >= S.rows) break;
    const long long lr = static_cast<long long>(b) * S.rows + r;
    const float* row = S.x + lr * P.D;
    bf16* o = S.out + lr * P.D;
    if constexpr (VPL > 0) {
      float4 v[VPL];
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        v[i] = ld4_stream(row + (i * 32 + lane) * 4);
        s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
      }
      const float mean = warp_sum(s) / P.D;
      float ss = 0.f;
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        const float a = v[i].x - mean, bq = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
        ss += (a * a + bq * bq) + (c * c + d * d);
      }
      const float rstd = rsqrtf(warp_sum(ss) / P.D + 1e-6f);
      if constexpr (kFp8) {
        float am = 0.f;
#pragma unroll
        for (int i = 0; i < VPL; ++i) {
          const int k = (i * 32 + lane) * 4;
          const float4 h = *reinterpret_cast<const float4*>(ln_mod + k), c = *reinterpret_cast<const float4*>(ln_mod + P.D + k);
          v[i] = make_float4((v[i].x - mean) * rstd * c.x + h.x, (v[i].y - mean) * rstd * c.y + h.y, (v[i].z - mean) * rstd * c.z + h.z,
                             (v[i].w - mean) * rstd * c.w + h.w);
          am = fmaxf(am, fmaxf(fmaxf(fabsf(v[i].x), fabsf(v[i].y)), fmaxf(fabsf(v[i].z), fabsf(v[i].w))));
        }
        am = warp_max(am);
        const float inv = fp8_row_inv_scale(am);
        uint8_t* o8 = S.out8 + lr * P.D;
#pragma unroll
        for (int i = 0; i < VPL; ++i)
          *reinterpret_cast<uint32_t*>(o8 + (i * 32 + lane) * 4) = pack_e4m3x4(v[i].x, v[i].y, v[i].z, v[i].w, inv);
        if (lane == 0) S.out_scale[lr] = fp8_row_scale(am);
      } else {
#pragma unroll
        for (int i = 0; i < VPL; ++i) {
          const int k = (i * 32 + lane) * 4;
          const float4 h = *reinterpret_cast<const float4*>(ln_mod + k), c = *reinterpret_cast<const float4*>(ln_mod + P.D + k);
          uint2 w;
          w.x = pack_bf16x2((v[i].x - mean) * rstd * c.x + h.x, (v[i].y - mean) * rstd * c.y + h.y);
          w.y = pack_bf16x2((v[i].z - mean) * rstd * c.z + h.z, (v[i].w - mean) * rstd * c.w + h.w);
          *reinterpret_cast<uint2*>(o + k) = w;
        }
      }
    } else {
      float mean, rstd;
      row_stats(row, P.D, lane, mean, rstd);
      if constexpr (kFp8) {  // generic width: one pass for the amax, one that recomputes the same values and stores the codes
        auto mod4 = [&](int k) {
          const float4 v = ld4(row + k), h = *reinterpret_cast<const float4*>(ln_mod + k), c = *reinterpret_cast<const float4*>(ln_mod + P.D + k);
          return make_float4((v.x - mean) * rstd * c.x + h.x, (v.y - mean) * rstd * c.y + h.y, (v.z - mean) * rstd * c.z + h.z,
                             (v.w - mean) * rstd * c.w + h.w);
        };
        float am = 0.f;
        for (int k = lane * 4; k < P.D; k += 128) {
          const float4 y = mod4(k);
          am = fmaxf(am, fmaxf(fmaxf(fabsf(y.x), fabsf(y.y)), fmaxf(fabsf(y.z), fabsf(y.w))));
        }
        am = warp_max(am);
        const float inv = fp8_row_inv_scale(am);
        uint8_t* o8 = S.out8 + lr * P.D;
        for (int k = lane * 4; k < P.D; k += 128) {
          const float4 y = mod4(k);
          *reinterpret_cast<uint32_t*>(o8 + k) = pack_e4m3x4(y.x, y.y, y.z, y.w, inv);
        }
        if (lane == 0) S.out_scale[lr] = fp8_row_scale(am);
      } else {
        for (int k = lane * 4; k < P.D; k += 128) {
          const float4 v = ld4(row + k), h = *reinterpret_cast<const float4*>(ln_mod + k), c = *reinterpret_cast<const float4*>(ln_mod + P.D + k);
          uint2 w;
          w.x = pack_bf16x2((v.x - mean) * rstd * c.x + h.x, (v.y - mean) * rstd * c.y + h.y);
          w.y = pack_bf16x2((v.z - mean) * rstd * c.z + h.z, (v.w - mean) * rstd * c.w + h.w);
          *reinterpret_cast<uint2*>(o + k) = w;
        }
      }
    }
  }
}

// norm_out (transformer_sd3.py:372-373) fused with the CFG combine of hidden_states_2 (modeling_sd3_pnt.py:545-548) and
// the token->pixel scramble of reshape_hidden_states_to_2d (:551).
__global__ void __launch_bounds__(256) norm_out_kernel(const float* __restrict__ x, bf16* __restrict__ xn,
                                                       const float* __restrict__ shift, const float* __restrict__ scale,
                                                       int mod_stride, int B, int cfg_pairs, int N, int D, int g, float guidance,
                                                       bf16* __restrict__ tpm_x, float* __restrict__ h2_out) {
  const int lane = threadIdx.x & 31;
  const long long r = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (r >= static_cast<long long>(B) * N) return;
  const int bl = static_cast<int>(r / N), n = static_cast<int>(r - static_cast<long long>(bl) * N);
  const int halves = cfg_pairs ? 2 : 1;
  float mean[2], rstd[2];
  const float* row[2];
  for (int hf = 0; hf < halves; ++hf) {
    row[hf] = x + (static_cast<long long>(bl + hf * B) * N + n) * D;
    row_stats(row[hf], D, lane, mean[hf], rstd[hf]);
  }
  const long long pix = tpm_x ? (static_cast<long long>(bl) * N + scramble_pixel(n, g)) * (2 * D) + D : 0;
  for (int k = lane * 4; k < D; k += 128) {
    float y[2][4];
    for (int hf = 0; hf < halves; ++hf) {
      const int bb = bl + hf * B;
      const float4 v = ld4(row[hf] + k), h = ld4(shift + static_cast<long long>(bb) * mod_stride + k),
                   c = ld4(scale + static_cast<long long>(bb) * mod_stride + k);
      y[hf][0] = (v.x - mean[hf]) * rstd[hf] * (1.f + c.x) + h.x;
      y[hf][1] = (v.y - mean[hf]) * rstd[hf] * (1.f + c.y) + h.y;
      y[hf][2] = (v.z - mean[hf]) * rstd[hf] * (1.f + c.z) + h.z;
      y[hf][3] = (v.w - mean[hf]) * rstd[hf] * (1.f + c.w) + h.w;
      const long long o = (static_cast<long long>(bb) * N + n) * D + k;
      uint2 w;
      w.x = pack_bf16x2(y[hf][0], y[hf][1]);
      w.y = pack_bf16x2(y[hf][2], y[hf][3]);
      *reinterpret_cast<uint2*>(xn + o) = w;
      if (h2_out) *reinterpret_cast<float4*>(h2_out + o) = make_float4(y[hf][0], y[hf][1], y[hf][2], y[hf][3]);
    }
    if (tpm_x) {
      float c4[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) c4[e] = cfg_pairs ? y[0][e] + guidance * (y[1][e] - y[0][e]) : y[0][e];
      uint2 w;
      w.x = pack_bf16x2(c4[0], c4[1]);
      w.y = pack_bf16x2(c4[2], c4[3]);
      *reinterpret_cast<uint2*>(tpm_x + pix + k) = w;
    }
  }
}

// diffusers RMSNorm on q/k heads (Attention.norm_q / norm_k / norm_added_q / norm_added_k; K9)
__global__ void __launch_bounds__(256) qk_rmsnorm_kernel(bf16* __restrict__ qkv, int Bt, int S, int row0, int rows, int H, int dp, int d,
                                                         const float* __restrict__ wq, const float* __restrict__ wk) {
  const int lane = threadIdx.x & 31;
  const long long item = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);  // (b, r, which, h)
  const long long total = static_cast<long long>(Bt) * rows * 2 * H;
  if (item >= total) return;
  const int h = static_cast<int>(item % H);
  const int which = static_cast<int>((item / H) % 2);
  const long long br = item / (2 * H);
  const int r = static_cast<int>(br % rows), b = static_cast<int>(br / rows);
  bf16* p = qkv + (static_cast<long long>(b) * S + row0 + r) * (3LL * H * dp) + static_cast<long long>(which) * H * dp + h * dp;
  const float* w = which ? wk : wq;
  float v[4];
  float ss = 0.f;
  const int per = dp / 32;  // 2 or 4
  for (int e = 0; e < per; ++e) {
    v[e] = __bfloat162float(p[lane * per + e]);
    ss += v[e] * v[e];
  }
  const float rs = rsqrtf(warp_sum(ss) / d + 1e-6f);
  for (int e = 0; e < per; ++e) p[lane * per + e] = __float2bfloat16(v[e] * rs * w[lane * per + e]);
}

// unpatchify (transformer_sd3.py:377-399) + CFG combine (modeling_sd3_pnt.py:537-538) + custom_step (model_utilis.py:61-69)
__global__ void __launch_bounds__(256) unpatchify_kernel(const float* __restrict__ pout, int B, int cfg_pairs, float guidance, int C,
                                                         int Hl, int Wl, float* __restrict__ velocity, float* __restrict__ latents,
                                                         const float* __restrict__ sigma, const float* __restrict__ sigma_next,
                                                         int sigma_stride, float* __restrict__ history) {
  const long long total = static_cast<long long>(B) * C * Hl * Wl;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int xx = static_cast<int>(i % Wl);
  const int yy = static_cast<int>((i / Wl) % Hl);
  const int c = static_cast<int>((i / (static_cast<long long>(Wl) * Hl)) % C);
  const int b = static_cast<int>(i / (static_cast<long long>(Wl) * Hl * C));
  const int gw = Wl / 2, N = gw * (Hl / 2);
  const int n = (yy >> 1) * gw + (xx >> 1);
  const int idx = (((yy & 1) << 1) | (xx & 1)) * C + c;
  float v = pout[(static_cast<long long>(b) * N + n) * (4 * C) + idx];
  if (cfg_pairs) {
    const float vc = pout[(static_cast<long long>(b + B) * N + n) * (4 * C) + idx];
    v = v + guidance * (vc - v);
  }
  if (velocity) velocity[i] = v;
  if (latents) {
    const float ds = sigma_next[b * sigma_stride] - sigma[b * sigma_stride];
    const float nv = latents[i] + ds * v;
    latents[i] = nv;
    if (history) history[i] = nv;
  }
}

__global__ void euler_kernel(const float* __restrict__ v, const float* __restrict__ sn, const float* __restrict__ s0,
                             const float* __restrict__ x, float* __restrict__ out, int B, long long n) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(B) * n) return;
  const int b = static_cast<int>(i / n);
  out[i] = x[i] + (sn[b] - s0[b]) * v[i];
}

__global__ void cfg_combine_kernel(const float* __restrict__ in, float* __restrict__ out, float* __restrict__ out2, int B, int n,
                                   float guidance) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(B) * n) return;
  const float u = in[i], c = in[i + static_cast<long long>(B) * n];
  const float r = u + guidance * (c - u);
  out[i] = r;
  if (out2) out2[i] = r;
}

// ------------------------------------------------------------------------------------------------------------
// TimePredictor tail (modeling_sd3_pnt.py:77-83, 104-115)
// ------------------------------------------------------------------------------------------------------------
__global__ void nchw_to_nhwc_bf16_kernel(const float* __restrict__ x, bf16* __restrict__ out, int B, int C, int g) {
  __shared__ float tile[32][33];
  const int P = g * g;
  const int b = blockIdx.z, c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, p = p0 + threadIdx.x;
    tile[i][threadIdx.x] = (c < C && p < P) ? x[(static_cast<long long>(b) * C + c) * P + p] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int p = p0 + i, c = c0 + threadIdx.x;
    if (c < C && p < P) out[(static_cast<long long>(b) * P + p) * C + c] = __float2bfloat16(tile[threadIdx.x][i]);
  }
}

__global__ void __launch_bounds__(256) gn_stats_kernel(const float* __restrict__ y, double* __restrict__ stats, long long n) {
  const int b = blockIdx.y;
  const float* p = y + static_cast<long long>(b) * n;
  float s = 0.f, ss = 0.f;
  for (long long i = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) * 4; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x * 4) {
    const float4 v = ld4(p + i);
    s += (v.x + v.y) + (v.z + v.w);
    ss += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
  }
  __shared__ float red[2][8];
  s = warp_sum(s);
  ss = warp_sum(ss);
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = s;
    red[1][threadIdx.x >> 5] = ss;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, c = 0;
    for (int i = 0; i < 8; ++i) {
      a += red[0][i];
      c += red[1][i];
    }
    atomicAdd(&stats[2 * b], a);
    atomicAdd(&stats[2 * b + 1], c);
  }
}

__global__ void __launch_bounds__(256) gn_mod_silu_kernel(const float* __restrict__ y, const double* __restrict__ stats,
                                                          const float* __restrict__ gn_w, const float* __restrict__ gn_b,
                                                          const float* __restrict__ emb, float* __restrict__ a, int B, int npix, int C) {
  const long long total = static_cast<long long>(B) * npix * C;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = static_cast<int>(i % C);
  const int b = static_cast<int>(i / (static_cast<long long>(npix) * C));
  const double cnt = static_cast<double>(npix) * C;
  const double mean = stats[2 * b] / cnt;
  const double var = stats[2 * b + 1] / cnt - mean * mean;
  const float rstd = rsqrtf(static_cast<float>(var > 0 ? var : 0) + 1e-6f);
  const float shift = emb[b * 2 * C + c], scale = emb[b * 2 * C + C + c];
  float v = (y[i] - static_cast<float>(mean)) * rstd * gn_w[c] + gn_b[c];
  v = v * (1.f + scale) + shift;
  a[i] = silu_f(v);
}

constexpr int kC2Pix = 4;
// Block = kC2Pix output pixels of one row; thread = (input-channel half, output channel).  The two halves are summed
// through shared memory.  512 blocks of 2*C threads for a 64x64 input: the first version (8 pixels, C threads, scalar
// LDS) ran 128 blocks and was latency-bound at 125 us.
__global__ void __launch_bounds__(256) conv3x3_s2_kernel(const float* __restrict__ a, const float* __restrict__ w,
                                                         const float* __restrict__ bias, float* __restrict__ y, int g, int C) {
  extern __shared__ __align__(16) float in_s[];  // [3][2*kC2Pix+1][C], then [kC2Pix][C] partial sums
  const int go = g / 2;
  const int b = blockIdx.z, oy = blockIdx.y, ox0 = blockIdx.x * kC2Pix;
  const int cols = 2 * kC2Pix + 1;
  for (int i = threadIdx.x; i < 3 * cols * C; i += blockDim.x) {
    const int c = i % C, col = (i / C) % cols, ky = i / (C * cols);
    const int iy = 2 * oy + ky - 1, ix = 2 * ox0 + col - 1;
    in_s[i] = (iy >= 0 && iy < g && ix >= 0 && ix < g) ? a[((static_cast<long long>(b) * g + iy) * g + ix) * C + c] : 0.f;
  }
  __syncthreads();
  const int oc = threadIdx.x % C, half = threadIdx.x / C;
  const int cb = half * (C / 2), ce = cb + C / 2;
  float acc[kC2Pix];
#pragma unroll
  for (int p = 0; p < kC2Pix; ++p) acc[p] = half == 0 ? bias[oc] : 0.f;
  for (int tap = 0; tap < 9; ++tap) {
    const int ky = tap / 3, kx = tap % 3;
    const float* wp = w + static_cast<long long>(tap) * C * C + oc;
    const float* ip = in_s + (ky * cols + kx) * C;
    for (int c0 = cb; c0 < ce; c0 += 8) {
      float wv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) wv[u] = wp[static_cast<long long>(c0 + u) * C];  // 8 independent (coalesced over oc) loads in flight
#pragma unroll
      for (int p = 0; p < kC2Pix; ++p) {
        const float4 i0 = *reinterpret_cast<const float4*>(ip + 2 * p * C + c0);  // broadcast LDS.128
        const float4 i1 = *reinterpret_cast<const float4*>(ip + 2 * p * C + c0 + 4);
        acc[p] = fmaf(wv[0], i0.x, acc[p]);
        acc[p] = fmaf(wv[1], i0.y, acc[p]);
        acc[p] = fmaf(wv[2], i0.z, acc[p]);
        acc[p] = fmaf(wv[3], i0.w, acc[p]);
        acc[p] = fmaf(wv[4], i1.x, acc[p]);
        acc[p] = fmaf(wv[5], i1.y, acc[p]);
        acc[p] = fmaf(wv[6], i1.z, acc[p]);
        acc[p] = fmaf(wv[7], i1.w, acc[p]);
      }
    }
  }
  float* part = in_s + 3 * cols * C;
  if (half == 1) {
#pragma unroll
    for (int p = 0; p < kC2Pix; ++p) part[p * C + oc] = acc[p];
  }
  __syncthreads();
  if (half == 0) {
#pragma unroll
    for (int p = 0; p < kC2Pix; ++p)
      if (ox0 + p < go) y[((static_cast<long long>(b) * go + oy) * go + ox0 + p) * C + oc] = acc[p] + part[p * C + oc];
  }
}

// adaptive_avg_pool2d(16,16) -> global max -> fc1 -> SiLU -> fc2 -> exp + eps.  One block of 1024 threads per sample:
// thread = (cell group 0..7, channel); each group reduces 32 of the 256 pooled cells, then a shared-memory max.
__global__ void __launch_bounds__(1024) tpm_tail_kernel(const float* __restrict__ y2, int go, int C, const float* __restrict__ fc1_w,
                                                        const float* __restrict__ fc1_b, const float* __restrict__ fc2_w,
                                                        const float* __restrict__ fc2_b, float eps, float* __restrict__ alpha_beta) {
  __shared__ float part[8][128];
  __shared__ float pooled[128];
  __shared__ float hid[128];
  const int b = blockIdx.x, t = threadIdx.x & 127, grp = threadIdx.x >> 7;
  const float* p = y2 + static_cast<long long>(b) * go * go * C;
  float mx = -INFINITY;
  if (t < C && go == 32) {
    // exact 2x2 windows: 8 cells (32 independent loads) in flight per batch.  The generic loop below has run-time window
    // bounds, is not unrolled and walked its 128 loads one DRAM/L2 round trip at a time (80 us for one block).
#pragma unroll
    for (int c8 = 0; c8 < 4; ++c8) {
      float v[8][4];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int cell = grp * 32 + c8 * 8 + u;
        const int i = cell >> 4, j = cell & 15;
        const float* q = p + (static_cast<long long>(2 * i) * 32 + 2 * j) * C + t;
        v[u][0] = q[0];
        v[u][1] = q[C];
        v[u][2] = q[32 * C];
        v[u][3] = q[33 * C];
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) mx = fmaxf(mx, (((v[u][0] + v[u][1]) + v[u][2]) + v[u][3]) / 4.f);
    }
  } else if (t < C) {
#pragma unroll 4
    for (int cell = grp * 32; cell < grp * 32 + 32; ++cell) {  // unrolled: the cells' loads are independent and stay in flight together
      const int i = cell >> 4, j = cell & 15;
      const int r0 = (i * go) / 16, r1 = ((i + 1) * go + 15) / 16;
      const int c0 = (j * go) / 16, c1 = ((j + 1) * go + 15) / 16;
      float s = 0.f;
      for (int r = r0; r < r1; ++r)
        for (int c = c0; c < c1; ++c) s += p[(static_cast<long long>(r) * go + c) * C + t];
      mx = fmaxf(mx, s / static_cast<float>((r1 - r0) * (c1 - c0)));
    }
  }
  part[grp][t] = mx;
  __syncthreads();
  if (threadIdx.x < 128) {
    float m = part[0][t];
#pragma unroll
    for (int g2 = 1; g2 < 8; ++g2) m = fmaxf(m, part[g2][t]);
    pooled[t] = m;
  }
  __syncthreads();
  // fc1: the 8 thread groups split the input channels (16 each), partial sums meet in shared memory; fc2: one warp per
  // output, lanes split the 128 hidden units.  (One thread per output walked 32 / 128 dependent-latency loads.)
  {
    float acc = 0.f;
    if (t < 128) {
      const int cpg = C / 8;  // C % 32 == 0 is checked by k_tpm_tail
      const float* wr = fc1_w + t * C + grp * cpg;
#pragma unroll 4
      for (int c = 0; c < cpg; c += 4) {
        const float4 w4 = ld4(wr + c);
        const float* pc = pooled + grp * cpg + c;
        acc = fmaf(w4.x, pc[0], fmaf(w4.y, pc[1], fmaf(w4.z, pc[2], fmaf(w4.w, pc[3], acc))));
      }
    }
    __syncthreads();  // everyone is done reading part[][] from the pooling phase
    part[grp][t] = acc;
  }
  __syncthreads();
  if (threadIdx.x < 128) {
    float acc = fc1_b[t];
#pragma unroll
    for (int g8 = 0; g8 < 8; ++g8) acc += part[g8][t];
    hid[t] = silu_f(acc);
  }
  __syncthreads();
  if (threadIdx.x < 64) {
    const int o = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float4 w4 = ld4(fc2_w + o * 128 + lane * 4);
    float acc = w4.x * hid[lane * 4] + w4.y * hid[lane * 4 + 1] + w4.z * hid[lane * 4 + 2] + w4.w * hid[lane * 4 + 3];
    acc = warp_sum(acc);
    if (lane == 0) alpha_beta[b * 2 + o] = expf(acc + fc2_b[o]) + eps;
  }
}

// Gamma(shape, 1) by Marsaglia-Tsang (shape < 1 boosted through Gamma(shape + 1) * U^(1/shape))
__device__ float gamma_draw(curandStatePhilox4_32_10_t* st, float shape) {
  float boost = 1.f;
  if (shape < 1.f) {
    boost = powf(curand_uniform(st), 1.f / shape);
    shape += 1.f;
  }
  const float d = shape - 1.f / 3.f, c = rsqrtf(9.f * d);
  for (int it = 0; it < 64; ++it) {
    const float x = curand_normal(st);
    float v = 1.f + c * x;
    if (v <= 0.f) continue;
    v = v * v * v;
    const float u = curand_uniform(st);
    if (logf(u) < 0.5f * x * x + d - d * v + d * logf(v)) return boost * d * v;
  }
  return boost * d;
}

// One sample's schedule update (modeling_sd3_pnt.py:557-590) from the raw TimePredictor outputs (p1, p2) at `sigma`.  The ratio
// is the Beta mode (predict), `given` (an injected draw) or Beta.sample() from the Philox stream (seed, sample, step * 1024);
// tpdm_sample_* and the device queue both key that stream by (sample or prompt, trajectory step), so both draw the same ratio.
enum RatioSource { kRatioMode, kRatioGiven, kRatioDraw };
struct ScheduleStep {
  float alpha, beta, ratio, sigma_next;
  double logprob;
};
__device__ __forceinline__ ScheduleStep schedule_step(float p1, float p2, float sigma, RatioSource src, float given, unsigned long long seed,
                                                      int sample, int step, int prediction_type, int relative, float epsilon) {
  ScheduleStep r;
  if (prediction_type == 0) {
    r.alpha = p1;
    r.beta = p2;
  } else {
    r.alpha = p1 * (p2 - 2.f) + 1.f;
    r.beta = (1.f - p1) * (p2 - 2.f) + 1.f;
  }
  float ratio;
  if (src == kRatioMode) {
    ratio = (r.alpha - 1.f) / (r.alpha + r.beta - 2.f);  // Beta.mode (:567)
  } else if (src == kRatioGiven) {
    ratio = given;
  } else {  // Beta.sample() (:569) = Ga / (Ga + Gb)
    curandStatePhilox4_32_10_t st;
    curand_init(seed, static_cast<unsigned long long>(sample), static_cast<unsigned long long>(step) * 1024ull, &st);
    const float ga = gamma_draw(&st, r.alpha), gb = gamma_draw(&st, r.beta);
    ratio = ga / (ga + gb);
  }
  if (relative) {
    ratio = fminf(fmaxf(ratio, epsilon), 1.f - epsilon);
    r.sigma_next = sigma * ratio;
  } else {
    ratio = fminf(fmaxf(ratio, epsilon), sigma);
    ratio = fminf(fmaxf(ratio, 0.f), 1.f - epsilon);
    r.sigma_next = sigma - ratio;
  }
  r.ratio = ratio;
  const double A = r.alpha, Bq = r.beta, rr = ratio;
  r.logprob = (A - 1.0) * log(rr) + (Bq - 1.0) * log1p(-rr) + lgamma(A + Bq) - lgamma(A) - lgamma(Bq);
  return r;
}

// schedule update of the lockstep batch (modeling_sd3_pnt.py:557-590, 608)
__global__ void schedule_kernel(const ScheduleArgs a) {
  const int i = threadIdx.x;
  int done = 1;
  if (i < a.B) {
    const float sigma = a.sigma_hist[i * (a.T + 1) + a.step];
    const RatioSource src = a.predict ? kRatioMode : (a.ratios ? kRatioGiven : kRatioDraw);
    const ScheduleStep r = schedule_step(a.alpha_beta[2 * i], a.alpha_beta[2 * i + 1], sigma, src,
                                         src == kRatioGiven ? a.ratios[i * a.T + a.step] : 0.f, a.seed, i, a.step, a.prediction_type,
                                         a.relative, a.epsilon);
    float sigma_next = r.sigma_next;
    int mask = 0;
    if (sigma < a.min_sigma) {
      mask = 1;
      if (a.predict) sigma_next = 0.f;
    }
    const int o = i * a.T + a.step;
    a.alphas[o] = r.alpha;
    a.betas[o] = r.beta;
    a.logprobs[o] = static_cast<float>(r.logprob);
    a.masks[o] = mask;
    a.sigma_hist[i * (a.T + 1) + a.step + 1] = sigma_next;
    done = sigma_next < a.min_sigma ? 1 : 0;
  }
  const int all = __syncthreads_and(done);
  if (i == 0) a.all_done[a.step] = all;
}

__global__ void __launch_bounds__(256) sum_partials_kernel(const float* __restrict__ part, int splits, long long n, const float* __restrict__ bias,
                                                           int C, float* __restrict__ y) {
  const long long i = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (i >= n) return;
  float4 acc = bias ? ld4(bias + static_cast<int>(i % C)) : make_float4(0.f, 0.f, 0.f, 0.f);
  for (int s = 0; s < splits; ++s) {
    const float4 v = ld4(part + s * n + i);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  *reinterpret_cast<float4*>(y + i) = acc;
}

// ---- device-side prompt queue ---------------------------------------------------------------------------------
// schedule update per slot (modeling_sd3_pnt.py:557-590), sigma kept per slot.  predict: ratio = Beta mode.  Rollouts
// (predict == 0): the prompt's injected ratio or a Philox draw keyed by (prompt, the slot's own trajectory step), recorded per
// prompt and step.
__global__ void queue_schedule_kernel(const QueueArgs a) {
  const int i = threadIdx.x;
  if (i >= a.B) return;
  const float sigma = a.sigma_cur[i];
  const int prompt = a.slot_prompt[i];
  if (prompt < 0) {  // idle slot: the Euler step is a no-op
    a.sigma_next[i] = sigma;
    return;
  }
  const int step = a.slot_step[i];
  const long long o = static_cast<long long>(prompt) * a.max_steps + step;
  const RatioSource src = a.predict ? kRatioMode : (a.ratios_all ? kRatioGiven : kRatioDraw);
  const ScheduleStep r = schedule_step(a.alpha_beta[2 * i], a.alpha_beta[2 * i + 1], sigma, src, src == kRatioGiven ? a.ratios_all[o] : 0.f,
                                       a.seed, prompt, step, a.prediction_type, a.relative, a.epsilon);
  float sigma_next = r.sigma_next;
  if (a.predict && sigma < a.min_sigma) sigma_next = 0.f;
  a.sigma_next[i] = sigma_next;
  if (a.rec_alphas) a.rec_alphas[o] = r.alpha;
  if (a.rec_betas) a.rec_betas[o] = r.beta;
  if (a.rec_logprobs) a.rec_logprobs[o] = static_cast<float>(r.logprob);
}

// rollout records of every occupied slot at its own (prompt, step): the CFG-combined temb [D] and the NHWC bf16 TimePredictor
// input [g][g][2D] (6.3 MB per slot at 512^2), 16-byte vector copies spread over gridDim.x blocks per slot
__global__ void __launch_bounds__(256) queue_record_kernel(const int* __restrict__ slot_prompt, const int* __restrict__ slot_step, int max_steps,
                                                           int D, const float* __restrict__ temb_cfg, float* __restrict__ tembs_all,
                                                           const uint4* __restrict__ tpm_x, uint4* __restrict__ tpm_all, long long tpm_vecs) {
  const int b = blockIdx.y;
  const int prompt = slot_prompt[b];
  if (prompt < 0) return;
  const long long o = static_cast<long long>(prompt) * max_steps + slot_step[b];
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  const long long t0 = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (tembs_all)
    for (long long k = t0 * 4; k < D; k += stride * 4) *reinterpret_cast<float4*>(tembs_all + o * D + k) = ld4(temb_cfg + static_cast<long long>(b) * D + k);
  if (tpm_all) {
    const uint4* src = tpm_x + b * tpm_vecs;
    uint4* dst = tpm_all + o * tpm_vecs;
    for (long long k = t0; k < tpm_vecs; k += stride) dst[k] = __ldg(src + k);
  }
}

// count the step of an occupied slot: returns true when its trajectory ended (final step count written), else moves it on
__device__ __forceinline__ bool queue_slot_retires(const QueueArgs& a, int i, int prompt) {
  const int step = a.slot_step[i] + 1;
  const float sn = a.sigma_next[i];
  if (a.out_sigmas) a.out_sigmas[static_cast<long long>(prompt) * (a.max_steps + 1) + step] = sn;
  if (sn < a.min_sigma || step >= a.max_steps) {   // the prompt-level form of the batch-wide exit test (:608)
    a.out_steps[prompt] = step;
    return true;
  }
  a.slot_step[i] = step;
  a.sigma_cur[i] = sn;
  return false;
}

// after the Euler step: count the step, retire finished trajectories, hand the freed slots their next ticket
__global__ void queue_advance_kernel(const QueueArgs a) {
  const int i = threadIdx.x;
  int holds = 0;
  if (i < a.B) {
    int prompt = a.slot_prompt[i], flush = -1, load = 0;
    bool need = a.init != 0;
    if (!a.init && prompt >= 0 && queue_slot_retires(a, i, prompt)) {
      flush = prompt;
      need = true;
    }
    if (need) {
      const int t = atomicAdd_system(a.ticket, 1);
      prompt = t < a.n_prompts ? (a.order ? a.order[t] : t) : -1;
      a.slot_prompt[i] = prompt;
      a.slot_step[i] = a.init_step;
      a.sigma_cur[i] = (a.init_sigma && prompt >= 0) ? a.init_sigma[prompt] : 1.0f;   // sigma = ones (:508) unless probed
      load = prompt >= 0 ? 1 : 0;
      if (prompt >= 0 && a.out_sigmas && a.init_step == 0) a.out_sigmas[static_cast<long long>(prompt) * (a.max_steps + 1)] = 1.0f;
    }
    a.slot_flush[i] = flush;
    a.slot_load[i] = load;
    holds = prompt >= 0 ? 1 : 0;
    a.slot_active[i] = holds;
  }
  const int n = __syncthreads_count(holds);
  if (i == 0) {
    *a.active = n;
    *a.idle_flag = n == 0 ? 1 : 0;
  }
}

// exclusive count of `flag` over the threads below this one (slot order) and the block total; every thread of the block calls it
__device__ __forceinline__ int block_rank(int flag, int* total, int* warp_counts) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const unsigned m = __ballot_sync(0xffffffffu, flag != 0);
  if (lane == 0) warp_counts[warp] = __popc(m);
  __syncthreads();
  int below = 0, all = 0;
  for (int w = 0; w < nwarps; ++w) {
    const int c = warp_counts[w];
    below += w < warp ? c : 0;
    all += c;
  }
  __syncthreads();  // warp_counts is reused by the next call
  *total = all;
  return below + __popc(m & ((1u << lane) - 1u));
}

// Stream mode of queue_advance_kernel.  The claim head is private to the stream, so tickets are handed out by rank in slot order
// (deterministic, no atomics); finished entries are appended to the completion log in the same order.
__global__ void stream_advance_kernel(const QueueArgs a, int admit) {
  __shared__ int warp_counts[32];
  const int i = threadIdx.x;
  const int submitted = a.counters[kStreamSubmitted], head = a.counters[kStreamClaimed], completed = a.counters[kStreamCompleted];
  const int ran = *a.active > 0 ? 1 : 0;   // slots held a prompt when the step began: it was not skipped
  int prompt = -1, flush = -1;
  if (i < a.B) {
    prompt = a.slot_prompt[i];
    if (!admit && prompt >= 0 && queue_slot_retires(a, i, prompt)) {
      flush = prompt;
      prompt = -1;
    }
  }
  const int need = i < a.B && prompt < 0 ? 1 : 0;
  int n_need = 0, n_flush = 0;
  const int r_need = block_rank(need, &n_need, warp_counts);
  const int r_flush = block_rank(flush >= 0, &n_flush, warp_counts);
  int holds = 0;
  if (i < a.B) {
    int load = 0;
    if (need) {
      const int t = head + r_need;
      prompt = t < submitted ? a.order[t % a.capacity] : -1;
      a.slot_prompt[i] = prompt;
      a.slot_step[i] = 0;
      a.sigma_cur[i] = 1.0f;   // sigma = ones (:508)
      load = prompt >= 0 ? 1 : 0;
      if (prompt >= 0 && a.out_sigmas) a.out_sigmas[static_cast<long long>(prompt) * (a.max_steps + 1)] = 1.0f;
    }
    if (flush >= 0) a.done_log[(completed + r_flush) % a.capacity] = flush;
    a.slot_flush[i] = flush;
    a.slot_load[i] = load;
    holds = prompt >= 0 ? 1 : 0;
    a.slot_active[i] = holds;
  }
  const int n = __syncthreads_count(holds);
  if (i == 0) {
    a.counters[kStreamClaimed] = head + n_need < submitted ? head + n_need : submitted;
    a.counters[kStreamCompleted] = completed + n_flush;
    if (!admit) a.counters[kStreamExecuted] += ran;
    *a.active = n;
    *a.idle_flag = n == 0 ? 1 : 0;
  }
}

__global__ void stream_publish_kernel(int* order, int* counters, int capacity, const StreamEntries e, int n) {
  const int s = counters[kStreamSubmitted];
  for (int k = 0; k < n; ++k) order[(s + k) % capacity] = e.id[k];
  counters[kStreamSubmitted] = s + n;
}

__global__ void __launch_bounds__(256) queue_move_kernel(const int* __restrict__ slot_prompt, const int* __restrict__ slot_flush,
                                                         const int* __restrict__ slot_load, int B, long long lat, long long ctx, int D,
                                                         float* __restrict__ latents, const float* __restrict__ noise_all,
                                                         float* __restrict__ out_latents, float* __restrict__ ctx0,
                                                         const float* __restrict__ ctx0_all, float* __restrict__ text_part,
                                                         const float* __restrict__ text_all) {
  const int b = blockIdx.y;
  const int flush = slot_flush[b], load = slot_load[b], prompt = slot_prompt[b];
  if (flush < 0 && !load) return;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x * 4;
  const long long t0 = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (flush >= 0)
    for (long long k = t0; k < lat; k += stride)
      *reinterpret_cast<float4*>(out_latents + flush * lat + k) = ld4(latents + b * lat + k);
  if (load) {
    for (long long k = t0; k < lat; k += stride) *reinterpret_cast<float4*>(latents + b * lat + k) = ld4(noise_all + prompt * lat + k);
    for (int half = 0; half < 2; ++half) {
      float* dst = ctx0 + (static_cast<long long>(half) * B + b) * ctx;
      const float* src = ctx0_all + (static_cast<long long>(prompt) * 2 + half) * ctx;
      for (long long k = t0; k < ctx; k += stride) *reinterpret_cast<float4*>(dst + k) = ld4(src + k);
      float* tdst = text_part + (static_cast<long long>(half) * B + b) * D;
      const float* tsrc = text_all + (static_cast<long long>(prompt) * 2 + half) * D;
      for (long long k = t0; k < D; k += stride) *reinterpret_cast<float4*>(tdst + k) = ld4(tsrc + k);
    }
  }
}

// LayerNorm + modulation with the rows STAGED THROUGH SHARED MEMORY by 1-D bulk async copies (cp.async.bulk, the TMA engine):
// every warp owns kLnSlots row slots and keeps that many rows in flight without spending registers on them -- while a row
// is reduced, normalised and stored, the copies of the warp's next rows are already running.  The register-only kernel
// above reaches 3.4 TB/s of DRAM reads (each warp waits out a full memory round trip per row); same block -> rows mapping.
constexpr int kLnSlots = 2;

__device__ __forceinline__ void bulk_load_row(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(smem_u32(smem_dst)),
               "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

template <int VPL, bool kFp8 = false>
__global__ void __launch_bounds__(256, 2) ln_modulate_bulk_kernel(const __grid_constant__ LnParams P) {
  pdl_launch_dependents();
  extern __shared__ __align__(128) float ln_smem[];  // [D] shift, [D] 1 + scale, then 8 warps x kLnSlots rows of D floats
  __shared__ uint64_t bars[8 * kLnSlots];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int D = VPL * 128;
  float* ring = ln_smem + 2 * D + warp * kLnSlots * D;
  if (lane == 0) {
    for (int i = 0; i < kLnSlots; ++i) mbar_init(&bars[warp * kLnSlots + i], 1);
    fence_barrier_init();
  }
  __syncwarp();
  pdl_wait();
  if (P.skip != nullptr && *P.skip != 0) return;
  const int si = static_cast<long long>(blockIdx.x) >= P.blocks0 ? 1 : 0;
  const LnSeg& S = P.seg[si];
  const int blk = blockIdx.x - (si ? static_cast<int>(P.blocks0) : 0);
  const int rb_per_batch = (S.rows + kLnRowsPerBlock - 1) / kLnRowsPerBlock;
  const int b = blk / rb_per_batch, r0 = (blk - b * rb_per_batch) * kLnRowsPerBlock;
  if (P.bmask != nullptr && P.bmask[b % P.bslots] == 0) return;  // emptied queue slot (uniform over the block)
  // this warp's rows: r0 + warp, r0 + warp + 8, ...  (kLnRowsPerBlock / 8 of them); start the first kLnSlots copies
  const long long row0 = static_cast<long long>(b) * S.rows;
  auto row_ok = [&](int j) { return j < kLnRowsPerBlock / 8 && r0 + warp + 8 * j < S.rows; };
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < kLnSlots; ++j)
      if (row_ok(j)) {
        mbar_arrive_expect_tx(&bars[warp * kLnSlots + j], D * 4);
        bulk_load_row(ring + j * D, S.x + (row0 + r0 + warp + 8 * j) * D, D * 4, &bars[warp * kLnSlots + j]);
      }
  }
  const float* sh = S.shift + static_cast<long long>(b) * S.mod_stride;
  const float* sc = S.scale + static_cast<long long>(b) * S.mod_stride;
  for (int k = threadIdx.x * 4; k < D; k += 256 * 4) {
    *reinterpret_cast<float4*>(ln_smem + k) = ld4(sh + k);
    float4 c = ld4(sc + k);
    c.x += 1.f; c.y += 1.f; c.z += 1.f; c.w += 1.f;
    *reinterpret_cast<float4*>(ln_smem + D + k) = c;
  }
  __syncthreads();
#pragma unroll 1
  for (int j = 0; j < kLnRowsPerBlock / 8; ++j) {
    if (!row_ok(j)) break;
    const int slot = j % kLnSlots;
    uint64_t* bar = &bars[warp * kLnSlots + slot];
    mbar_wait(bar, (j / kLnSlots) & 1);
    const float* src = ring + slot * D;
    float4 v[VPL];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      v[i] = *reinterpret_cast<const float4*>(src + (i * 32 + lane) * 4);
      s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
    __syncwarp();
    if (lane == 0 && row_ok(j + kLnSlots)) {  // the slot is free again: refill it for the row after next
      fence_proxy_async();                  // generic-proxy reads above are ordered before the async-proxy write below
      mbar_arrive_expect_tx(bar, D * 4);
      bulk_load_row(ring + slot * D, S.x + (row0 + r0 + warp + 8 * (j + kLnSlots)) * D, D * 4, bar);
    }
    const float mean = warp_sum(s) / D;
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const float a = v[i].x - mean, bq = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
      ss += (a * a + bq * bq) + (c * c + d * d);
    }
    const float rstd = rsqrtf(warp_sum(ss) / D + 1e-6f);
    if constexpr (kFp8) {
      float am = 0.f;
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        const int k = (i * 32 + lane) * 4;
        const float4 h = *reinterpret_cast<const float4*>(ln_smem + k), c = *reinterpret_cast<const float4*>(ln_smem + D + k);
        v[i] = make_float4((v[i].x - mean) * rstd * c.x + h.x, (v[i].y - mean) * rstd * c.y + h.y, (v[i].z - mean) * rstd * c.z + h.z,
                           (v[i].w - mean) * rstd * c.w + h.w);
        am = fmaxf(am, fmaxf(fmaxf(fabsf(v[i].x), fabsf(v[i].y)), fmaxf(fabsf(v[i].z), fabsf(v[i].w))));
      }
      am = warp_max(am);
      const float inv = fp8_row_inv_scale(am);
      const long long lr = row0 + r0 + warp + 8 * j;
      uint8_t* o8 = S.out8 + lr * D;
#pragma unroll
      for (int i = 0; i < VPL; ++i)
        *reinterpret_cast<uint32_t*>(o8 + (i * 32 + lane) * 4) = pack_e4m3x4(v[i].x, v[i].y, v[i].z, v[i].w, inv);
      if (lane == 0) S.out_scale[lr] = fp8_row_scale(am);
      continue;
    }
    bf16* o = S.out + (row0 + r0 + warp + 8 * j) * D;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const int k = (i * 32 + lane) * 4;
      const float4 h = *reinterpret_cast<const float4*>(ln_smem + k), c = *reinterpret_cast<const float4*>(ln_smem + D + k);
      uint2 w;
      w.x = pack_bf16x2((v[i].x - mean) * rstd * c.x + h.x, (v[i].y - mean) * rstd * c.y + h.y);
      w.y = pack_bf16x2((v[i].z - mean) * rstd * c.z + h.z, (v[i].w - mean) * rstd * c.w + h.w);
      *reinterpret_cast<uint2*>(o + k) = w;
    }
  }
}

// one warp per row: amax pass, then the codes (weights at load time, so the second read of the row is not worth avoiding)
__global__ void __launch_bounds__(256) quantize_fp8_rows_kernel(const float* __restrict__ x, int rows, int K, uint8_t* __restrict__ codes,
                                                                float* __restrict__ scales) {
  const int lane = threadIdx.x & 31;
  const long long r = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (r >= rows) return;
  const float* row = x + r * K;
  float am = 0.f;
  for (int k = lane * 4; k < K; k += 128) {
    const float4 v = ld4(row + k);
    am = fmaxf(am, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
  }
  am = warp_max(am);
  const float inv = fp8_row_inv_scale(am);
  for (int k = lane * 4; k < K; k += 128) {
    const float4 v = ld4(row + k);
    *reinterpret_cast<uint32_t*>(codes + r * K + k) = pack_e4m3x4(v.x, v.y, v.z, v.w, inv);
  }
  if (lane == 0) scales[r] = fp8_row_scale(am);
}

inline unsigned blocks_for(long long n, int per) { return static_cast<unsigned>((n + per - 1) / per); }

}  // namespace

// ------------------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------------------
int k_cast_bf16(const float* in, bf16* out, long long n, cudaStream_t s) {
  if (n <= 0) return 0;
  long long blocks = (n / 4 + 255) / 256;
  blocks = blocks < 1 ? 1 : (blocks > 148 * 16 ? 148 * 16 : blocks);
  cast_bf16_kernel<<<static_cast<unsigned>(blocks), 256, 0, s>>>(in, out, n);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_timestep_embedding(const float* timestep, int t_stride, float scale, float* out, int Bt, int rep, cudaStream_t s) {
  timestep_embedding_kernel<<<Bt, 128, 0, s>>>(timestep, t_stride, scale, out, Bt, rep);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_gemv_f32(const float* W, const float* bias, const float* x, int ldx, const float* addend, float* y, int ldy, int Bt, int J, int K,
               int act, cudaStream_t s) {
  return gemv_launch<float>(W, bias, x, ldx, addend, y, ldy, Bt, J, K, act, s);
}
int k_gemv_bf16(const bf16* W, const float* bias, const float* x, int ldx, const float* addend, float* y, int ldy, int Bt, int J, int K,
                int act, cudaStream_t s) {
  prof_begin(3, 2.0 * J * K, s);  // profile class 3: the weight matrix is read once
  const int st = gemv_launch<bf16>(W, bias, x, ldx, addend, y, ldy, Bt, J, K, act, s);
  prof_end(s);
  return st;
}

int k_patchify(const float* latents, const float* Wp, const float* bias, const float* pos_table, int pos_max, float* x, int Bl, int dup,
               int C, int Hl, int Wl, int D, float* h1_out, bf16* tpm_x, cudaStream_t s) {
  const int N = (Hl / 2) * (Wl / 2);
  TPDM_CHECK(C * 4 == 64, TPDM_ERR_SHAPE, "patchify: in_channels*patch^2 must be 64 (got %d)", C * 4);
  TPDM_CHECK(N % kPatchTok == 0, TPDM_ERR_SHAPE, "patchify: token count %d must be a multiple of %d", N, kPatchTok);
  TPDM_CHECK(Hl / 2 <= pos_max && Wl / 2 <= pos_max, TPDM_ERR_SHAPE, "patchify: grid %dx%d exceeds pos_embed_max_size %d", Hl / 2,
             Wl / 2, pos_max);
  dim3 grid(N / kPatchTok, Bl, (D + 255) / 256);  // one output channel per thread: (N/32) x Bl x D/256 blocks
  const size_t smem = (kPatchTok * 64 + 64 * 257) * sizeof(float);  // input patches + transposed weight slice
  static bool attr_set = false;
  if (!attr_set) {
    TPDM_CUDA_OK(cudaFuncSetAttribute(patchify_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    attr_set = true;
  }
  patchify_kernel<<<grid, 256, smem, s>>>(latents, Wp, bias, pos_table, pos_max, x, Bl, dup, C, Hl, Wl, D, h1_out, tpm_x);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_quantize_fp8_rows(const float* x, int rows, int K, uint8_t* codes, float* scales, cudaStream_t s) {
  TPDM_CHECK(rows > 0 && K > 0 && K % 4 == 0, TPDM_ERR_SHAPE, "quantize_fp8_rows: rows=%d, K=%d (K must be a positive multiple of 4)", rows, K);
  TPDM_CHECK((reinterpret_cast<uintptr_t>(x) & 15) == 0, TPDM_ERR_ARG, "quantize_fp8_rows: the input must be 16-byte aligned");
  quantize_fp8_rows_kernel<<<blocks_for(rows, 8), 256, 0, s>>>(x, rows, K, codes, scales);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_ln_modulate(const LnSeg* segs, int nseg, int D, cudaStream_t s) {
  TPDM_CHECK(nseg >= 1 && nseg <= 2 && D % 4 == 0, TPDM_ERR_ARG, "ln_modulate: bad arguments");
  const bool fp8 = segs[0].out8 != nullptr;
  TPDM_CHECK(nseg == 1 || (segs[1].out8 != nullptr) == fp8, TPDM_ERR_ARG, "ln_modulate: segments of one launch share the output type");
  for (int i = 0; i < nseg; ++i)
    TPDM_CHECK(!fp8 || segs[i].out_scale != nullptr, TPDM_ERR_ARG, "ln_modulate: an E4M3 output needs its row scales");
  LnParams P;
  P.nseg = nseg;
  P.D = D;
  P.skip = skip_flag();
  P.bmask = batch_mask();
  P.bslots = batch_mask_slots();
  P.seg[0] = segs[0];
  P.seg[1] = nseg > 1 ? segs[1] : segs[0];
  auto blocks_of = [](const LnSeg& g) { return static_cast<long long>(g.batch) * ((g.rows + kLnRowsPerBlock - 1) / kLnRowsPerBlock); };
  P.blocks0 = blocks_of(segs[0]);
  P.blocks_total = P.blocks0 + (nseg > 1 ? blocks_of(segs[1]) : 0);
  const unsigned grid = static_cast<unsigned>(P.blocks_total);
  const size_t smem = static_cast<size_t>(2) * D * sizeof(float);
  TPDM_CHECK(smem <= 48 * 1024, TPDM_ERR_SHAPE, "ln_modulate: D=%d too large", D);
  double bytes = 0;  // profile class 2: algorithmic bytes = one fp32 read + one bf16 (E4M3) write per element
  for (int i = 0; i < nseg; ++i) bytes += (fp8 ? 5.0 : 6.0) * segs[i].batch * segs[i].rows * D;
  prof_begin(2, bytes, s);
  static const bool bulk = getenv("TPDM_LN_BULK") == nullptr || atoi(getenv("TPDM_LN_BULK")) != 0;
  if (fp8) {
    if (D == 1536 && bulk) {
      const size_t smem_b = (2 + 8 * kLnSlots) * static_cast<size_t>(D) * sizeof(float);
      static bool attr = false;
      if (!attr) {
        TPDM_CUDA_OK(cudaFuncSetAttribute(ln_modulate_bulk_kernel<12, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem_b)));
        attr = true;
      }
      TPDM_CUDA_OK(launch_pdl(ln_modulate_bulk_kernel<12, true>, dim3(grid), dim3(256), smem_b, s, P));
    } else if (D == 1536)
      TPDM_CUDA_OK(launch_pdl(ln_modulate_kernel<12, true>, dim3(grid), dim3(256), smem, s, P));
    else if (D == 384)
      TPDM_CUDA_OK(launch_pdl(ln_modulate_kernel<3, true>, dim3(grid), dim3(256), smem, s, P));
    else
      TPDM_CUDA_OK(launch_pdl(ln_modulate_kernel<0, true>, dim3(grid), dim3(256), smem, s, P));
  } else if (D == 1536 && bulk) {
    const size_t smem_b = (2 + 8 * kLnSlots) * static_cast<size_t>(D) * sizeof(float);
    static bool attr = false;
    if (!attr) {
      TPDM_CUDA_OK(cudaFuncSetAttribute(ln_modulate_bulk_kernel<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem_b)));
      attr = true;
    }
    TPDM_CUDA_OK(launch_pdl(ln_modulate_bulk_kernel<12>, dim3(grid), dim3(256), smem_b, s, P));
  } else if (D == 1536)
    TPDM_CUDA_OK(launch_pdl(ln_modulate_kernel<12>, dim3(grid), dim3(256), smem, s, P));
  else if (D == 384)
    TPDM_CUDA_OK(launch_pdl(ln_modulate_kernel<3>, dim3(grid), dim3(256), smem, s, P));
  else
    TPDM_CUDA_OK(launch_pdl(ln_modulate_kernel<0>, dim3(grid), dim3(256), smem, s, P));
  prof_end(s);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_norm_out(const float* x, bf16* xn, const float* shift, const float* scale, int mod_stride, int B, int cfg_pairs, int N, int D,
               int g, float guidance, bf16* tpm_x, float* h2_out, cudaStream_t s) {
  norm_out_kernel<<<blocks_for(static_cast<long long>(B) * N, 8), 256, 0, s>>>(x, xn, shift, scale, mod_stride, B, cfg_pairs, N, D, g,
                                                                               guidance, tpm_x, h2_out);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_qk_rmsnorm(bf16* qkv, int Bt, int S, int row0, int rows, int H, int dp, int d, const float* wq, const float* wk, cudaStream_t s) {
  const long long total = static_cast<long long>(Bt) * rows * 2 * H;
  qk_rmsnorm_kernel<<<blocks_for(total, 8), 256, 0, s>>>(qkv, Bt, S, row0, rows, H, dp, d, wq, wk);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_unpatchify(const float* pout, int B, int cfg_pairs, float guidance, int C, int Hl, int Wl, float* velocity, float* latents,
                 const float* sigma, const float* sigma_next, int sigma_stride, float* history, cudaStream_t s) {
  const long long total = static_cast<long long>(B) * C * Hl * Wl;
  unpatchify_kernel<<<blocks_for(total, 256), 256, 0, s>>>(pout, B, cfg_pairs, guidance, C, Hl, Wl, velocity, latents, sigma, sigma_next,
                                                          sigma_stride, history);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_euler(const float* v, const float* sigma_next, const float* sigma, const float* sample, float* prev, int B, long long n,
            cudaStream_t s) {
  euler_kernel<<<blocks_for(static_cast<long long>(B) * n, 256), 256, 0, s>>>(v, sigma_next, sigma, sample, prev, B, n);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_cfg_combine(const float* in, float* out, float* out2, int B, int n, float guidance, cudaStream_t s) {
  cfg_combine_kernel<<<blocks_for(static_cast<long long>(B) * n, 256), 256, 0, s>>>(in, out, out2, B, n, guidance);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_nchw_to_nhwc_bf16(const float* x, bf16* out, int B, int C, int g, cudaStream_t s) {
  dim3 grid((g * g + 31) / 32, (C + 31) / 32, B), block(32, 8);
  nchw_to_nhwc_bf16_kernel<<<grid, block, 0, s>>>(x, out, B, C, g);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_gn_stats(const float* y, double* stats, int B, long long n, cudaStream_t s) {
  TPDM_CHECK(n % 4 == 0, TPDM_ERR_SHAPE, "gn_stats: n must be a multiple of 4");
  dim3 grid(64, B);
  gn_stats_kernel<<<grid, 256, 0, s>>>(y, stats, n);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_gn_mod_silu(const float* y, const double* stats, const float* gn_w, const float* gn_b, const float* emb, float* a, int B, int npix,
                  int C, cudaStream_t s) {
  gn_mod_silu_kernel<<<blocks_for(static_cast<long long>(B) * npix * C, 256), 256, 0, s>>>(y, stats, gn_w, gn_b, emb, a, B, npix, C);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_conv3x3_s2(const float* a, const float* w, const float* bias, float* y, int B, int g, int C, cudaStream_t s) {
  TPDM_CHECK(C <= 1024 && C % 8 == 0 && g % 2 == 0, TPDM_ERR_SHAPE, "conv3x3_s2: unsupported shape");
  const int go = g / 2;
  dim3 grid((go + kC2Pix - 1) / kC2Pix, go, B);
  TPDM_CHECK(C % 16 == 0 && 2 * C <= 256, TPDM_ERR_SHAPE, "conv3x3_s2: channels %d must be a multiple of 16 and <= 128", C);
  const size_t smem = static_cast<size_t>(3 * (2 * kC2Pix + 1) + kC2Pix) * C * sizeof(float);
  conv3x3_s2_kernel<<<grid, 2 * C, smem, s>>>(a, w, bias, y, g, C);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_tpm_tail(const float* y2, int B, int go, int C, const float* fc1_w, const float* fc1_b, const float* fc2_w, const float* fc2_b,
               float eps, float* alpha_beta, cudaStream_t s) {
  TPDM_CHECK(C <= 128 && C % 32 == 0, TPDM_ERR_SHAPE, "tpm_tail: conv_out_channels %d must be a multiple of 32, <= 128", C);
  tpm_tail_kernel<<<B, 1024, 0, s>>>(y2, go, C, fc1_w, fc1_b, fc2_w, fc2_b, eps, alpha_beta);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_sum_partials(const float* part, int splits, long long n, const float* bias, int C, float* y, cudaStream_t s) {
  TPDM_CHECK(n % 4 == 0 && C % 4 == 0 && splits >= 1, TPDM_ERR_SHAPE, "sum_partials: n and C must be multiples of 4");
  sum_partials_kernel<<<blocks_for(n / 4, 256), 256, 0, s>>>(part, splits, n, bias, C, y);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_queue_schedule(const QueueArgs& a, cudaStream_t s) {
  TPDM_CHECK(a.B <= 1024, TPDM_ERR_SHAPE, "queue: %d slots > 1024", a.B);
  queue_schedule_kernel<<<1, ((a.B + 31) / 32) * 32, 0, s>>>(a);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_queue_advance(const QueueArgs& a, cudaStream_t s) {
  TPDM_CHECK(a.B <= 1024, TPDM_ERR_SHAPE, "queue: %d slots > 1024", a.B);
  queue_advance_kernel<<<1, ((a.B + 31) / 32) * 32, 0, s>>>(a);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_stream_advance(const QueueArgs& a, int admit, cudaStream_t s) {
  TPDM_CHECK(a.B <= 1024, TPDM_ERR_SHAPE, "queue: %d slots > 1024", a.B);
  TPDM_CHECK(a.counters && a.done_log && a.order && a.capacity > 0, TPDM_ERR_STATE, "stream_advance: the plan has no open stream");
  stream_advance_kernel<<<1, ((a.B + 31) / 32) * 32, 0, s>>>(a, admit);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_stream_publish(int* order, int* counters, int capacity, const StreamEntries& e, int n, cudaStream_t s) {
  TPDM_CHECK(n >= 0 && n <= kStreamPublishMax, TPDM_ERR_ARG, "stream_publish: %d entries per launch (at most %d)", n, kStreamPublishMax);
  stream_publish_kernel<<<1, 1, 0, s>>>(order, counters, capacity, e, n);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_queue_record(const int* slot_prompt, const int* slot_step, int B, int max_steps, int D, const float* temb_cfg, float* tembs_all,
                   const bf16* tpm_x, bf16* tpm_all, long long tpm_elems, cudaStream_t s) {
  TPDM_CHECK(D % 4 == 0 && tpm_elems % 8 == 0, TPDM_ERR_SHAPE, "queue_record: D and the TimePredictor input must be whole 16-byte vectors");
  TPDM_CHECK((reinterpret_cast<uintptr_t>(tembs_all) & 15) == 0 && (reinterpret_cast<uintptr_t>(tpm_all) & 15) == 0, TPDM_ERR_ARG,
             "queue_record: record buffers must be 16-byte aligned");
  queue_record_kernel<<<dim3(64, B), 256, 0, s>>>(slot_prompt, slot_step, max_steps, D, temb_cfg, tembs_all, reinterpret_cast<const uint4*>(tpm_x),
                                                  reinterpret_cast<uint4*>(tpm_all), tpm_elems / 8);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_queue_move(const int* slot_prompt, const int* slot_flush, const int* slot_load, int B, long long lat, long long ctx, int D,
                 float* latents, const float* noise_all, float* out_latents, float* ctx0, const float* ctx0_all, float* text_part,
                 const float* text_all, cudaStream_t s) {
  TPDM_CHECK(lat % 4 == 0 && ctx % 4 == 0 && D % 4 == 0, TPDM_ERR_SHAPE, "queue: sizes must be multiples of 4 floats");
  queue_move_kernel<<<dim3(64, B), 256, 0, s>>>(slot_prompt, slot_flush, slot_load, B, lat, ctx, D, latents, noise_all, out_latents, ctx0, ctx0_all,
                                               text_part, text_all);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

// sigma_hist[b][0] = 1 (modeling_sd3_pnt.py:508), the rest of the per-trajectory state zeroed: one launch, no host staging buffer
__global__ void sample_init_kernel(float* __restrict__ sigma_hist, int* __restrict__ masks, int* __restrict__ all_done, int B, int T) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B * (T + 1)) sigma_hist[i] = (i % (T + 1)) == 0 ? 1.0f : 0.0f;
  if (i < B * T) masks[i] = 0;
  if (i < T) all_done[i] = 0;
}

int k_sample_init(float* sigma_hist, int* masks, int* all_done, int B, int T, cudaStream_t s) {
  sample_init_kernel<<<blocks_for(static_cast<long long>(B) * (T + 1), 256), 256, 0, s>>>(sigma_hist, masks, all_done, B, T);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

int k_schedule(const ScheduleArgs& a, cudaStream_t s) {
  TPDM_CHECK(a.B <= 1024, TPDM_ERR_SHAPE, "schedule: batch %d > 1024", a.B);
  const int threads = ((a.B + 31) / 32) * 32;
  schedule_kernel<<<1, threads, 0, s>>>(a);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace tpdm
