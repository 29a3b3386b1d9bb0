// tpdm_b200 -- epilogue of the tcgen05 GEMM kernels, shared by the 1-CTA (gemm_tcgen05.cu) and the CTA-pair
// (gemm2_tcgen05.cu) variants: one warp drains its 32 accumulator rows x BN columns from TMEM in 32-column chunks and
// applies bias / GELU-tanh / x += gate * (acc + bias).
//   bf16 outputs are stored straight from the accumulator registers (lane = row, 64 contiguous bytes per chunk).  Staging
//     them through shared memory for fully coalesced stores measured 2-6 % SLOWER on every SD3-medium GEMM shape: the
//     staging traffic competes with the MMA operand reads and the TMA writes for shared-memory bandwidth.
//   fp32 outputs (and the fp32 residual read of the gate mode) go through a padded shared-memory transpose so that global
//     traffic is row-contiguous 16-byte accesses: lane = row with 128-byte rows measured 0.68x (32 lines per request).
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"
#include "host.h"

namespace tpdm {

constexpr int kStagePad = 36;  // floats per staged row: 16-byte aligned rows, conflict-free 128-bit access

// `wait_accumulator()` blocks until the tile's accumulator is complete; `release_accumulator()` is called by the whole warp
// once its last TMEM load has landed in registers.
// The warp handles the 32-column chunks [c_begin, c_end) of the tile (all of them in the 1-CTA kernel; half of them in the
// CTA-pair kernel, where two warps share each TMEM lane quarter).  sbias holds 2 * 32 * (c_end - c_begin) floats.
// kScaled (E4M3 operands): y = acc * a_scale[b][row] * w_scale[col] + bias before the store; w_scale is staged in the gate half
// of sbias, which the bf16 / plain fp32 modes leave unused, and each lane reads its row's a_scale once per tile.
template <int BN, bool kScaled = false, typename WaitFn, typename ReleaseFn>
__device__ __forceinline__ void gemm_epilogue_tile(const GemmOp& G, int batch_idx, int row_base, int n0, uint32_t tmem_acc, float* st,
                                                   float* sbias, int lane, int c_begin, int c_end, WaitFn wait_accumulator,
                                                   ReleaseFn release_accumulator) {
  int n_chunks = (G.N - n0 + 31) / 32;
  n_chunks = n_chunks > c_end ? c_end : n_chunks;
  const int ncol = (c_end - c_begin) * 32;  // columns staged in sbias
  if (n_chunks <= c_begin) {  // nothing to store for this warp (N tail), but the accumulator hand-shake must still happen
    wait_accumulator();
    tc_fence_after();
    tc_fence_before();
    __syncwarp();
    release_accumulator();
    return;
  }
      int rows = G.rows_per_batch - row_base;
      rows = rows > 32 ? 32 : rows;
      const bool f32_out = G.epi == EPI_BIAS_F32 || G.epi == EPI_GATE_RESIDUAL;
      const bool add_bf16 = G.epi == EPI_BIAS_ADD_BF16;
      const bool resid = G.epi == EPI_GATE_RESIDUAL;
      // fp32 path, after the transpose: a lane owns 4 consecutive columns of one row, so a warp-wide access covers whole
      // 128-byte row segments of 4 rows
      const int vec = 4;
      const int cg = lane % 8;    // this lane's column group within the 32-column chunk
      const int r_in = lane / 8;  // this lane's row within a pass (8 passes of 4 rows)
      const float* gate_row = resid ? G.gate + static_cast<long long>(batch_idx) * G.gate_stride : nullptr;
      const long long tile_o0 = static_cast<long long>(batch_idx) * G.out_batch_stride + static_cast<long long>(row_base) * G.ldo + n0;

      // residual mode: the read half of out += gate * (acc + bias) does not depend on the accumulator.  While the MMA
      // warp is still working on this tile, pull the warp's 32 x BN fp32 block towards L2 and the first chunk into
      // registers; inside the chunk loop the next chunk's rows are always in flight while the current one is combined.
      auto load_resv = [&](int c, float4 (&rv)[8]) {
        const int col = n0 + c * 32 + cg * 4;
        if (col < G.N) {
          const float* o = reinterpret_cast<const float*>(G.out) + tile_o0 + c * 32 + cg * 4;
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            const int r = it * 4 + r_in;
            rv[it] = r < rows ? *reinterpret_cast<const float4*>(o + static_cast<long long>(r) * G.ldo) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
      };
      // bias / gate of the tile's columns: fetched once per tile into shared memory while the MMA is still running (loading
      // them per 32-column chunk put an L2 round trip on the critical path of every chunk)
      for (int k = lane * 4; k < ncol; k += 128) {
        const int col = n0 + c_begin * 32 + k;
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f), g4 = b4;
        if (col < G.N) {
          if (G.bias) b4 = *reinterpret_cast<const float4*>(G.bias + col);
          if (resid) g4 = *reinterpret_cast<const float4*>(gate_row + col);
          if constexpr (kScaled) g4 = *reinterpret_cast<const float4*>(G.w_scale + col);
        }
        *reinterpret_cast<float4*>(sbias + k) = b4;
        *reinterpret_cast<float4*>(sbias + ncol + k) = g4;
      }
      __syncwarp();
      // kScaled: a_s = this lane's row scale (bf16 path, lane = row); a_r[it] = the scale of row it * 4 + r_in (fp32 path)
      float a_s = 0.f, a_r[8];
      if constexpr (kScaled) {
        if (lane < rows) a_s = G.a_scale[static_cast<long long>(batch_idx) * G.rows_per_batch + row_base + lane];
#pragma unroll
        for (int it = 0; it < 8; ++it) a_r[it] = __shfl_sync(0xffffffffu, a_s, it * 4 + r_in);
      }
      float4 resv_a[8], resv_b[8];
      if (resid) {
        if (lane < rows) {
          const float* o = reinterpret_cast<const float*>(G.out) + tile_o0 + static_cast<long long>(lane) * G.ldo;
          for (int c = c_begin + 1; c < n_chunks; ++c) asm volatile("prefetch.global.L2 [%0];" ::"l"(o + c * 32));
        }
        load_resv(c_begin, resv_a);
      }
      wait_accumulator();
      tc_fence_after();

      auto process_chunk = [&](int c, const float4 (&resv)[8]) {
        const int col = n0 + c * 32 + cg * vec;
        const bool col_ok = col < G.N && rows > 0;
        const long long o0 = tile_o0 + c * 32 + cg * vec;
        float bias[4], gate[4];  // fp32 path only (the bf16 path reads its 32 columns' bias as it goes)
        {
          const float* sb = sbias + (c - c_begin) * 32 + cg * 4;
          const float4 b0 = *reinterpret_cast<const float4*>(sb);
          bias[0] = b0.x; bias[1] = b0.y; bias[2] = b0.z; bias[3] = b0.w;
          const float4 g4 = *reinterpret_cast<const float4*>(sb + ncol);
          gate[0] = g4.x; gate[1] = g4.y; gate[2] = g4.z; gate[3] = g4.w;
        }
        uint32_t v[32];
        tmem_ld_32x32(tmem_acc + c * 32, v);
        tmem_wait_ld();
        if (c == n_chunks - 1) {
          tc_fence_before();
          __syncwarp();
          release_accumulator();
        }
        if (!f32_out) {
          if (lane < rows && n0 + c * 32 < G.N) {
            const bool gelu = G.epi == EPI_BIAS_GELU_BF16;
            const float* sb = sbias + (c - c_begin) * 32;
            __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(G.out) + tile_o0 + c * 32 + static_cast<long long>(lane) * G.ldo;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float4 b0 = *reinterpret_cast<const float4*>(sb + 8 * q);
              const float4 b1 = *reinterpret_cast<const float4*>(sb + 8 * q + 4);
              float y[8] = {__uint_as_float(v[8 * q]) + b0.x,     __uint_as_float(v[8 * q + 1]) + b0.y,
                            __uint_as_float(v[8 * q + 2]) + b0.z, __uint_as_float(v[8 * q + 3]) + b0.w,
                            __uint_as_float(v[8 * q + 4]) + b1.x, __uint_as_float(v[8 * q + 5]) + b1.y,
                            __uint_as_float(v[8 * q + 6]) + b1.z, __uint_as_float(v[8 * q + 7]) + b1.w};
              if constexpr (kScaled) {
                const float4 s0 = *reinterpret_cast<const float4*>(sb + ncol + 8 * q);
                const float4 s1 = *reinterpret_cast<const float4*>(sb + ncol + 8 * q + 4);
                const float ws[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w}, bs[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                for (int e = 0; e < 8; ++e) y[e] = fmaf(__uint_as_float(v[8 * q + e]) * a_s, ws[e], bs[e]);
              }
              if (gelu) {
#pragma unroll
                for (int e = 0; e < 8; ++e) y[e] = gelu_tanh(y[e]);
              }
              if (add_bf16 && n0 + c * 32 + 8 * q < G.N) {
                const uint4 a = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(G.res) + (o - reinterpret_cast<__nv_bfloat16*>(G.out)) + 8 * q);
                y[0] += __uint_as_float(a.x << 16); y[1] += __uint_as_float(a.x & 0xffff0000u);
                y[2] += __uint_as_float(a.y << 16); y[3] += __uint_as_float(a.y & 0xffff0000u);
                y[4] += __uint_as_float(a.z << 16); y[5] += __uint_as_float(a.z & 0xffff0000u);
                y[6] += __uint_as_float(a.w << 16); y[7] += __uint_as_float(a.w & 0xffff0000u);
              }
              uint4 w;
              w.x = pack_bf16x2(y[0], y[1]);
              w.y = pack_bf16x2(y[2], y[3]);
              w.z = pack_bf16x2(y[4], y[5]);
              w.w = pack_bf16x2(y[6], y[7]);
              if (n0 + c * 32 + 8 * q < G.N) *reinterpret_cast<uint4*>(o + 8 * q) = w;
            }
          }
          return;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j)
          *reinterpret_cast<uint4*>(st + lane * kStagePad + 4 * j) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        __syncwarp();
        if (col_ok) {
          {
            float* o = reinterpret_cast<float*>(G.out) + o0;
#pragma unroll
            for (int it = 0; it < 8; ++it) {
              const int r = it * 4 + r_in;
              if (r < rows) {
                const float4 x = *reinterpret_cast<const float4*>(st + r * kStagePad + cg * 4);
                float4 y = make_float4(x.x + bias[0], x.y + bias[1], x.z + bias[2], x.w + bias[3]);
                if constexpr (kScaled)
                  y = make_float4(fmaf(x.x * a_r[it], gate[0], bias[0]), fmaf(x.y * a_r[it], gate[1], bias[1]), fmaf(x.z * a_r[it], gate[2], bias[2]),
                                  fmaf(x.w * a_r[it], gate[3], bias[3]));
                if (resid)
                  y = make_float4(resv[it].x + gate[0] * y.x, resv[it].y + gate[1] * y.y, resv[it].z + gate[2] * y.z,
                                  resv[it].w + gate[3] * y.w);
                *reinterpret_cast<float4*>(o + static_cast<long long>(r) * G.ldo) = y;
              }
            }
          }
        }
        __syncwarp();
      };

      for (int c = c_begin; c < n_chunks; c += 2) {
        if (resid && c + 1 < n_chunks) load_resv(c + 1, resv_b);
        process_chunk(c, resv_a);
        if (c + 1 < n_chunks) {
          if (resid && c + 2 < n_chunks) load_resv(c + 2, resv_a);
          process_chunk(c + 1, resv_b);
        }
      }
}

}  // namespace tpdm
