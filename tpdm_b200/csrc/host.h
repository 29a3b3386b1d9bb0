// tpdm_b200 -- host-side helpers shared by the translation units of libtpdm_b200.so
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <utility>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <string>

#include "../../include/tpdm_b200.h"

namespace tpdm {

void set_last_error(const std::string& msg);
int fail(int code, const char* fmt, ...);

#define TPDM_CUDA_OK(expr)                                                                           \
  do {                                                                                               \
    cudaError_t _e = (expr);                                                                         \
    if (_e != cudaSuccess)                                                                           \
      return ::tpdm::fail(TPDM_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

#define TPDM_CHECK(cond, code, ...)                     \
  do {                                                  \
    if (!(cond)) return ::tpdm::fail(code, __VA_ARGS__); \
  } while (0)

#define TPDM_TRY(expr)       \
  do {                       \
    int _s = (expr);         \
    if (_s != 0) return _s;  \
  } while (0)

int num_sms();

// launch accounting + optional CUDA-event brackets per kernel class (bench.py roofline); class 0 = GEMM, 1 = attention
void count_launch();
void count_launches(long long n);  // kernels replayed through a CUDA graph
long long launches_so_far();
bool profiling_active();  // between tpdm_profile_start and tpdm_profile_stop
void prof_begin(int cls, double flops, cudaStream_t s);
void prof_end(cudaStream_t s);

// Device flag checked at the top of the heavy kernels: when *flag != 0 the launch returns immediately.  Used so that a
// denoising step enqueued speculatively after the trajectory has finished costs only empty launches.
void set_skip_flag(const int* device_flag);
const int* skip_flag();
// Per-slot activity mask of the device-side prompt queue: slot_active[b % slots] == 0 makes the heavy kernels skip the tiles /
// CTAs / rows of batch entry b (an emptied slot at the tail of the queue then costs nothing).  nullptr = everything runs.
void set_batch_mask(const int* slot_active, int slots);
const int* batch_mask();
int batch_mask_slots();

// Launch with programmatic stream serialization (see pdl_wait in common.cuh); TPDM_PDL=0 turns the attribute off.
bool pdl_enabled();
template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr{};
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = &attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// bf16 tiled tensor map with 128-byte swizzle.  dims/strides innermost first; strides (bytes) for dims 1..rank-1.
int encode_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                     const uint32_t* box);
// the same for any element type (E4M3 operands use CU_TENSOR_MAP_DATA_TYPE_UINT8)
int encode_tmap(CUtensorMap* out, CUtensorMapDataType dtype, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                const uint32_t* box);

// ------------------------------------------------------------------------------------------------------------
// GEMM  (gemm_tcgen05.cu):  out = epilogue(A[rows x K] * W[N x K]^T)
// ------------------------------------------------------------------------------------------------------------
enum GemmEpilogue : int {
  EPI_BIAS_BF16 = 0,       // out(bf16) = acc + bias
  EPI_BIAS_F32 = 1,        // out(f32)  = acc + bias
  EPI_BIAS_GELU_BF16 = 2,  // out(bf16) = gelu_tanh(acc + bias)
  EPI_GATE_RESIDUAL = 3,   // out(f32) += gate[b, n] * (acc + bias)
  EPI_BIAS_ADD_BF16 = 4,   // out(bf16) = acc + bias + res(bf16)   (VAE resnet / attention skip connections)
};

struct alignas(64) GemmOp {
  CUtensorMap tmA;  // normal: (K, rows_per_batch, batch) box (64,128,1); conv: (C, x, y, b) box (64, g, 128/g, 1)
  CUtensorMap tmB;  // (K, N) box (64, BN)
  CUtensorMap tmB2; // (K, N) box (64, 128): half of a 256-wide N tile, for the CTA-pair kernel (gemm2_tcgen05.cu)
  int rows_per_batch, batch, N, K;
  int tiles_m_per_batch, tiles_n, num_tiles, block_n;
  int conv, conv_by, kb_per_tap, epi;  // conv: 0 plain, 1 conv3x3 forward, 2 conv3x3 weight gradient
  int conv_bx = 0, conv_xt = 1;        // conv 1: pixels per tile row segment, tile segments per image row
  int ksplit = 1;                      // 1-CTA kernel: K is cut into `ksplit` ranges, range s writes out + (s*batch + b)*out_batch_stride
                                       // (partial sums, to be added by the consumer); see gemm_op_set_ksplit
  // E4M3 operands (gemm_op_init_fp8, CTA-pair kernel only): out = epilogue(acc * a_scale[b][row] * w_scale[n] + bias).  The two
  // scale pointers share storage with `res` / `gate`, which no FP8 epilogue reads, so the struct keeps its 512 bytes.
  int fp8 = 0;
  union {
    const void* res = nullptr;         // EPI_BIAS_ADD_BF16: bf16 addend, indexed exactly like `out` (may alias it)
    const float* w_scale;              // fp8: [N]
  };
  int wg_px, wg_bpr, wg_ctiles, wg_pad;
  void* out;
  long long out_batch_stride;  // elements between batches of the output
  int ldo;                     // output leading dimension (elements)
  int gate_stride;             // elements between batches of gate
  const float* bias;           // [N] or null
  union {
    const float* gate;         // [batch][gate_stride] (EPI_GATE_RESIDUAL)
    const float* a_scale;      // fp8: [batch][rows_per_batch]
  };
};
static_assert(sizeof(GemmOp) == 512, "GemmOp is a kernel parameter: its size sets the indexing of GemmParams::op[]");

// A: bf16, element (b, r, k) at A + b*a_batch_stride + r*a_row_stride + k.   W: bf16 [N][K] row-major.
int gemm_op_init(GemmOp* op, const void* A, long long a_row_stride, long long a_batch_stride, int rows_per_batch, int batch,
                 int K, const void* W, int N, int epi, void* out, long long out_batch_stride, int ldo, const float* bias,
                 const float* gate, int gate_stride);
// A: E4M3 codes, element (b, r, k) at A + b*a_batch_stride + r*a_row_stride + k (strides in elements = bytes), a_scale fp32
// [batch][rows_per_batch];  W: E4M3 [N][K] row-major, w_scale fp32 [N].  epi: EPI_BIAS_BF16, EPI_BIAS_F32 or EPI_BIAS_GELU_BF16;
// N > 128 (256-wide N tiles of the CTA-pair kernel); K tails beyond a 128-element k-block are zero-filled by TMA.
int gemm_op_init_fp8(GemmOp* op, const void* A, long long a_row_stride, long long a_batch_stride, const float* a_scale, int rows_per_batch,
                     int batch, int K, const void* W, const float* w_scale, int N, int epi, void* out, long long out_batch_stride, int ldo,
                     const float* bias);
// implicit-GEMM 3x3 / pad 1 / stride 1 convolution over NHWC bf16 X[b][g][g][C]; W packed [N][9*C] (tap-major, tap=ky*3+kx).
int gemm_op_init_conv3x3(GemmOp* op, const void* X, int batch, int g, int C, const void* W, int N, int epi, void* out,
                         int ldo, const float* bias);
// same over a rectangular image X[b][H][Wd][C]: a 128-pixel M tile is a 128-wide segment of one row (Wd >= 128, Wd % 128 == 0)
// or 128 / Wd whole rows (Wd a power of two < 128); `res` as in GemmOp
int gemm_op_init_conv3x3_hw(GemmOp* op, const void* X, int batch, int H, int Wd, int C, const void* W, int N, int epi, void* out,
                            int ldo, const float* bias, const void* res);
// conv3x3 (pad 1, stride 1) weight gradient as a GEMM: dW[m][tap][c] = sum_{sample,pix} dYt[sample][m][pix] * X[sample][c][pix+tap]
// dYt bf16 [samples][M][g*g]; X bf16 as THREE x-shifted NCHW copies [samples][3][C][g][g], copy k holding X[.., x + k - 1]
// (zero outside), so no TMA load needs an unaligned innermost coordinate; dW fp32 [M][9][C] (overwritten)
int gemm_op_init_conv3x3_wgrad(GemmOp* op, const void* dYt, const void* Xnchw, int samples, int g, int C, int M, float* dW);
// split K of a bias-free fp32-output op of the 1-CTA kernel into `ksplit` partial products (more CTAs for few-tile problems)
int gemm_op_set_ksplit(GemmOp* op, int ksplit);
// one persistent launch over up to two ops (e.g. image stream + text stream)
int gemm_launch(const GemmOp* ops, int n_ops, cudaStream_t stream);
// CTA-pair (cta_group::2) kernel for plain GEMMs with 256-wide N tiles; gemm_launch dispatches to it
int gemm2_launch(const GemmOp* ops, int n_ops, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------------------
// joint attention (attention_tcgen05.cu)
// ------------------------------------------------------------------------------------------------------------
struct alignas(64) AttnOp {
  CUtensorMap tmQ, tmK, tmV;  // (dp, S, H, Bt) views of the token-major qkv buffer, box (64, 128, 1, 1)
  int S, H, Bt, dp;           // dp = padded head dim (64 or 128)
  int q_tiles, head_dim;
  float scale_log2;           // log2(e) / sqrt(head_dim)
  const int* skip;            // see set_skip_flag
  const int* bmask = nullptr; // see set_batch_mask
  int bslots = 1;
  __nv_bfloat16* out;         // [Bt][S][H*dp]
  int* redo = nullptr;        // [Bt*H*q_tiles] flags: CTAs that recomputed their tile with the exact softmax
};
int attn_op_init(AttnOp* op, const void* qkv, int Bt, int S, int H, int dp, int head_dim, void* out);
int attn_launch(const AttnOp* op, cudaStream_t stream);
long long attn_redo_total();  // diagnostic, synchronises: CTAs that took the exact pass since the library was loaded
int attn_redo_count();  // diagnostic, synchronises: CTAs of the last launch recomputed with the exact softmax (-1: no flag buffer)

}  // namespace tpdm
